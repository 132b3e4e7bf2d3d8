"""Whole-image validation of a network on a ``DeviceDataset`` (the reference selects its checkpoint on validation
metrics and drives ``ReduceLROnPlateau`` / ``EarlyStopping`` from them, ``__main__.py:240-257``).

The reference's validation loader is not available, so the definition here is stated: every image is seen whole, as
``predict.py`` sees it -- batch-1 semantics, eval-mode network (BatchNorm on its running statistics, no dropout) in
predict's storage precision (``models.DEFAULT_PRECISION``), logits upsampled bicubically to the image's own size -- and
each figure is a mean over images of the per-image value:

* ``loss``: the training loss on the full-resolution logits (``weighted_ce``, ``lovasz`` or ``mixed`` = ce / 4 + lovasz);
* ``miou``: ``lovasz_losses.iou`` of the argmax (EMPTY = 1, in %), averaged over the three classes;
* ``f1``: ``PixelWiseF1`` per class: argmax, ``remove_small_zones`` (150 pixels), F1 with the absent-class rule.

A chunk of equally wide images costs one ragged network pass (``Plan.forward_ragged``, bit-identical per image to a
forward of that image alone) and one ``ops.eval_ragged`` call, which gives every image's loss, confusion matrices and
region-removal counts exactly as the per-image ops would (bicubic upsample, loss forward, argmax, confusion matrix,
region removal); everything is read back once at the end.

With ``tta`` ('h' or 'hv', ``ops.tta_views``) a chunk runs one ``ops.flip_ragged`` per mirrored view and one network pass
per view, and ``ops.eval_ragged_views`` scores the views' mean logits (each view flipped back after the bicubic upsample):
the same figures for the test-time-augmented prediction ``predict --tta`` writes.

As a command, it scores a checkpoint on a labelled folder and writes one row per image (see ``main``):

    python -m neuralbarkcalculator_b200.evaluate ROOT --model best_model.pt [--split all|train|valid|test] [--seed 0]
        [--loss lovasz|weighted_ce|mixed] [--exclude_nodes] [--chunk 8] [--block 256] [--out evaluation.tsv]
        [--device cuda:0] [--tta none|h|hv]"""
import argparse
import os

import numpy as np
import torch

from . import ops
from .lovasz_losses import iou_from_confusion
from .models import DEFAULT_PRECISION, NeuralBarkCalculator, fcn_resnet50
from .utils import f1_from_confusion, get_pos_weight

LOSSES = ('weighted_ce', 'lovasz', 'mixed')


def model_keys(state_dict):
    """The 326 keys of ``fcn_resnet50`` in module order; raises when ``state_dict`` does not have exactly those."""
    with torch.device('meta'):
        keys = list(fcn_resnet50(pretrained=False).state_dict().keys())
    if set(keys) != set(state_dict.keys()):
        raise RuntimeError('evaluate: the state_dict does not have the 326 keys of fcn_resnet50')
    return keys


def make_plan(state_dict, device, precision=DEFAULT_PRECISION):
    """The inference plan of a 326-key ``fcn_resnet50`` state_dict, with predict's normalisation."""
    keys = model_keys(state_dict)
    tensors = [state_dict[k].detach().to(device) if state_dict[k].dtype == torch.int64
               else state_dict[k].detach().to(device=device, dtype=torch.float32) for k in keys]
    return ops.Plan(tensors, NeuralBarkCalculator.DEFAULT_MEAN, NeuralBarkCalculator.DEFAULT_STD, device, precision)


def image_logits(plan, ds, indices, chunk=8):
    """Yields (dataset index, full-resolution logits f32 [1,3,h,w], classes u8 [1,h,w]) for every index, in chunks of
    up to ``chunk`` images of one width (one ragged network pass each)."""
    indices = [int(i) for i in indices]
    widths = sorted({int(ds.sizes[i, 1]) for i in indices})
    for w in widths:
        same = [i for i in indices if ds.sizes[i, 1] == w]
        for start in range(0, len(same), chunk):
            part = same[start:start + chunk]
            hs = [int(ds.sizes[i, 0]) for i in part]
            sel = torch.tensor(part, dtype=torch.int64, device=ds.device)
            canvas = ds.images.index_select(0, sel)[:, :max(hs), :w].contiguous()
            heights = torch.tensor(hs, dtype=torch.int32, device=ds.device)
            low = plan.forward_ragged(canvas, heights=heights)
            for j, (i, h) in enumerate(zip(part, hs)):
                full = ops.upsample_bicubic(low[j:j + 1, :, :(h + 7) // 8].contiguous(), (h, w))
                yield i, full, ds.classes[i:i + 1, :h, :w].contiguous()


def _width_chunks(ds, indices, chunk):
    """Lists of up to ``chunk`` indices of one width, widths ascending, each width in the order of ``indices``."""
    widths = sorted({int(ds.sizes[i, 1]) for i in indices})
    for w in widths:
        same = [i for i in indices if ds.sizes[i, 1] == w]
        for start in range(0, len(same), chunk):
            yield w, same[start:start + chunk]


def image_row(index, loss, ce, lov, cm_raw, cm_rsz, counts):
    """One image's row from what ``ops.eval_ragged`` gives for it (f32 losses, 3x3 matrices cm[label, prediction])."""
    value = {'weighted_ce': ce, 'lovasz': lov, 'mixed': np.float32(ce) / np.float32(4) + np.float32(lov)}[loss]   # f32, as MixedLoss
    iou = iou_from_confusion(cm_raw)
    return {'index': index, 'loss': float(value), 'miou': float(np.mean(iou)), 'f1': f1_from_confusion(cm_rsz), 'iou': iou,
            'cm_rsz': cm_rsz, 'counts': counts}


def evaluate_plan(plan, ds, indices, loss='lovasz', class_weights=None, chunk=8, tta='none'):
    """``evaluate`` with a plan made beforehand: one ``forward_ragged`` and one ``ops.eval_ragged`` per chunk of up to
    ``chunk`` equally wide images, one read-back at the end.  Rows are grouped by width, as ``image_logits`` yields them;
    besides 'index', 'loss', 'miou' and 'f1' each row has 'iou' (the three per-class IoU behind 'miou'), 'cm_rsz' (the
    3x3 confusion matrix after region removal, behind 'f1') and 'counts' (the class counts of that mask).  tta 'h' / 'hv':
    one flip and one ``forward_ragged`` per view, then one ``ops.eval_ragged_views`` per chunk."""
    flags = ops.tta_views(tta)[1]
    if loss not in LOSSES:
        raise ValueError("loss must be 'weighted_ce', 'lovasz' or 'mixed'")
    if len(indices) == 0:
        raise RuntimeError('evaluate: no images')
    if int(chunk) < 1:
        raise ValueError('evaluate: chunk must be at least 1')
    bits = {'weighted_ce': ops.EVAL_WCE, 'lovasz': ops.EVAL_LOVASZ, 'mixed': ops.EVAL_WCE | ops.EVAL_LOVASZ}[loss]
    dev = ds.device
    indices = [int(i) for i in indices]
    with torch.cuda.device(dev):
        wts = (get_pos_weight() if class_weights is None else class_weights).to(device=dev, dtype=torch.float32).contiguous()
        order, outs, ws = [], [], None
        for w, part in _width_chunks(ds, indices, int(chunk)):
            hs = [int(ds.sizes[i, 0]) for i in part]
            sel = torch.tensor(part, dtype=torch.int64, device=dev)
            heights = torch.tensor(hs, dtype=torch.int32, device=dev)
            canvas = ds.images.index_select(0, sel)[:, :max(hs), :w].contiguous()
            labels = ds.classes.index_select(0, sel)[:, :max(hs), :w].contiguous()
            lows = [plan.forward_ragged(canvas if f == 0 else ops.flip_ragged(canvas, heights, f), heights=heights) for f in flags]
            need = ops._lib.load().nbc_eval_workspace_bytes(len(part), max(hs), w)
            if ws is None or ws.numel() < need:
                ws = None
                ws = torch.empty(need, dtype=torch.uint8, device=dev)
            if len(lows) == 1:
                outs.append(ops.eval_ragged(lows[0], heights, labels, wts, bits, workspace=ws))
            else:
                outs.append(ops.eval_ragged_views(lows, flags, heights, labels, wts, bits, workspace=ws))
            order.extend(part)
        host = {k: torch.cat([o[k] for o in outs]).cpu().numpy() for k in outs[0]}
    rows = [image_row(i, loss, host['loss_wce'][j], host['loss_lovasz'][j], host['cm_raw'][j], host['cm_rsz'][j],
                      host['counts'][j]) for j, i in enumerate(order)]
    return summary(rows)


def summary(rows):
    """{'loss', 'miou', 'f1', 'rows'}: the means over ``rows`` in their order (the order fixes the float sums)."""
    return {'loss': float(np.mean([r['loss'] for r in rows])), 'miou': float(np.mean([r['miou'] for r in rows])),
            'f1': np.mean([r['f1'] for r in rows], axis=0), 'rows': rows}


def width_order(ds, indices):
    """``indices`` in the row order of ``evaluate_plan``: widths ascending, each width in the order given."""
    return [i for _, part in _width_chunks(ds, [int(i) for i in indices], max(len(indices), 1)) for i in part]


def evaluate_sharded(plan, ds, indices, loss='lovasz', class_weights=None, chunk=8, tta='none'):
    """``evaluate_plan`` spread over the ranks of the torch.distributed process group: ``indices`` are put in
    ``evaluate_plan``'s row order, each rank evaluates a contiguous shard of that order (``distributed.shard_bounds``;
    a shard may be empty, the rank still joins the gather) and every rank gets all rows back.  Rows are per-image exact,
    so every rank returns what ``evaluate_plan`` returns in one process for the same network, bit for bit.  Every rank
    must call it with the same ``indices``; without a group of more than one process it is ``evaluate_plan``."""
    import torch.distributed as dist
    from .distributed import shard_bounds
    views = {} if tta == 'none' else {'tta': tta}      # fit's validation makes the call without it
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return evaluate_plan(plan, ds, indices, loss, class_weights, chunk, **views)
    if loss not in LOSSES:      # checked on every rank before the shards part: a rank must not leave the gather
        raise ValueError("loss must be 'weighted_ce', 'lovasz' or 'mixed'")
    ops.tta_views(tta)
    if len(indices) == 0:
        raise RuntimeError('evaluate: no images')
    if int(chunk) < 1:
        raise ValueError('evaluate: chunk must be at least 1')
    order = width_order(ds, indices)
    start, end = shard_bounds(len(order), dist.get_rank(), dist.get_world_size())
    mine = evaluate_plan(plan, ds, order[start:end], loss, class_weights, chunk, **views)['rows'] if end > start else []
    gathered = [None] * dist.get_world_size()
    dist.all_gather_object(gathered, mine)
    return summary([r for part in gathered for r in part])


def evaluate(state_dict, ds, indices, loss='lovasz', class_weights=None, precision=DEFAULT_PRECISION, chunk=8, tta='none'):
    """Validation of ``state_dict`` on the items ``indices`` of ``ds`` (see the module docstring for the definition).
    Returns {'loss', 'miou', 'f1' (3 values): means over the images, 'rows': one dict per image with the same keys and
    'index'} (rows grouped by width; ``evaluate_plan`` lists the further keys of a row)."""
    if loss not in LOSSES:
        raise ValueError("loss must be 'weighted_ce', 'lovasz' or 'mixed'")
    if len(indices) == 0:
        raise RuntimeError('evaluate: no images')
    with torch.cuda.device(ds.device):
        plan = make_plan(state_dict, ds.device, precision)
    return evaluate_plan(plan, ds, indices, loss, class_weights, chunk, tta)


# ---- the command -------------------------------------------------------------------------------------------------
SPLITS = ('all', 'train', 'valid', 'test')
HEADER = ['Name', 'Type', 'Height', 'Width', 'Loss', 'IoU 0', 'IoU 1', 'IoU 2', 'mIoU', 'F1 0', 'F1 1', 'F1 2',
          'Label Bark %', 'Output Bark %', 'Label Node %', 'Output Node %']


def _pct(n, n_pixels):
    """A class's share in the float32 arithmetic and format of ``NeuralBarkCalculator._stats_strings``."""
    return '{:.5f}'.format(np.float32(n) / np.float32(n_pixels) * np.float32(100))


def percent_rows(cm_rsz, counts, height, width, exclude_nodes=False):
    """[Label Bark %, Output Bark %, Label Node %, Output Node %] of one image.  The output shares come from the region
    removal's class counts, as ``final_stats.csv`` reports them; the label shares from the rows of the confusion matrix
    after region removal (cm[label, prediction]: every labelled pixel is counted once).  With ``exclude_nodes`` predict
    rewrites node to bark after the region removal, so both sides are folded the same way: (c0, c1 + c2, 0)."""
    lab = [int(v) for v in np.asarray(cm_rsz).reshape(3, 3).sum(1)]
    out = [int(v) for v in counts]
    if exclude_nodes:
        lab = [lab[0], lab[1] + lab[2], 0]
        out = [out[0], out[1] + out[2], 0]
    n = int(height) * int(width)
    return [_pct(lab[1], n), _pct(out[1], n), _pct(lab[2], n), _pct(out[2], n)]


def table_row(name, wood, height, width, row, exclude_nodes=False):
    """One line of the evaluation file: metrics as ``repr(float)``, as ``fit``'s log writes them."""
    return ([name, wood, str(int(height)), str(int(width)), repr(float(row['loss']))]
            + [repr(float(v)) for v in row['iou']] + [repr(float(row['miou']))] + [repr(float(v)) for v in row['f1']]
            + percent_rows(row['cm_rsz'], row['counts'], height, width, exclude_nodes))


def mean_row(rows):
    """The final line: the mean of every metric column over ``rows`` (in their order), and in the Output Bark % /
    Output Node % columns the mean absolute difference between the label and output percentages."""
    metrics = np.array([[float(v) for v in r[4:12]] for r in rows], dtype=np.float64)
    bark = np.mean([abs(float(r[12]) - float(r[13])) for r in rows])
    node = np.mean([abs(float(r[14]) - float(r[15])) for r in rows])
    return (['mean', '', '', ''] + [repr(float(v)) for v in metrics.mean(0)]
            + ['', '{:.5f}'.format(bark), '', '{:.5f}'.format(node)])


def select_items(items, split, seed):
    """Dataset indices (ascending) of ``split``: every item, or ``fit``'s split for ``seed`` (``np.random.seed`` then
    ``utils.get_splits`` on the dual images' labelled-pixel counts).  Under torch.distributed rank 0 computes it and
    broadcasts the list."""
    if split == 'all':
        return list(range(len(items)))
    import torch.distributed as dist
    distributed = dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
    box = [None]
    if not distributed or dist.get_rank() == 0:
        from .augment import label_classes
        from .dataset import pil_loader
        from .utils import get_splits
        label_pixels = np.array([np.count_nonzero(label_classes(pil_loader(t, grayscale=True))) for _, t, _, _ in items],
                                dtype=np.int64)
        np.random.seed(seed)
        parts = get_splits([(None, None, f, w) for _, _, f, w in items], label_pixels=label_pixels)
        box[0] = sorted(int(i) for i in parts[SPLITS.index(split) - 1])
    if distributed:
        dist.broadcast_object_list(box, src=0)
    return box[0]


def check_folder(items, root):
    if not items:
        raise RuntimeError('evaluate: no images under %s/samples' % root)
    missing = [f for _, t, f, _ in items if not t]
    if missing:
        raise RuntimeError('evaluate: %d samples have no dual image under %s/duals (first: %s)' % (len(missing), root, missing[0]))


def main(args):
    """Scores ``--model`` on the labelled folder ROOT and writes ``--out``: a header, one row per image of the split in
    dataset order (``HEADER``), then ``mean_row``.  Under ``torchrun`` each rank evaluates a contiguous shard on
    cuda:LOCAL_RANK and rank 0 merges the rows, so the file equals a one-GPU run.  Images are loaded and evaluated in
    blocks of ``--block``, so device memory does not grow with the folder."""
    import torch
    from . import distributed as ndist
    from .augment import load_dataset
    from .dataset import make_dataset
    items = make_dataset(args.root)
    check_folder(items, args.root)
    if not os.path.isfile(args.model):
        raise RuntimeError('evaluate: --model %s: no such file' % args.model)
    state_dict = torch.load(args.model, map_location='cpu')
    model_keys(state_dict)
    rank, local_rank, world = ndist.env_world()
    device = args.device
    if world > 1:
        device = 'cuda:%d' % local_rank
        ndist.init_from_env('cuda')
        ndist.bind_to_gpu_numa(local_rank)
    selected = select_items(items, args.split, args.seed)
    if not selected:
        raise RuntimeError('evaluate: the %s split of %s is empty' % (args.split, args.root))
    start, end = ndist.shard_bounds(len(selected), rank, world)
    mine = selected[start:end]
    rows = []
    if mine:
        with torch.cuda.device(torch.device(device)):
            plan = make_plan(state_dict, device)
            for b in range(0, len(mine), args.block):
                sub = mine[b:b + args.block]
                ds = load_dataset(args.root, device, items=sub)
                res = evaluate_plan(plan, ds, range(len(sub)), args.loss, chunk=args.chunk, tta=getattr(args, 'tta', 'none'))
                by = {r['index']: r for r in res['rows']}
                for j, i in enumerate(sub):
                    _, _, fname, wood = items[i]
                    h, w = ds.sizes[j]
                    rows.append(table_row(fname, wood, h, w, by[j], args.exclude_nodes))
                del ds, res
    merged = ndist.merge_rows(rows, start, len(selected))
    if rank == 0:
        with open(args.out, 'w') as f:
            for r in [HEADER] + merged + [mean_row(merged)]:
                f.write('\t'.join(r) + '\n')
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()
    return merged


def parse_args(argv=None):
    parser = argparse.ArgumentParser(prog='python -m neuralbarkcalculator_b200.evaluate')
    parser.add_argument('root', help='labelled folder with samples/<wood>/ and duals/<wood>/')
    parser.add_argument('--model', default='best_model.pt', help='326-key state_dict (torch.save file)')
    parser.add_argument('--split', default='all', choices=SPLITS, help="all items, or fit's split for --seed")
    parser.add_argument('--seed', type=int, default=0)
    parser.add_argument('--loss', default='lovasz', choices=list(LOSSES))
    parser.add_argument('--exclude_nodes', action='store_true', default=False,
                        help='count nodes as bark in the percentages, as predict --exclude_nodes does')
    parser.add_argument('--chunk', type=int, default=8, help='images per batched pass')
    parser.add_argument('--block', type=int, default=256, help='images loaded onto the GPU at a time')
    parser.add_argument('--out', default='evaluation.tsv')
    parser.add_argument('--device', default='cuda:0', help='CUDA device (cuda, cuda:N)')
    parser.add_argument('--tta', default='none', choices=list(ops.TTA_MODES),
                        help="flip test-time augmentation, as predict --tta: none, h or hv")
    args = parser.parse_args(argv)
    if not args.device.startswith('cuda'):
        parser.error('--device %s: only CUDA devices are supported (no CPU path)' % args.device)
    if args.chunk < 1 or args.block < 1:
        parser.error('--chunk and --block must be at least 1')
    return args


if __name__ == '__main__':
    main(parse_args())
