"""Train a network from a labelled folder and write the checkpoint ``predict.py`` reads (the epoch loop of the
reference's ``__main__.py:199-291``, which runs it through Poutyne).

    python -m neuralbarkcalculator_b200.fit ROOT --init SD.pt|random [--out best_model.pt] [--epochs 30] [--crop 512]
        [--batch 5] [--accumulate 1] [--freeze none] [--loss lovasz] [--lr 5e-4] [--weight-decay 2e-3] [--dropout 0.8]
        [--seed 0] [--device cuda:0] [--state run.state [--resume]]
    torchrun --nproc_per_node W -m neuralbarkcalculator_b200.fit ROOT ...      (data parallel, one GPU per rank)

ROOT holds ``samples/<wood>/*`` and ``duals/<wood>/*`` (processed images and their dual label images, any height up to
``--target``).  The dataset is loaded once onto the GPU; ``utils.get_splits`` makes the 80 / 10 / 10 split per wood type
and the sampling weights.  Each epoch draws its batches with ``utils.weighted_epoch_batches``, augments each on the GPU
(``augment.augment_ragged``: pad_resize, colour jitter, crop, flips) and runs ``Trainer.step``; the training loss is read
back once per epoch.  Then ``evaluate`` scores the validation split whole-image, as predict would run it; a row goes to
the log (epoch, lr, loss, val_loss, val_miou, val_f1 x 3, seconds), the learning rate follows ``ReduceLROnPlateau`` on
val_loss, training stops early when val_loss has not improved for ``--early-stop-patience`` epochs, and the 326-key
state_dict is saved to ``--out`` whenever val_miou improves.  At the end the best checkpoint is evaluated on the test
split and logged.

The reference's values are used where SURVEY records them (Adam lr 5e-4, weight decay 2e-3, Dropout 0.8, crop 512,
batch 5, 30 epochs, Lovasz loss).  It does not record the parameters of its ``ReduceLROnPlateau`` and ``EarlyStopping``:
the plateau rule takes torch's defaults (factor 0.1, patience 10), and early stopping waits 20 epochs, twice the plateau
patience, so that the learning rate is lowered before training gives up.  Normalisation is predict's
(``NeuralBarkCalculator.DEFAULT_MEAN / DEFAULT_STD``): the checkpoint carries none.  ``--init random`` starts from
torchvision's initialisation (ImageNet weights would need a download).

Data parallel and gradient accumulation.  ``--batch`` is the micro-batch, the size the network step runs at; under
``torchrun`` with W ranks (rank r on cuda:LOCAL_RANK, NCCL) and ``--accumulate K`` one optimizer step covers the global
batch G = W * K * batch.  Every rank loads the whole folder and draws the same epoch batches of G and the same
augmentation parameters of each (same seeds: no communication); micro-batch j is the slice [j * batch, (j + 1) * batch)
of both, and rank r runs micro-batches r * K .. r * K + K - 1, accumulating their gradients, before one all-reduce and one
Adam step on the mean.  Micro-batch j's dropout seed depends on j and the step only (``train.dropout_seed``), so a W-GPU
run is the same training as a one-GPU run with ``--accumulate`` W * K, draw for draw, except for the BatchNorm running
statistics: each rank updates its own once per micro-batch, and at the end of each epoch they are averaged over the
ranks (one small all-reduce), where the one-GPU run updates one set once per micro-batch in sequence.  As in torch DDP
without SyncBatchNorm, the BatchNorm batch statistics and the Lovasz sort see the micro-batch, not the global batch,
and ``--lr`` is not rescaled with G.  W = 1 and K = 1 make exactly the draws and calls of a one-GPU run.  The epoch's
training loss is the mean over all micro-batches of all ranks (one all-reduce per epoch).  Validation is sharded over
the ranks (``evaluate.evaluate_sharded``) and gives every rank the figures of a one-GPU evaluation bit for bit, so the
plateau and early-stopping decisions agree; rank 0 alone writes ``--log`` and ``--out``.  Every rank keeps the best
state_dict in host memory and evaluates the test split from it, sharded.  On stdout, rank 0 reports each epoch's
optimizer steps, training-loop and validation seconds, and every rank its dataset load time.

Fine-tuning a checkpoint.  ``--freeze stem|layer1|layer2|layer3|layer4`` freezes the backbone from the stem through
that stage (``--init`` must then be a checkpoint, not ``random``).  The frozen units run as eval-mode BatchNorm with
the checkpoint's running statistics (torchvision's FrozenBatchNorm2d, with ``requires_grad_(False)`` on their weights):
their weights, running statistics and ``num_batches_tracked`` stay exactly as loaded, Adam and its weight decay never
touch them, the backward stops at the first trainable block, and the epoch-end average of the running statistics over
the ranks covers only the trainable units.  Dropout, the loss and the sampling are unchanged; the checkpoint is the same
326-key state_dict.  Rank 0 prints the number of trainable parameters.

Resuming an interrupted run.  With ``--state FILE``, rank 0 writes FILE at the end of every epoch, after the log row and
the checkpoint: a format version, the run-defining arguments (the folder's items with their wood types and sizes,
--crop --batch --accumulate, the world size, --freeze --target --loss --lr --weight-decay --dropout --plateau-*
--early-stop-patience --seed), the epoch just finished, ``Trainer.training_state()`` (weights and running statistics,
Adam moments, step count, learning rate, ``num_batches_tracked``), the plateau and early-stopping counters, the best
val_miou and its state_dict, the log rows so far, the epoch-sampling ``torch.Generator`` and the augmentation
``numpy`` generator states, and whether the run stopped early.  The file is written to a temporary file in the same
directory, flushed, fsynced and renamed over FILE, so a kill during the write leaves the previous state intact.  At an
epoch boundary every rank holds the same state (same all-reduced gradients, same Adam step, averaged running
statistics); fit checks this with a digest of each rank's buffers before each write and stops if they differ.
``--resume`` continues from FILE: it refuses, naming each field, if a run-defining argument or the folder differs
(``--epochs``, ``--log``, ``--out``, ``--device`` and ``--init`` may change; a larger ``--epochs`` continues a finished
run), recomputes the splits as at the start, restores all of the above, rewrites ``--log`` as the header plus the saved
epochs' rows and ``--out`` from the saved best state_dict, and continues with the next epoch.  A run that had stopped
early only re-runs the test evaluation.  The weight-gradient reductions are deterministic, so a resumed run writes
exactly the log (but for ``seconds``), checkpoint and state of the run that was never interrupted (same GPU model,
world size and library build)."""
import argparse
import math
import os
import time

import numpy as np

from .train import FREEZE


class Plateau:
    """``torch.optim.lr_scheduler.ReduceLROnPlateau(mode='min', threshold_mode='rel')`` for one learning rate: after
    more than ``patience`` epochs without a relative improvement of ``threshold``, lr = max(lr * factor, min_lr)."""

    def __init__(self, lr, factor=0.1, patience=10, threshold=1e-4, cooldown=0, min_lr=0.0, eps=1e-8):
        if factor >= 1.0:
            raise ValueError('Plateau: factor must be below 1')
        self.lr, self.factor, self.patience, self.threshold = float(lr), float(factor), int(patience), float(threshold)
        self.cooldown, self.min_lr, self.eps = int(cooldown), float(min_lr), float(eps)
        self.best = math.inf
        self.num_bad_epochs = 0
        self.cooldown_counter = 0

    def step(self, metric):
        current = float(metric)
        if current < self.best * (1.0 - self.threshold):
            self.best = current
            self.num_bad_epochs = 0
        else:
            self.num_bad_epochs += 1
        if self.cooldown_counter > 0:
            self.cooldown_counter -= 1
            self.num_bad_epochs = 0
        if self.num_bad_epochs > self.patience:
            new_lr = max(self.lr * self.factor, self.min_lr)
            if self.lr - new_lr > self.eps:
                self.lr = new_lr
            self.cooldown_counter = self.cooldown
            self.num_bad_epochs = 0
        return self.lr


    def state_dict(self):
        return {'lr': self.lr, 'best': self.best, 'num_bad_epochs': self.num_bad_epochs, 'cooldown_counter': self.cooldown_counter}

    def load_state_dict(self, d):
        self.lr, self.best = float(d['lr']), float(d['best'])
        self.num_bad_epochs, self.cooldown_counter = int(d['num_bad_epochs']), int(d['cooldown_counter'])


class EarlyStopping:
    """Poutyne's ``EarlyStopping(mode='min', min_delta=0)``: stop once the metric has not decreased for ``patience``
    epochs in a row."""

    def __init__(self, patience=20):
        self.patience = int(patience)
        self.best = math.inf
        self.wait = 0

    def step(self, metric):
        """True when training should stop after this epoch."""
        if float(metric) < self.best:
            self.best = float(metric)
            self.wait = 0
            return False
        self.wait += 1
        return self.wait >= self.patience

    def state_dict(self):
        return {'best': self.best, 'wait': self.wait}

    def load_state_dict(self, d):
        self.best, self.wait = float(d['best']), int(d['wait'])


LOG_HEADER = ['epoch', 'lr', 'loss', 'val_loss', 'val_miou', 'val_f1_0', 'val_f1_1', 'val_f1_2', 'seconds']


def _log(path, fields):
    with open(path, 'a') as f:
        f.write('\t'.join(str(v) for v in fields) + '\n')


STATE_VERSION = 1
# run-defining fields of the state file and how a refusal names them
RUN_FIELDS = {'version': 'the state format version', 'items': 'the folder (item names, wood types, sizes)',
              'world': 'the world size', 'crop': '--crop', 'batch': '--batch', 'accumulate': '--accumulate',
              'freeze': '--freeze', 'target': '--target', 'loss': '--loss', 'lr': '--lr', 'weight_decay': '--weight-decay',
              'dropout': '--dropout', 'plateau_factor': '--plateau-factor', 'plateau_patience': '--plateau-patience',
              'early_stop_patience': '--early-stop-patience', 'seed': '--seed'}


def run_config(args, items, world):
    """The arguments a resumed run must share with the run that wrote the state.  ``items``: [(name, wood type,
    height, width)] of the folder in dataset order."""
    cfg = {k: getattr(args, k) for k in RUN_FIELDS if hasattr(args, k)}
    cfg.update(version=STATE_VERSION, items=[(str(n), str(w), int(h), int(wd)) for n, w, h, wd in items], world=int(world))
    return cfg


def check_resume(saved, current):
    """Raise naming every run-defining field in which ``current`` differs from ``saved``."""
    bad = [k for k in RUN_FIELDS if saved.get(k) != current.get(k)]
    if bad:
        def show(v):
            return '%d items' % len(v) if isinstance(v, list) else repr(v)
        raise RuntimeError('fit --resume: the state was written by a different run; it differs in ' + '; '.join(
            '%s (saved %s, now %s)' % (RUN_FIELDS[k], show(saved.get(k)), show(current.get(k))) for k in bad))


def write_state(path, state):
    """torch.save ``state`` to ``path`` atomically: a temporary file in the same directory, flushed and fsynced, then
    renamed over ``path``.  An exception or a kill before the rename leaves the previous file as it was."""
    import torch
    d = os.path.dirname(os.path.abspath(path))
    tmp = os.path.join(d, '.%s.tmp%d' % (os.path.basename(path), os.getpid()))
    try:
        with open(tmp, 'wb') as f:
            torch.save(state, f)
            f.flush()
            os.fsync(f.fileno())
        os.replace(tmp, path)
    finally:
        if os.path.exists(tmp):
            os.remove(tmp)


def read_state(path):
    import torch
    if not os.path.isfile(path):
        raise RuntimeError('fit --resume: no state file %s' % path)
    return torch.load(path, map_location='cpu', weights_only=False)


def rewrite_log(path, rows):
    """--log as the header plus ``rows`` (the saved epochs): drops whatever a killed run appended after its last
    state, and the test row of a finished run."""
    with open(path, 'w') as f:
        f.write('\t'.join(LOG_HEADER) + '\n')
        for r in rows:
            f.write('\t'.join(str(v) for v in r) + '\n')


def state_digest(trainer):
    """int64 sums of the bit patterns of the weights, statistics and Adam moments: equal on every rank when the
    ranks hold the same training state."""
    import torch
    bufs = (trainer.params, trainer.stats, trainer.adam_m, trainer.adam_v)
    return torch.stack([b.view(torch.int32).to(torch.int64).sum() for b in bufs])


def initial_state_dict(init, dropout):
    import torch
    from .models import fcn_resnet50
    if init == 'random':
        return fcn_resnet50(pretrained=False, dropout=dropout).state_dict()
    if not os.path.isfile(init):
        raise RuntimeError('--init %s: no such file (give a state_dict saved with torch.save, or "random")' % init)
    return torch.load(init, map_location='cpu')


def average_running_stats(stats, stats_off, world):
    """BatchNorm running statistics averaged over the ranks, in place, for the trainable units only (``stats_off`` on):
    a mean of identical values is not always exact ((x + x + x) / 3), and frozen statistics must stay bit-identical."""
    import torch.distributed as dist
    trainable = stats[stats_off:]
    dist.all_reduce(trainable)
    trainable.div_(world)


def rank_micro_batches(batches, rng, rank, accumulate, batch, n_sources, crop, target):
    """This rank's share of each global batch of the epoch.  ``batches``: int64 [steps, G] sources from
    ``utils.weighted_epoch_batches``; per row, the augmentation parameters of all G samples are drawn from ``rng``
    (every rank makes the same draws), and the row's micro-batches j = rank * accumulate .. (rank + 1) * accumulate - 1
    are yielded as [(j, params[j * batch:(j + 1) * batch])]."""
    from . import augment
    for row in batches:
        params = augment.draw_params(rng, len(row), n_sources, crop, target, sources=row.numpy())
        yield [(j, params[j * batch:(j + 1) * batch]) for j in range(rank * accumulate, (rank + 1) * accumulate)]


def _items(ds):
    return [(f, w, int(h), int(wd)) for f, w, (h, wd) in zip(ds.fnames, ds.wood_types, ds.sizes)]


def main(args):
    import torch
    from . import augment, distributed as ndist, utils
    from .evaluate import evaluate_sharded, make_plan
    from .train import Trainer
    rank, local_rank, world = ndist.env_world()
    device = args.device
    if world > 1:
        import torch.distributed as dist
        device = 'cuda:%d' % local_rank
        torch.cuda.set_device(local_rank)
        ndist.init_from_env('cuda')
        ndist.bind_to_gpu_numa(local_rank)
    torch.manual_seed(args.seed)
    np.random.seed(args.seed)            # get_splits shuffles with numpy's global generator, as the reference
    target = (args.target, args.target)
    t0 = time.perf_counter()
    ds = augment.load_dataset(args.root, device)       # every rank: any rank may be handed any source
    print('fit: rank %d loaded %d images in %.3f s' % (rank, len(ds), time.perf_counter() - t0), flush=True)
    train_split, valid_split, test_split, train_weights = utils.get_splits(ds.split_items(), label_pixels=ds.label_pixels)
    if len(valid_split) == 0:
        raise RuntimeError('fit: the validation split is empty (a wood type needs at least 10 images for one)')
    saved = read_state(args.state) if args.resume else None
    if saved is not None:
        check_resume(saved['config'], run_config(args, _items(ds), world))
    init_sd = saved['trainer']['model'] if saved is not None else initial_state_dict(args.init, args.dropout)
    trainer = Trainer(init_sd, args.batch, args.crop, args.crop, device=device,
                      lr=args.lr, weight_decay=args.weight_decay, dropout=args.dropout, loss=args.loss, seed=args.seed,
                      freeze=args.freeze)
    if rank == 0:
        print('fit: --freeze %s: %d of %d parameters trainable' % (
            args.freeze, trainer.params.numel() - trainer.param_off, trainer.params.numel()), flush=True)
    generator = torch.Generator().manual_seed(args.seed)
    rng = np.random.default_rng(args.seed)
    plateau = Plateau(args.lr, factor=args.plateau_factor, patience=args.plateau_patience)
    stopper = EarlyStopping(args.early_stop_patience)
    global_batch = world * args.accumulate * args.batch
    best_miou, best_sd, log_rows, first_epoch, stopped = -math.inf, None, [], 1, False
    if saved is not None:
        trainer.load_training_state(saved['trainer'])
        plateau.load_state_dict(saved['plateau'])
        stopper.load_state_dict(saved['early_stopping'])
        generator.set_state(saved['generator'])
        rng.bit_generator.state = saved['rng']
        best_miou, best_sd, log_rows = saved['best_miou'], saved['best_model'], saved['log']
        first_epoch, stopped = saved['epoch'] + 1, saved['stopped']
        if rank == 0:
            if best_sd is not None:
                torch.save(best_sd, args.out)
            print('fit: resuming from %s after epoch %d%s' % (args.state, saved['epoch'],
                  ' (the run had stopped early: only the test evaluation runs)' if stopped else ''), flush=True)
        del saved
    if rank == 0:
        rewrite_log(args.log, log_rows)
    reported = False
    for epoch in range(first_epoch, args.epochs + 1):
        if stopped:
            break
        t0 = time.perf_counter()
        lr = trainer.lr
        batches = utils.weighted_epoch_batches(train_split, train_weights, global_batch, generator=generator)
        if len(batches) == 0:
            raise RuntimeError('fit: the training split gives no full global batch of %d' % global_batch)
        with torch.cuda.device(trainer.device):
            total = torch.zeros((), dtype=torch.float32, device=trainer.device)
            for micro in rank_micro_batches(batches, rng, rank, args.accumulate, args.batch, len(ds), args.crop, target):
                for i, (j, params) in enumerate(micro):
                    images, classes = augment.augment_ragged(ds, params, args.crop, target)
                    total += trainer.forward_backward(images, classes, seed=trainer.dropout_seed(j), accumulate=i > 0)
                trainer.optimizer_step()
            if world > 1:
                dist.all_reduce(total)
                average_running_stats(trainer.stats, trainer.stats_off, world)
            train_loss = float(total) / (len(batches) * world * args.accumulate)
        t_train = time.perf_counter() - t0
        with torch.cuda.device(trainer.device):
            sd = trainer.state_dict()
            val = evaluate_sharded(make_plan(sd, trainer.device), ds, valid_split, loss=args.loss,
                                   class_weights=trainer.class_weights)
        row = ([epoch, repr(lr), repr(train_loss), repr(val['loss']), repr(val['miou'])] + [repr(float(v)) for v in val['f1']]
               + ['%.3f' % (time.perf_counter() - t0)])
        log_rows.append(row)
        if rank == 0:
            _log(args.log, row)
            print('fit: epoch %d: %d steps of %d samples, training %.3f s, validation %.3f s'
                  % (epoch, len(batches), global_batch, t_train, time.perf_counter() - t0 - t_train), flush=True)
        if val['miou'] > best_miou:
            best_miou = val['miou']
            best_sd = {k: v.cpu() for k, v in sd.items()}
            if rank == 0:
                torch.save(best_sd, args.out)
        del sd
        trainer.lr = plateau.step(val['loss'])
        stopped = stopper.step(val['loss'])
        if args.state:
            if world > 1:
                with torch.cuda.device(trainer.device):
                    digest = state_digest(trainer)
                    lo, hi = digest.clone(), digest.clone()
                    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
                    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
                    if not torch.equal(lo, hi):
                        raise RuntimeError('fit: the ranks hold different training states after epoch %d' % epoch)
            if rank == 0:
                t1 = time.perf_counter()
                write_state(args.state, {
                    'config': run_config(args, _items(ds), world), 'epoch': epoch, 'trainer': trainer.training_state(),
                    'plateau': plateau.state_dict(), 'early_stopping': stopper.state_dict(), 'best_miou': best_miou,
                    'best_model': best_sd, 'log': log_rows, 'generator': generator.get_state(),
                    'rng': rng.bit_generator.state, 'stopped': stopped})
                if not reported:
                    print('fit: state %s: %.1f MB, written in %.3f s' % (
                        args.state, os.path.getsize(args.state) / 1e6, time.perf_counter() - t1), flush=True)
                    reported = True
        if stopped:
            break
    if len(test_split):
        t0 = time.perf_counter()
        with torch.cuda.device(trainer.device):
            test = evaluate_sharded(make_plan(best_sd, trainer.device), ds, test_split, loss=args.loss)
        if rank == 0:
            _log(args.log, ['test', '', '', repr(test['loss']), repr(test['miou'])] + [repr(float(v)) for v in test['f1']]
                 + ['%.3f' % (time.perf_counter() - t0)])
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return best_miou


def parse_args(argv=None):
    parser = argparse.ArgumentParser(prog='python -m neuralbarkcalculator_b200.fit')
    parser.add_argument('root', help='labelled folder with samples/<wood>/ and duals/<wood>/')
    parser.add_argument('--init', required=True, help='initial state_dict (torch.save file), or "random"')
    parser.add_argument('--out', default='best_model.pt', help='checkpoint written when val_miou improves')
    parser.add_argument('--log', default='log.tsv', help='one tab-separated row per epoch, then the test row')
    parser.add_argument('--epochs', type=int, default=30)
    parser.add_argument('--crop', type=int, default=512)
    parser.add_argument('--batch', type=int, default=5, help='micro-batch: the size one network step runs at')
    parser.add_argument('--accumulate', type=int, default=1,
                        help='micro-batches per rank summed into one optimizer step (global batch = ranks x this x --batch)')
    parser.add_argument('--freeze', default='none', choices=list(FREEZE),
                        help='freeze the backbone from the stem through this stage (eval-mode BatchNorm; needs --init SD.pt)')
    parser.add_argument('--target', type=int, default=1024, help='pad_resize size of every image')
    parser.add_argument('--loss', default='lovasz', choices=['lovasz', 'weighted_ce', 'mixed'])
    parser.add_argument('--lr', type=float, default=5e-4)
    parser.add_argument('--weight-decay', type=float, default=2e-3)
    parser.add_argument('--dropout', type=float, default=0.8)
    parser.add_argument('--plateau-factor', type=float, default=0.1)
    parser.add_argument('--plateau-patience', type=int, default=10)
    parser.add_argument('--early-stop-patience', type=int, default=20)
    parser.add_argument('--seed', type=int, default=0)
    parser.add_argument('--device', default='cuda:0', help='CUDA device (cuda, cuda:N); under torchrun cuda:LOCAL_RANK')
    parser.add_argument('--state', default=None, help='training state written at the end of every epoch (for --resume)')
    parser.add_argument('--resume', action='store_true', help='continue the run whose --state file is given')
    args = parser.parse_args(argv)
    if not args.device.startswith('cuda'):
        parser.error('--device %s: only CUDA devices are supported (no CPU path)' % args.device)
    if args.epochs < 1 or args.batch < 1 or args.crop < 1 or args.crop > args.target:
        parser.error('--epochs and --batch must be positive and --crop within [1, --target]')
    if args.accumulate < 1:
        parser.error('--accumulate must be at least 1')
    if args.resume and not args.state:
        parser.error('--resume needs --state FILE')
    if args.freeze != 'none' and args.init == 'random' and not args.resume:
        parser.error('--freeze %s needs --init SD.pt: freezing randomly initialised layers is almost certainly a mistake'
                     % args.freeze)
    return args


if __name__ == '__main__':
    main(parse_args())
