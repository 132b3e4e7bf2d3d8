"""``predict.py`` of the reference (predict.py:1-81) on the B200 path.

    python -m neuralbarkcalculator_b200.predict ROOT_DIR [--device cuda:0] [--exclude_nodes] [--only_preprocess]
        [--tta none|h|hv]

Same arguments, same ``processed/`` and ``results/`` layout, weights from ``./best_model.pt``.  ``--tta`` adds flip
test-time augmentation (``h``: the image and its column mirror, ``hv``: also the row mirrors; the class map is the argmax
of the views' mean logits); without it every file is the one the plain network gives.  ``--device`` accepts
``cuda`` / ``cuda:N``; ``cpu`` is rejected (this build has no CPU path -- use the reference for that)."""
import argparse
import os

from .models import NeuralBarkCalculator
from .ops import TTA_MODES

ALL_WOOD_TYPES = ['epinette_gelee', 'epinette_non_gelee', 'sapin']


def generate_folders(root_path, only_preprocess):
    """predict.py:10-48: processed/samples/<wood> and results/{combined_images,outputs}/<wood> for present woods."""
    present = [w for w in ALL_WOOD_TYPES if w in set(os.listdir(os.path.join(root_path, 'samples')))]
    trees = [('processed', ['samples'])] + ([] if only_preprocess else [('results', ['combined_images', 'outputs'])])
    for top, levels in trees:
        for level in levels:
            os.makedirs(os.path.join(root_path, top, level), exist_ok=True)
            for wood in present:
                os.makedirs(os.path.join(root_path, top, level, wood), exist_ok=True)


def main(args, state_dict=None):
    """predict.py:51-58.  Every folder goes through the streaming FolderPipeline -- preprocessing and prediction fused
    into one pass with batched GPU work and threaded file IO.  Folders of standard scans (4096x4096 24-bit BMP) take its
    uniform route, any other folder its mixed route; both write the files the per-image path of models.py
    (``Preprocessor`` + ``NeuralBarkCalculator.predict``) writes.

    Under ``torchrun`` (one process per GPU) every rank takes a contiguous shard of the dataset order on cuda:LOCAL_RANK --
    images are independent, there is no collective on the data path -- and rank 0 merges the CSV rows back into dataset
    order, so the files are identical to a single-GPU run."""
    import csv
    import time
    from . import distributed as ndist
    from . import pipeline
    from .dataset import make_dataset
    rank, local_rank, world = ndist.env_world()
    device = args.device
    if world > 1:
        device = 'cuda:%d' % local_rank
        ndist.init_from_env('cuda')
        ndist.bind_to_gpu_numa(local_rank)
    t0 = time.perf_counter()
    if rank == 0:
        generate_folders(args.root_path, args.only_preprocess)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    items = make_dataset(args.root_path)
    model = NeuralBarkCalculator(None if state_dict is not None else './best_model.pt', device, state_dict=state_dict,
                                 load_weights=not args.only_preprocess, tta=getattr(args, 'tta', 'none'))
    if os.environ.get('NBC_TIMING'):
        print('[nbc] folders + model construction: %.3f s' % (time.perf_counter() - t0))
    pipe = pipeline.FolderPipeline(model)
    shard = ndist.shard_bounds(len(items), rank, world) if world > 1 else None
    out = pipe.run(args.root_path, args.exclude_nodes, args.only_preprocess, shard=shard)
    if world > 1 and not args.only_preprocess:
        rows = ndist.merge_rows(out, shard[0], len(items))
        out = None
        if rank == 0:
            out = [pipeline.CSV_HEADER] + rows
            with open(os.path.join(args.root_path, 'results', 'final_stats.csv'), 'w') as f:   # models.py:360-364
                csv.writer(f, delimiter='\t').writerows(out)
    if os.environ.get('NBC_TIMING'):
        print('[nbc] folder pipeline timing: %s' % pipe.last_timing)
    return out


def parse_args(argv=None):
    parser = argparse.ArgumentParser()
    parser.add_argument('root_path', type=str, help='root directory path.')
    parser.add_argument('--device', type=str, default='cuda:0', help='Which CUDA device to run on (cuda, cuda:N).')
    parser.add_argument('--exclude_nodes', action='store_true', default=False)
    parser.add_argument('--only_preprocess', action='store_true', default=False)
    parser.add_argument('--tta', default='none', choices=list(TTA_MODES),
                        help='flip test-time augmentation: none, h (image + column mirror) or hv (+ row mirrors)')
    args = parser.parse_args(argv)
    if not args.device.startswith('cuda'):
        parser.error("--device %s: only CUDA devices are supported by this build (no CPU path)" % args.device)
    if args.only_preprocess and args.tta != 'none':
        parser.error('--tta %s: --only_preprocess runs no network' % args.tta)
    return args


if __name__ == '__main__':
    main(parse_args())
