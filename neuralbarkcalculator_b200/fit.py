"""Train a network from a labelled folder and write the checkpoint ``predict.py`` reads (the epoch loop of the
reference's ``__main__.py:199-291``, which runs it through Poutyne).

    python -m neuralbarkcalculator_b200.fit ROOT --init SD.pt|random [--out best_model.pt] [--epochs 30] [--crop 512]
        [--batch 5] [--loss lovasz] [--lr 5e-4] [--weight-decay 2e-3] [--dropout 0.8] [--seed 0] [--device cuda:0]

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
(``NeuralBarkCalculator.DEFAULT_MEAN / DEFAULT_STD``): the checkpoint carries none.  One GPU; ``--init random`` starts
from torchvision's initialisation (ImageNet weights would need a download)."""
import argparse
import math
import os
import time

import numpy as np


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


LOG_HEADER = ['epoch', 'lr', 'loss', 'val_loss', 'val_miou', 'val_f1_0', 'val_f1_1', 'val_f1_2', 'seconds']


def _log(path, fields):
    with open(path, 'a') as f:
        f.write('\t'.join(str(v) for v in fields) + '\n')


def initial_state_dict(init, dropout):
    import torch
    from .models import fcn_resnet50
    if init == 'random':
        return fcn_resnet50(pretrained=False, dropout=dropout).state_dict()
    if not os.path.isfile(init):
        raise RuntimeError('--init %s: no such file (give a state_dict saved with torch.save, or "random")' % init)
    return torch.load(init, map_location='cpu')


def main(args):
    import torch
    from . import augment, utils
    from .evaluate import evaluate
    from .train import Trainer
    torch.manual_seed(args.seed)
    np.random.seed(args.seed)            # get_splits shuffles with numpy's global generator, as the reference
    target = (args.target, args.target)
    ds = augment.load_dataset(args.root, args.device)
    train_split, valid_split, test_split, train_weights = utils.get_splits(ds.split_items(), label_pixels=ds.label_pixels)
    if len(valid_split) == 0:
        raise RuntimeError('fit: the validation split is empty (a wood type needs at least 10 images for one)')
    trainer = Trainer(initial_state_dict(args.init, args.dropout), args.batch, args.crop, args.crop, device=args.device,
                      lr=args.lr, weight_decay=args.weight_decay, dropout=args.dropout, loss=args.loss, seed=args.seed)
    generator = torch.Generator().manual_seed(args.seed)
    rng = np.random.default_rng(args.seed)
    plateau = Plateau(args.lr, factor=args.plateau_factor, patience=args.plateau_patience)
    stopper = EarlyStopping(args.early_stop_patience)
    with open(args.log, 'w') as f:
        f.write('\t'.join(LOG_HEADER) + '\n')
    best_miou = -math.inf
    for epoch in range(1, args.epochs + 1):
        t0 = time.perf_counter()
        lr = trainer.lr
        batches = utils.weighted_epoch_batches(train_split, train_weights, args.batch, generator=generator)
        if len(batches) == 0:
            raise RuntimeError('fit: the training split gives no full batch of %d' % args.batch)
        with torch.cuda.device(trainer.device):
            total = torch.zeros((), dtype=torch.float32, device=trainer.device)
            for row in batches:
                params = augment.draw_params(rng, args.batch, len(ds), args.crop, target, sources=row.numpy())
                images, classes = augment.augment_ragged(ds, params, args.crop, target)
                total += trainer.step(images, classes)
            train_loss = float(total) / len(batches)
        val = trainer.evaluate(ds, valid_split)
        _log(args.log, [epoch, repr(lr), repr(train_loss), repr(val['loss']), repr(val['miou'])]
             + [repr(float(v)) for v in val['f1']] + ['%.3f' % (time.perf_counter() - t0)])
        if val['miou'] > best_miou:
            best_miou = val['miou']
            torch.save({k: v.cpu() for k, v in trainer.state_dict().items()}, args.out)
        trainer.lr = plateau.step(val['loss'])
        if stopper.step(val['loss']):
            break
    if len(test_split):
        t0 = time.perf_counter()
        test = evaluate(torch.load(args.out, map_location='cpu'), ds, test_split, loss=args.loss)
        _log(args.log, ['test', '', '', repr(test['loss']), repr(test['miou'])] + [repr(float(v)) for v in test['f1']]
             + ['%.3f' % (time.perf_counter() - t0)])
    return best_miou


def parse_args(argv=None):
    parser = argparse.ArgumentParser(prog='python -m neuralbarkcalculator_b200.fit')
    parser.add_argument('root', help='labelled folder with samples/<wood>/ and duals/<wood>/')
    parser.add_argument('--init', required=True, help='initial state_dict (torch.save file), or "random"')
    parser.add_argument('--out', default='best_model.pt', help='checkpoint written when val_miou improves')
    parser.add_argument('--log', default='log.tsv', help='one tab-separated row per epoch, then the test row')
    parser.add_argument('--epochs', type=int, default=30)
    parser.add_argument('--crop', type=int, default=512)
    parser.add_argument('--batch', type=int, default=5)
    parser.add_argument('--target', type=int, default=1024, help='pad_resize size of every image')
    parser.add_argument('--loss', default='lovasz', choices=['lovasz', 'weighted_ce', 'mixed'])
    parser.add_argument('--lr', type=float, default=5e-4)
    parser.add_argument('--weight-decay', type=float, default=2e-3)
    parser.add_argument('--dropout', type=float, default=0.8)
    parser.add_argument('--plateau-factor', type=float, default=0.1)
    parser.add_argument('--plateau-patience', type=int, default=10)
    parser.add_argument('--early-stop-patience', type=int, default=20)
    parser.add_argument('--seed', type=int, default=0)
    parser.add_argument('--device', default='cuda:0', help='CUDA device (cuda, cuda:N)')
    args = parser.parse_args(argv)
    if not args.device.startswith('cuda'):
        parser.error('--device %s: only CUDA devices are supported (no CPU path)' % args.device)
    if args.epochs < 1 or args.batch < 1 or args.crop < 1 or args.crop > args.target:
        parser.error('--epochs and --batch must be positive and --crop within [1, --target]')
    return args


if __name__ == '__main__':
    main(parse_args())
