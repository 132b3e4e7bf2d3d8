"""Worker of tests/test_gpu_train_freeze.py::test_two_rank_frozen_step (launched with torch.distributed.run, one process
per GPU): with layer2 frozen, a data-parallel step with one micro-batch per rank gives, after the exchange, the gradient
of one Trainer that accumulates the same micro-batches, in both exchange modes; Adam leaves identical weights on every
rank; and the epoch-end average of the running statistics leaves the frozen ones bit-identical."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    from oracle import model as omodel, synth
    from neuralbarkcalculator_b200.fit import average_running_stats
    from neuralbarkcalculator_b200.train import Trainer, dropout_seed, gradient_segments
    os.environ.pop('NBC_TRAIN_BUCKETS', None)
    rank, world = int(os.environ['RANK']), int(os.environ['WORLD_SIZE'])
    local = int(os.environ['LOCAL_RANK'])
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    dist.init_process_group('nccl', device_id=dev)
    g = np.load(os.path.join(ROOT, 'tests', 'golden', 'model_small.npz'))
    sd = omodel.synthetic_state_dict(seed=int(g['state_dict_seed']), head=(g['head_w'], g['head_b']))
    N, H, W, base, freeze = 2, 64, 96, 11, 'layer2'
    micro = [(torch.from_numpy(np.stack([synth.texture_u8(H, W, 10 * j + i) for i in range(N)])).to(dev),
              torch.from_numpy(np.stack([synth.class_mask(H, W, 50 + 10 * j + i) for i in range(N)])).to(dev))
             for j in range(world)]
    ref = Trainer(sd, N, H, W, device=str(dev), loss='lovasz', seed=base, freeze=freeze)
    for j, (x, t) in enumerate(micro):
        ref.forward_backward(x, t, seed=dropout_seed(base, j, 0), accumulate=j > 0)
    torch.cuda.synchronize()
    want = ref.grads.clone()
    segments = [s for s in gradient_segments(ref.lib, ref.handle) if s[1] > 0]
    del ref
    for bucket_mb in (0.0, 16.0):
        tr = Trainer(sd, N, H, W, device=str(dev), loss='lovasz', seed=base, bucket_mb=bucket_mb, freeze=freeze)
        x, t = micro[rank]
        before, stats0 = tr.params.clone(), tr.stats.clone()
        tr.forward_backward(x, t, seed=tr.dropout_seed())
        tr.optimizer_step()
        average_running_stats(tr.stats, tr.stats_off, world)
        torch.cuda.synchronize()
        assert torch.equal(tr.grads[:tr.param_off], torch.zeros_like(tr.grads[:tr.param_off]))
        for i, (off, cnt) in enumerate(segments):
            a, b = tr.grads[off:off + cnt], want[off:off + cnt]
            rel = ((a - b).norm() / (b.norm() + 1e-30)).item()
            assert rel <= 1e-3, 'bucket_mb %g: segment %d differs from one-GPU accumulation by %.3g (relative)' % (bucket_mb, i, rel)
        ps = [torch.empty_like(tr.params) for _ in range(world)]
        dist.all_gather(ps, tr.params)
        assert all(torch.equal(ps[0], p) for p in ps[1:]), 'weights diverged across ranks (bucket_mb %g)' % bucket_mb
        assert torch.equal(tr.params[:tr.param_off], before[:tr.param_off]), 'a frozen weight moved'
        assert not torch.equal(tr.params[tr.param_off:], before[tr.param_off:]), 'Adam did not move the weights'
        assert torch.equal(tr.stats[:tr.stats_off], stats0[:tr.stats_off]), 'a frozen running statistic changed'
        del tr
    if rank == 0:
        print('FREEZE_PARALLEL_OK world=%d grad_norm=%.6g' % (world, float(want.norm())))
    dist.barrier()
    dist.destroy_process_group()


if __name__ == '__main__':
    main()
