"""Worker of tests/test_gpu_fit_parallel.py::test_two_rank_step_equals_one_gpu_accumulation (launched with
torch.distributed.run, one process per GPU): a data-parallel step with one micro-batch per rank gives, after the
exchange, the gradient of one Trainer that accumulates the same micro-batches with the same dropout seeds, in both
exchange modes (one all-reduce, buckets behind the backward), and Adam leaves identical weights on every rank."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    from oracle import model as omodel, synth
    from neuralbarkcalculator_b200.train import Trainer, dropout_seed, gradient_segments
    os.environ.pop('NBC_TRAIN_BUCKETS', None)
    rank, world = int(os.environ['RANK']), int(os.environ['WORLD_SIZE'])
    local = int(os.environ['LOCAL_RANK'])
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    dist.init_process_group('nccl', device_id=dev)
    g = np.load(os.path.join(ROOT, 'tests', 'golden', 'model_small.npz'))
    sd = omodel.synthetic_state_dict(seed=int(g['state_dict_seed']), head=(g['head_w'], g['head_b']))
    N, H, W, base = 2, 64, 96, 11
    micro = [(torch.from_numpy(np.stack([synth.texture_u8(H, W, 10 * j + i) for i in range(N)])).to(dev),
              torch.from_numpy(np.stack([synth.class_mask(H, W, 50 + 10 * j + i) for i in range(N)])).to(dev))
             for j in range(world)]
    # one GPU, world-fold accumulation (forward_backward only: its optimizer_step would join the group's all-reduce)
    ref = Trainer(sd, N, H, W, device=str(dev), loss='lovasz', seed=base)
    for j, (x, t) in enumerate(micro):
        ref.forward_backward(x, t, seed=dropout_seed(base, j, 0), accumulate=j > 0)
    torch.cuda.synchronize()
    want = ref.grads.clone()
    segments = gradient_segments(ref.lib, ref.handle)
    assert ref.micro_batches == world
    del ref
    for bucket_mb in (0.0, 16.0):
        tr = Trainer(sd, N, H, W, device=str(dev), loss='lovasz', seed=base, bucket_mb=bucket_mb)
        assert bucket_mb == 0 or len(tr.gradient_buckets()) >= 3
        x, t = micro[rank]
        before = tr.params.clone()
        tr.forward_backward(x, t, seed=tr.dropout_seed())          # rank r runs global micro-batch j = r
        tr.optimizer_step()                                        # exchange, then Adam on the mean
        torch.cuda.synchronize()
        for i, (off, cnt) in enumerate(segments):
            a, b = tr.grads[off:off + cnt], want[off:off + cnt]
            rel = ((a - b).norm() / (b.norm() + 1e-30)).item()
            assert rel <= 1e-3, 'bucket_mb %g: segment %d differs from one-GPU accumulation by %.3g (relative)' % (bucket_mb, i, rel)
        ps = [torch.empty_like(tr.params) for _ in range(world)]
        dist.all_gather(ps, tr.params)
        assert all(torch.equal(ps[0], p) for p in ps[1:]), 'weights diverged across ranks (bucket_mb %g)' % bucket_mb
        assert not torch.equal(tr.params, before), 'Adam did not move the weights'
        del tr
    if rank == 0:
        print('FIT_PARALLEL_OK world=%d grad_norm=%.6g' % (world, float(want.norm())))
    dist.barrier()
    dist.destroy_process_group()


if __name__ == '__main__':
    main()
