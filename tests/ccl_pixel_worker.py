"""K5 calls for tests/test_gpu_ccl_patterns.py, in this process or as a child process.

``run_job`` hands one dense batch or ragged canvas to K5 four times, each time on a dirty workspace:
  1. every byte 0x00;
  2. each int32 of each of the four label / counter arrays equal to its own index, with exclude_nodes;
  3. the leftovers of call 2, on the canvas mirrored left to right (a different mask of the same shape);
  4. the leftovers of call 3, with exclude_nodes.
Every poison keeps labels[i] <= i (call 2 and 3 leftovers are clamped at 0: the per-pixel kernels write -1 outside the
set), so a kernel that reads a label it never wrote finds a wrong root inside the buffer, not a fault.  Call 1's mask and
counts are returned; calls 2 to 4 must give the same result, mirrored or with class 2 folded into 1, including the
untouched rows below each image's height.

As a script (``python ccl_pixel_worker.py IN.npz OUT.npz``) it runs every job of IN.npz and writes the results to
OUT.npz.  The test starts it with NBC_CCL_RUNS=0, so that every width takes the per-pixel kernels."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def run_job(canvas, heights, threshold, device):
    """canvas u8 [N, H, W]; heights int32 [N] (ragged) or None (dense).  Returns (mask, counts, problems)."""
    import torch
    from neuralbarkcalculator_b200 import _lib, ops
    lib = _lib.load()
    N, H, W = canvas.shape
    need = lib.nbc_ccl_workspace_bytes(N, H, W)
    ws = torch.empty(need, dtype=torch.uint8, device=device)
    ws32 = ws.view(torch.int32)
    per_array = -(-N * H * W * 4 // 256) * 256 // 4      # int32 entries from one label / counter array to the next
    hd = None if heights is None else torch.from_numpy(np.ascontiguousarray(heights, np.int32)).to(device)
    rows = torch.arange(H, device=device).view(1, H, 1)
    valid = torch.ones((N, H, 1), dtype=torch.bool, device=device) if hd is None else rows < hd.view(N, 1, 1)
    src = torch.from_numpy(np.ascontiguousarray(canvas)).to(device)

    def call(m, exclude):
        m = m.clone()
        if hd is None:
            _, counts = ops.remove_small_zones_u8(m, threshold, exclude, workspace=ws)
        else:
            _, counts = ops.remove_small_zones_ragged(m, hd, threshold, exclude, workspace=ws)
        return m, counts

    ws.zero_()
    first, first_counts = call(src, False)
    folded = torch.where(valid & (first == 2), torch.ones_like(first), first)
    folded_counts = first_counts.clone()
    folded_counts[:, 1] += folded_counts[:, 2]
    folded_counts[:, 2] = 0
    ws32.copy_(torch.arange(ws32.numel(), device=device, dtype=torch.int32) % per_array)
    expect = [('index poison, exclude_nodes', src, True, folded, folded_counts),
              ('leftovers, mirrored', src.flip(2), False, first.flip(2), first_counts),
              ('leftovers, exclude_nodes', src, True, folded, folded_counts)]
    problems = []
    for j, (what, m, exclude, exp, exp_counts) in enumerate(expect):
        if j > 0:
            ws32.clamp_(min=0)
        out, counts = call(m, exclude)
        if not torch.equal(out, exp):
            bad = (out != exp).nonzero()[0].tolist()
            problems.append('%s: %d bytes differ from the 0x00 call, first at %s' % (what, int((out != exp).sum()), bad))
        if not torch.equal(counts, exp_counts):
            problems.append('%s: counts differ from the 0x00 call' % what)
    torch.cuda.synchronize(device)
    return first.cpu().numpy(), first_counts.cpu().numpy(), problems


def main(src, dst):
    import torch
    from neuralbarkcalculator_b200 import _lib
    _lib.require_device(0)
    dev = torch.device('cuda:0')
    jobs = np.load(src)
    out = {}
    for k in range(int(jobs['count'])):
        heights = jobs['heights%d' % k] if 'heights%d' % k in jobs.files else None
        mask, counts, problems = run_job(jobs['canvas%d' % k], heights, int(jobs['threshold%d' % k]), dev)
        out['mask%d' % k], out['counts%d' % k] = mask, counts
        out['problems%d' % k] = np.array(problems, dtype=str)
    np.savez(dst, **out)


if __name__ == '__main__':
    main(sys.argv[1], sys.argv[2])
