"""The network pass bench.py's roofline is quoted on -- a dense [8,624,1024,3] chunk -- run `iters` times (for ncu).
usage: python tools/prof_forward.py [N] [H] [W] [iters]"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import neuralbarkcalculator_b200 as nbc  # noqa: E402
from oracle import model as omodel, synth  # noqa: E402

N = int(sys.argv[1]) if len(sys.argv) > 1 else 8
H = int(sys.argv[2]) if len(sys.argv) > 2 else 624
W = int(sys.argv[3]) if len(sys.argv) > 3 else 1024
iters = int(sys.argv[4]) if len(sys.argv) > 4 else 3
root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
g = np.load(os.path.join(root, 'tests', 'golden', 'model_small.npz'))
sd = omodel.synthetic_state_dict(seed=0, head=(g['head_w'], g['head_b']))
dev = torch.device('cuda:0')
m = nbc.fcn_resnet50(pretrained=False)
m.load_state_dict(sd)
m.to(dev).eval()
m.set_normalisation(omodel.DEFAULT_MEAN, omodel.DEFAULT_STD)
plan = m.native_plan()
img = torch.from_numpy(synth.texture_u8(H, W, 5)).to(dev).unsqueeze(0).repeat(N, 1, 1, 1).contiguous()
out = plan.forward(img)          # warm-up (plan creation, first-launch attributes)
torch.cuda.synchronize()
t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
t0.record()
for _ in range(iters):
    out = plan.forward(img)
t1.record()
torch.cuda.synchronize()
ms = t0.elapsed_time(t1) / iters
print('forward x%d done, logits %s: %.3f ms per pass, %.3f ms per image' % (iters, tuple(out.shape), ms, ms / N))
