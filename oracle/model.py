"""Oracle for the network (reference ``models.py:27-43, 113-139, 221-223, 269-270``).  Test infrastructure only.

The FCN-ResNet50 of the reference is torchvision's ``resnet50(replace_stride_with_dilation=[False, True, True])``
wrapped by ``IntermediateLayerGetter({'layer4': 'out'})`` + the reference's own ``FCNHead`` + a *bicubic*
``F.interpolate`` to the input size.  torch / torchvision are present, so this is the reference's own code path
executed by the same library family, in ``.eval()`` (the reference forgets ``.eval()`` -- SURVEY.md D5 -- which makes
its own output non-deterministic; eval mode is the one deliberate deviation, as in ``__main__.py:299-300``).

Pinned by ``oracle/make_golden.py``: the reference's ``models.fcn_resnet50`` (imported with stubbed plotting /
skimage modules) gives bit-identical logits to ``fcn_resnet50`` below for the same state_dict and input.
"""
import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F
from torchvision.models import resnet
from torchvision.models._utils import IntermediateLayerGetter

DEFAULT_MEAN = [0.7399, 0.6139, 0.4401]   # models.py:208
DEFAULT_STD = [0.1068, 0.1272, 0.1271]    # models.py:209


class FCNHead(nn.Sequential):
    """models.py:113-124."""

    def __init__(self, in_channels, channels, dropout=0.1):
        inter = in_channels // 4
        super().__init__(nn.Conv2d(in_channels, inter, 3, padding=1, bias=False), nn.BatchNorm2d(inter), nn.ReLU(),
                         nn.Dropout(dropout), nn.Conv2d(inter, channels, 1))


class SimpleSegmentationModel(nn.Module):
    """models.py:27-43."""

    def __init__(self, backbone, classifier):
        super().__init__()
        self.backbone = backbone
        self.classifier = classifier

    def features(self, x):
        return self.classifier(self.backbone(x)["out"])

    def forward(self, x):
        size = x.shape[-2:]
        return F.interpolate(self.features(x), size=size, mode='bicubic', align_corners=False)


def fcn_resnet50(dropout=0.1):
    """models.py:127-139 with pretrained=False (predict path, models.py:221)."""
    backbone = resnet.resnet50(weights=None, replace_stride_with_dilation=[False, True, True])
    backbone = IntermediateLayerGetter(backbone, return_layers={'layer4': 'out'})
    return SimpleSegmentationModel(backbone, FCNHead(2048, 3, dropout))


def synthetic_state_dict(seed=0, logit_std=1.5, class_bias=(1.6, 0.2, -2.2), head=None, branch_gain=0.5, calibration='whiten'):
    """Seeded random-init weights with *randomised BatchNorm* (SURVEY.md 8d config 0).

    Default torchvision init leaves BN at gamma=1, beta=0, mean=0, var=1, so a wrong BN fold would still pass and
    eval-mode logits are ~0.04 in magnitude.  Here BN gamma ~ U(0.5,1.5), beta ~ N(0,0.1), running_mean ~ N(0,0.1),
    running_var ~ U(0.5,1.5); ``classifier.4`` is then calibrated (whitened) on one synthetic image so the class logits are
    decorrelated with standard deviation ``logit_std`` and mean ``class_bias[c]`` (class frequencies skewed like the reference's
    prior, utils.py:72-73).  ``head=(weight, bias)`` skips the calibration forward and installs a stored head
    (used by the golden fixtures so the state_dict is reproducible to the bit on any machine)."""
    g = torch.Generator().manual_seed(seed)
    torch.manual_seed(seed)
    model = fcn_resnet50()
    sd = model.state_dict()
    for k in sd:
        v = sd[k]
        if k.endswith('running_mean'):
            v.copy_(torch.randn(v.shape, generator=g) * 0.1)
        elif k.endswith('running_var'):
            v.copy_(torch.rand(v.shape, generator=g) + 0.5)
        elif ('bn' in k or 'downsample.1' in k or k.startswith('classifier.1')) and k.endswith('.weight'):
            v.copy_(torch.rand(v.shape, generator=g) + 0.5)
        elif ('bn' in k or 'downsample.1' in k or k.startswith('classifier.1')) and k.endswith('.bias'):
            v.copy_(torch.randn(v.shape, generator=g) * 0.1)
    # The last BN of each bottleneck feeds the residual sum; keep the stream from exploding over 16 blocks.
    # branch_gain: 0.5 (default) is a deliberately HARSH test network -- every block still changes the stream by ~50 %, so
    # rounding noise is re-amplified 16 times; trained ResNets (and torchvision's zero_init_residual) sit near 0.1.
    for k in sd:
        if k.endswith('bn3.weight'):
            sd[k].mul_(branch_gain)
    if head is None and calibration == 'features':
        # Classifier = three random directions on the STANDARDISED 512 head features, each class rescaled (diagonally) to
        # logit_std / class_bias.  Unlike 'whiten' below -- which multiplies the raw logits by cov^(-1/2) and so blows the
        # low-variance directions of three strongly correlated outputs, and any rounding noise in them, up by orders of
        # magnitude -- this head has the noise gain of an ordinary trained linear layer.
        from . import synth
        model.load_state_dict(sd)
        model.eval()
        with torch.no_grad():
            feats = model.backbone(normalise_u8(synth.texture_u8(256, 256, seed=1234 + seed)))['out']
            for layer in list(model.classifier.children())[:4]:      # conv3x3, BN, ReLU, Dropout (identity in eval)
                feats = layer(feats)
        F_ = feats.permute(0, 2, 3, 1).reshape(-1, feats.shape[1]).double()
        mu_f, sd_f = F_.mean(0), F_.std(0)
        alive = sd_f > 0.1 * sd_f.median()          # (nearly) constant channels carry no signal: weight 0, not 1/eps
        R = torch.randn(3, feats.shape[1], generator=g).double()
        Wd = torch.where(alive, R / sd_f.clamp_min(1e-12), torch.zeros_like(R))
        L = (F_ - mu_f) @ Wd.T
        scale = logit_std / L.std(0)
        Wd = Wd * scale[:, None]
        sd['classifier.4.weight'].copy_(Wd.float().view(3, -1, 1, 1))
        sd['classifier.4.bias'].copy_(torch.tensor(class_bias) - (Wd @ mu_f).float())
    elif head is None:
        from . import synth
        model.load_state_dict(sd)
        model.eval()
        with torch.no_grad():
            low = model.features(normalise_u8(synth.texture_u8(256, 256, seed=1234 + seed)))
        L = low.permute(0, 2, 3, 1).reshape(-1, 3).double()
        mu = L.mean(0)
        cov = torch.cov((L - mu).T)
        evals, evecs = torch.linalg.eigh(cov)
        A = (logit_std * (evecs @ torch.diag(evals.rsqrt()) @ evecs.T)).float()     # whitening: decorrelate classes
        W = sd['classifier.4.weight'].view(3, -1)
        b0 = sd['classifier.4.bias'].clone()
        sd['classifier.4.weight'].copy_((A @ W).view(3, -1, 1, 1))
        sd['classifier.4.bias'].copy_(torch.tensor(class_bias) + A @ (b0 - mu.float()))
    else:
        sd['classifier.4.weight'].copy_(torch.as_tensor(head[0]))
        sd['classifier.4.bias'].copy_(torch.as_tensor(head[1]))
    return {k: v.clone() for k, v in sd.items()}


def load_model(state_dict):
    m = fcn_resnet50()
    m.load_state_dict(state_dict, strict=True)
    return m.eval()


def normalise_u8(img_u8, mean=DEFAULT_MEAN, std=DEFAULT_STD):
    """ToTensor + Normalize (dataset.py:181-190 with models.py:233-237): u8 HWC -> f32 [1,3,H,W]."""
    x = torch.from_numpy(np.ascontiguousarray(img_u8)).permute(2, 0, 1).float().div(255)
    m = torch.tensor(mean, dtype=torch.float32).view(3, 1, 1)
    s = torch.tensor(std, dtype=torch.float32).view(3, 1, 1)
    return ((x - m) / s).unsqueeze(0)


@torch.no_grad()
def lowres_logits(model, x):
    """Classifier output before the upsample: f32 [N,3,ceil(H/8),ceil(W/8)]."""
    return model.features(x)


@torch.no_grad()
def upsample_argmax(logits_lowres, size):
    """models.py:38-41 + models.py:270: bicubic (A=-0.75, align_corners=False) then argmax(dim=1), ties -> lowest."""
    up = F.interpolate(logits_lowres, size=size, mode='bicubic', align_corners=False)
    return up, torch.argmax(up, dim=1)


def bicubic_weights_f32(in_size, out_size, clamp=True):
    """Restated index / weight arithmetic of torch's upsample_bicubic2d (align_corners=False), all in float32.

    scale = in/out (f32); src = scale * (dst + 0.5) - 0.5 (f32); i0 = floor(src); t = src - i0; taps i0-1..i0+2
    clamped to [0, in-1]; cubic convolution coefficients with A = -0.75 (SURVEY.md a7).  ``clamp=False`` returns the
    unclamped tap indices (a deliberately wrong variant for negative controls)."""
    A = np.float32(-0.75)
    scale = np.float32(in_size) / np.float32(out_size)
    dst = np.arange(out_size, dtype=np.float32)
    src = scale * (dst + np.float32(0.5)) - np.float32(0.5)
    i0 = np.floor(src)
    t = (src - i0).astype(np.float32)
    i0 = i0.astype(np.int64)

    def c1(x):  # |x| <= 1
        return ((A + np.float32(2)) * x - (A + np.float32(3))) * x * x + np.float32(1)

    def c2(x):  # 1 < |x| < 2
        return ((A * x - np.float32(5) * A) * x + np.float32(8) * A) * x - np.float32(4) * A

    one = np.float32(1)
    w = np.stack([c2(t + one), c1(t), c1(one - t), c2((one - t) + one)], axis=1).astype(np.float32)
    idx = i0[:, None] + np.arange(-1, 3)[None, :]
    return (np.clip(idx, 0, in_size - 1) if clamp else idx), w


def upsample_bicubic_restated(low, size):
    """Bit-exact specification of the CUDA upsample kernel (head.cu): torch's bicubic arithmetic restated in float32
    with one rounding per operation (no fma) and a fixed summation order:

        inner_i = ((v[i,0]*wx0 + v[i,1]*wx1) + v[i,2]*wx2) + v[i,3]*wx3      (x taps, per source row i)
        out     = ((inner_0*wy0 + inner_1*wy1) + inner_2*wy2) + inner_3*wy3

    low: f32 array [N,C,h,w] -> f32 [N,C,H,W].  torch's own kernel differs from this by float round-off only
    (<= ~2e-6 relative; checked in tests/test_oracle.py)."""
    low = np.asarray(low, dtype=np.float32)
    N, C, h, w = low.shape
    H, W = size
    iy, wy = bicubic_weights_f32(h, H)
    ix, wx = bicubic_weights_f32(w, W)
    out = None
    for i in range(4):
        rows = low[:, :, iy[:, i], :]                      # [N,C,H,w]
        inner = None
        for j in range(4):
            term = (rows[:, :, :, ix[:, j]] * wx[None, None, None, :, j]).astype(np.float32)
            inner = term if inner is None else (inner + term).astype(np.float32)
        t = (inner * wy[None, None, :, i, None]).astype(np.float32)
        out = t if out is None else (out + t).astype(np.float32)
    return out


def argmax_lowest(up):
    """torch.argmax(dim=1) semantics: first (lowest) index among ties."""
    return np.argmax(np.asarray(up), axis=1).astype(np.uint8)
