"""Shared helpers for the tests (synthetic inputs identical to tests/golden/_ref_worker.py)."""
import hashlib

import numpy as np
import torch


def synth(n, h, w, classes, seed=123, device="cpu"):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn((n, 3, h, w), generator=g)
    y = torch.randint(0, classes, (n, h, w), generator=g)
    ign = torch.rand((n, h, w), generator=g) < 0.05
    y[ign] = 255
    return x.to(device), y.to(device)


def rel_l2(a, b):
    a = torch.as_tensor(np.asarray(a) if not torch.is_tensor(a) else a.detach()).double().flatten().cpu()
    b = torch.as_tensor(np.asarray(b) if not torch.is_tensor(b) else b.detach()).double().flatten().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))


def build_pspnet(layers=50, classes=150, seed=0, **kw):
    from semseg_b200.pspnet import PSPNet
    torch.manual_seed(seed)
    return PSPNet(layers=layers, classes=classes, zoom_factor=8, dropout=0.0, pretrained=False, **kw)


def build_psanet(layers=50, classes=150, seed=0, mask=9, **kw):
    from semseg_b200.psanet import PSANet
    torch.manual_seed(seed)
    return PSANet(layers=layers, classes=classes, zoom_factor=8, dropout=0.0, psa_type=2, compact=False,
                  shrink_factor=2, mask_h=mask, mask_w=mask, pretrained=False, **kw)


def oracle_from(model, arch, **kw):
    """fp32 oracle sharing (clones of) the model's parameters and buffers."""
    from oracle.torch_oracle import Oracle
    params = {k for k, _ in model.named_parameters()}
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    for k, v in sd.items():
        if k in params:
            v.requires_grad_(True)
    return Oracle(sd, arch=arch, **kw), sd


class TinySegNet(torch.nn.Module):
    """Deterministic stand-in network of the sliding-window goldens (identical to tests/golden/_ref_worker.py)."""

    def __init__(self, classes=5, stride=1, seed=5):
        super().__init__()
        g = torch.Generator().manual_seed(seed)
        self.weight = torch.nn.Parameter(torch.randn((classes, 3, 3, 3), generator=g) * 0.6)
        self.bias = torch.nn.Parameter(torch.randn((classes,), generator=g) * 0.1)
        self.stride = stride

    def forward(self, x):
        if self.stride > 1:
            x = torch.nn.functional.avg_pool2d(x, self.stride)
        return torch.nn.functional.conv2d(x, self.weight, self.bias, padding=1)


SW_CFG = dict(classes=5, base_size=64, crop_h=33, crop_w=33, scales=[0.75, 1.0, 1.5],
              mean=[0.485 * 255, 0.456 * 255, 0.406 * 255], std=[0.229 * 255, 0.224 * 255, 0.225 * 255])


def sw_image(seed=9, h=40, w=60):
    rng = np.random.default_rng(seed)
    return (rng.random((h, w, 3)) * 255).astype(np.float32)


def metric_case(seed, shape, K, ignore=255):
    """Synthetic (prediction, target) pair of the metric goldens (identical to tests/golden/_ref_worker.py)."""
    rng = np.random.default_rng(seed)
    target = rng.integers(0, K, size=shape).astype(np.int64)
    pred = np.where(rng.random(shape) < 0.6, target, rng.integers(0, K, size=shape)).astype(np.int64)
    target[rng.random(shape) < 0.07] = ignore
    return pred, target


METRIC_CASES = [(1, (2, 33, 47), 150), (2, (1, 65, 65), 19), (3, (4000,), 2), (4, (3, 17), 300)]


# psa_mask geometries (n, h, w, mask_h, mask_w) of the goldens recorded from the reference's own compiled CPU and CUDA
# extensions (tests/golden/make_golden_ext.py)
PSAMASK_EXT_CPU_CASES = [(2, 4, 5, 7, 9), (1, 6, 7, 5, 3), (2, 5, 5, 9, 9), (1, 30, 30, 59, 59), (1, 3, 9, 5, 17),
                         (1, 1, 1, 1, 1)]
PSAMASK_EXT_GPU_CASES = [(2, 30, 30, 59, 59), (1, 9, 12, 9, 7), (3, 5, 40, 9, 79), (1, 13, 13, 25, 25)]


def psamask_key(geom, psa_type):
    return "n%d_h%d_w%d_mh%d_mw%d_t%d" % (tuple(geom) + (psa_type,))


def psamask_cpu_ext_cases():
    """(key, psa_type, mask_h, mask_w, x, dout) of the CPU-extension goldens (float32 ndarrays, one seeded stream)."""
    rng = np.random.default_rng(11)
    for geom in PSAMASK_EXT_CPU_CASES:
        n, h, w, mh, mw = geom
        for t in (0, 1):
            x = rng.standard_normal((n, mh * mw, h, w)).astype(np.float32)
            dout = rng.standard_normal((n, h * w, h, w)).astype(np.float32)
            yield psamask_key(geom, t), t, mh, mw, x, dout


def psamask_gpu_ext_inputs(geom, psa_type):
    """(x, dout) of the CUDA-extension goldens, drawn on the GPU from a seeded generator."""
    n, h, w, mh, mw = geom
    g = torch.Generator(device="cuda").manual_seed(h * 31 + w + psa_type)
    x = torch.randn((n, mh * mw, h, w), device="cuda", generator=g)
    dout = torch.randn((n, h * w, h, w), device="cuda", generator=g)
    return x, dout


def _np(a):
    return a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a)


def sha256(a):
    return hashlib.sha256(np.ascontiguousarray(_np(a)).tobytes()).hexdigest()


def check_psamask_golden(g, key, x, dout, out, din):
    """out / din bit-identical to the golden entry `key` (written by tests/golden/make_golden_ext.py), whose inputs must
    be x / dout."""
    assert sha256(x) == str(g[key + "/x_sha"]) and sha256(dout) == str(g[key + "/dout_sha"]), \
        "%s: inputs differ from those the golden was recorded with" % key
    if key + "/out" in g:
        assert np.array_equal(_np(out), g[key + "/out"]), key
        assert np.array_equal(_np(din), g[key + "/din"]), key
    assert sha256(out) == str(g[key + "/out_sha"]), key
    assert sha256(din) == str(g[key + "/din_sha"]), key
