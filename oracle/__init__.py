"""ORACLE — TEST INFRASTRUCTURE ONLY (never imported by semseg_b200/).

CPU restatements of the reference's hot path, used by tests/, __graft_entry__.smoke() and the
cpu_baseline / --impl reference legs of bench.py as the checker / CPU baseline:

  - psamask_oracle.c  : plain-C restatement of lib/psa/src/cpu/psamask.cpp (bit-exact data movement)
  - torch_oracle.py   : fp32 CPU restatement of model/pspnet.py, model/psanet.py, model/resnet.py on top of
                        torch.nn.functional (the reference's arithmetic *is* PyTorch's ATen)
  - _ref/             : the reference's own psamask.cpp compiled in place from /root/reference (git-ignored)

Parity pin: see tests/test_oracle_cpu.py and tests/golden/make_golden.py.
"""
import ctypes
import importlib.util
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "liboracle_psamask.so")
_REF_DIR = os.path.join(_HERE, "_ref")

_lib = None


def _load():
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB):
            from . import build
            build.build_oracle()
        _lib = ctypes.CDLL(_LIB)
        for name in ("oracle_psamask_fwd", "oracle_psamask_bwd"):
            fn = getattr(_lib, name)
            fn.restype = None
            fn.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p] + [ctypes.c_int] * 5
    return _lib


def psamask_fwd(x, psa_type, mask_h, mask_w):
    """x: float32 ndarray [N, mH*mW, H, W] -> [N, H*W, H, W]."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    n, c, h, w = x.shape
    assert c == mask_h * mask_w
    out = np.empty((n, h * w, h, w), dtype=np.float32)
    _load().oracle_psamask_fwd(psa_type, x.ctypes.data, out.ctypes.data, n, h, w, mask_h, mask_w)
    return out


def psamask_bwd(dout, psa_type, mask_h, mask_w):
    """dout: float32 ndarray [N, H*W, H, W] -> [N, mH*mW, H, W]."""
    dout = np.ascontiguousarray(dout, dtype=np.float32)
    n, hw, h, w = dout.shape
    assert hw == h * w
    din = np.empty((n, mask_h * mask_w, h, w), dtype=np.float32)
    _load().oracle_psamask_bwd(psa_type, dout.ctypes.data, din.ctypes.data, n, h, w, mask_h, mask_w)
    return din


def ref_psamask_module(device="cpu"):
    """The reference's own CPU or GPU extension (oracle/_ref/psamask_ref_{cpu,gpu}*.so) or None if it was not built."""
    if not os.path.isdir(_REF_DIR):
        return None
    import torch  # noqa: F401  (the extension links against libtorch)
    name = "psamask_ref_" + device
    for f in sorted(os.listdir(_REF_DIR)):
        if f.startswith(name) and f.endswith(".so"):
            spec = importlib.util.spec_from_file_location(name, os.path.join(_REF_DIR, f))
            mod = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(mod)
            return mod
    return None
