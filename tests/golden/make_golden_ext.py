"""Generate psamask_ref_cpu.npz / psamask_ref_gpu.npz from the reference's own compiled psa_mask extensions
(oracle/_ref/psamask_ref_{cpu,gpu}*.so, which __graft_entry__.build() compiles from the reference's lib/psa/src where
the reference tree exists):

    python tests/golden/make_golden_ext.py cpu [OUT_DIR]     # lib/psa/src/cpu/psamask.cpp
    python tests/golden/make_golden_ext.py gpu [OUT_DIR]     # lib/psa/src/gpu/psamask_cuda.cu, needs a CUDA device

Each kernel is called the way lib/psa/functions/psamask.py calls it (zero-filled output, then the kernel) on the inputs
of tests/util.py. Per case the fixture holds the sha256 of inputs and outputs, and the outputs themselves when small.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

import oracle  # noqa: E402
from tests import util  # noqa: E402

MAX_STORED = 20000          # outputs up to this many elements are stored whole


def record(res, key, x, dout, out, din):
    res[key + "/x_sha"], res[key + "/dout_sha"] = util.sha256(x), util.sha256(dout)
    res[key + "/out_sha"], res[key + "/din_sha"] = util.sha256(out), util.sha256(din)
    if out.numel() <= MAX_STORED:
        res[key + "/out"], res[key + "/din"] = out.cpu().numpy(), din.cpu().numpy()


def run(ref, t, mh, mw, x, dout):
    n, _, h, w = x.shape
    out = torch.zeros((n, h * w, h, w), device=x.device)
    ref.psamask_forward(t, x, out, n, h, w, mh, mw, (mh - 1) // 2, (mw - 1) // 2)
    din = torch.zeros((n, mh * mw, h, w), device=x.device)
    ref.psamask_backward(t, dout, din, n, h, w, mh, mw, (mh - 1) // 2, (mw - 1) // 2)
    return out, din


def main():
    device = sys.argv[1]
    out_dir = sys.argv[2] if len(sys.argv) > 2 else HERE
    ref = oracle.ref_psamask_module(device)
    if ref is None:
        sys.exit("oracle/_ref/psamask_ref_%s*.so is not built" % device)
    res = {}
    if device == "cpu":
        for key, t, mh, mw, x, dout in util.psamask_cpu_ext_cases():
            x, dout = torch.from_numpy(x), torch.from_numpy(dout)
            record(res, key, x, dout, *run(ref, t, mh, mw, x, dout))
        res["provenance"] = "lib/psa/src/cpu/psamask.cpp, torch %s" % torch.__version__
    else:
        for geom in util.PSAMASK_EXT_GPU_CASES:
            for t in (0, 1):
                x, dout = util.psamask_gpu_ext_inputs(geom, t)
                key = util.psamask_key(geom, t)
                record(res, key, x, dout, *run(ref, t, geom[3], geom[4], x, dout))
        res["provenance"] = "lib/psa/src/gpu/psamask_cuda.cu on %s, torch %s" % (torch.cuda.get_device_name(),
                                                                                  torch.__version__)
    os.makedirs(out_dir, exist_ok=True)
    path = os.path.join(out_dir, "psamask_ref_%s.npz" % device)
    np.savez_compressed(path, **res)
    print(path, res["provenance"])


if __name__ == "__main__":
    main()
