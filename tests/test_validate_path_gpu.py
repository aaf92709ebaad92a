"""GPU tier: the reference's validate() call pattern (tool/train.py:353-359) — `model.eval()` then `model(input)` with
autograd ENABLED and every parameter requiring grad, followed by `criterion(output, target)`; nothing is back-propagated.
The eval-mode BatchNorm path folds conv + BN (+ residual, ReLU) into one kernel that has no backward, so it must neither
raise nor change the numbers relative to the torch.no_grad() call that tool/test.py makes."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests import util

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("arch", ["psp", "psa"])
def test_eval_forward_with_autograd_enabled_equals_no_grad(arch):
    build = util.build_pspnet if arch == "psp" else util.build_psanet
    model = build(50, 21).cuda().eval()
    assert all(p.requires_grad for p in model.parameters())
    x, y = util.synth(2, 65, 65, 21, device="cuda")
    with torch.no_grad():
        ref = model(x)
    assert torch.is_grad_enabled()
    out = model(x)                                   # what validate() does
    assert tuple(out.shape) == tuple(ref.shape) == (2, 21, 65, 65)
    assert bool(torch.isfinite(out).all())
    assert torch.allclose(out.detach(), ref, rtol=0.0, atol=1e-6)
    loss = F.cross_entropy(out, y, ignore_index=255)     # criterion(output, target), tool/train.py:360
    assert bool(torch.isfinite(loss))


@pytest.mark.parametrize("geom", util.PSAMASK_EXT_GPU_CASES)
@pytest.mark.parametrize("psa_type", [0, 1])
def test_psamask_bit_identical_to_the_references_cuda_kernel(geom, psa_type, golden_dir):
    """psa_mask forward / backward against the reference's stock GPU kernel (lib/psa/src/gpu/psamask_cuda.cu:8-128) called
    the way lib/psa/functions/psamask.py:17-35 calls it (zero-filled output, then the kernel): bit-identical. The
    stock kernel's outputs were recorded on a B200 by tests/golden/make_golden_ext.py (psamask_ref_gpu.npz)."""
    from semseg_b200 import ops
    g = np.load(os.path.join(golden_dir, "psamask_ref_gpu.npz"))
    _, _, _, mh, mw = geom
    x, go = util.psamask_gpu_ext_inputs(geom, psa_type)
    util.check_psamask_golden(g, util.psamask_key(geom, psa_type), x, go, ops.psamask_fwd(x, psa_type, mh, mw),
                              ops.psamask_bwd(go, psa_type, mh, mw))
