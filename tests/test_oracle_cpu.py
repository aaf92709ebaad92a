"""CPU tier: pin the oracle (oracle/) against the reference — golden fixtures made from the real reference
(tests/golden/make_golden.py) and from the reference's own compiled psamask extension
(tests/golden/make_golden_ext.py)."""
import hashlib
import json
import os

import numpy as np
import torch

import oracle
from oracle import torch_oracle
from tests import util

CASES = [(2, 4, 5, 7, 9), (1, 6, 7, 5, 3), (2, 5, 5, 9, 9), (1, 30, 30, 59, 59)]


def test_psamask_oracle_matches_reference_goldens(golden_dir):
    g = np.load(os.path.join(golden_dir, "psamask.npz"))
    rng = np.random.default_rng(7)  # same stream as _ref_worker.golden_psamask
    for (n, h, w, mh, mw) in CASES:
        for t in (0, 1):
            key = "n%d_h%d_w%d_mh%d_mw%d_t%d" % (n, h, w, mh, mw, t)
            x = rng.standard_normal((n, mh * mw, h, w)).astype(np.float32)
            out = oracle.psamask_fwd(x, t, mh, mw)
            dout = rng.standard_normal(out.shape).astype(np.float32)
            din = oracle.psamask_bwd(dout, t, mh, mw)
            assert hashlib.sha256(out.tobytes()).hexdigest() == str(g[key + "/out_sha"]), key
            assert hashlib.sha256(din.tobytes()).hexdigest() == str(g[key + "/din_sha"]), key
            if key + "/out" in g:
                assert np.array_equal(out, g[key + "/out"])
                assert np.array_equal(din, g[key + "/din"])


def test_psamask_oracle_matches_compiled_reference(golden_dir):
    """Bit-identical to the reference's own compiled CPU extension (lib/psa/src/cpu/psamask.cpp), whose outputs
    tests/golden/make_golden_ext.py recorded in psamask_ref_cpu.npz."""
    g = np.load(os.path.join(golden_dir, "psamask_ref_cpu.npz"))
    for key, t, mh, mw, x, dout in util.psamask_cpu_ext_cases():
        util.check_psamask_golden(g, key, x, dout, oracle.psamask_fwd(x, t, mh, mw),
                                  oracle.psamask_bwd(dout, t, mh, mw))


def test_psamask_torch_restatement_matches_c_oracle():
    rng = np.random.default_rng(3)
    for (n, h, w, mh, mw) in CASES[:3] + [(1, 7, 6, 13, 11)]:
        for t in (0, 1):
            x = rng.standard_normal((n, mh * mw, h, w)).astype(np.float32)
            xt = torch.from_numpy(x).requires_grad_(True)
            o = torch_oracle.psa_mask_torch(xt, t, mh, mw)
            assert np.array_equal(o.detach().numpy(), oracle.psamask_fwd(x, t, mh, mw))
            g = rng.standard_normal(tuple(o.shape)).astype(np.float32)
            o.backward(torch.from_numpy(g))
            assert np.array_equal(xt.grad.numpy(), oracle.psamask_bwd(g, t, mh, mw))


def test_collect_distribute_transpose_property():
    rng = np.random.default_rng(5)
    n, h, w = 2, 6, 5
    x = rng.standard_normal((n, (2 * h - 1) * (2 * w - 1), h, w)).astype(np.float32)
    col = oracle.psamask_fwd(x, 0, 2 * h - 1, 2 * w - 1)
    dis = oracle.psamask_fwd(x, 1, 2 * h - 1, 2 * w - 1)
    assert np.array_equal(dis, col.reshape(n, h * w, h * w).transpose(0, 2, 1).reshape(n, h * w, h, w))


def _check_model(tag, arch, golden_dir, build, okw):
    g = np.load(os.path.join(golden_dir, tag + ".npz"))
    meta = json.load(open(os.path.join(golden_dir, "meta.json")))
    torch.set_num_threads(8)
    model = build()
    # identical construction order => identical seeded weights as the reference (checksummed)
    wsum = meta["%s50_wsum" % ("pspnet" if arch == "psp" else "psanet")]
    sdm = model.state_dict()
    for k, (a, s) in wsum.items():
        assert abs(float(sdm[k].double().abs().sum()) - a) <= 1e-9 * max(1.0, abs(a)), k
        assert abs(float(sdm[k].double().sum()) - s) <= 1e-6 * max(1.0, abs(a)), k
    orc, sd = util.oracle_from(model, arch, layers=50, classes=150, **okw)
    x, y = util.synth(2, 65, 65, 150, seed=123 if arch == "psp" else 321)
    orc.train()
    out, main_loss, aux_loss = orc.forward(x, y)
    (main_loss + 0.4 * aux_loss).backward()
    assert abs(main_loss.item() - float(g["main_loss"])) < 2e-5
    assert abs(aux_loss.item() - float(g["aux_loss"])) < 2e-5
    # argmax in train mode: the reference itself flips 0.014 % of pixels between thread counts (SURVEY §7)
    mism = (out.numpy().astype(np.int16) != g["argmax"]).mean()
    assert mism < 2e-3, mism
    for k in g.files:
        if k.startswith("gradnorm/"):
            name = k[len("gradnorm/"):]
            got = sd[name].grad.double().norm().item()
            assert abs(got - float(g[k])) <= 2e-3 * float(g[k]) + 1e-9, (name, got, float(g[k]))
    tot = float(torch.sqrt(sum((v.grad.double() ** 2).sum() for v in sd.values() if v.grad is not None)))
    assert abs(tot - float(g["gradnorm_total"])) <= 1e-3 * float(g["gradnorm_total"])
    orc.eval()
    with torch.no_grad():
        logits = orc.forward(x)
    assert util.rel_l2(logits[:, :, ::8, ::8], g["eval_logits_s8"]) < 1e-4
    assert util.rel_l2(sd["layer4.2.bn3.running_mean"][:32], g["running_mean/layer4.2.bn3"]) < 1e-5


def test_torch_oracle_pspnet50_matches_reference_goldens(golden_dir):
    _check_model("pspnet50_65", "psp", golden_dir, lambda: util.build_pspnet(50, 150), {})


def test_torch_oracle_psanet50_matches_reference_goldens(golden_dir):
    _check_model("psanet50_65", "psa", golden_dir, lambda: util.build_psanet(50, 150, mask=9),
                 dict(mask_h=9, mask_w=9))


def test_metric_oracle_matches_reference_goldens(golden_dir):
    """oracle/metrics.py vs the reference's own numpy intersectionAndUnion (util/util.py:40-52), incl. K > ignore_index
    where label 255 is a countable class."""
    from oracle import metrics as om
    g = np.load(os.path.join(golden_dir, "metrics.npz"))
    for seed, shape, K in util.METRIC_CASES:
        pred, target = util.metric_case(seed, shape, K)
        i, u, t, _ = om.intersection_and_union(pred, target, K, 255)
        key = "s%d" % seed
        assert np.array_equal(i, g[key + "/i"]) and np.array_equal(u, g[key + "/u"]) and np.array_equal(t, g[key + "/t"])
