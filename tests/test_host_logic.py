"""CPU tier: host-side logic of the drop-in modules (no kernels run)."""
import json
import os

import pytest
import torch
import torch.nn as nn

from tests import util


def test_state_dict_keys_and_shapes_match_reference(golden_dir):
    meta = json.load(open(os.path.join(golden_dir, "meta.json")))
    for tag, build in (("pspnet50", lambda: util.build_pspnet(50, 150)),
                       ("psanet50", lambda: util.build_psanet(50, 150, mask=9)),
                       ("pspnet101", lambda: util.build_pspnet(101, 19))):
        sd = build().state_dict()
        ref = meta[tag + "_keys"]
        assert list(sd.keys()) == list(ref.keys()), tag
        for k, v in sd.items():
            assert list(v.shape) == ref[k], (tag, k)


def test_drop_in_import_paths_and_signatures():
    import inspect
    from model.pspnet import PSPNet, PPM
    from model.psanet import PSANet, PSA
    import model.resnet as models
    import lib.psa.functional as PF
    import semseg_b200.pspnet
    assert PSPNet is semseg_b200.pspnet.PSPNet
    sig = inspect.signature(PSPNet.__init__)
    assert list(sig.parameters)[1:] == ["layers", "bins", "dropout", "classes", "zoom_factor", "use_ppm",
                                       "criterion", "pretrained"]
    sig = inspect.signature(PSANet.__init__)
    assert list(sig.parameters)[1:] == ["layers", "dropout", "classes", "zoom_factor", "use_psa", "psa_type",
                                       "compact", "shrink_factor", "mask_h", "mask_w", "normalization_factor",
                                       "psa_softmax", "criterion", "pretrained"]
    assert list(inspect.signature(PF.psa_mask).parameters) == ["input", "psa_type", "mask_H_", "mask_W_"]
    assert hasattr(models, "resnet50") and hasattr(models, "resnet101") and hasattr(models, "resnet152")


def test_trainer_contract_attributes_and_param_groups():
    """tool/train.py:125-140 builds 8 SGD groups from these attributes."""
    m = util.build_pspnet(50, 21)
    groups = [m.layer0, m.layer1, m.layer2, m.layer3, m.layer4, m.ppm, m.cls, m.aux]
    n = sum(p.numel() for g in groups for p in g.parameters())
    assert n == sum(p.numel() for p in m.parameters())
    opt = torch.optim.SGD([dict(params=g.parameters(), lr=0.01) for g in groups], lr=0.01, momentum=0.9,
                          weight_decay=1e-4)
    assert len(opt.param_groups) == 8
    # dilation patch (model/pspnet.py:49-58)
    c = m.layer3[0].conv2
    assert c.stride == (1, 1) and c.dilation == (2, 2) and c.padding == (2, 2)
    c = m.layer4[2].conv2
    assert c.stride == (1, 1) and c.dilation == (4, 4) and c.padding == (4, 4)
    assert m.layer4[0].downsample[0].stride == (1, 1)
    assert m.layer2[0].conv2.stride == (2, 2)


def test_convert_sync_batchnorm_keeps_structure():
    m = util.build_pspnet(50, 21)
    keys = list(m.state_dict().keys())
    m2 = nn.SyncBatchNorm.convert_sync_batchnorm(m)
    assert list(m2.state_dict().keys()) == keys
    assert isinstance(m2.layer3[0].bn2, nn.SyncBatchNorm)
    assert isinstance(m2.layer0[1], nn.SyncBatchNorm)
    assert type(m2.layer0).__name__ == "Stem"


def test_pretrained_loads_initmodel_relative_to_cwd(tmp_path, monkeypatch):
    import semseg_b200.resnet as R
    torch.manual_seed(1)
    src = R.resnet50(pretrained=False)
    (tmp_path / "initmodel").mkdir()
    torch.save(src.state_dict(), tmp_path / "initmodel" / "resnet50_v2.pth")
    monkeypatch.chdir(tmp_path)
    torch.manual_seed(2)
    dst = R.resnet50(pretrained=True)
    assert torch.equal(dst.layer3[0].conv2.weight, src.layer3[0].conv2.weight)


def test_conv_taps():
    from semseg_b200 import ops
    t = ops.conv_taps(3, 4)
    assert len(t) == 9 and t[0] == (-4, -4, 0) and t[4] == (0, 0, 4) and t[8] == (4, 4, 8)
    td = ops.conv_taps(3, 2, transpose=True)
    assert td[0] == (2, 2, 0) and td[8] == (-2, -2, 8)
    assert ops.conv_taps(1, 1) == [(0, 0, 0)]


def test_ops_fail_loudly_without_cuda():
    """No CPU fallback: CPU tensors are rejected instead of silently taking another path."""
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from semseg_b200 import ops, _lib
    with pytest.raises(_lib.SemsegError):
        ops.psamask_fwd(torch.zeros(1, 9, 2, 2), 0, 3, 3)
    with pytest.raises(_lib.SemsegError):
        ops.pack_weights(torch.zeros(64, 64, 1, 1))
    m = util.build_pspnet(50, 21)
    with pytest.raises(_lib.SemsegError):
        m(torch.zeros(2, 3, 65, 65), torch.zeros(2, 65, 65, dtype=torch.long))


def test_product_package_never_imports_oracle():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for d in ("semseg_b200", "model", "lib"):
        for dirpath, _, files in os.walk(os.path.join(root, d)):
            for f in files:
                if f.endswith(".py"):
                    src = open(os.path.join(dirpath, f)).read()
                    assert "import oracle" not in src and "from oracle" not in src, os.path.join(dirpath, f)


def test_bench_reference_runner_environment(monkeypatch):
    """bench.py's reference-module runner (baseline/run_reference.py) starts with the reference tree ALONE on PYTHONPATH,
    without the torchrun rendezvous variables, and — for the GPU leg — pinned to the one GPU the bench process measures on
    (nn.DataParallel, tool/train.py:159, would otherwise spread over every visible GPU of a multi-GPU box)."""
    import argparse
    import subprocess
    import bench
    seen = {}

    class Done:
        returncode, stdout, stderr = 0, 'noise\n{"images_per_sec": 1.0}\n', ""

    def fake_run(cmd, cwd=None, env=None, **kw):
        seen.update(cmd=cmd, cwd=cwd, env=env)
        return Done()

    monkeypatch.setattr(subprocess, "run", fake_run)
    args = argparse.Namespace(arch="psp", layers=50, classes=150, size=473)
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "3,5")
    monkeypatch.setenv("LOCAL_RANK", "1")
    monkeypatch.setenv("RANK", "1")
    monkeypatch.setenv("WORLD_SIZE", "2")
    assert bench.run_reference_modules(args, "cuda", 16, 5, 3) == {"images_per_sec": 1.0}
    assert seen["env"]["CUDA_VISIBLE_DEVICES"] == "5"
    assert seen["env"]["PYTHONPATH"] == bench.REF_DIR and seen["cwd"] == bench.REF_DIR
    assert not any(k in seen["env"] for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"))
    assert seen["cmd"][1].endswith("baseline/run_reference.py") and "--device" in seen["cmd"]
    monkeypatch.delenv("CUDA_VISIBLE_DEVICES")
    monkeypatch.setenv("LOCAL_RANK", "0")
    bench.run_reference_modules(args, "cuda", 16, 5, 3)
    assert seen["env"]["CUDA_VISIBLE_DEVICES"] == "0"
    bench.run_reference_modules(args, "cpu", 2, 2, 1, threads=8)
    assert "CUDA_VISIBLE_DEVICES" not in seen["env"] and seen["cmd"][seen["cmd"].index("--threads") + 1] == "8"


def test_bench_dump_outputs_writes_float32_and_samples_the_same_positions(tmp_path, monkeypatch):
    """bench.py --dump-outputs: every array is float32; one larger than DUMP_MAX_ELEMS is sampled at the same positions
    in every run, so that two builds can be compared output for output."""
    import numpy as np
    import bench
    monkeypatch.setattr(bench, "DUMP_MAX_ELEMS", 64)
    m = torch.nn.Conv2d(3, 8, 3)                      # 224 weights + 8 biases, more than 64
    for p in m.parameters():
        p.grad = torch.full_like(p, 0.5)
    pred = torch.arange(60, dtype=torch.long).reshape(1, 6, 10)
    outputs = (pred, torch.tensor(1.5), torch.tensor(2.0), torch.tensor(2.3))
    bench.dump_outputs(str(tmp_path / "a"), outputs, m)
    bench.dump_outputs(str(tmp_path / "b"), outputs, m)
    flat = torch.cat([p.detach().reshape(-1) for p in m.parameters()])
    for name in ("pred", "main_loss", "aux_loss", "loss", "grads", "params"):
        a, b = np.load(tmp_path / "a" / (name + ".npy")), np.load(tmp_path / "b" / (name + ".npy"))
        assert a.dtype == np.float32 and np.array_equal(a, b), name
    assert np.array_equal(np.load(tmp_path / "a" / "pred.npy"), pred.float().numpy())
    assert float(np.load(tmp_path / "a" / "loss.npy")) == np.float32(2.3)
    grads, params = np.load(tmp_path / "a" / "grads.npy"), np.load(tmp_path / "a" / "params.npy")
    assert grads.shape == params.shape == (64,) and (grads == 0.5).all()
    assert np.isin(params, flat.numpy()).all() and len(np.unique(params)) > 32


def test_precision_mode_switch_and_graph_gates(monkeypatch):
    """Host-side switches: the operand policy (semseg_b200/precision.py) and the CUDA-graph gate (graphs.enabled /
    train_step declining anything that is not a CUDA training call)."""
    from semseg_b200 import graphs, precision
    assert precision.get_mode() in precision.MODES
    before = precision.get_mode()
    with precision.mode("bf16x3"):
        assert precision.split_enabled() and precision.get_mode() == "bf16x3"
        with precision.mode("bf16"):
            assert not precision.split_enabled()
        assert precision.split_enabled()
    assert precision.get_mode() == before
    with pytest.raises(ValueError):
        precision.set_mode("fp8")
    with pytest.raises(ValueError):
        with precision.mode("tf32"):
            pass
    assert precision.get_mode() == before
    monkeypatch.setenv("SEMSEG_B200_GRAPH", "0")
    assert not graphs.enabled()
    monkeypatch.delenv("SEMSEG_B200_GRAPH")
    assert graphs.enabled() and not graphs.capturing()
    # a CPU call, a call without target and a call under no_grad are never captured: the caller runs its eager path
    x, y = torch.zeros((1, 3, 9, 9)), torch.zeros((1, 9, 9), dtype=torch.long)
    m = torch.nn.Conv2d(3, 3, 1)
    assert graphs.train_step(m, None, x, y) is None
    assert graphs.launches_per_step(m) == 0
    t = torch.ones(3, requires_grad=True)
    assert graphs.note_boundary(t) is t           # outside a capture: identity, nothing recorded
