#!/usr/bin/env python
"""Benchmark of the semseg training hot path (BASELINE.json metric: PSPNet50 473x473 training images/sec).

    python bench.py --gpus N --steps K --warmup W            # B200-native arm (this repository)
    python bench.py --impl reference --gpus N ...            # reference arm: the reference's OWN modules
                                                             # (baseline/_ref/model/pspnet.py) on the host cores

A "step" is the body of the reference's training loop, tool/train.py:267-276: H2D of a pinned synthetic batch,
model(input, target) (forward incl. both cross-entropy losses and the argmax), loss = main + 0.4*aux, zero_grad,
backward, SGD step. Workload = BASELINE configs[1]: PSPNet50, 473x473, 150 classes, 16 images per GPU
(weak scaling: per-GPU batch fixed; N>1 uses SyncBatchNorm + DistributedDataParallel exactly as
tool/train.py:141-157). Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# SURVEY.md §8(d): fwd+bwd conv FLOPs (2*MAC) per image of the measured configurations
CONV_GFLOP_PER_IMG_TRAIN = {("psp", 50, 473, 150): 1022.8, ("psp", 101, 473, 150): 1431.9,
                            ("psp", 101, 713, 19): 3217.6, ("psa", 50, 465, 150): 1071.0}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=16, help="images per GPU")
    ap.add_argument("--size", type=int, default=473)
    ap.add_argument("--classes", type=int, default=150)
    ap.add_argument("--layers", type=int, default=50)
    ap.add_argument("--arch", default="psp", choices=["psp", "psa"])
    ap.add_argument("--cpu-batch", type=int, default=2, help="images per step of the CPU arms (bounded sample)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-stock-gpu", action="store_true")
    ap.add_argument("--no-parity-mode", action="store_true")
    ap.add_argument("--parity-mode-multi", action="store_true", help="also time the bf16x3 leg when --gpus > 1")
    ap.add_argument("--optimizer", default="torch", choices=["torch", "fused"],
                    help="torch.optim.SGD (the reference's, tool/train.py:140) or semseg_b200.optim.FusedSGD (one launch)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed as DIR/<name>.npy (rank 0; B200 arm only)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to the b200 arm")
    return args


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(bf16_tflops=d.get("bf16_tflops", 1590.0), bf16_tflops_sustained=d.get("bf16_tflops_sustained",
                    1400.0), hbm_gbs=d.get("hbm_gbs", 6650.0), source="measured (MEASURED_PEAKS.json)")
    return dict(bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, hbm_gbs=6650.0, source="fallback")


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU with NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:      # noqa: BLE001
            pass

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:      # noqa: BLE001
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:      # noqa: BLE001
                pass
            time.sleep(0.1)

    def result(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def synth_batch(n, size, classes, seed):
    import torch
    g = torch.Generator().manual_seed(seed)
    x = torch.randn((n, 3, size, size), generator=g)
    y = torch.randint(0, classes, (n, size, size), generator=g)
    y[torch.rand((n, size, size), generator=g) < 0.05] = 255
    return x, y


DUMP_MAX_ELEMS = 4 * 1024 * 1024      # per array: 16 MB as float32, so a dump of three arrays and scalars stays < 64 MB


def dump_sample(t):
    """`t` itself when it has at most DUMP_MAX_ELEMS elements, else that many of its elements (flattened) at positions
    drawn from a fixed seed, the same positions for the same size in every run."""
    import torch
    if t.numel() <= DUMP_MAX_ELEMS:
        return t
    idx = torch.randint(t.numel(), (DUMP_MAX_ELEMS,), generator=torch.Generator().manual_seed(0)).sort().values
    return t.reshape(-1)[idx.to(t.device)]


def dump_outputs(out_dir, outputs, model):
    """Writes what one training step hands back, as float32 .npy files: the prediction and both losses of
    model(input, target), the loss it back-propagated, and the parameter gradients and updated parameters (all
    parameters flattened in model.parameters() order and sampled by dump_sample)."""
    import numpy as np
    import torch
    pred, main_loss, aux_loss, loss = outputs
    params = list(model.parameters())
    grads = [p.grad if p.grad is not None else torch.zeros_like(p) for p in params]
    arrays = {"pred": dump_sample(pred), "main_loss": main_loss, "aux_loss": aux_loss, "loss": loss,
              "grads": dump_sample(torch.cat([g.reshape(-1) for g in grads])),
              "params": dump_sample(torch.cat([p.detach().reshape(-1) for p in params]))}
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


def build_optimizer(model, arch, kind="torch"):
    """The reference's 8 SGD parameter groups (tool/train.py:125-140)."""
    import torch
    ori = [model.layer0, model.layer1, model.layer2, model.layer3, model.layer4]
    new = [model.ppm if arch == "psp" else model.psa, model.cls, model.aux]
    groups = [dict(params=m.parameters(), lr=0.01) for m in ori] + [dict(params=m.parameters(), lr=0.1) for m in new]
    if kind == "fused":
        from semseg_b200.optim import FusedSGD
        return FusedSGD(groups, lr=0.01, momentum=0.9, weight_decay=1e-4)
    return torch.optim.SGD(groups, lr=0.01, momentum=0.9, weight_decay=1e-4)


# ---------------------------------------------------------------------------------------------------- reference arms
REF_DIR = os.path.join(ROOT, "baseline", "_ref")


def reference_available():
    """The unmodified reference tree under baseline/_ref (baseline/install_reference.py; git-ignored, travels with the
    snapshot). In the build container it is (re)created from /root/reference on demand."""
    if not os.path.isdir(os.path.join(REF_DIR, "model")):
        try:
            sys.path.insert(0, os.path.join(ROOT, "baseline"))
            import install_reference
            install_reference.install()
        except Exception:      # noqa: BLE001
            pass
        finally:
            sys.path.pop(0)
    return os.path.isdir(os.path.join(REF_DIR, "model"))


def run_reference_modules(args, device, batch, steps, warmup, threads=0, timeout=1500):
    """The reference's own model/pspnet.py / model/psanet.py stepping on `device` in a subprocess whose cwd and
    PYTHONPATH are baseline/_ref only (its `model` package must not meet this repository's). -> dict from the runner."""
    import subprocess
    env = dict(os.environ)
    env["PYTHONPATH"] = REF_DIR
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT", "TORCHELASTIC_RUN_ID"):
        env.pop(k, None)
    if device == "cuda":
        # nn.DataParallel (tool/train.py:159) spreads over every visible GPU: pin the runner to the ONE GPU this bench
        # process measures on, so that "same GPU, same workload" holds on a multi-GPU box too
        vis = [v for v in os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",") if v.strip()]
        lr = int(os.environ.get("LOCAL_RANK", "0"))
        env["CUDA_VISIBLE_DEVICES"] = vis[lr] if lr < len(vis) else str(lr)
    cmd = [sys.executable, os.path.join(ROOT, "baseline", "run_reference.py"), "--device", device, "--arch", args.arch,
           "--layers", str(args.layers), "--classes", str(args.classes), "--size", str(args.size), "--batch",
           str(batch), "--steps", str(steps), "--warmup", str(warmup), "--threads", str(threads)]
    r = subprocess.run(cmd, cwd=REF_DIR, env=env, capture_output=True, text=True, timeout=timeout)
    if r.returncode != 0:
        raise RuntimeError("reference runner failed: %s" % r.stderr.strip().splitlines()[-1:])
    return json.loads(r.stdout.strip().splitlines()[-1])


def cpu_reference_run(args, steps, warmup):
    """The reference's CPU PyTorch path on the host cores: its own modules from baseline/_ref (kind "reference"); the
    fp32 oracle restatement (kind "port") only where the reference tree is absent."""
    # oneDNN scales poorly past ~32 threads on a 2-image batch (128 threads were 10x slower than 32 on the GPU box),
    # so the CPU arms use min(host cores, 32) threads and report that number as `cores`.
    cores = min(os.cpu_count() or 1, 32)
    if reference_available():
        d = run_reference_modules(args, "cpu", args.cpu_batch, steps, warmup, threads=cores)
        return dict(value=d["images_per_sec"], seconds=d["seconds"], cores=d["threads"], kind="reference",
                    what="reference modules %s (baseline/_ref), fp32, torch %s" % (d["module_file"], d["torch"]))
    import torch
    from oracle.torch_oracle import Oracle
    from semseg_b200.pspnet import PSPNet
    from semseg_b200.psanet import PSANet
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    if args.arch == "psp":
        m = PSPNet(layers=args.layers, classes=args.classes, zoom_factor=8, pretrained=False)   # weights only
        okw = {}
    else:
        mk = 2 * ((args.size - 1) // 16 + 1) - 1
        m = PSANet(layers=args.layers, classes=args.classes, zoom_factor=8, mask_h=mk, mask_w=mk, pretrained=False)
        okw = dict(mask_h=mk, mask_w=mk)
    params = {k for k, _ in m.named_parameters()}
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    plist = []
    for k, v in sd.items():
        if k in params:
            v.requires_grad_(True)
            plist.append(v)
    orc = Oracle(sd, arch=args.arch, layers=args.layers, classes=args.classes, dropout=0.1, **okw).train()
    opt = torch.optim.SGD(plist, lr=0.01, momentum=0.9, weight_decay=1e-4)
    x, y = synth_batch(args.cpu_batch, args.size, args.classes, 0)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        _, ml, al = orc.forward(x, y)
        loss = ml + 0.4 * al
        opt.zero_grad()
        loss.backward()
        opt.step()
        times.append(time.perf_counter() - t0)
    t = sum(times[warmup:])
    return dict(value=args.cpu_batch * steps / t, seconds=t, cores=cores, kind="port",
                what="oracle/torch_oracle.py restatement (baseline/_ref absent)")


def workload_name(args):
    return "%s%d %s-shape %dx%d, %d classes, synthetic training step (tool/train.py:267-276), %d images/GPU" % (
        "PSPNet" if args.arch == "psp" else "PSANet", args.layers, "ADE20K" if args.classes == 150 else "Cityscapes"
        if args.classes == 19 else "custom", args.size, args.size, args.classes, args.batch)


def metric_name(args):
    return "%s%d %dx%d training images/sec" % ("PSPNet" if args.arch == "psp" else "PSANet", args.layers, args.size,
                                                 args.size)


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = max(1, min(args.steps, 8)), max(1, min(args.warmup, 2))
    r = cpu_reference_run(args, steps, warmup)
    sample = "%d timed steps (of --steps %d) x %d images of the workload, fp32, min(host cores, 32) threads; %s" % (
        steps, args.steps, args.cpu_batch, r["what"])
    line = {
        "impl": "reference", "metric": metric_name(args), "value": r["value"], "unit": "images/sec",
        "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": 1e3 * r["seconds"] / steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args),
                   "sample": "CPU arm times %d images/step of that workload (bounded sample)" % args.cpu_batch},
        "cpu_baseline": {"value": r["value"], "unit": "images/sec", "cores": r["cores"], "kind": r["kind"],
                         "sample": sample},
        "e2e": {"value": r["value"], "unit": "images/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------- B200 arm
def run_b200_arm(args):
    import torch
    import torch.distributed as dist
    import torch.nn as nn
    from semseg_b200 import _lib, ops
    from model.pspnet import PSPNet
    from model.psanet import PSANet

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    assert world == args.gpus, "launch with torchrun --nproc-per-node %d (WORLD_SIZE=%d)" % (args.gpus, world)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    torch.manual_seed(0)
    if args.arch == "psp":
        model = PSPNet(layers=args.layers, classes=args.classes, zoom_factor=8, pretrained=False)
    else:
        mk = 2 * ((args.size - 1) // 16 + 1) - 1
        model = PSANet(layers=args.layers, classes=args.classes, zoom_factor=8, mask_h=mk, mask_w=mk,
                       pretrained=False)
    opt = build_optimizer(model, args.arch, args.optimizer)
    if world > 1:
        model = nn.SyncBatchNorm.convert_sync_batchnorm(model)
        model = nn.parallel.DistributedDataParallel(model.cuda(), device_ids=[local_rank])
    else:
        model = model.cuda()
    model.train()

    x_host, y_host = synth_batch(args.batch, args.size, args.classes, 100 + rank)
    x_host, y_host = x_host.pin_memory(), y_host.pin_memory()
    x_dev, y_dev = x_host.to(dev), y_host.to(dev)
    h2d = x_host.numel() * 4 + y_host.numel() * 8

    last = []               # outputs of the latest step, kept for --dump-outputs only

    def step(inp, tgt):
        pred, main_loss, aux_loss = model(inp, tgt)
        loss = main_loss + 0.4 * aux_loss
        opt.zero_grad()
        loss.backward()
        opt.step()
        if args.dump_outputs:
            last[:] = (pred, main_loss, aux_loss, loss)
        return loss

    def step_e2e():
        inp = x_host.to(dev, non_blocking=True)
        tgt = y_host.to(dev, non_blocking=True)
        return step(inp, tgt).item()            # D2H read of the step's loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    from semseg_b200 import graphs
    inner = model.module if world > 1 else model
    n_warm = max(3, args.warmup) + (graphs.WARMUP_CALLS + 1 if graphs.enabled() else 0)   # eager warm-up + graph capture
    for _ in range(n_warm):
        step(x_dev, y_dev)
    sampler = ClockSampler(local_rank)
    sampler.start()
    l0 = _lib.launch_count()
    ms_dev = timed(lambda: step(x_dev, y_dev), args.steps)
    launches = _lib.launch_count() - l0
    if args.dump_outputs and rank == 0:
        # before any further step: a replayed step graph rewrites the same static output buffers every time
        dump_outputs(args.dump_outputs, last, inner)
    graphed = graphs.launches_per_step(inner)
    if graphed:                      # kernels replayed from the captured step graphs are not counted by the library
        launches += graphed * args.steps
    step_e2e()
    ms_e2e = timed(step_e2e, args.steps)
    sampler.stop_flag = True
    sampler.join(2)

    n_img = args.batch * world * args.steps
    value = n_img / (ms_dev / 1e3)
    e2e_value = n_img / (ms_e2e / 1e3)

    # ---- the same step in the parity-precision operand mode (bf16x3: hi/lo bf16 pairs, three MMA segments per K block;
    #      the mode whose eval logits match the fp32 reference to 1e-3 with identical argmax, tests/test_parity_x3_gpu.py)
    parity = None
    if not args.no_parity_mode and (world == 1 or args.parity_mode_multi):
        # N > 1: off by default — the scaling runs measure the speed configuration only; the parity mode's multi-rank
        # correctness is covered by tests/test_multigpu_gpu.py, its throughput by the N = 1 line
        from semseg_b200 import precision
        psteps = max(1, min(args.steps, 5))
        try:
            with precision.mode("bf16x3"):
                for _ in range(2 + (graphs.WARMUP_CALLS + 1 if graphs.enabled() else 0)):
                    step(x_dev, y_dev)
                ms_p = timed(lambda: step(x_dev, y_dev), psteps)
            parity = {"dtype": "bf16x3", "value": args.batch * world * psteps / (ms_p / 1e3), "unit": "images/sec",
                      "ms_per_step": ms_p / psteps, "steps": psteps,
                      "what": "same training step with (hi, lo) bf16 activations / weights and x_hi*w_hi + x_lo*w_hi + "
                              "x_hi*w_lo accumulation in fp32 (16-bit mantissa operands >= the reference's TF32 cuDNN path)"}
        except Exception as e:      # noqa: BLE001
            parity = {"dtype": "bf16x3", "error": str(e)[:300]}

    # ---- roofline of the dominant kernel: the cls-head 3x3 conv 4096->512 fprop, timed alone with CUDA events
    pk = peaks()
    roof = None
    if rank == 0:
        fmap = (args.size - 1) // 8 + 1
        g = torch.Generator(device=dev).manual_seed(0)
        xa = torch.randn((args.batch, fmap, fmap, 4096), device=dev, generator=g).to(torch.bfloat16)
        w = torch.randn((512, 4096, 3, 3), device=dev, generator=g) * 0.01
        pw = ops.pack_weights(w, need_dgrad=False)
        taps = ops.conv_taps(3, 1)
        flush = torch.empty(512 * 1024 * 1024, dtype=torch.uint8, device=dev)
        for _ in range(3):
            ops.conv_fprop(xa, pw.wf, 512, taps, stats=True)
        ts = []
        for _ in range(10):
            flush.zero_()                       # flush the 126 MB L2 between timed launches
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            ops.conv_fprop(xa, pw.wf, 512, taps, stats=True)
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        t_k = sum(ts) / len(ts)
        flops = 2.0 * args.batch * fmap * fmap * 4096 * 512 * 9
        ach = flops / (t_k * 1e-3) / 1e12
        roof = {"bound": "tensor", "kernel": "conv_igemm_kernel<256> (cls 3x3 4096->512 fprop, bs%d %dx%d)" % (
                    args.batch, fmap, fmap), "achieved": ach, "peak": pk["bf16_tflops"], "unit": "TFLOP/s",
                "frac": ach / pk["bf16_tflops"],
                # dram__bytes_read.sum + dram__bytes_write.sum of this kernel at this shape from the committed
                # `ncu --set full` capture of the final build (profiles/r1_ncu_full_final_key_metrics.csv, first row):
                # 738.1 MB + 72.5 MB per launch; the algorithmic bytes are 510 MB in + 59 MB out.
                "traffic": 810.6e6 if (args.batch, fmap) == (16, 60) else None, "traffic_unit": "bytes/launch",
                "traffic_source": "ncu --set full capture of round 1 (profiles/r1_ncu_full_final_key_metrics.csv); the "
                                  "bf16 instantiation of this kernel and its tiling are unchanged in round 2",
                "ms_per_launch": t_k, "peak_source": pk["source"] +
                " burst bf16 (kernel timed alone)"}
        del xa, w, pw, flush

    if world > 1:
        dist.barrier()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    gflop_img = CONV_GFLOP_PER_IMG_TRAIN.get((args.arch, args.layers, args.size, args.classes))
    step_tflops = gflop_img * args.batch * world * args.steps / (ms_dev / 1e3) / 1e3 if gflop_img else None
    line = {
        "metric": metric_name(args), "value": value, "unit": "images/sec", "n_gpus": world, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": ms_dev / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "dtype_note": "value / e2e: single-pass bf16 operands (speed configuration); parity_mode: bf16x3 (the "
                      "reference-precision configuration)",
        "parity_mode": parity,
        "config": {"workload": workload_name(args),
                   "global_batch": args.batch * world, "parallelism": "dp%d" % world,
                   "l2": "inputs larger than L2: each step streams > 10 GB of activations through the 126 MB L2",
                   "optimizer": "%s, momentum 0.9 wd 1e-4, 8 param groups" % (
                       "torch.optim.SGD" if args.optimizer == "torch" else "semseg_b200.optim.FusedSGD (one launch)"),
                   "sync_bn": world > 1,
                   "execution": ("forward and backward replayed as two CUDA graphs (%d kernels per step) behind one "
                                 "autograd node" % graphed) if graphed else "eager launches",
                   "syncbn_exchange": __import__("semseg_b200.p2p", fromlist=["x"]).exchange_kind()},
        "e2e": {"value": e2e_value, "unit": "images/sec", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": int(launches),
        "clocks": sampler.result(),
        "roofline": roof,
        "step_conv_tflops": step_tflops,
        "step_conv_frac_of_sustained_peak": step_tflops / (pk["bf16_tflops_sustained"] * world) if step_tflops else None,
    }
    if world == 1 and not args.no_stock_gpu:
        try:
            line["stock_gpu_baseline"] = stock_gpu_baseline(args, dev)
        except Exception as e:      # noqa: BLE001
            line["stock_gpu_baseline"] = {"error": str(e)[:200]}
    if world == 1 and not args.no_cpu_baseline:
        r = cpu_reference_run(args, 2, 1)
        line["cpu_baseline"] = {"value": r["value"], "unit": "images/sec", "cores": r["cores"], "kind": r["kind"],
                                "sample": "2 timed steps x %d images of the same workload, fp32, min(host cores, 32) "
                                          "threads; %s" % (args.cpu_batch, r["what"])}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def stock_gpu_baseline(args, dev):
    """The optimisation target's denominator (BASELINE.md §4.1): the reference's own modules on the same GPU and workload
    — fp32 NCHW, cuDNN, torch default flags (TF32 convolutions), nn.DataParallel as tool/train.py:159 — through
    baseline/run_reference.py. Informational extra field (the driver's ratio uses the CPU reference arm)."""
    import torch
    torch.cuda.empty_cache()
    if not reference_available():
        return {"error": "baseline/_ref absent"}
    d = run_reference_modules(args, "cuda", args.batch, 5, 3)
    ms = 1e3 * d["seconds"] / d["steps"]
    return {"value": d["images_per_sec"], "unit": "images/sec", "ms_per_step": ms, "kind": "reference",
            "what": "reference modules %s under nn.DataParallel on the same GPU: fp32 NCHW, cuDNN, torch default flags "
                    "(TF32 convs %s), bs%d, H2D of the pinned batch inside the step" % (d["module_file"],
                                                                                      d["tf32_conv"], args.batch)}


def main():
    args = parse()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_b200_arm(args)


if __name__ == "__main__":
    main()
