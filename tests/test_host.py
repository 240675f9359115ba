"""CPU: host-side logic, import surface, C-ABI export list, no-fallback guarantees."""
import ctypes
import os
import re
import subprocess
import sys

import pytest
import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_import_paths():
    from models import cifar10 as cifar_models, imagenet as imagenet_models              # train.py:27-28
    from models.imagenet.resnet_bi_imagenet_set_2 import HardBinaryConv_react           # train.py:30
    from models.imagenet.resnet_bi_imagenet_set_2_2 import HardBinaryConv               # train.py:31
    from models.bin_module.binarized_modules import HardBinaryConv_cifar, BinarizeConv2d  # train.py:32
    from kurtosis import KurtosisWeight                                                  # train.py:29
    from utils.KD_loss import DistributionLoss, DistributionLoss_layer                   # train.py:34
    names = sorted(n for n in imagenet_models.__dict__
                   if n.islower() and not n.startswith("__") and callable(imagenet_models.__dict__[n]))
    assert "resnet18" in names and "resnet34" in names                                   # train.py:53-56
    assert callable(cifar_models.__dict__["resnet20"])
    for cls in (HardBinaryConv, HardBinaryConv_react, HardBinaryConv_cifar):
        assert issubclass(cls, BinarizeConv2d) and issubclass(cls, nn.Conv2d)
    assert KurtosisWeight and DistributionLoss and DistributionLoss_layer


def test_module_contract_and_hook_selection():
    import models
    from bdbnn_b200.step import StepConfig, select_hooked_weights
    m = models.imagenet.resnet18(False)
    hooked = select_hooked_weights(m, StepConfig(w_kurtosis=True))
    assert len(hooked) == 19                                          # train.py:467-470
    assert "conv1.weight" not in hooked and "layer2.0.downsample.0.weight" in hooked
    for n, p in hooked.items():
        assert p.ndim == 4 and p.requires_grad and n.endswith(".weight")
    assert sum(p.numel() for p in m.parameters()) == 11689512
    sd = m.state_dict()
    assert "layer1.0.conv1.weight" in sd and not any(k.endswith(".k") or k.endswith(".t") for k in sd)
    m2 = models.cifar10.resnet20()
    assert len(select_hooked_weights(m2, StepConfig(w_kurtosis=True))) == 18
    conv = m2.layer1[0].conv1
    conv.k, conv.t = torch.tensor([3.0]), torch.tensor([0.3])          # EDE assignment, train.py:414-415
    hooked = select_hooked_weights(m, StepConfig(w_kurtosis=True, remove_weight_name=["downsample"]))
    assert 16 <= len(hooked) < 19                                     # buggy in-loop remove kept (train.py:395)


def test_cpu_tensors_are_rejected_no_fallback():
    from bdbnn_b200 import BinarizeConv2d, KurtosisWeight, DistributionLoss
    conv = BinarizeConv2d(4, 4)
    with pytest.raises(RuntimeError, match="CUDA"):
        conv(torch.randn(1, 4, 5, 5))
    kw = KurtosisWeight(torch.randn(4, 4, 3, 3), "w", 1.8)
    with pytest.raises(RuntimeError, match="CUDA"):
        kw.fn_regularization()
    with pytest.raises(RuntimeError, match="CUDA"):
        DistributionLoss()(torch.randn(2, 3), torch.randn(2, 3))
    with pytest.raises(ValueError, match="should not require gradients"):
        DistributionLoss()(torch.randn(2, 3), torch.randn(2, 3, requires_grad=True))


def test_product_never_imports_oracle():
    bad = []
    prod = [os.path.join(ROOT, "kurtosis.py")]
    for d in ("bdbnn_b200", "models", "utils"):
        for dp, _, fs in os.walk(os.path.join(ROOT, d)):
            prod += [os.path.join(dp, f) for f in fs if f.endswith(".py")]
    for f in prod:
        src = open(f).read()
        if re.search(r"^\s*(from|import)\s+oracle\b", src, re.M) or re.search(r"from\s+\.+\s*import\s+oracle", src):
            bad.append(f)
    assert not bad, bad


def _declared_symbols():
    hdr = open(os.path.join(ROOT, "include", "bdbnn.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    return sorted(set(re.findall(r"\b(bdbnn_[a-z0-9_]+)\s*\(", hdr)))


def test_capi_library_exports_every_declared_symbol():
    from bdbnn_b200 import build, _lib
    path = build.build()
    syms = _declared_symbols()
    assert len(syms) >= 18
    assert sorted(_lib.SIGNATURES) == syms, "ctypes SIGNATURES out of sync with include/bdbnn.h"
    h = ctypes.CDLL(path)
    for s in syms:
        assert hasattr(h, s), f"{s} not exported"
    h.bdbnn_version.restype = ctypes.c_int
    assert h.bdbnn_version() >= 1000
    out = subprocess.run(["nm", "-D", "--defined-only", path], capture_output=True, text=True).stdout
    exported = set(re.findall(r"\sT\s+(bdbnn_\w+)", out))
    assert exported == set(syms), exported ^ set(syms)


def test_library_is_sm100a():
    from bdbnn_b200 import build
    path = build.build()
    out = subprocess.run(["cuobjdump", "-lelf", path], capture_output=True, text=True).stdout
    assert "sm_100a" in out, out[:400]


def test_cpu_oracle_step_runs_and_learns():
    """Config 1 shape (ResNet-20 CIFAR) on the shared step driver with the oracle ops."""
    from bdbnn_b200.step import StepConfig, TrainStep, make_optimizer
    from oracle.models_ref import RefOps, resnet20_ref
    torch.manual_seed(0)
    m = resnet20_ref()
    step = TrainStep(m, make_optimizer(m, "cifar10", lr=0.05), StepConfig(w_kurtosis=True), ops=RefOps)
    x, y = torch.randn(16, 3, 32, 32), torch.randint(0, 10, (16,))
    l0 = float(step(x, y)["loss"])
    for _ in range(5):
        out = step(x, y)
    assert float(out["loss"]) < l0
    assert all(p.grad is not None for p in m.parameters())          # DDP needs every param to get a grad


def _ddp_worker(rank, world, port, outdir, use_shim=True):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from bdbnn_b200.ddp import FlatGradOptimizerShim, GradAllReduce
    from bdbnn_b200.step import StepConfig, TrainStep, make_optimizer
    from oracle.models_ref import RefOps, resnet20_ref
    torch.manual_seed(100 + rank)                     # different init per rank: broadcast must fix it
    m = resnet20_ref()
    red = GradAllReduce(m)
    g = torch.Generator().manual_seed(5)
    x = torch.randn(8, 3, 32, 32, generator=g)
    y = torch.randint(0, 10, (8,), generator=g)
    xs, ys = x[rank * 4:(rank + 1) * 4], y[rank * 4:(rank + 1) * 4]
    if use_shim:
        opt = FlatGradOptimizerShim(make_optimizer(m, "cifar10", lr=0.1), red)
        step = TrainStep(m, opt, StepConfig(w_kurtosis=True), ops=RefOps, grad_sync=red)
        for _ in range(2):
            step(xs, ys)
    else:
        # a caller that wraps nothing: torch's own zero_grad() (set_to_none=True drops the flat-buffer views), plain
        # backward, the reducer, the optimizer — must give the same result (ADVICE r1: no silent stale all-reduce)
        opt = make_optimizer(m, "cifar10", lr=0.1)
        step = TrainStep(m, opt, StepConfig(w_kurtosis=True), ops=RefOps)      # no grad_sync: drives nothing itself
        hooked = list(step.hooked.values())
        for _ in range(2):
            opt.zero_grad()
            loss = torch.nn.functional.cross_entropy(m(xs), ys) + RefOps.kurtosis(hooked, [1.8] * len(hooked), "avg",
                                                                                 len(hooked), 1.0)
            loss.backward()
            red()
            opt.step()
    torch.save((red.flat.clone(), torch.cat([p.detach().reshape(-1) for p in m.parameters()])),
               os.path.join(outdir, f"r{rank}_{int(use_shim)}.pt"))
    dist.destroy_process_group()


def test_gloo_world2_gradient_allreduce(tmp_path):
    """Two gloo ranks, two steps: averaged gradients and updated parameters are bit-identical across ranks, with the
    flat-buffer shim AND for a caller that uses torch's own optimizer.zero_grad() (views dropped, re-bound by the
    reducer) — and both ways give the same parameters."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    res = {}
    for use_shim in (True, False):
        port = 29500 + os.getpid() % 2000 + int(use_shim)
        procs = [ctx.Process(target=_ddp_worker, args=(r, 2, port, str(tmp_path), use_shim)) for r in range(2)]
        for p in procs:
            p.start()
        for p in procs:
            p.join(300)
            assert p.exitcode == 0
        (g0, p0), (g1, p1) = [torch.load(os.path.join(tmp_path, f"r{r}_{int(use_shim)}.pt")) for r in range(2)]
        assert torch.equal(g0, g1) and torch.equal(p0, p1)     # averaged grads and updated params identical
        assert g0.abs().sum() > 0
        res[use_shim] = p0
    torch.testing.assert_close(res[True], res[False], rtol=1e-6, atol=1e-7)


def test_allreduce_bucket_accounting_with_side_stream_gradients():
    """Host logic of GradAllReduce's bucket scheduling (no process group, `_launch` recorded instead of issued): a
    bucket is issued one event AFTER its last parameter was accounted for; a conv weight whose gradient is written by
    a side-stream GEMM (`side_target`) and ALSO receives an autograd term (kurtosis) is counted once; the lagged
    issue therefore still happens after that term's accumulation hook; a gradient arriving after its bucket was
    issued raises; `__call__`-time reset re-arms everything."""
    import torch.nn as nn
    from bdbnn_b200.ddp import GradAllReduce
    m = nn.Sequential(nn.Conv2d(4, 4, 3, bias=False), nn.BatchNorm2d(4), nn.Conv2d(4, 4, 3, bias=False), nn.BatchNorm2d(4))
    red = GradAllReduce(m, broadcast_params=False, n_buckets=2)           # world 1: no hooks registered, no NCCL
    assert len(red.buckets) == 2
    red.overlap = True                                                     # drive the scheduling by hand
    issued = []
    red._launch = lambda b: (issued.append(b), red._works.__setitem__(b, "work"))
    w1, g1, b1, w2, g2, b2 = list(m.parameters())
    order = list(reversed(red.params))                                     # flat layout = reverse registration
    assert [id(p) for p in order] == [id(p) for p in (b2, g2, w2, b1, g1, w1)]
    assert [red._bucket_of[id(p)] for p in order] == [0, 0, 0, 1, 1, 1]    # 152 + 152 elements
    # --- backward of the last unit: side-stream wgrad of w2, then the autograd hooks of its BN parameters
    buf = red.side_target(w2, stream=None)
    assert buf is not None and buf.shape == w2.shape and buf.data_ptr() != red._view[id(w2)].data_ptr()
    assert red.wflat is not None and float(red.wflat.abs().sum()) == 0.0
    for p in (g2, b2):
        p.grad = red._view[id(p)]
        red._hook(p)
    assert issued == [] and red._armed == [0]                              # complete, but not issued yet
    # w2's kurtosis term: its post-accumulate hook is the next event — the accumulation is already enqueued, so the
    # flush inside this hook covers it; w2 itself is counted once
    red._hook(w2)
    assert issued == [0] and red._pending == [0, 3]
    # --- next unit
    red.side_target(w1, stream=None)
    for p in (g1, b1):
        red._hook(p)
    assert issued == [0] and red._armed == [1] and red._pending == [0, 0]
    # a gradient for an already-issued bucket is an error, not a silent stale reduce
    try:
        red._hook(b2)
        raise AssertionError("late gradient accepted")
    except RuntimeError as e:
        assert "after its bucket" in str(e)
    # the remaining bucket goes out in __call__ (world 1: nothing to reduce) and the state is re-armed
    red.world = 2
    red.scale = False
    red._works = [type("W", (), {"wait": lambda self: None})() if w is not None else None for w in red._works]
    red._launch = lambda b: (issued.append(b), red._works.__setitem__(b, type("W", (), {"wait": lambda self: None})()))
    red()
    assert sorted(issued) == [0, 1]
    assert red._pending == [b[2] for b in red.buckets] and not red._done and not red._armed and not red._side_now
    assert set(red._side_ever) == {id(w1), id(w2)}


def test_ede_attributes_and_activation_rule():
    """train.py:412-415 assigns .k/.t onto every nn.Conv2d; only the cifar class reacts, and only
    after both were assigned."""
    import torch.nn as nn
    from bdbnn_b200.modules import HardBinaryConv, HardBinaryConv_cifar
    from bdbnn_b200.step import apply_ede
    c, h = HardBinaryConv_cifar(16, 16), HardBinaryConv(16, 16)
    assert isinstance(c, nn.Conv2d) and not c.ede_active and not h.ede_active
    assert float(c.k) == 1.0 and float(c.t) == 1.0                 # readable defaults
    net = nn.Sequential(c, h, nn.Conv2d(16, 16, 1))
    t, k = apply_ede(net, 5, 10, device="cpu")
    assert c.ede_active and not h.ede_active
    assert c.k is k and c.t is t and net[2].k is k
    assert "k" not in c.state_dict() and "_ede_k" not in c.state_dict()


def test_make_optimizer_cpu_is_plain_torch_and_fused_rejects_cpu():
    """No CPU path in the product optimizers: CPU models get torch's, FusedAdam on CPU tensors raises."""
    import torch.nn as nn
    from bdbnn_b200.optim import FusedAdam
    from bdbnn_b200.step import make_optimizer
    m = nn.Sequential(nn.Conv2d(3, 4, 3), nn.BatchNorm2d(4))
    assert type(make_optimizer(m, "imagenet")).__module__.startswith("torch.optim")
    assert type(make_optimizer(m, "cifar10")).__module__.startswith("torch.optim")
    o = make_optimizer(m, "imagenet")
    assert [g.get("weight_decay", 0) for g in o.param_groups] == [0, 1e-4]       # train.py:331-334
    p = torch.zeros(3, requires_grad=True)
    p.grad = torch.ones(3)
    with pytest.raises(RuntimeError, match="CUDA"):
        FusedAdam([p]).step()


def test_wgrad_tiling_plans_are_sane_for_every_network_layer():
    """Host-only sweep of the wgrad planner (no GPU): every binary-conv geometry of the ResNet-18/34/20 shells,
    both gradient operand widths — shared memory within the 227 KB CTA limit, one wave of CTAs, the
    workspace large enough for the split the launch will use."""
    import ctypes
    from bdbnn_b200 import _lib
    from bdbnn_b200.functional import conv_shape
    L = _lib.lib()
    shapes = []
    for n in (1, 7, 256):
        shapes += [((n, 64, 56, 56), (64, 64, 3, 3), 1), ((n, 64, 56, 56), (128, 64, 3, 3), 2),
                   ((n, 128, 28, 28), (128, 128, 3, 3), 1), ((n, 128, 28, 28), (256, 128, 3, 3), 2),
                   ((n, 256, 14, 14), (256, 256, 3, 3), 1), ((n, 256, 14, 14), (512, 256, 3, 3), 2),
                   ((n, 512, 7, 7), (512, 512, 3, 3), 1),
                   ((n, 64, 28, 28), (128, 64, 1, 1), 1), ((n, 256, 7, 7), (512, 256, 1, 1), 1),       # packed shortcuts
                   ((n, 16, 32, 32), (16, 16, 3, 3), 1), ((n, 16, 32, 32), (32, 16, 3, 3), 2),
                   ((n, 32, 16, 16), (32, 32, 3, 3), 1), ((n, 32, 16, 16), (64, 32, 3, 3), 2),
                   ((n, 64, 8, 8), (64, 64, 3, 3), 1)]
    for xs, ws, stride in shapes:
        pad = 1 if ws[2] == 3 else 0
        sh = conv_shape(xs, ws, stride, pad)
        need = int(L.bdbnn_wgrad_tc_workspace_bytes(ctypes.byref(sh)))
        for halves in (1, 2):
            out = (ctypes.c_int32 * 12)()
            assert L.bdbnn_debug_wgrad_plan(ctypes.byref(sh), halves, out, 12) == 0
            ok, ksplit, ks_cap, mgroups, ntiles, smem, G, BN, UW, halo, k_stage, stages = list(out)
            assert ok == 1, (xs, ws, stride, halves)
            assert smem <= 227 * 1024 and stages >= 2 and k_stage % 16 == 0 and k_stage > 0
            assert 1 <= ksplit <= ks_cap and ksplit * mgroups * ntiles <= 148           # one wave on a B200
            assert UW in (16, 32, 64) and G * BN <= 512                                 # TMEM columns
            assert need >= ksplit * ws[0] * ws[1] * ws[2] * ws[3] * 4, (xs, ws, halves, need, ksplit)
    # unsupported geometry is reported, not planned
    out = (ctypes.c_int32 * 12)()
    sh = conv_shape((1, 40, 8, 8), (64, 40, 3, 3), 1, 1)
    assert L.bdbnn_debug_wgrad_plan(ctypes.byref(sh), 1, out, 12) == 0 and out[0] == 0


def test_conv_tiling_plans_are_sane_for_every_network_layer():
    """Host-only sweep of the persistent forward / dgrad kernel's planner (no GPU): TMEM columns, shared memory
    (dynamic + the kernel's static 6.5 KB of BN-statistics scratch in the forward) and ring depth."""
    import ctypes
    from bdbnn_b200 import _lib
    from bdbnn_b200.functional import conv_shape
    L = _lib.lib()
    layers = [((64, 56, 56), 64, 1), ((64, 56, 56), 128, 2), ((128, 28, 28), 128, 1), ((128, 28, 28), 256, 2),
              ((256, 14, 14), 256, 1), ((256, 14, 14), 512, 2), ((512, 7, 7), 512, 1), ((64, 8, 8), 64, 1)]
    planned = 0
    for n in (2, 256, 512):
        for (cin, h, w), cout, stride in layers:
            sh = conv_shape((n, cin, h, w), (cout, cin, 3, 3), stride, 1)
            for mode, halves in ((0, 1), (1, 1), (1, 2), (2, 1)):
                out = (ctypes.c_int32 * 12)()
                assert L.bdbnn_debug_conv_plan(ctypes.byref(sh), mode, halves, out, 12) == 0
                ok, halo, TS, NB, BN, n_tiles, supers, stages, smem, grid, stage_bytes, patch = list(out)
                if not ok:
                    assert mode == 2 and cin % 128 != 0 or n == 2, (cin, cout, stride, mode)   # fp8 needs Cin % 128
                    continue
                planned += 1
                assert TS * BN * NB <= 512 and BN in (64, 128, 256) and NB in (1, 2)
                assert stages >= 2 and 1 <= grid <= 148 and supers >= 1
                static = 7 * 1024 if mode != 1 else 1024
                assert smem + static <= 227 * 1024, (cin, cout, stride, mode, smem)
                assert BN * n_tiles == (cin if mode == 1 else cout)
    assert planned > 60
    # 16/32-channel layers are served by the one-tile kernel: the probe says "not planned"
    out = (ctypes.c_int32 * 12)()
    sh = conv_shape((4, 16, 32, 32), (16, 16, 3, 3), 1, 1)
    assert L.bdbnn_debug_conv_plan(ctypes.byref(sh), 0, 1, out, 12) == 0 and out[0] == 0


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs beside the GPU arm) prints ONE JSON line with
    the keys of the bench contract; bounded sample so it finishes in seconds."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--model", "resnet20",
                        "--steps", "1", "--warmup", "1", "--cpu-batch", "4"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
              "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "images/sec" and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["value"] > 0
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0


def test_bench_dump_outputs_writes_the_step_outputs_within_budget(tmp_path, monkeypatch):
    """`bench.py --dump-outputs`: every returned tensor and every floating-point state entry as <name>.npy (float64
    kept, the rest float32, shapes kept); above the byte budget, the largest arrays become the same seeded sample
    of their flattened elements on every run."""
    import numpy as np
    import bench
    torch.manual_seed(0)
    m = bench.build_model("resnet20", ref=True)
    out = {"loss": torch.tensor(2.5), "acc1": torch.tensor(50.0, dtype=torch.float64), "kurt": 0,
           "output": torch.randn(8, 10, dtype=torch.float16)}
    bench.dump_outputs(str(tmp_path / "all"), out, m)
    names = {f[:-4] for f in os.listdir(tmp_path / "all")}
    assert names == {"loss", "acc1", "output"} | {f"model.{k}" for k, v in m.state_dict().items() if v.is_floating_point()}
    assert np.load(tmp_path / "all" / "acc1.npy").dtype == np.float64 and np.load(tmp_path / "all" / "loss.npy").shape == ()
    assert np.array_equal(np.load(tmp_path / "all" / "output.npy"), out["output"].float().numpy())
    w = m.state_dict()["layer3.0.conv2.weight"]
    assert np.array_equal(np.load(tmp_path / "all" / "model.layer3.0.conv2.weight.npy"), w.numpy())
    monkeypatch.setattr(bench, "DUMP_BYTES", 64 << 10)
    for d in ("cut", "cut2"):
        bench.dump_outputs(str(tmp_path / d), out, m)
    sizes = {f: np.load(tmp_path / "cut" / f).nbytes for f in os.listdir(tmp_path / "cut")}
    assert sum(sizes.values()) <= 64 << 10 and sizes["loss.npy"] == 4
    cut = np.load(tmp_path / "cut" / "model.layer3.0.conv2.weight.npy")
    assert cut.ndim == 1 and 0 < cut.size < w.numel() and set(cut.tolist()) <= set(w.reshape(-1).tolist())
    assert np.array_equal(cut, np.load(tmp_path / "cut2" / "model.layer3.0.conv2.weight.npy"))
