#!/usr/bin/env python
"""bench.py — ResNet-18 1W/1A training throughput (images/sec) on N B200s of one node.

    python bench.py --gpus 1 --steps 20 --warmup 5            # this repo (CUDA kernels)
    torchrun ... bench.py --gpus N --steps K --warmup W       # one rank per GPU, NCCL
    python bench.py --impl reference ...                      # reference arm: the CPU oracle step
    python bench.py --gpus 1 --steps 20 --warmup 5 --dump-outputs DIR   # + the last timed step's outputs as .npy

A "step" = one full optimisation step of the restated train.py body (bdbnn_b200.step.TrainStep:
forward, losses, backward, gradient all-reduce, optimizer) on one synthetic batch.  Workload at N=1 is
BASELINE.json configs[1]: ResNet-18 1W/1A, synthetic 224x224, batch 256 per GPU.

Prints ONE JSON line (rank 0).  `value` = images/sec with inputs resident in HBM; `e2e` = the same
step fed from pinned host memory (H2D copy of every batch + D2H read of the loss inside the timed
region); `roofline` = achieved algorithmic GB/s of the dominant CUDA kernel family measured with CUDA
events on the launching stream inside the timed region; `cpu_baseline` = the CPU oracle step timed on
this box's host cores on a bounded sample.
"""
import argparse
import gc
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "reference-gpu"],
                    help="b200 = this repo; reference = the reference's CPU path (oracle port) on the host cores; "
                         "reference-gpu = the same pure-PyTorch oracle modules on cuda (stock eager cuDNN/ATen)")
    ap.add_argument("--model", default="resnet18", choices=["resnet18", "resnet34", "resnet20"])
    ap.add_argument("--batch", type=int, default=None, help="per-GPU batch (default 256; 128 for resnet20)")
    ap.add_argument("--workload", default="ce", choices=["ce", "kurt_kd"],
                    help="ce = BASELINE configs[1]; kurt_kd = configs[2] (kurtosis + KD, fp32 teacher)")
    ap.add_argument("--conv-impl", default=None, choices=[None, "auto", "xnor", "tc"])
    ap.add_argument("--ede", action="store_true",
                    help="EDE backward (train.py:409-415) at epoch 40/120; acts on HardBinaryConv_cifar (resnet20)")
    ap.add_argument("--cpu-batch", type=int, default=None,
                    help="images per CPU step (default: the full per-GPU batch, cut only if the run would exceed ~4 min)")
    ap.add_argument("--no-graph", action="store_true",
                    help="launch every kernel from Python each step instead of replaying the captured CUDA graph")
    ap.add_argument("--no-eager-gpu", action="store_true", help="skip the eager-cuDNN comparator line (N=1)")
    ap.add_argument("--no-secondary", action="store_true", help="skip the bf16x2 gradient-mode secondary value")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--profile-mode", action="store_true",
                    help="for runs under ncu: 1 warm-up step, no e2e / cpu legs (numbers printed are not bench values)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of --impl b200")
    return args


TRAFFIC_KERNEL = {  # KernelTimer family -> kernel-name prefixes in profiles/*_dram_traffic.json (ncu --set full)
    "binconv_dgrad_tc": ("tc_conv2_kernel<1", "tc_conv64_kernel<1"),
    "binconv_fwd_tc": ("tc_conv2_kernel<0", "tc_conv64_kernel<0, 0, 1, 0"),
    "binconv_fwd_tc8": ("tc_conv2_kernel<0",), "binconv_wgrad_tc": ("tc_wgrad_kernel",),
    "bn_fwd": ("bn_apply_add_pack_kernel<1",), "bn_bwd_pack": ("bn_bwd_pack_kernel<3",),
}


def ncu_traffic(family, calls_per_step):
    """dram__bytes_read+write of the family's kernels over ONE step of the newest committed ncu capture, divided by
    the family's API calls per step (a stride-2 dgrad is four phase launches; the three 1x1 shortcut dgrads run the
    same kernel and are included, so the figure is an upper bound for the family)."""
    import glob
    import re
    nat = lambda f: [int(t) if t.isdigit() else t for t in re.split(r"(\d+)", os.path.basename(f))]
    files = sorted((f for f in glob.glob(os.path.join(ROOT, "profiles", "*_dram_traffic.json")) if "losses" not in f),
                   key=nat)                                                     # r1_step9 < r1_step10 < r2_final
    if not files or family not in TRAFFIC_KERNEL or not calls_per_step:
        return None, None
    with open(files[-1]) as fh:
        d = json.load(fh)
    tot = sum(e["launches"] * e["dram_bytes_per_launch"] for k, e in d.items()
              if any(k.startswith(pre) for pre in TRAFFIC_KERNEL[family]))
    return (round(tot / calls_per_step), os.path.basename(files[-1])) if tot else (None, None)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as fh:
            d = json.load(fh)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled every 200 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []
        self.t0 = self.t1 = None          # host-time window of the timed region (mark_begin / mark_end)

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        # the sampler is started before the warm-up (process start-up must not land in the timed region);
        # only samples taken inside the timed window count (all of them if the window saw fewer than 2)
        inside = [ln for ts, ln in self.lines if self.t0 is None or (self.t0 <= ts <= (self.t1 or ts) + 0.2)]
        if len(inside) < 2:
            inside = [ln for _, ln in self.lines][-3:]
        for ln in inside:
            f = [t.strip() for t in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


DUMP_BYTES = 60 << 20          # all arrays of --dump-outputs together, under 64 MB with the .npy headers


def dump_outputs(dirname, out, model):
    """Write what one training step computed as DIR/<name>.npy: every tensor the step returns (`loss`, `ce`,
    `acc1`, `acc5`, the logits as `output`, and the kurtosis / KD terms when they are on) and the floating-point
    state the step updated (`model.<state_dict name>`, parameters and BatchNorm statistics, in their logical
    NCHW / OIHW order).  float64 stays float64, everything else is written as float32.  When the whole set would
    exceed DUMP_BYTES, every array above an equal share of what is left is cut to a fixed sample of its flattened
    elements: the first k positions of a permutation seeded with 0, in ascending order.  With the same arguments
    the inputs are the same on every run.  So are the outputs of the default ResNet-18 CE workload, which runs no
    cuDNN (tests/test_gpu_step.py repeats three such steps bit for bit); workloads that run
    cuDNN under cudnn.benchmark=True (the kurt_kd teacher, the ResNet-20 stem) may time their way to another
    algorithm on another run and then differ."""
    import numpy as np
    arrays = {k: v for k, v in out.items() if torch.is_tensor(v)}
    arrays.update({f"model.{k}": v for k, v in model.state_dict().items() if v.is_floating_point()})
    arrays = {k: v.detach().to("cpu", torch.float64 if v.dtype == torch.float64 else torch.float32).contiguous()
              for k, v in arrays.items()}
    nbytes = lambda t: t.numel() * t.element_size()
    left, cap = DUMP_BYTES, None
    for i, v in enumerate(sorted(arrays.values(), key=nbytes)):       # smallest first: each takes at most its share
        if nbytes(v) > left // (len(arrays) - i):
            cap = left // (len(arrays) - i)
            break
        left -= nbytes(v)
    os.makedirs(dirname, exist_ok=True)
    for k, v in arrays.items():
        if cap is not None and nbytes(v) > cap:
            keep = torch.randperm(v.numel(), generator=torch.Generator().manual_seed(0))[:cap // v.element_size()]
            v = v.reshape(-1)[keep.sort().values]
        np.save(os.path.join(dirname, f"{k}.npy"), v.numpy())


def build_model(name, conv_impl=None, ref=False):
    if ref:
        from oracle import models_ref
        return {"resnet18": models_ref.resnet18_ref, "resnet34": models_ref.resnet34_ref,
                "resnet20": models_ref.resnet20_ref}[name]()
    from bdbnn_b200 import resnet
    from bdbnn_b200.modules import BinarizeConv2d
    m = {"resnet18": resnet.resnet18, "resnet34": resnet.resnet34, "resnet20": resnet.resnet20}[name]()
    for mod in m.modules():
        if isinstance(mod, BinarizeConv2d):
            mod.impl = conv_impl
    return m


def build_teacher(name):
    """fp32 teacher, random init (no checkpoints offline), eval, no grads (train.py:250-277)."""
    import torchvision
    if name == "resnet20":
        from oracle import models_ref  # noqa: F401  (not used on the GPU arm)
        raise SystemExit("kurt_kd workload is defined for the ImageNet models")
    t = {"resnet18": torchvision.models.resnet18, "resnet34": torchvision.models.resnet34}[name]()
    t.eval()
    for p in t.parameters():
        p.requires_grad = False
    return t


def shapes(model_name, batch):
    if model_name == "resnet20":
        return (batch, 3, 32, 32), 10, "cifar10"
    return (batch, 3, 224, 224), 1000, "imagenet"


def step_config(workload):
    from bdbnn_b200.step import StepConfig
    if workload == "kurt_kd":
        return StepConfig(w_kurtosis=True, teacher_student=True, alpha=0.9, beta=200.0, w_lambda_ce=1.0)
    return StepConfig()


def host_threads():
    """Threads this process may use: affinity mask capped by the cgroup CPU quota."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        with open("/sys/fs/cgroup/cpu.max") as fh:
            quota, period = fh.read().split()
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period) + 0.5)))
    except Exception:
        pass
    return n


def cpu_reference_run(args, steps, warmup, batch, budget_s=240.0):
    """The reference arm / cpu_baseline: restated train.py step on the pure-PyTorch oracle modules.
    Thread count: the fastest of {16, 32, 64, all usable} on one probe step each (oversubscribing a
    small batch across 128 SMT threads is far slower than 32), then `steps` timed steps at that count.
    Runs the FULL per-GPU batch; only if `steps` of them would not fit `budget_s` is the batch halved
    (returned, so the caller can say what the sample was)."""
    from oracle import step_ref as S
    n_all = host_threads()
    torch.set_num_threads(min(n_all, 16))
    torch.manual_seed(0)
    ishape, ncls, dataset = shapes(args.model, batch)
    model = build_model(args.model, ref=True)
    if getattr(args, "ede", False):
        from oracle.binconv_ref import cpt_tk
        t, k = cpt_tk(40, 120)
        for m in model.modules():                 # train.py:409-415
            if isinstance(m, torch.nn.Conv2d):
                m.k, m.t = k, t
    teacher = None
    kd = args.workload == "kurt_kd"
    if kd:
        teacher = build_teacher(args.model)
    hooked = S.ref_hooked_weights(model) if kd else {}
    opt = S.ref_make_optimizer(model, dataset, 0.1 if dataset != "imagenet" else 1e-3)
    # the oracle's restatement of the reference loop body (oracle/step_ref.py; pinned to the reference's own
    # train() / train_teacher_student() by tests/test_ref_train.py)
    step = lambda xs, ys: S.ref_train_step(model, opt, xs, ys, hooked=hooked, targets=[1.8] * len(hooked),
                                           kurt_on=kd, teacher=teacher, alpha=0.9, beta=200.0)
    g = torch.Generator().manual_seed(0)
    x = torch.randn(ishape, generator=g)
    y = torch.randint(0, ncls, (batch,), generator=g)
    step(x, y)                                   # allocator / oneDNN primitive warm-up
    best_t, best_n = None, torch.get_num_threads()
    for n in sorted({c for c in (16, 32, 64, n_all) if c <= n_all}):
        torch.set_num_threads(n)
        t0 = time.perf_counter()
        float(step(x, y)["loss"])
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best_t, best_n = dt, n
        elif dt > 1.3 * best_t:
            break                                # past the scaling knee: stop probing
    torch.set_num_threads(best_n)
    while best_t * (steps + max(0, warmup - 1)) > budget_s and batch > 8:
        batch //= 2                              # bounded sample: a slice of the batch
        x, y = x[:batch].contiguous(), y[:batch].contiguous()
        t0 = time.perf_counter()
        float(step(x, y)["loss"])
        best_t = time.perf_counter() - t0
    for _ in range(max(0, warmup - 1)):
        step(x, y)
    t0 = time.perf_counter()
    for _ in range(steps):
        out = step(x, y)
        float(out["loss"])
    dt = time.perf_counter() - t0
    return batch * steps / dt, dt / steps * 1e3, torch.get_num_threads(), batch


def eager_gpu_run(args, steps, warmup, batch, dev):
    """The same-box GPU comparator (SURVEY.md §6): the pure-PyTorch oracle modules and the oracle's restated
    loop body on `dev` — stock eager PyTorch, cuDNN convolutions on +-1 fp32 tensors, ATen elementwise,
    torch.optim, cudnn.benchmark=True as train.py:368.  None of this repo's kernels run on this path."""
    from oracle import step_ref as S
    torch.backends.cudnn.benchmark = True
    torch.manual_seed(0)
    ishape, ncls, dataset = shapes(args.model, batch)
    model = build_model(args.model, ref=True).to(dev).to(memory_format=torch.channels_last)
    kd = args.workload == "kurt_kd"
    teacher = build_teacher(args.model).to(dev).to(memory_format=torch.channels_last) if kd else None
    hooked = S.ref_hooked_weights(model) if kd else {}
    opt = S.ref_make_optimizer(model, dataset, 0.1 if dataset != "imagenet" else 1e-3)
    g = torch.Generator().manual_seed(0)
    x = torch.randn(ishape, generator=g).to(dev).contiguous(memory_format=torch.channels_last)
    y = torch.randint(0, ncls, (batch,), generator=g).to(dev)
    step = lambda: S.ref_train_step(model, opt, x, y, hooked=hooked, targets=[1.8] * len(hooked), kurt_on=kd,
                                    teacher=teacher, alpha=0.9, beta=200.0)
    for _ in range(max(3, warmup)):
        step()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        out = step()
    e1.record()
    torch.cuda.synchronize(dev)
    float(out["loss"])
    ms = e0.elapsed_time(e1) / steps
    del model, opt, teacher
    torch.cuda.empty_cache()
    return batch / (ms / 1e3), ms


def finish(world):
    """Leave without tearing NCCL down: with captured graphs holding collectives alive,
    dist.destroy_process_group() / interpreter teardown can block forever (seen at N=2: the JSON line was printed and
    the processes never exited).  Everything is flushed; a hard exit is the documented-safe way out of a benchmark."""
    sys.stdout.flush()
    sys.stderr.flush()
    if world > 1:
        os._exit(0)


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    batch = args.batch or (128 if args.model == "resnet20" else 256)
    workload = (f"{args.model} 1W/1A synthetic {'32x32' if args.model == 'resnet20' else '224x224'} "
                f"batch {batch}/GPU, {'CE' if args.workload == 'ce' else 'CE+kurtosis+KD(fp32 teacher)'}"
                f"{' +EDE backward' if args.ede else ''} full train step")

    if args.impl == "reference":
        if rank != 0:
            return
        cb = min(args.cpu_batch or batch, batch)
        v, ms, cores, cb = cpu_reference_run(args, max(1, args.steps), max(0, args.warmup), cb)
        line = {"impl": "reference", "metric": "images/sec", "value": round(v, 3), "unit": "images/sec",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 3),
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic", "config": {"workload": workload, "parallelism": "cpu",
                                                "same_config": cb == batch, "cpu_batch": cb},
                "cpu_baseline": {"value": round(v, 3), "unit": "images/sec", "cores": cores, "kind": "port",
                                 "sample": (f"{args.steps} steps of the full {batch}-image batch" if cb == batch else
                                            f"{args.steps} steps of a {cb}-image slice of the {batch}-image batch") +
                                           " (oracle/step_ref.py: the reference loop body restated on the pure-PyTorch "
                                           "oracle modules, pinned to the reference's own train() by "
                                           "tests/test_ref_train.py; train.py itself needs CUDA and the absent "
                                           "models/ package, SURVEY.md §0.3)"},
                "e2e": {"value": round(v, 3), "unit": "images/sec", "h2d_bytes_per_step": 0,
                        "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 path has no CPU fallback "
                         "(use --impl reference for the CPU arm)")
    if args.impl == "reference-gpu":
        if rank != 0:
            return
        dev = torch.device("cuda", local_rank)
        torch.cuda.set_device(dev)
        v, ms = eager_gpu_run(args, max(1, args.steps), max(3, args.warmup), batch, dev)
        print(json.dumps({"impl": "reference-gpu", "metric": "images/sec", "value": round(v, 2), "unit": "images/sec",
                          "n_gpus": 1, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": round(ms, 3),
                          "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                          "dtype": "f32 (cuDNN default: TF32 tensor-core convolutions allowed)", "data": "synthetic",
                          "config": {"workload": workload, "parallelism": "dp1",
                                     "path": "oracle modules on cuda: stock eager PyTorch (cuDNN + ATen + torch.optim)"},
                          "gpu_launches": 0}))
        return
    import torch.distributed as dist
    from bdbnn_b200 import _lib
    from bdbnn_b200.ddp import FlatGradOptimizerShim, GradAllReduce
    from bdbnn_b200.functional import KernelTimer
    from bdbnn_b200.step import GraphedTrainStep, TrainStep, make_optimizer

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # NCCL prints its version banner (and NCCL_DEBUG output) on stdout: keep stdout to the one JSON line.
        # NCCL_DEBUG_FILE is only honoured above the VERSION level, so a bare VERSION setting becomes WARN.
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=dev)
    torch.backends.cudnn.benchmark = True            # train.py:368
    torch.manual_seed(0)
    ishape, ncls, dataset = shapes(args.model, batch)
    # parameters stay in their native dense (OIHW) layout: the kernels of this repo read and write weights and
    # weight gradients in that layout (a channels_last parameter would cost one layout copy per weight and per
    # gradient every step); activations are NHWC from the input batch on
    model = build_model(args.model, args.conv_impl).to(dev)
    if args.model == "resnet20":      # its fp32 3x3 stem runs on cuDNN, which wants NHWC filters for NHWC inputs
        model.conv1.to(memory_format=torch.channels_last)
    if args.ede:
        from bdbnn_b200.step import apply_ede
        apply_ede(model, 40, 120)
    cfg = step_config(args.workload)
    teacher = None
    if cfg.teacher_student:
        teacher = build_teacher(args.model).to(dev).to(memory_format=torch.channels_last)
    opt = make_optimizer(model, dataset)
    reducer = None
    if world > 1:
        fold = hasattr(opt, "grad_scale")       # FusedAdam / FusedSGD apply 1/world inside the update kernel
        if fold:
            opt.grad_scale = 1.0 / world
        # BDBNN_DDP_BUCKETS=k: k reverse-order buckets all-reduced from post-accumulate hooks while the backward
        # runs (overlap); 0: ONE all-reduce of the flat buffer after the backward
        nb = int(os.environ.get("BDBNN_DDP_BUCKETS", "2"))
        reducer = GradAllReduce(model, scale=not fold, n_buckets=max(1, nb), overlap=nb > 0)
        opt = FlatGradOptimizerShim(opt, reducer)
    step_eager = TrainStep(model, opt, cfg, teacher=teacher, grad_sync=reducer)
    use_graph = not args.no_graph and not args.profile_mode
    # whole step captured once as a CUDA graph and replayed (bdbnn_b200.step.GraphedTrainStep)
    step = GraphedTrainStep(step_eager) if use_graph else step_eager

    g = torch.Generator().manual_seed(rank)
    x_host = torch.randn(ishape, generator=g).contiguous(memory_format=torch.channels_last).pin_memory()
    y_host = torch.randint(0, ncls, (batch,), generator=g).pin_memory()
    x_dev = x_host.to(dev, non_blocking=True)
    y_dev = y_host.to(dev, non_blocking=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return ms

    # ---- device-resident timing (value) -----------------------------------------------------------
    if args.profile_mode:
        args.no_e2e = args.no_cpu_baseline = True
    n_warm = 2 if args.profile_mode else max(3, args.warmup)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    graph_note = None
    try:
        for _ in range(n_warm):
            step(x_dev, y_dev)
    except Exception as exc:
        if not use_graph:
            raise
        # capture failed (e.g. a collective that cannot be captured on this software stack): measure the eager step
        graph_note = f"CUDA graph capture failed, eager launch used: {repr(exc)[:200]}"
        use_graph = False
        step = step_eager
        torch.cuda.synchronize()
        for _ in range(n_warm):
            step(x_dev, y_dev)
    if use_graph:
        # inputs resident in HBM: the graph's own static input buffers (no per-step copy in the `value` loop)
        step.static_images.copy_(x_dev); step.static_target.copy_(y_dev)
        x_dev, y_dev = step.static_images, step.static_target
    if args.profile_mode:
        torch.cuda.synchronize()
        torch.cuda.profiler.start()          # ncu --profile-from-start off: only the timed step(s)
    barrier()
    if not use_graph:
        KernelTimer.start()
    n0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    gc.collect()
    gc.disable()                 # a generation-2 collection inside the loop stalls the launch thread for tens of ms
    sampler.mark_begin()
    e0.record()
    for _ in range(args.steps):
        out = step(x_dev, y_dev)
    e1.record()
    barrier()
    sampler.mark_end()
    gc.enable()
    if args.profile_mode:
        torch.cuda.profiler.stop()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    launches = _lib.launch_count() - n0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out, model)     # before the legs below take further steps on the model
    if use_graph:
        # per-kernel CUDA events cannot be recorded inside a graph: the roofline figures come from the SAME step
        # launched eagerly (identical kernels, identical arguments) right after the timed region
        for _ in range(2):
            step_eager(x_dev, y_dev)
        barrier()
        KernelTimer.start()
        kt0 = torch.cuda.Event(enable_timing=True); kt1 = torch.cuda.Event(enable_timing=True)
        kt0.record()
        for _ in range(args.steps):
            step_eager(x_dev, y_dev)
        kt1.record()
        kern = KernelTimer.stop()
        ms_total_eager = kt0.elapsed_time(kt1)
    else:
        kern = KernelTimer.stop()
        ms_total_eager = None
    clocks = sampler.stop() if rank == 0 else None
    ms_step = ms_total / args.steps
    value = batch * world * args.steps / (ms_total / 1e3)

    # ---- end-to-end: pinned host batch -> H2D (prefetched on a copy stream) -> step -> D2H loss -----
    e2e = None
    if not args.no_e2e:
        copy_stream = torch.cuda.Stream()
        bufs = [(torch.empty_like(x_dev), torch.empty_like(y_dev)) for _ in range(2)]
        ready = [torch.cuda.Event(), torch.cuda.Event()]
        consumed = [torch.cuda.Event(), torch.cuda.Event()]

        diag = os.environ.get("BDBNN_E2E_DIAG", "")      # attribution runs only (scripts/): "noh2d", "nod2d"

        def prefetch(i):
            b = i % 2
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(consumed[b])
                if diag != "noh2d":
                    bufs[b][0].copy_(x_host, non_blocking=True)
                    bufs[b][1].copy_(y_host, non_blocking=True)
                ready[b].record(copy_stream)

        loss_pin = [torch.empty((), dtype=torch.float32).pin_memory() for _ in range(2)]
        loss_evt = [torch.cuda.Event(), torch.cuda.Event()]

        def e2e_loop(n):
            # every step: H2D of its batch (prefetched one step ahead on the copy stream) and a D2H read of its loss
            # (train.py:519 `loss.item()`).  The read is asynchronous — copied to pinned memory right behind the step
            # and consumed by the host after the NEXT step has been launched — so the host never leaves the GPU idle.
            for b in range(2):
                consumed[b].record()
            prefetch(0)
            last, pending = None, None
            for i in range(n):
                b = i % 2
                if i + 1 < n:
                    prefetch(i + 1)
                torch.cuda.current_stream().wait_event(ready[b])
                if diag == "nod2d" and getattr(step, "static_images", None) is not None:
                    out = step(step.static_images, step.static_target)
                else:
                    out = step(bufs[b][0], bufs[b][1])
                consumed[b].record()
                loss_pin[b].copy_(out["loss"], non_blocking=True)
                loss_evt[b].record()
                if pending is not None:
                    loss_evt[pending].synchronize()
                    last = float(loss_pin[pending])
                pending = b
            loss_evt[pending].synchronize()
            last = float(loss_pin[pending])
            return last

        e2e_loop(2)
        barrier()
        gc.collect()
        gc.disable()
        e0.record()
        e2e_loop(args.steps)
        e1.record()
        barrier()
        gc.enable()
        ms_e2e = max_over_ranks(e0.elapsed_time(e1))
        e2e = {"value": round(batch * world * args.steps / (ms_e2e / 1e3), 2), "unit": "images/sec",
               "ms_per_step": round(ms_e2e / args.steps, 3),
               "h2d_bytes_per_step": int(x_host.numel() * 4 + y_host.numel() * 8) * world,
               "d2h_bytes_per_step": 4 * world,
               "note": "whole job (all ranks): pinned fp32 batch, H2D double-buffered on a copy stream; every "
                       "step's loss is copied to pinned host memory and read by the host one launch later"}

    # ---- secondary value: the fp32-class gradient operand mode (bf16 hi+lo pair, two MMAs per K step) -------
    from bdbnn_b200.functional import grad_mode
    secondary = None
    if not args.no_secondary and not args.profile_mode and grad_mode()[0] == "fp16s":
        os.environ["BDBNN_GRAD_MODE"] = "bf16x2"
        try:
            step2 = GraphedTrainStep(step_eager) if use_graph else step_eager
            for _ in range(3):
                step2(x_dev, y_dev)
            barrier()
            ns = max(3, min(10, args.steps))
            gc.collect(); gc.disable()
            e0.record()
            for _ in range(ns):
                step2(x_dev, y_dev)
            e1.record()
            barrier()
            gc.enable()
            ms2 = max_over_ranks(e0.elapsed_time(e1)) / ns
            secondary = {"grad_mode": "bf16x2", "value": round(batch * world / (ms2 / 1e3), 2), "unit": "images/sec",
                         "ms_per_step": round(ms2, 3), "steps": ns,
                         "note": "gradient operand = bf16 hi+lo pair (fp32-class, 5e-5 of max|grad| vs fp64; "
                                 "tests/test_gpu_tc.py), everything else identical"}
        finally:
            os.environ["BDBNN_GRAD_MODE"] = "fp16s"
            step2 = None

    if world > 1:
        barrier()                     # every rank has finished its timed regions before anyone leaves
    if rank != 0:
        finish(world)
        return

    # ---- same-box GPU comparator: stock eager PyTorch on the oracle modules (N=1 only) ----------------------
    eager = None
    if world == 1 and not args.no_eager_gpu and not args.profile_mode:
        del step, step_eager, model, opt
        torch.cuda.empty_cache()
        try:
            ve, mse = eager_gpu_run(args, max(3, min(10, args.steps)), 3, batch, dev)
            eager = {"value": round(ve, 2), "unit": "images/sec", "ms_per_step": round(mse, 3),
                     "path": "pure-PyTorch oracle modules on cuda: eager cuDNN convs on +-1 fp32 tensors (TF32 allowed, "
                             "cudnn.benchmark=True as train.py:368) + ATen elementwise + torch.optim; same batch, "
                             "same loop body (oracle/step_ref.py)",
                     "speedup_value_over_eager": round(value / ve, 3)}
        except Exception as exc:                      # the comparator must never take the bench line down
            eager = {"error": repr(exc)[:300]}

    # ---- roofline of the dominant kernel family ---------------------------------------------------
    peak, peak_src = peaks()
    fam = {}
    for (family, key), d in kern.items():
        f = fam.setdefault(family, {"ms": 0.0, "launches": 0, "bytes": 0})
        f["ms"] += d["ms"]; f["launches"] += d["launches"]; f["bytes"] += d["bytes"] * d["launches"]
    kernels = []
    for family, f in sorted(fam.items(), key=lambda kv: -kv[1]["ms"]):
        kernels.append({"kernel": family, "ms_per_step": round(f["ms"] / args.steps, 4),
                        "launches_per_step": f["launches"] // args.steps,
                        "achieved_gbs": round(f["bytes"] / 1e9 / (f["ms"] / 1e3), 1) if f["ms"] > 0 else None,
                        "share_of_step": round(f["ms"] / (ms_total_eager or ms_total), 4)})
    roofline = None
    timed = [k for k in kernels if k["achieved_gbs"]]       # families with algorithmic bytes (not the cuDNN teacher)
    if timed:
        top = timed[0]
        traffic, traffic_src = ncu_traffic(top["kernel"], top["launches_per_step"])
        roofline = {"bound": "hbm", "kernel": top["kernel"], "achieved": top["achieved_gbs"], "peak": peak,
                    "unit": "GB/s", "frac": round(top["achieved_gbs"] / peak, 4), "traffic": traffic,
                    "traffic_source": traffic_src,
                    "peak_source": peak_src,
                    "how": "sum of per-launch algorithmic bytes (DESIGN.md §4) / sum of CUDA-event durations "
                           "of that kernel family over " + ("the timed region" if not use_graph else
                           f"{args.steps} steps of the same step launched eagerly right after the graph-replayed "
                           "timed region (events cannot be recorded inside a CUDA graph)")}

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        cb = min(args.cpu_batch or batch, batch)
        v, ms, cores, cb = cpu_reference_run(args, 2, 1, cb, budget_s=60.0)
        cpu = {"value": round(v, 3), "unit": "images/sec", "cores": cores, "kind": "port",
               "sample": f"2 timed steps (1 warm-up) of " +
                         (f"the full {batch}-image batch" if cb == batch else f"a {cb}-image slice of the {batch}-image batch") +
                         f", {ms:.0f} ms/step, oracle CPU step (oracle/step_ref.py)"}

    gname = grad_mode()[0]
    dtype_str = {"fp16s": "f16 (+-1 operands exact; gradient = fp16 x per-call 2^e scale), f32 accumulate",
                 "bf16x2": "bf16 (+-1 operands exact; gradient = bf16 hi+lo pair), f32 accumulate",
                 "bf16": "bf16 (+-1 operands exact; gradient = bf16), f32 accumulate"}[gname]
    line = {"metric": "images/sec", "value": round(value, 2), "unit": "images/sec", "n_gpus": world,
            "steps": args.steps, "warmup": n_warm, "ms_per_step": round(ms_step, 3),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": dtype_str,
            "data": "synthetic",
            "config": {"workload": workload, "global_batch": batch * world,
                       "parallelism": f"dp{world}", "ddp_buckets": os.environ.get("BDBNN_DDP_BUCKETS", "2") if world > 1 else None,
                       "optimizer": "Adam (train.py:323-336)" if dataset == "imagenet"
                       else "SGD (train.py:319-321)", "conv_impl": args.conv_impl or "auto", "grad_mode": gname,
                       "launch": "CUDA graph replay (whole step captured once)" if use_graph else
                                 (graph_note or "eager (Python/ctypes per kernel)"),
                       "l2_policy": "per-step working set (>3 GB of activations) exceeds the 126 MB L2; no flush"},
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roofline,
            "kernels": kernels, "cpu_baseline": cpu, "eager_gpu": eager, "secondary": secondary}
    print(json.dumps(line))
    finish(world)


if __name__ == "__main__":
    main()
