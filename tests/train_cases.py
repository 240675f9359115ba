"""Shared definition of the whole-step parity cases (used by tests/golden/make_train_golden.py, which runs
the REFERENCE's train() / train_teacher_student() on them, and by the CPU / GPU tests that replay them)."""
import torch

# name -> (arch, dataset, batch, image size, teacher?, args overrides for the reference parser)
CASES = {
    # CIFAR shell with one block per stage (6 binary convs): small enough to store every gradient
    "cifar_kurt": dict(arch="cifar_n1", dataset="cifar10", batch=16, hw=32, teacher=False,
                       args=dict(w_kurtosis=True, w_kurtosis_target=1.8, kurtosis_mode="avg", lr=0.1)),
    "cifar_kurt_max": dict(arch="cifar_n1", dataset="cifar10", batch=8, hw=32, teacher=False,
                           args=dict(w_kurtosis=True, w_kurtosis_target=1.4, kurtosis_mode="max",
                                     w_lambda_kurtosis=0.5, lr=0.05)),
    "cifar_ts": dict(arch="cifar_n1", dataset="cifar10", batch=16, hw=32, teacher=True,
                     args=dict(w_kurtosis=True, w_kurtosis_target=1.8, kurtosis_mode="sum", lr=0.1,
                               imagenet_setting_step_2_ts=True, alpha=0.9, beta=200.0)),
    "cifar_ts_react": dict(arch="cifar_n1", dataset="cifar10", batch=8, hw=32, teacher=True,
                           args=dict(w_kurtosis=False, lr=0.1, imagenet_setting_step_2_ts=True, react=True)),
    # the configuration the headline times: ResNet-18, 224x224, Adam with conv-only weight decay
    "r18_ce": dict(arch="resnet18", dataset="imagenet", batch=4, hw=224, teacher=False,
                   args=dict(w_kurtosis=False, lr=1e-3)),
    "r18_kurt_ts": dict(arch="resnet18", dataset="imagenet", batch=4, hw=224, teacher=True,
                        args=dict(w_kurtosis=True, diffkurt=True, kurtosis_mode="avg", lr=1e-3,
                                  imagenet_setting_step_2_ts=True, alpha=0.9, beta=200.0)),
}
SUMMARY_ONLY = ("r18_ce", "r18_kurt_ts")      # 11.7 M parameters: store per-parameter summaries, not tensors
N_SAMPLES = 64
# intra-op threads of every fp32 CPU step that makes or replays a fixture: oneDNN splits its convolution reductions
# by thread count, and the replay tolerances (1e-6 of max|reference|) hold for the summation order of this count
CPU_THREADS = 8


def build_oracle(case, seed=0):
    """(student, teacher or None) on the pure-PyTorch oracle modules, deterministic from `seed`."""
    import torch.nn as nn
    from oracle import models_ref as M
    c = CASES[case]
    torch.manual_seed(seed)
    if c["arch"] == "cifar_n1":
        stud = M.RefResNetCifar(1)
    else:
        stud = M.resnet18_ref()
    teacher = None
    if c["teacher"]:
        torch.manual_seed(seed + 1)
        if c["arch"] == "cifar_n1":
            teacher = M.RefResNetCifar(1, conv_cls=lambda i, o, k, s, p: nn.Conv2d(i, o, k, s, p, bias=False))
        else:
            import torchvision
            teacher = torchvision.models.resnet18()
        teacher.eval()
        for p in teacher.parameters():
            p.requires_grad = False                       # train.py:275-277
    return stud, teacher


def build_product(case):
    """The same architectures on the product modules (CUDA kernels); weights are loaded by the caller."""
    import torch.nn as nn
    from bdbnn_b200 import resnet as R
    c = CASES[case]
    if c["arch"] == "cifar_n1":
        stud = R.ResNetCifar(1)
        teacher = R.ResNetCifar(1, conv_cls=lambda i, o, k, s, p: nn.Conv2d(i, o, k, s, p, bias=False)) \
            if c["teacher"] else None
    else:
        stud = R.resnet18()
        teacher = None
        if c["teacher"]:
            import torchvision
            teacher = torchvision.models.resnet18()
    if teacher is not None:
        teacher.eval()
        for p in teacher.parameters():
            p.requires_grad = False
    return stud, teacher


def make_batch(case, seed=7):
    c = CASES[case]
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(c["batch"], 3, c["hw"], c["hw"], generator=g)
    y = torch.randint(0, 10 if c["dataset"] == "cifar10" else 1000, (c["batch"],), generator=g)
    return x, y


def state_checksum(module):
    return state_checksum_from(module.state_dict())


def state_checksum_from(state):
    """Order-sensitive fp64 checksum of a state_dict (verifies that a seed regenerated the same weights)."""
    tot = 0.0
    for i, (k, v) in enumerate(state.items()):
        tot += (i + 1) * float(v.double().sum()) + float(v.double().abs().sum())
    return tot


def sample_index(numel, n=N_SAMPLES):
    """Fixed pseudo-random positions inside a tensor of `numel` elements."""
    g = torch.Generator().manual_seed(numel % 100003)
    return torch.randint(0, numel, (min(n, numel),), generator=g)


def summarize(tensors):
    """{name: dict(norm, sum, absmax, samples)} — what is stored for the ResNet-18 cases."""
    out = {}
    for n, t in tensors.items():
        f = t.detach().double().reshape(-1).cpu()
        out[n] = {"norm": float(f.norm()), "sum": float(f.sum()), "absmax": float(f.abs().max()),
                  "samples": f[sample_index(f.numel())].float().clone()}
    return out


def step_kwargs(case, hooked_len):
    """Arguments of the restated steps (oracle.step_ref.ref_train_step / bdbnn_b200.step.StepConfig) that
    correspond to the reference parser overrides of the case."""
    c = CASES[case]
    a = c["args"]
    if a.get("diffkurt"):
        from oracle.step_ref import TS_DIFFKURT, IMAGENET_DIFFKURT, CIFAR_DIFFKURT
        if c["teacher"]:
            targets = TS_DIFFKURT                                        # train.py:586-589
        else:
            targets = IMAGENET_DIFFKURT if c["dataset"] == "imagenet" else CIFAR_DIFFKURT
    else:
        targets = [a.get("w_kurtosis_target", 1.8)] * hooked_len
    return dict(targets=list(targets)[:hooked_len] if hooked_len <= len(targets) else list(targets),
                kurtosis_mode=a.get("kurtosis_mode", "avg"), lam_kurt=a.get("w_lambda_kurtosis", 1.0),
                kurt_on=bool(a.get("w_kurtosis")), alpha=a.get("alpha", 0.9), beta=a.get("beta", 200.0),
                react=bool(a.get("react")))
