"""Whole-step parity against the REFERENCE's own loop code (SURVEY.md §8 a9, VERDICT r1 item 2).

tests/golden/train_step_<case>.pt were produced by tests/golden/make_train_golden.py, which imports the
reference's train.py unmodified (tests/ref_launcher.py) and calls its `train()` /
`train_teacher_student()` on CPU; tests/golden/reference_interface.json records what that train.py imports
from this repo's drop-in packages.  Neither generator is needed to run the tests.  Here:
  * CPU: the oracle's restated step (oracle/step_ref.py) and the product's step driver
    (bdbnn_b200.step.TrainStep with CPU loss ops) must reproduce those fixtures, and the reference's import
    block must resolve against this repo's drop-in packages.
  * GPU (tests/test_gpu_ref_train.py): the CUDA path replays the same fixtures."""
import importlib
import json
import os
import sys
import types

import pytest
import torch

import train_cases as TC

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
SMALL = [c for c in TC.CASES if c not in TC.SUMMARY_ONLY]


@pytest.fixture(autouse=True)
def fixture_threads():
    """Replay the fp32 CPU steps with the thread count the fixtures were computed with (train_cases.CPU_THREADS)."""
    n = torch.get_num_threads()
    torch.set_num_threads(TC.CPU_THREADS)
    yield
    torch.set_num_threads(n)


def load_golden(case):
    return torch.load(os.path.join(GOLD, f"train_step_{case}.pt"), weights_only=False)


def check_terms(out, gold, rtol=1e-6, atol=1e-7):
    """Loss terms / accuracies the reference loop fed to its AverageMeters (train.py:519-524, 638-646)."""
    m = gold["meters"]
    pairs = [("loss", "Loss"), ("ce", "Loss_ce"), ("kurt", "Loss_kurt"), ("kl", "Loss_kl"), ("kl_c", "Loss_kl_c"),
             ("acc1", "Acc@1"), ("acc5", "Acc@5")]
    for ours, theirs in pairs:
        if theirs in m:
            got = float(torch.as_tensor(out[ours]).reshape(-1)[0])
            assert got == pytest.approx(m[theirs][-1], rel=rtol, abs=atol), (ours, got, m[theirs][-1])
    assert gold["scalars"]["Train Loss"][-1] == pytest.approx(float(out["loss"]), rel=rtol, abs=atol)


def check_tensors(got, gold, tol, what):
    """Full tensors (small nets): max error relative to max|reference| per tensor."""
    assert got.keys() == gold.keys()
    for n, ref in gold.items():
        scale = ref.abs().max().item() + 1e-12
        err = (got[n].detach().cpu().float() - ref).abs().max().item()
        assert err <= tol * scale, (what, n, err, scale)


def check_summaries(got, gold, tol, what):
    """Per-parameter summaries (ResNet-18): norm, sum and 64 sampled entries."""
    assert got.keys() == gold.keys()
    for n, ref in gold.items():
        f = got[n].detach().double().reshape(-1).cpu()
        scale = ref["absmax"] + 1e-12
        assert abs(float(f.norm()) - ref["norm"]) <= tol * max(ref["norm"], 1e-12), (what, n, "norm")
        s = f[TC.sample_index(f.numel())].float()
        assert (s - ref["samples"]).abs().max().item() <= tol * scale, (what, n, "samples")


def oracle_step(case, gold):
    from oracle import step_ref as S
    c = TC.CASES[case]
    stud, teacher = TC.build_oracle(case)
    if "init" in gold:
        stud.load_state_dict(gold["init"])
        if teacher is not None:
            teacher.load_state_dict(gold["teacher_state"])
        x = gold["x"]
    else:
        assert TC.state_checksum(stud) == pytest.approx(gold["init_checksum"], rel=1e-12), "seeded init differs"
        x = TC.make_batch(case)[0]
        assert float(x.double().sum()) == pytest.approx(gold["x_checksum"], rel=1e-12)
    y = gold["y"]
    hooked = S.ref_hooked_weights(stud) if c["args"].get("w_kurtosis") else {}
    assert list(hooked) == gold["hooked"]
    kw = TC.step_kwargs(case, len(hooked))
    opt = S.ref_make_optimizer(stud, c["dataset"], c["args"]["lr"])
    out = S.ref_train_step(stud, opt, x, y, hooked=hooked, teacher=teacher, **kw)
    return stud, out


@pytest.mark.parametrize("case", list(TC.CASES))
def test_oracle_step_reproduces_reference_loop(case):
    """oracle/step_ref.py == the reference's train()/train_teacher_student() on the stored fixtures."""
    gold = load_golden(case)
    stud, out = oracle_step(case, gold)
    check_terms(out, gold)
    grads = {n: p.grad for n, p in stud.named_parameters()}
    after = dict(stud.named_parameters())
    if case in TC.SUMMARY_ONLY:
        check_summaries(grads, gold["grads"], 1e-5, "grad")
        check_summaries(after, gold["after"], 1e-6, "param")
    else:
        check_tensors(grads, gold["grads"], 1e-6, "grad")
        check_tensors(after, gold["after"], 1e-6, "param")
        check_tensors(dict(stud.named_buffers()), gold["buffers"], 1e-6, "buffer")


@pytest.mark.parametrize("case", SMALL)
def test_product_step_driver_reproduces_reference_loop_on_cpu(case):
    """bdbnn_b200.step.TrainStep (hook selection, loss assembly, optimizer construction) driven on CPU with
    the oracle's loss ops and modules: same fixtures, so the host logic of the product is pinned too."""
    from bdbnn_b200.step import StepConfig, TrainStep, make_optimizer
    from oracle.models_ref import RefOps
    gold = load_golden(case)
    c = TC.CASES[case]
    a = c["args"]
    stud, teacher = TC.build_oracle(case)
    stud.load_state_dict(gold["init"])
    if teacher is not None:
        teacher.load_state_dict(gold["teacher_state"])
    cfg = StepConfig(w_kurtosis=bool(a.get("w_kurtosis")), w_kurtosis_target=a.get("w_kurtosis_target", 1.8),
                     w_lambda_kurtosis=a.get("w_lambda_kurtosis", 1.0), kurtosis_mode=a.get("kurtosis_mode", "avg"),
                     teacher_student=c["teacher"], react=bool(a.get("react")), alpha=a.get("alpha", 0.9),
                     beta=a.get("beta", 200.0))
    step = TrainStep(stud, make_optimizer(stud, c["dataset"], lr=a["lr"]), cfg, teacher=teacher, ops=RefOps)
    assert list(step.hooked) == gold["hooked"]
    out = step(gold["x"], gold["y"])
    check_terms(out, gold)
    check_tensors({n: p.grad for n, p in stud.named_parameters()}, gold["grads"], 1e-6, "grad")
    check_tensors(dict(stud.named_parameters()), gold["after"], 1e-6, "param")


def _module_or_attr(module, name):
    mod = importlib.import_module(module)
    return getattr(mod, name) if hasattr(mod, name) else importlib.import_module(f"{module}.{name}")


def test_reference_import_block_resolves_against_the_dropin_packages():
    """Every name the reference's train.py imports from the drop-in packages (`from utils import utils`,
    `from models import ...`, `from kurtosis import KurtosisWeight, ...`, `from utils import KD_loss`; recorded in
    golden/reference_interface.json by golden/make_interface_golden.py) binds to THIS repo's files and objects,
    the drop-in modules carry every attribute train.py reads on them, the model-name lists train.py builds
    from `models` are unchanged, and bdbnn_b200.step.StepConfig defaults to the reference parser's values."""
    import bdbnn_b200
    from bdbnn_b200.step import StepConfig
    with open(os.path.join(GOLD, "reference_interface.json")) as fh:
        gold = json.load(fh)
    for imp in gold["imports"]:
        obj = _module_or_attr(imp["module"], imp["name"])
        src = obj if isinstance(obj, types.ModuleType) else sys.modules[obj.__module__]
        assert os.path.abspath(src.__file__).startswith(ROOT + os.sep), (imp, src.__file__)
    assert _module_or_attr("kurtosis", "KurtosisWeight") is bdbnn_b200.KurtosisWeight
    assert _module_or_attr("models.imagenet.resnet_bi_imagenet_set_2_2", "HardBinaryConv") is bdbnn_b200.HardBinaryConv
    assert _module_or_attr("utils", "KD_loss").DistributionLoss is bdbnn_b200.DistributionLoss
    for module, names in gold["attributes"].items():
        mod = importlib.import_module(module)
        assert [n for n in names if not hasattr(mod, n)] == [], module
    for pkg, names in gold["model_names"].items():
        m = importlib.import_module(f"models.{pkg}")
        assert sorted(n for n in vars(m) if n.islower() and not n.startswith("__") and callable(vars(m)[n])) == names
    assert "resnet18" in gold["model_names"]["imagenet"] and "resnet20" in gold["model_names"]["cifar10"]
    # weight_name defaults to the `all` the reference README's recipes pass (parser default: None); w_lambda_ce is
    # read by train.py but only assigned under --react
    defaults, cfg = gold["parser_defaults"], StepConfig()
    assert defaults.pop("weight_name") is None and tuple(cfg.weight_name) == ("all",) and cfg.w_lambda_ce == 1.0
    assert defaults["alpha"] == 0.9 and defaults["beta"] == 200
    assert {k: getattr(cfg, k) for k in defaults} == defaults


def test_dropin_utils_match_reference_semantics():
    """utils/utils.py helpers the loop calls: meters' running average and rendering, accuracy, parameter lookup."""
    from utils import utils as U
    m = U.AverageMeter("Loss", ":.4e")
    m.update(2.0, 4)
    m.update(1.0, 12)
    assert m.avg == pytest.approx(1.25) and m.get_avg() == m.avg and m.count == 16 and m.val == 1.0
    assert str(m) == "Loss 1.0000e+00 (1.2500e+00)"
    lines = []

    class Lg:
        def info(self, s):
            lines.append(s)
    U.ProgressMeter(391, [m], Lg(), prefix="Epoch: [3]").display(7)
    assert lines == ["Epoch: [3][  7/391]\tLoss 1.0000e+00 (1.2500e+00)"]
    out = torch.tensor([[0.1, 0.9, 0.0], [0.8, 0.1, 0.1], [0.2, 0.3, 0.5]])
    acc1, acc2 = U.accuracy(out, torch.tensor([1, 2, 2]), topk=(1, 2))
    assert float(acc1) == pytest.approx(200.0 / 3) and float(acc2) == pytest.approx(200.0 / 3)
    lin = torch.nn.Linear(2, 2)
    assert U.find_weight_tensor_by_name(lin, "bias") is lin.bias and U.find_weight_tensor_by_name(lin, "nope") is None
    from kurtosis import RidgeRegularization, WeightRegularization
    w = torch.tensor([[0.5, -2.0], [1.0, 0.0]])
    r = RidgeRegularization(w, "w")
    assert r.l2_regularization() is None and float(r.l2_loss) == pytest.approx(5.25)
    q = WeightRegularization(w, "w")
    assert q.w_regularization() is None and q.size == 4
    assert float(q.wr_loss) == pytest.approx((0.25 + 1.0 + 0.0 + 1.0) ** 0.5)
