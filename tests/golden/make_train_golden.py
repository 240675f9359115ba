"""Generate whole-step golden fixtures by executing the REFERENCE's own `train()` and
`train_teacher_student()` (train.py:441-554, 556-675), imported unmodified through
tests/ref_launcher.py in "reference" mode: train.py, kurtosis.py, utils/utils.py and utils/KD_loss.py are
the reference's files; only the `models` package (absent upstream) and the network under test (oracle
modules, CPU) come from this repo.  Build container only.

    python tests/golden/make_train_golden.py        ->  tests/golden/train_step_<case>.pt

Per case: the batch, the initial state (small nets) or its checksum (ResNet-18, regenerated from the
seed), every value the loop fed to its AverageMeters (loss, CE, kurtosis, KL terms, top-1/5), every
parameter gradient and every updated parameter (tensors for the small nets, summaries for ResNet-18)."""
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import ref_launcher as RL        # noqa: E402
import train_cases as TC         # noqa: E402


def record_meters(train):
    """Subclass the reference's own AverageMeter so that every update() is also appended to a log
    (the loop keeps its meters in locals; train.py:442-448, 557-565)."""
    base = train.utils.AverageMeter
    log = {}

    class Recording(base):
        def update(self, val, n=1):
            if self.name not in ("Time", "Data"):            # wall-clock meters: not part of the result
                log.setdefault(self.name, []).append(float(val))
            return super().update(val, n)

    train.utils.AverageMeter = Recording
    return log, base


def run_case(case):
    c = TC.CASES[case]
    train = RL.import_reference_train("reference")
    stud, teacher = TC.build_oracle(case)
    init = {k: v.clone() for k, v in stud.state_dict().items()}
    t_state = {k: v.clone() for k, v in teacher.state_dict().items()} if teacher is not None else None
    args = RL.make_args(train, dataset=c["dataset"], **{k: v for k, v in c["args"].items() if k != "lr"})
    args.lr = c["args"]["lr"]
    from oracle.step_ref import ref_make_optimizer        # optimizer construction lives inside main_worker
    opt = ref_make_optimizer(stud, c["dataset"], args.lr, args.momentum, args.weight_decay)
    x, y = TC.make_batch(case)
    log, base = record_meters(train)
    try:
        out = RL.run_reference_loop(train, stud, opt, [(x, y)], args, teacher=teacher)
    finally:
        train.utils.AverageMeter = base
    grads = {n: p.grad.detach().clone() for n, p in stud.named_parameters()}
    after = {n: p.detach().clone() for n, p in stud.named_parameters()}
    buffers = {n: b.detach().clone() for n, b in stud.named_buffers()}
    rec = {"case": case, "config": c, "x_checksum": float(x.double().sum()), "y": y, "meters": log, "scalars": out["scalars"],
           "hooked": list(out["hooked"].keys()), "sources": train.__bdbnn_sources__,
           "init_checksum": TC.state_checksum_from(init), "torch": torch.__version__}
    if case in TC.SUMMARY_ONLY:
        rec.update(grads=TC.summarize(grads), after=TC.summarize(after), buffers=TC.summarize(buffers))
    else:
        rec.update(x=x, init=init, teacher_state=t_state, grads=grads, after=after, buffers=buffers)
    torch.save(rec, os.path.join(os.environ.get("BDBNN_GOLDEN_OUT", HERE), f"train_step_{case}.pt"))
    print(case, {k: v for k, v in log.items() if k not in ("Time", "Data")}, out["scalars"])


if __name__ == "__main__":
    torch.set_num_threads(TC.CPU_THREADS)
    for name in (sys.argv[1:] or TC.CASES):
        run_case(name)
