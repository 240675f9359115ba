"""GPU, 2 ranks over NCCL (skipped when fewer than 2 devices are visible):
the product's data-parallel path — GradAllReduce's post-accumulate hooks issuing async bucket all-reduces
from the autograd thread into the flat .grad views, 1/world folded into FusedAdam (train.py:304, 527-529).

Checked: (1) gradients and updated parameters are BIT-IDENTICAL on both ranks; (2) they equal a
single-process run over the concatenated batch.  BatchNorm makes (2) exact only if the statistics do not
depend on the batch split, so the models run with BN in eval mode (frozen running statistics, the per-sample
map is then batch-independent) — the binary convs, fused losses, all-reduce and optimizer are the real ones;
(3) the fail-safe: plain `optimizer.zero_grad()` (set_to_none=True) without the shim still yields the same
result (ADVICE r1: stale flat buffer)."""
import os
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _worker(rank, world, port, outdir, use_shim):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    from bdbnn_b200.ddp import FlatGradOptimizerShim, GradAllReduce
    from bdbnn_b200.resnet import ResNetCifar
    from bdbnn_b200.step import StepConfig, TrainStep, make_optimizer
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    torch.manual_seed(100 + rank)                      # different init per rank: the broadcast must fix it
    m = ResNetCifar(1).to(dev).to(memory_format=torch.channels_last)
    red = GradAllReduce(m, scale=False, n_buckets=3)
    m.eval()                                           # BN on running statistics (see module docstring)
    opt = make_optimizer(m, "imagenet", lr=1e-2)       # FusedAdam, conv-only weight decay (train.py:323-336)
    opt.grad_scale = 1.0 / world
    cfg = StepConfig(w_kurtosis=True)
    step = TrainStep(m, FlatGradOptimizerShim(opt, red) if use_shim else opt, cfg, grad_sync=red if use_shim else None)
    g = torch.Generator().manual_seed(5)
    x = torch.randn(16, 3, 32, 32, generator=g)
    y = torch.randint(0, 10, (16,), generator=g)
    per = 16 // world
    xs = x[rank * per:(rank + 1) * per].to(dev).contiguous(memory_format=torch.channels_last)
    ys = y[rank * per:(rank + 1) * per].to(dev)
    init = torch.cat([p.detach().reshape(-1) for p in m.parameters()]).cpu()
    grads1 = None
    if use_shim:
        for it in range(2):
            step(xs, ys)
            if it == 0:
                grads1 = torch.cat([p.grad.reshape(-1) for p in m.parameters()]).cpu() / world
    else:
        # a user who wraps nothing: torch's own zero_grad (drops the views), backward, all-reduce, step
        for it in range(2):
            opt.zero_grad()                            # set_to_none=True by default
            out = m(xs)
            loss = torch.nn.functional.cross_entropy(out, ys)
            from bdbnn_b200.losses import kurtosis_regularization
            hooked = list(step.hooked.values())
            loss = loss + kurtosis_regularization(hooked, [1.8] * len(hooked), "avg", len(hooked), 1.0)[0]
            loss.backward()
            red()
            opt.step()
            if it == 0:
                grads1 = torch.cat([p.grad.reshape(-1) for p in m.parameters()]).cpu() / world
    torch.cuda.synchronize()
    torch.save({"flat": red.flat.cpu(), "params": torch.cat([p.detach().reshape(-1) for p in m.parameters()]).cpu(),
                "init": init, "grads1": grads1}, os.path.join(outdir, f"r{rank}_{int(use_shim)}.pt"))
    dist.destroy_process_group()


def _single(outdir, init_flat):
    """Single-process run on the concatenated batch, starting from the rank-0 initial parameters."""
    from bdbnn_b200.resnet import ResNetCifar
    from bdbnn_b200.step import StepConfig, TrainStep, make_optimizer
    dev = torch.device("cuda", 0)
    m = ResNetCifar(1).to(dev).to(memory_format=torch.channels_last)
    off = 0
    with torch.no_grad():
        for p in m.parameters():
            p.copy_(init_flat[off:off + p.numel()].view_as(p))
            off += p.numel()
    m.eval()
    step = TrainStep(m, make_optimizer(m, "imagenet", lr=1e-2), StepConfig(w_kurtosis=True))
    g = torch.Generator().manual_seed(5)
    x = torch.randn(16, 3, 32, 32, generator=g).to(dev).contiguous(memory_format=torch.channels_last)
    y = torch.randint(0, 10, (16,), generator=g).to(dev)
    step(x, y)
    return torch.cat([p.grad.reshape(-1) for p in m.parameters()]).cpu()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("use_shim", [True, False])
def test_nccl_world2_grads_and_params_identical_and_match_single_process(tmp_path, use_shim):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    port = 29600 + os.getpid() % 2000 + int(use_shim)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, str(tmp_path), use_shim)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(600)
        assert p.exitcode == 0
    r0, r1 = [torch.load(os.path.join(tmp_path, f"r{r}_{int(use_shim)}.pt")) for r in range(2)]
    assert torch.equal(r0["init"], r1["init"])                       # construction broadcast (DDP semantics)
    assert torch.equal(r0["flat"], r1["flat"]) and r0["flat"].abs().sum() > 0
    assert torch.equal(r0["params"], r1["params"])                   # bit-identical replicas after two steps
    assert torch.equal(r0["grads1"], r1["grads1"])
    single = _single(str(tmp_path), r0["init"])
    # averaged gradient of the two half batches vs the gradient of the whole batch in one process: the same
    # arithmetic up to fp32 summation order and the per-call power-of-two scale of the fp16 gradient operand
    # (Adam's sign-like first update would amplify these into O(lr) parameter differences, so the comparison
    # is made on the gradient the optimizer consumes, after step 1)
    scale = single.abs().max().item()
    assert scale > 0
    assert (single - r0["grads1"]).abs().max().item() <= 5e-3 * scale
