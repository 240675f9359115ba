"""GPU: whole training step (BASELINE.json config 1 shape, reduced batch) vs the CPU oracle step,
and the kernel-launch counter bench.py reports."""
import copy

import pytest
import torch

pytestmark = pytest.mark.gpu


def _grads(m):
    return {n: p.grad.detach().cpu().clone() for n, p in m.named_parameters()}


@pytest.mark.parametrize("ts,ede", [(False, False), (True, False), (False, True)])
def test_resnet20_step_matches_cpu_oracle(ts, ede):
    import torchvision
    from bdbnn_b200 import _lib
    from bdbnn_b200.resnet import resnet20
    from bdbnn_b200.step import StepConfig, TrainStep, make_optimizer
    from oracle.models_ref import resnet20_fp32, resnet20_ref
    from oracle import step_ref as S
    torch.manual_seed(0)
    ref = resnet20_ref()
    gpu = resnet20()
    gpu.load_state_dict(ref.state_dict())
    gpu = gpu.cuda().to(memory_format=torch.channels_last)
    teacher_ref = teacher_gpu = None
    if ts:
        import torch.nn as nn
        from bdbnn_b200.resnet import ResNetCifar
        fp32_conv = lambda i, o, k, s, p: nn.Conv2d(i, o, k, s, p, bias=False)   # fp32 teacher (train.py:250-277)
        torch.manual_seed(1)
        teacher_ref = resnet20_fp32().eval()          # same names/shapes as the student (KD_loss.py:63)
        for p in teacher_ref.parameters():
            p.requires_grad = False                   # train.py:275-276
        teacher_gpu = ResNetCifar(3, conv_cls=fp32_conv)
        teacher_gpu.load_state_dict(teacher_ref.state_dict())
        teacher_gpu = teacher_gpu.cuda().to(memory_format=torch.channels_last).eval()
        for p in teacher_gpu.parameters():
            p.requires_grad = False
    if ede:                                           # train.py:409-415 at epoch 40 of 120
        from bdbnn_b200.step import apply_ede
        t, k = apply_ede(gpu, 40, 120)
        for m in ref.modules():                       # the oracle's own restatement of train.py:409-415
            if isinstance(m, torch.nn.Conv2d):
                m.k, m.t = k.cpu(), t.cpu()
        assert all(m.ede_active for m in gpu.modules() if hasattr(m, "ede_active"))
    cfg = StepConfig(w_kurtosis=True, teacher_student=ts, beta=200.0, alpha=0.9)
    # lr=0: compare gradients of one step without the update moving the weights.  The CPU side is the
    # oracle's independent restatement of the loop body (oracle/step_ref.py, pinned to the reference's own
    # train() by tests/test_ref_train.py) — not the product's step driver.
    hooked = S.ref_hooked_weights(ref)
    s_ref = lambda xs, ys: S.ref_train_step(ref, S.ref_make_optimizer(ref, "cifar10", 0.0), xs, ys, hooked=hooked,
                                            targets=[1.8] * len(hooked), kurt_on=True, teacher=teacher_ref,
                                            alpha=0.9, beta=200.0)
    s_gpu = TrainStep(gpu, make_optimizer(gpu, "cifar10", lr=0.0), cfg, teacher=teacher_gpu)
    g = torch.Generator().manual_seed(3)
    x = torch.randn(16, 3, 32, 32, generator=g)
    y = torch.randint(0, 10, (16,), generator=g)
    n0 = _lib.launch_count()
    o_ref = s_ref(x, y)
    o_gpu = s_gpu(x.cuda().contiguous(memory_format=torch.channels_last), y.cuda())
    assert _lib.launch_count() - n0 >= 18 * 6      # 18 binary convs x (pack, wpack x2, fwd, dgrad, wgrad)
    # Whole-network tolerances are looser than the per-kernel ones (tests/test_gpu_kernels.py,
    # test_gpu_tc.py): BatchNorm runs in cuDNN on the GPU and oneDNN on the CPU, so a handful of
    # activations within fp32 round-off of 0 (or of +-1) take the other sign / STE-mask value, a discrete
    # difference that propagates through the remaining layers.
    for k in ("loss", "ce", "kurt") + (("kl", "kl_c") if ts else ()):
        torch.testing.assert_close(o_gpu[k].cpu(), o_ref[k], rtol=5e-4, atol=1e-5)
    torch.testing.assert_close(o_gpu["output"].cpu(), o_ref["output"], rtol=5e-3, atol=5e-4)
    gr, gg = _grads(ref), _grads(gpu)
    assert gr.keys() == gg.keys()
    for n in gr:
        scale = gr[n].abs().max().item() + 1e-12
        err = (gg[n] - gr[n]).abs().max().item()
        assert err <= 2e-2 * scale, (n, err, scale)


def test_resnet18_steps_are_bit_reproducible():
    """The same inputs give the same steps, bit for bit.  In a binarised network a last-bit difference flips signs
    and grows over the following steps; BatchNorm statistics combined through fp32 atomics differed in the last bit
    from run to run (2 % of max|logit| after one step).  The fp64 combine leaves order effects in the last fp64 bits,
    which the fp32 statistics almost never see."""
    from bdbnn_b200.resnet import resnet18
    from bdbnn_b200.step import StepConfig, TrainStep, make_optimizer
    g = torch.Generator().manual_seed(0)
    x = torch.randn(64, 3, 224, 224, generator=g).cuda().contiguous(memory_format=torch.channels_last)
    y = torch.randint(0, 1000, (64,), generator=g).cuda()
    runs = []
    for _ in range(2):
        torch.manual_seed(0)
        m = resnet18().cuda()
        step = TrainStep(m, make_optimizer(m, "imagenet"), StepConfig())
        outs = [{k: v.clone() for k, v in step(x, y).items() if torch.is_tensor(v)} for _ in range(3)]
        torch.cuda.synchronize()
        runs.append((outs, {k: v.clone() for k, v in m.state_dict().items()}))
    for a, b in zip(runs[0][0], runs[1][0]):
        for k in a:
            assert torch.equal(a[k], b[k]), k
    for k, v in runs[0][1].items():
        assert torch.equal(v, runs[1][1][k]), k
