"""End-to-end parity of the B200 ResNet path against the CPU oracle (fp32) on the same weights and inputs."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def _models(seed=0, **kw):
    from deeplearning_b200.classification.resnet.models.networks import resnet50

    torch.manual_seed(seed)
    m = resnet50(**kw)
    state = {k: v.clone() for k, v in m.state_dict().items()}
    return m.cuda(), state


def _torch_ref(state, layers=(3, 4, 6, 3)):
    import torchvision

    ref = torchvision.models.ResNet(torchvision.models.resnet.Bottleneck, list(layers)).cuda()
    ref.load_state_dict(state)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    return ref


def _autocast_yardstick(state, x, train, labels=None, layers=(3, 4, 6, 3)):
    """What bf16 storage costs the reference itself: PyTorch bf16 autocast vs PyTorch fp32 on the same weights/input.
    Returns (max-abs logit error, {param: grad rel-L2 error}) (grads only when labels are given)."""
    ref = _torch_ref(state, layers)
    ref.train(train)
    xg = x.cuda()
    outs, grads = [], []
    for amp in (False, True):
        ref.load_state_dict(state)
        ref.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp):
            with torch.set_grad_enabled(labels is not None):
                o = ref(xg).float()
        outs.append(o.detach())
        if labels is not None:
            F.cross_entropy(o, labels.cuda()).backward()
            grads.append({n: p.grad.detach().clone() for n, p in ref.named_parameters()})
    gerr = {}
    if labels is not None:
        gerr = {n: float((grads[1][n] - grads[0][n]).norm() / (grads[0][n].norm() + 1e-12)) for n in grads[0]}
    return float((outs[1] - outs[0]).abs().max()), gerr


def test_resnet50_eval_logits_parity():
    """Eval-mode logits vs the fp32 oracle, after calibrating the running statistics on one batch (at the raw init
    running_var = 1 makes eval-mode activations explode to |logit| ~ 100, where 1e-2 absolute is below bf16 resolution)."""
    from oracle.resnet import resnet_forward

    m, state = _models()
    xc = torch.randn(32, 3, 224, 224, generator=torch.Generator().manual_seed(3))
    with torch.no_grad():
        resnet_forward(state, xc, train=True, momentum=1.0)  # running stats := batch stats
    m.load_state_dict(state)
    m.eval()
    x = torch.randn(8, 3, 224, 224, generator=torch.Generator().manual_seed(1))
    with torch.no_grad():
        ref = resnet_forward(state, x, train=False)
        got = m(x.cuda()).float().cpu()
    err = float((got - ref).abs().max())
    yard, _ = _autocast_yardstick(state, x, False)
    print(f"eval logits max-abs err {err:.4g} (|ref| max {float(ref.abs().max()):.3g}); torch bf16 autocast on the same input: {yard:.4g}")
    assert err <= max(1e-2, 1.5 * yard), (err, yard)  # north_star: 1e-2 for bf16, or no worse than the reference's own bf16


def _train_step_check(layers, B, hw, grad_slack):
    from deeplearning_b200.classification.resnet.models.networks import Bottleneck, ResNet
    from oracle.resnet import train_step_grads

    torch.manual_seed(0)
    m = ResNet(Bottleneck, list(layers))
    state = {k: v.clone() for k, v in m.state_dict().items()}
    m = m.cuda().train()
    x = torch.randn(B, 3, hw, hw, generator=torch.Generator().manual_seed(1))
    labels = torch.randint(0, 1000, (B,), generator=torch.Generator().manual_seed(2))
    state_before = {k: v.clone() for k, v in state.items()}
    ref_logits, ref_loss, ref_grads = train_step_grads(state, x, labels)
    out = m(x.cuda())
    loss = F.cross_entropy(out, labels.cuda())
    loss.backward()
    err = float((out.detach().float().cpu() - ref_logits).abs().max())
    yard, gyard = _autocast_yardstick(state_before, x, True, labels, layers)
    print(f"layers={layers}: train logits max-abs err {err:.4g} (|ref| max {float(ref_logits.abs().max()):.3g}, torch-bf16 "
          f"yardstick {yard:.4g}); loss {float(loss.detach()):.5f} vs {float(ref_loss):.5f}")
    assert err <= max(1e-2, 1.5 * yard), (err, yard)
    assert abs(float(loss.detach()) - float(ref_loss)) <= 1e-2
    worst = (0.0, "")
    for name, p in m.named_parameters():
        g, r = p.grad.float().cpu(), ref_grads[name]
        rel = float((g - r).norm() / (r.norm() + 1e-12))
        worst = max(worst, (rel / (gyard[name] + 1e-3), name))
        assert rel <= grad_slack * gyard[name] + 0.02, f"{name}: grad rel-L2 error {rel:.3g} vs torch-bf16 yardstick {gyard[name]:.3g}"
    print(f"worst grad error relative to the torch-bf16 yardstick: {worst[0]:.2f}x at {worst[1]}")
    sd = m.state_dict()
    shallow = sum(layers) <= 4
    for k in state:
        # deep layers of the 50-layer net see inputs that already differ by tens of percent (bf16 chaos, see above)
        if "running_" in k and (shallow or k.startswith(("bn1.", "layer1."))):
            assert torch.allclose(sd[k].cpu(), state[k], rtol=2e-2, atol=2e-3), k
        if "num_batches" in k:
            assert int(sd[k]) == int(state[k])


def test_resnet14_train_step_parity():
    """Shallow Bottleneck net: bf16 rounding noise stays small, so gradients must agree with the fp32 oracle closely."""
    _train_step_check((1, 1, 1, 1), 32, 128, grad_slack=2.0)


def test_resnet50_train_step_parity():
    """Full ResNet-50: at random init train-mode BN amplifies any bf16 rounding ~1.25x per block (the reference's own
    autocast run shows the same), so the gate is 'no worse than torch bf16 autocast', measured on the same input."""
    _train_step_check((3, 4, 6, 3), 64, 224, grad_slack=2.0)


def test_resnet50_head_surgery_and_small_classes():
    """model.fc = nn.Linear(2048, 5) as the reference fine-tune script does (classification/resnet/train.py:79-80)."""
    m, _ = _models()
    m.fc = torch.nn.Linear(2048, 5).cuda()
    m.train()
    x = torch.randn(4, 3, 64, 64, device="cuda")
    out = m(x)
    assert out.shape == (4, 5)
    out.sum().backward()
    assert m.fc.weight.grad.shape == (5, 2048) and torch.isfinite(m.fc.weight.grad).all()
    assert m.conv1.weight.grad.shape == (64, 3, 7, 7)


def test_cpu_tensor_raises():
    m, _ = _models()
    with pytest.raises(RuntimeError):
        m(torch.randn(1, 3, 32, 32))


def test_reference_evaluate_and_train_loops_run_on_the_dropin():
    """SURVEY 8(f)-3 / B4: the reference's `evaluate` and `train_one_epoch` (classification/resnet/utils.py:61-83,28-57, as
    restated in oracle/train_loop.py, which returns what the reference's own loops return: tests/test_oracle_golden.py) drive
    the drop-in module; the eval pass runs with BatchNorm folded into the conv epilogues and agrees with the fp32 oracle on
    the same weights."""
    from oracle import train_loop as utils
    from oracle.resnet import resnet_forward

    m, state = _models()
    xc = torch.randn(32, 3, 224, 224, generator=torch.Generator().manual_seed(3))
    with torch.no_grad():
        resnet_forward(state, xc, train=True, momentum=1.0)       # calibrate the running statistics
    m.load_state_dict(state)
    g = torch.Generator().manual_seed(5)
    batches = [(torch.randn(8, 3, 224, 224, generator=g), torch.randint(0, 1000, (8,), generator=g)) for _ in range(2)]
    loss_fn = torch.nn.CrossEntropyLoss()
    loss, acc = utils.evaluate(m, batches, torch.device("cuda"), loss_fn)
    with torch.no_grad():
        ref = sum(float(F.cross_entropy(resnet_forward(state, x, train=False), y)) for x, y in batches) / len(batches)
    assert abs(loss - ref) < 2e-2, (loss, ref)
    opt = torch.optim.SGD(m.parameters(), lr=0.01, momentum=0.9, weight_decay=5e-5)
    tl, ta = utils.train_one_epoch(m, batches, torch.device("cuda"), opt, loss_fn)
    assert tl == tl and 0.0 <= ta <= 1.0   # finite loss, loop ran to the end


def test_gpu_input_pipeline_uint8_nhwc_equals_cpu_totensor_normalize():
    """SURVEY 8(f)-1: a decoded uint8 NHWC batch fed straight to the drop-in (ToTensor + Normalize fused into the stem's
    space-to-depth operand; 4x less host->device traffic) gives the logits of the reference's CPU preprocessing
    (classification/resnet/train.py:46-71: ToTensor, Normalize([0.485, 0.456, 0.406], [0.229, 0.224, 0.225])) + float input."""
    from deeplearning_b200 import ops

    m, _ = _models()
    m.eval()
    g = torch.Generator().manual_seed(9)
    u8 = torch.randint(0, 256, (4, 64, 64, 3), generator=g, dtype=torch.uint8)
    mean, std = torch.tensor(ops.IMAGENET_MEAN), torch.tensor(ops.IMAGENET_STD)
    xf = ((u8.float() / 255.0 - mean) / std).permute(0, 3, 1, 2).contiguous()
    with torch.no_grad():
        a = m(u8.cuda()).float().cpu()
        b = m(xf.cuda()).float().cpu()
    assert float((a - b).abs().max()) <= 2e-2 * max(1.0, float(b.abs().max())), float((a - b).abs().max())
    z1 = ops.stem_s2d_u8(u8.cuda())
    z2 = ops.stem_s2d(xf.cuda())
    assert float((z1.float() - z2.float()).abs().max()) <= 2e-2        # same operand up to one bf16 rounding of (u8*a + b)
    y = ops.normalize_u8_nhwc(u8.cuda())
    assert torch.allclose(y.cpu(), xf, rtol=1e-5, atol=1e-5)
