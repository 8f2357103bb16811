"""GPU parity tests of the individual sm_100a kernels against a plain PyTorch fp32 reference of the same op.

Inputs are rounded to bf16 first so that the only differences are accumulation order and the bf16 rounding of outputs.
"""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def _ops():
    from deeplearning_b200 import ops

    return ops


def _rand(*shape, scale=1.0, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.randn(*shape, device="cuda", generator=g) * scale).to(torch.bfloat16)


def _ref_conv(x_nhwc, w_oihw, ksize, stride):
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    x = x_nhwc.float().permute(0, 3, 1, 2).contiguous()
    return F.conv2d(x, w_oihw.float(), stride=stride, padding=ksize // 2)


def _close(a, b, rtol, atol, what):
    a, b = a.float(), b.float()
    err = (a - b).abs()
    tol = atol + rtol * b.abs()
    bad = err > tol
    assert not bad.any(), f"{what}: {int(bad.sum())}/{bad.numel()} bad, max abs err {float(err.max()):.4g} (ref max {float(b.abs().max()):.4g})"


CONV_CASES = [
    # B, H, W, Cin, Cout, k, s
    (2, 8, 8, 64, 64, 1, 1),
    (3, 7, 7, 128, 256, 1, 1),
    (2, 14, 14, 256, 1000, 1, 1),
    (4, 1, 1, 72, 40, 1, 1),
    (2, 56, 56, 64, 64, 3, 1),
    (24, 56, 56, 64, 64, 3, 1),   # 588 pixel tiles: several per CTA of the resident-weight kernel (conv_tap64.cuh)
    (2, 14, 14, 128, 128, 3, 1),
    (3, 7, 7, 64, 192, 3, 1),
    (2, 28, 28, 128, 128, 3, 2),
    (2, 14, 14, 64, 64, 3, 2),
    (2, 28, 28, 64, 128, 1, 2),
    (1, 9, 11, 64, 64, 3, 1),
    (1, 10, 6, 64, 64, 3, 2),
]


@pytest.mark.parametrize("B,H,W,Cin,Cout,k,s", CONV_CASES)
def test_conv_fwd(B, H, W, Cin, Cout, k, s):
    ops = _ops()
    x = _rand(B, H, W, Cin, seed=1)
    w = _rand(Cout, Cin, k, k, scale=(Cin * k * k) ** -0.5, seed=2)
    wp = ops.pack_weight(w.float())
    y, stats = ops.conv2d_fwd(x, wp, k, s, want_stats=True)
    ref = _ref_conv(x, w, k, s).permute(0, 2, 3, 1)
    _close(y, ref, 1e-2, 1e-2, "conv fwd")
    # statistics of the stored (bf16) output
    yf = y.float().reshape(-1, Cout)
    _close(stats[:, 0].sum(0), yf.sum(0), 1e-3, 1e-2, "stats sum")
    _close(stats[:, 1].sum(0), (yf * yf).sum(0), 1e-3, 1e-2, "stats sumsq")


@pytest.mark.parametrize("B,H,W,Cin,Cout,k,s", CONV_CASES)
def test_conv_dgrad(B, H, W, Cin, Cout, k, s):
    ops = _ops()
    w = _rand(Cout, Cin, k, k, scale=(Cout * k * k) ** -0.5, seed=3)
    Ho, Wo = ops.out_hw(H, k, s), ops.out_hw(W, k, s)
    dy = _rand(B, Ho, Wo, Cout, seed=4)
    wd = ops.pack_weight(w.float(), mode=1)
    x = torch.zeros(B, Cin, H, W, device="cuda", requires_grad=True)
    torch.backends.cudnn.allow_tf32 = False
    yr = F.conv2d(x, w.float(), stride=s, padding=k // 2)
    (gx,) = torch.autograd.grad(yr, x, dy.float().permute(0, 3, 1, 2))
    ref = gx.permute(0, 2, 3, 1)
    if k == 1 and s == 2:
        base = _rand(B, H, W, Cin, seed=5)
        out = base.clone()
        dx = ops.conv2d_dgrad(dy, wd, (H, W), k, s, residual=out, out=out)
        ref = ref + base.float()
    else:
        res = _rand(B, H, W, Cin, seed=6)
        dx = ops.conv2d_dgrad(dy, wd, (H, W), k, s, residual=res)
        ref = ref + res.float()
    _close(dx, ref, 1e-2, 2e-2, "conv dgrad")


@pytest.mark.parametrize("B,H,W,Cin,Cout,k,s", CONV_CASES)
def test_conv_wgrad(B, H, W, Cin, Cout, k, s):
    ops = _ops()
    x = _rand(B, H, W, Cin, seed=7)
    Ho, Wo = ops.out_hw(H, k, s), ops.out_hw(W, k, s)
    dy = _rand(B, Ho, Wo, Cout, seed=8)
    w = torch.zeros(Cout, Cin, k, k, device="cuda", requires_grad=True)
    torch.backends.cudnn.allow_tf32 = False
    yr = F.conv2d(x.float().permute(0, 3, 1, 2), w, stride=s, padding=k // 2)
    (gw,) = torch.autograd.grad(yr, w, dy.float().permute(0, 3, 1, 2))
    dw = ops.conv2d_wgrad(dy, x, k, s)
    scale = float(gw.abs().max()) + 1e-6
    _close(dw / scale, gw / scale, 1e-3, 2e-3, "conv wgrad")


def test_linear_epilogues():
    ops = _ops()
    M, K, N = 300, 200, 136
    x = _rand(M, 1, 1, K, seed=11)
    w = _rand(N, K, scale=K ** -0.5, seed=12)
    b = torch.randn(N, device="cuda")
    res = _rand(M, 1, 1, N, seed=13)
    wp = ops.pack_weight(w.float())
    ref = x.float().reshape(M, K) @ w.float().t() + b
    y, _ = ops.conv2d_fwd(x, wp, bias=b, act=2, residual=res)
    _close(y.reshape(M, N), F.gelu(ref) + res.float().reshape(M, N), 1e-2, 1e-2, "bias+gelu+res")
    y, _ = ops.conv2d_fwd(x, wp, bias=b, act=1)
    _close(y.reshape(M, N), F.relu(ref), 1e-2, 1e-2, "bias+relu")
    y, _ = ops.conv2d_fwd(x, wp, bias=b, out_f32=True)
    _close(y.reshape(M, N), ref, 1e-4, 1e-4, "fp32 out")


@pytest.mark.parametrize("rows,C", [(2 * 56 * 56, 64), (1000, 256), (98, 2048)])
def test_batchnorm_train_fwd_bwd(rows, C):
    ops = _ops()
    x = _rand(rows, 1, 1, C, seed=21) * 1.5 + 0.3
    x = x.to(torch.bfloat16)
    g = _rand(rows, 1, 1, C, seed=22)
    res = _rand(rows, 1, 1, C, seed=23)
    gamma = torch.rand(C, device="cuda") + 0.5
    beta = torch.randn(C, device="cuda") * 0.1
    # identity-weight 1x1 conv just to get the statistics partials through the real epilogue path
    eye = torch.eye(C, device="cuda").reshape(C, C, 1, 1)
    y_raw, stats = ops.conv2d_fwd(x, ops.pack_weight(eye), want_stats=True)
    assert torch.equal(y_raw, x)
    rm, rv = torch.zeros(C, device="cuda"), torch.ones(C, device="cuda")
    nbt = torch.zeros((), dtype=torch.int64, device="cuda")
    co = ops.bn_finalize(stats, rows, gamma, beta, 1e-5, 0.1, rm, rv, nbt)
    xr = x.float().reshape(rows, C).clone().requires_grad_(True)
    gr, br = gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True)
    rm2, rv2 = torch.zeros(C, device="cuda"), torch.ones(C, device="cuda")
    bn = F.batch_norm(xr, rm2, rv2, gr, br, True, 0.1, 1e-5)
    _close(rm, rm2, 1e-4, 1e-5, "running_mean")
    _close(rv, rv2, 1e-4, 1e-5, "running_var")
    assert int(nbt) == 1
    for use_res in (False, True):
        out_ref = F.relu(bn + res.float().reshape(rows, C)) if use_res else F.relu(bn)
        y = ops.bn_apply(x, co, relu=True, residual=res if use_res else None)
        _close(y.reshape(rows, C), out_ref, 1e-2, 1e-2, "bn apply")
        gx, ggam, gbet = torch.autograd.grad(out_ref, (xr, gr, br), g.float().reshape(rows, C), retain_graph=True)
        dx, dgam, dbet, dz = ops.bn_backward(g, x, co, relu=True, y_out=y if use_res else None, want_dz=use_res)
        # masks can differ where the bf16 output rounds to exactly 0; tolerate through norms
        sc = float(gx.abs().max())
        assert float((dx.float().reshape(rows, C) - gx).abs().max()) < 0.05 * sc + 1e-3
        _close(dgam, ggam, 2e-2, 2e-2 * float(ggam.abs().max()), "dgamma")
        _close(dbet, gbet, 2e-2, 2e-2 * float(gbet.abs().max()), "dbeta")


@pytest.mark.parametrize("B,H,W,C", [(2, 16, 16, 64), (3, 14, 10, 64), (2, 7, 9, 64), (5, 56, 56, 64)])
def test_stem_pool_and_avgpool(B, H, W, C):
    ops = _ops()
    x = _rand(B, H, W, C, seed=31)
    co = ops.BnCoeffs(C, "cuda")
    co.scale.copy_(torch.rand(C, device="cuda") + 0.5)
    co.shift.copy_(torch.randn(C, device="cuda") * 0.2)
    y, idx = ops.bn_relu_maxpool_fwd(x, co)
    a = F.relu(x.float() * co.scale + co.shift).to(torch.bfloat16).float().permute(0, 3, 1, 2).requires_grad_(True)
    ref = F.max_pool2d(a, 3, 2, 1)
    assert torch.equal(y.float(), ref.permute(0, 2, 3, 1))
    g = _rand(B, (H - 1) // 2 + 1, (W - 1) // 2 + 1, C, seed=32)
    (ga,) = torch.autograd.grad(ref, a, g.float().permute(0, 3, 1, 2))
    gin = ops.maxpool_bwd(g, idx, (H, W))
    # ties between equal bf16 activations may route to a different (equal-valued) element: compare window sums
    # (every input gradient is rounded to bf16 once: the noise of a sum over H*W entries grows with sqrt(H*W))
    _close(gin.float().sum((1, 2)), ga.permute(0, 2, 3, 1).sum((1, 2)), 1e-2, 5e-2 + 4e-3 * (H * W) ** 0.5, "maxpool bwd mass")
    nz = (a.permute(0, 2, 3, 1) > 0)
    match = ((gin.float() - ga.permute(0, 2, 3, 1)).abs() < 1e-2) | ~nz
    assert match.float().mean() > 0.98
    z = _rand(3, 7, 7, 128, seed=33)
    p = ops.avgpool_fwd(z)
    _close(p, z.float().mean((1, 2)), 1e-2, 1e-2, "avgpool")
    gz = ops.avgpool_bwd(p, (7, 7))
    _close(gz, (p.float() / 49)[:, None, None, :].expand(3, 7, 7, 128), 1e-2, 1e-3, "avgpool bwd")


def test_softmax_xent_and_sgd():
    ops = _ops()
    B, N = 37, 1000
    logits = torch.randn(B, N, device="cuda") * 3
    labels = torch.randint(0, N, (B,), device="cuda")
    lr_ = logits.clone().requires_grad_(True)
    ref = F.cross_entropy(lr_, labels)
    (gl,) = torch.autograd.grad(ref, lr_)
    loss, d, correct = ops.softmax_xent(logits, labels)
    assert abs(float(loss) - float(ref)) < 1e-4
    _close(d[:, :N], gl, 1e-2, 1e-5, "dlogits")
    assert torch.equal(correct.bool(), logits.argmax(1) == labels)
    n = 100003
    p = torch.randn(n, device="cuda")
    g = torch.randn(n, device="cuda")
    pr = p.clone().requires_grad_(True)
    opt = torch.optim.SGD([pr], lr=0.1, momentum=0.9, weight_decay=5e-5)
    buf = torch.zeros(n, device="cuda")
    for step in range(3):
        pr.grad = g.clone()
        opt.step()
        ops.sgd_momentum_(p, g, buf, 0.1, 0.9, 5e-5, first_step=(step == 0))
    _close(p, pr.detach(), 1e-5, 1e-6, "sgd")


def test_stem_im2col():
    ops = _ops()
    x = torch.randn(2, 3, 32, 32, device="cuda")
    w = torch.randn(64, 3, 7, 7, device="cuda") * 0.1
    a, Ho, Wo = ops.im2col_nchw(x, 7, 7, 2, 3, 160)
    wp = ops.pack_weight(w, ld=160)
    y, _ = ops.conv2d_fwd(a.reshape(-1, 1, 1, 160), wp)
    ref = F.conv2d(x.to(torch.bfloat16).float(), w.to(torch.bfloat16).float(), stride=2, padding=3).permute(0, 2, 3, 1)
    _close(y.reshape(2, Ho, Wo, 64), ref, 1e-2, 1e-2, "stem conv")


@pytest.mark.parametrize("B,H,W", [(2, 224, 224), (3, 64, 96), (1, 32, 32)])
def test_stem_space_to_depth_conv(B, H, W):
    """conv1 7x7/2/pad3 (3 -> 64) through the space-to-depth operand and overlapping TMA rows: forward, BN statistics
    partials and weight gradient against F.conv2d on the bf16-rounded operands."""
    ops = _ops()
    from deeplearning_b200 import _lib

    x = torch.randn(B, 3, H, W, device="cuda")
    w = torch.randn(64, 3, 7, 7, device="cuda") * 0.1
    z = ops.stem_s2d(x)
    assert z.shape == (B, H // 2 + 3, W // 2 + 3, 16)
    xp = F.pad(x, (3, 3, 3, 3)).to(torch.bfloat16)
    for dy in range(2):
        for dx in range(2):
            for c in range(3):
                assert torch.equal(z[..., (dy * 2 + dx) * 3 + c], xp[:, c, dy::2, dx::2][:, :H // 2 + 3, :W // 2 + 3])
    assert float(z[..., 12:].abs().max()) == 0.0
    # pack through the multi-tensor packer (mode 2)
    lib = _lib.load()
    wp = torch.empty(64, 256, dtype=torch.bfloat16, device="cuda")
    table = torch.tensor([[w.data_ptr(), wp.data_ptr(), 64, 3, 49, 2, 256, 0, 64, 0]], dtype=torch.int64, device="cuda")
    _lib.check(lib.b200_pack_weights_multi(table.data_ptr(), 1, 64, torch.cuda.current_stream().cuda_stream), "pack")
    y, stats = ops.stem_s2d_conv_fwd(z, wp, want_stats=True)
    xr = x.to(torch.bfloat16).float().requires_grad_(True)
    wr = w.to(torch.bfloat16).float().requires_grad_(True)
    ref = F.conv2d(xr, wr, stride=2, padding=3)
    _close(y, ref.permute(0, 2, 3, 1), 1e-2, 2e-2, "stem conv fwd")
    yf = y.float().reshape(-1, 64)
    _close(stats[:, 0].sum(0), yf.sum(0), 1e-3, 1e-1, "stem stats sum")
    _close(stats[:, 1].sum(0), (yf * yf).sum(0), 1e-3, 1e-1, "stem stats sumsq")
    dy_ = _rand(B, H // 2, W // 2, 64, seed=5)
    (gw,) = torch.autograd.grad(ref, wr, dy_.float().permute(0, 3, 1, 2))
    dw = ops.stem_s2d_conv_wgrad(dy_, z)
    sc = float(gw.abs().max())
    _close(dw / sc, gw / sc, 2e-3, 2e-3, "stem conv wgrad")


@pytest.mark.parametrize("O,I,kh,mode,ld_pad,rows_pad,scaled", [
    (64, 64, 3, 0, 0, 0, False), (64, 64, 3, 1, 0, 0, False), (192, 96, 1, 0, 0, 0, False), (192, 96, 1, 1, 0, 0, True),
    (40, 72, 1, 1, 8, 0, False), (1000, 2048, 1, 0, 0, 24, False), (128, 128, 3, 1, 16, 0, True), (96, 48, 2, 0, 8, 32, True),
    (96, 48, 2, 1, 0, 0, False), (33, 17, 3, 1, 7, 3, False), (24, 3, 7, 0, 13, 0, False), (24, 3, 7, 1, 0, 0, False)])
def test_pack_weights_multi_matches_single(O, I, kh, mode, ld_pad, rows_pad, scaled):
    """The one-launch model packer (shared-memory tiled layouts) == the plain per-tensor packer, padding zeroed."""
    from deeplearning_b200 import _lib
    ops = _ops()
    lib = _lib.load()
    torch.manual_seed(O * 131 + I)
    ws = [torch.randn(O, I, kh, kh, device="cuda"), torch.randn(O + 8, I, kh, kh, device="cuda")]
    scales = [torch.rand(w.shape[0], device="cuda") + 0.5 for w in ws]
    rows, outs, first = [], [], 0
    for w, sc in zip(ws, scales):
        o = w.shape[0]
        taps = kh * kh
        nrow = (o if mode == 0 else I) + rows_pad
        ld = taps * (I if mode == 0 else o) + ld_pad
        dst = torch.full((nrow, ld), 7.0, dtype=torch.bfloat16, device="cuda")
        outs.append(dst)
        rows.append([w.data_ptr(), dst.data_ptr(), o, I, taps, mode, ld, first, nrow, sc.data_ptr() if scaled else 0])
        first += 5
    table = torch.tensor(rows, dtype=torch.int64, device="cuda")
    _lib.check(lib.b200_pack_weights_multi(table.data_ptr(), len(rows), first, torch.cuda.current_stream().cuda_stream), "pack")
    for w, sc, dst in zip(ws, scales, outs):
        o = w.shape[0]
        ref = ops.pack_weight(w * sc.view(-1, 1, 1, 1) if scaled else w, mode=mode)
        nrow, ncol = ref.shape
        assert torch.equal(dst[:nrow, :ncol], ref)
        assert float(dst[nrow:].float().abs().max() if dst.shape[0] > nrow else 0.0) == 0.0
        assert float(dst[:, ncol:].float().abs().max() if dst.shape[1] > ncol else 0.0) == 0.0


@pytest.mark.parametrize("B,H,W,Cin,Cout,k,s", [(3, 9, 7, 64, 200, 1, 1), (4, 14, 14, 96, 384, 1, 1), (2, 16, 16, 64, 64, 3, 1),
                                                  (2, 14, 14, 96, 192, 2, 2), (37, 1, 1, 768, 2304, 1, 1),
                                                  (256, 197, 1, 768, 2304, 1, 1)])
def test_wgrad_bias_sums_from_the_dy_tiles(B, H, W, Cin, Cout, k, s):
    """conv2d_wgrad(bias_out=...) = column sums of dy (the layer's bias gradient), added up by the extra warps of the wgrad
    kernel from the dy tiles it already stages in shared memory; the weight gradient itself is unchanged.  The ViT-B/16 qkv
    shape (bs 256) has more work items than SMs, so CTAs run several items, some of whose tiles they do not sum."""
    from deeplearning_b200 import ops

    g = torch.Generator(device="cuda").manual_seed(5)
    x = torch.randn(B, H, W, Cin, device="cuda", generator=g).to(torch.bfloat16)
    Ho, Wo = ops.out_hw(H, k, s), ops.out_hw(W, k, s)
    dy = torch.randn(B, Ho, Wo, Cout, device="cuda", generator=g).to(torch.bfloat16)
    ref_w = ops.conv2d_wgrad(dy, x, k, s)
    bias = torch.full((Cout,), float("nan"), device="cuda")
    got_w = ops.conv2d_wgrad(dy, x, k, s, bias_out=bias)
    assert torch.equal(ref_w, got_w)
    ref_b = dy.double().sum((0, 1, 2))
    err = float((bias.double() - ref_b).abs().max())
    assert err <= 1e-5 * float(dy.double().abs().sum((0, 1, 2)).max()), err   # fp32 sums of the same values: ~1e-8 of it
    again = torch.full((Cout,), float("nan"), device="cuda")
    ops.conv2d_wgrad(dy, x, k, s, bias_out=again)
    assert torch.equal(bias, again)   # fixed summation order


def _bn_coeffs(ops, c, gamma, beta):
    """BnCoeffs of train-mode BatchNorm over the raw conv output c (bf16 NHWC)."""
    C = c.shape[-1]
    cf = c.float().reshape(-1, C)
    co = ops.BnCoeffs(C, c.device)
    co.mean.copy_(cf.mean(0))
    co.invstd.copy_((cf.var(0, unbiased=False) + 1e-5).rsqrt())
    co.scale.copy_(gamma * co.invstd)
    co.shift.copy_(beta - co.mean * co.scale)
    return co


@pytest.mark.parametrize("B,H,W,Cin,Cout,k", [(4, 56, 56, 64, 64, 3), (3, 14, 14, 256, 256, 3), (2, 9, 11, 128, 128, 3),
                                               (2, 28, 28, 128, 512, 1)])
def test_dgrad_with_fused_bn_backward_reduce(B, H, W, Cin, Cout, k):
    """conv2d_dgrad(bn_mask=(c, co)): the dgrad epilogue masks its output with relu'(bn(c)) and sums dz, dz * c per channel -
    bn_backward_from_sums then gives the same dx / dgamma / dbeta as the two-pass bn_backward on the unmasked gradient."""
    from deeplearning_b200 import ops

    dy = _rand(B, H, W, Cout, seed=3)
    w = _rand(Cout, Cin, k, k, scale=(Cout * k * k) ** -0.5, seed=4)
    wd = ops.pack_weight(w.float(), mode=1)
    c = _rand(B, H, W, Cin, seed=5) + 0.25
    g = torch.Generator(device="cuda").manual_seed(6)
    gamma = torch.rand(Cin, device="cuda", generator=g) + 0.5
    beta = torch.randn(Cin, device="cuda", generator=g) * 0.3
    co = _bn_coeffs(ops, c, gamma, beta)
    g_ref = ops.conv2d_dgrad(dy, wd, (H, W), k, 1)
    dx_ref, dgamma_ref, dbeta_ref, dz_ref = ops.bn_backward(g_ref, c, co, relu=True, want_dz=True)
    dz, sums = ops.conv2d_dgrad(dy, wd, (H, W), k, 1, bn_mask=(c, co))
    assert torch.equal(dz, dz_ref)
    dx, dgamma, dbeta = ops.bn_backward_from_sums(dz, sums, c, co)
    scale = float(dgamma_ref.abs().max())
    assert torch.allclose(dbeta, dbeta_ref, rtol=1e-3, atol=1e-3 * float(dbeta_ref.abs().max()))
    assert torch.allclose(dgamma, dgamma_ref, rtol=2e-3, atol=2e-3 * scale), float((dgamma - dgamma_ref).abs().max())
    _close(dx, dx_ref, 2e-2, 2e-2 * float(dx_ref.float().abs().max()), "dx")


def test_dual_gemm_with_fused_bn_backward_reduce():
    from deeplearning_b200 import ops

    px, K0, K1, N = 2 * 28 * 28, 512, 128, 128
    a0, a1 = _rand(2, 28, 28, K0, seed=1), _rand(2, 28, 28, K1, seed=2)
    wcat = _rand(N, K0 + K1, scale=(K0 + K1) ** -0.5, seed=3)
    bias = _rand(N, seed=4).float()
    c = _rand(2, 28, 28, N, seed=5)
    co = _bn_coeffs(ops, c, torch.ones(N, device="cuda"), torch.zeros(N, device="cuda"))
    g_ref = ops.gemm_dual(a0, a1, wcat, bias)
    dx_ref, dgamma_ref, dbeta_ref, dz_ref = ops.bn_backward(g_ref, c, co, relu=True, want_dz=True)
    dz, sums = ops.gemm_dual(a0, a1, wcat, bias, bn_mask=(c, co))
    assert torch.equal(dz, dz_ref)
    dx, dgamma, dbeta = ops.bn_backward_from_sums(dz, sums, c, co)
    assert torch.allclose(dbeta, dbeta_ref, rtol=1e-3, atol=1e-3 * float(dbeta_ref.abs().max()))
    assert torch.allclose(dgamma, dgamma_ref, rtol=2e-3, atol=2e-3 * float(dgamma_ref.abs().max()))
    _close(dx, dx_ref, 2e-2, 2e-2 * float(dx_ref.float().abs().max()), "dx")
