"""The persistent kernels at shapes where each CTA runs several work items, against fp64 references.

Almost every hot kernel here is persistent: the grid is capped at the SM count and each CTA loops over tiles, window pairs
or row blocks, carrying ring positions, mbarrier phases, the double-buffered TMEM accumulator and per-CTA statistics from
one item to the next.  None of that state matters until a CTA runs its second item, so every case below

* computes, with the same rules as the dispatch code, how many items each CTA (or CTA pair) runs and asserts that the case
  reaches the multi-item path (printed as "items/CTA");
* compares with an fp64 reference computed on the exact operands the kernel read (bf16 inputs, fp32 vectors, the kernel's
  own bf16 intermediates), under an error bound  |got - ref| <= u_out |ref| + c S + floor  where S is the same computation
  over absolute values; no element may exceed its bound, and the largest err / bound is printed;
* calls the kernel twice on the same inputs and requires identical bits (DESIGN.md section 4), partial statistics included.

Bounds: u_out = 2^-8 for bf16 outputs and 2^-23 for fp32 ones; c = 2^-16 for fp32-accumulated GEMMs (about 16x the typical
accumulation error at K <= 4608, while any tile-level mistake is of order S / sqrt(K)); per-CTA column sums are compared
with fp64 sums of the kernel's own stored output at 2^-18 of the absolute-value sum.  Window attention multiplies bf16
probabilities and bf16 dS tiles on the tensor core by design, which puts its error near 2^-9 S: it uses c = 2^-7, and its
log-sum-exp, a log of summed bf16 exponentials, gets an absolute floor of 2^-8 log2(e).

Run with -s to see the item counts and err / bound ratios.
"""
import math
import os
import subprocess
import sys

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

F64 = torch.float64
BF16 = torch.bfloat16
U_BF16 = 2.0 ** -8
U_F32 = 2.0 ** -23
C_GEMM = 2.0 ** -16
C_SUM = 2.0 ** -18
C_ATTN = 2.0 ** -7


def _ops():
    from deeplearning_b200 import ops

    return ops


def _lib():
    from deeplearning_b200 import _lib

    return _lib.load()


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _rand(*shape, scale=1.0, seed=0, dtype=BF16):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.randn(*shape, device="cuda", generator=g) * scale).to(dtype)


def _items(what, least, most=None, need=3):
    """Report the items per CTA of a case and fail if the case no longer reaches the multi-item path."""
    most = least if most is None else most
    print(f"\n  {what}: items/CTA {least}..{most}", flush=True)
    assert least >= need, f"{what}: only {least} items per CTA (need >= {need}); the case no longer tests the persistent loop"


def _check(what, got, ref, S, u_out, c=C_GEMM, floor=0.0, keep=None):
    """Every element within u_out |ref| + c S + floor (optionally only where `keep`); prints the largest err / bound."""
    err = (got.double() - ref).abs()
    bound = u_out * ref.abs() + c * S + floor
    if keep is not None:
        err, bound = err[keep], bound[keep]
    ratio = torch.where(err == 0, torch.zeros_like(err), err / bound)
    worst = float(ratio.max()) if ratio.numel() else 0.0
    print(f"  {what}: max err/bound {worst:.3g}", flush=True)
    if not worst <= 1.0:
        bad = ratio > 1
        raise AssertionError(f"{what}: {int(bad.sum())}/{bad.numel()} elements over the bound, max err/bound {worst:.3g}, "
                             f"max err {float(err.max()):.4g}, max |ref| {float(ref.abs().max()):.4g}")


def _same(what, a, b):
    for i, (x, y) in enumerate(zip(a, b)):
        if x is None:
            continue
        assert torch.equal(x, y), f"{what}: output {i} differs between two calls on the same inputs"


def _mm64(a, w, chunk=1 << 14):
    """(a @ w^T, |a| @ |w|^T) in fp64 for bf16 a [rows, K] and w [N, K], in row chunks."""
    w64 = w.double()
    wa = w64.abs()
    rows = a.shape[0]
    ref = torch.empty(rows, w.shape[0], dtype=F64, device=a.device)
    S = torch.empty_like(ref)
    for r0 in range(0, rows, chunk):
        a64 = a[r0:r0 + chunk].double()
        ref[r0:r0 + chunk] = a64 @ w64.t()
        S[r0:r0 + chunk] = a64.abs() @ wa.t()
    return ref, S


# ------------------------------------------------------------------------------------------------- tile geometry (host rules)
def _choose_box(d1, d2, d3, P=128):
    """abi_conv.cu choose_box: the (w, h, n) pixel box of one tile."""
    best, best_cost = (P, 1, 1), -1.0
    b1 = 1
    while b1 <= P:
        b2 = 1
        while b1 * b2 <= P:
            b3 = P // (b1 * b2)
            if b1 <= 256 and b2 <= 256 and b3 <= 256:
                cost = float(-(-d1 // b1) * b1) * (-(-d2 // b2) * b2) * (-(-d3 // b3) * b3)
                if best_cost < 0 or cost < best_cost - 0.5 or (
                        cost < best_cost + 0.5 and (b1 > best[0] or (b1 == best[0] and b2 > best[1]))):
                    best_cost, best = cost, (b1, b2, b3)
            b2 <<= 1
        b1 <<= 1
    return best


class _Geom:
    """Tile schedule of one conv_gemm_kernel launch: output view dims (d1 = w, d2 = h, d3 = n), N channels, grid in CTAs
    (pair: in CTA pairs)."""

    def __init__(self, dims, N, stats, pair=False):
        self.dims, self.N, self.pair = dims, N, pair
        self.box = _choose_box(*dims)
        self.tiles = [-(-d // b) for d, b in zip(dims, self.box)]
        self.m_tiles = self.tiles[0] * self.tiles[1] * self.tiles[2]
        self.BN = 64 if N <= 64 else (128 if N <= 128 else 256)
        self.n_tiles = -(-N // self.BN)
        sms = _sms()
        if pair:
            self.items = (self.m_tiles + 1) // 2 * self.n_tiles
            g = min(sms // 2, self.items)
        else:
            self.items = self.m_tiles * self.n_tiles
            g = min(sms, self.items)
        self.grid = g // self.n_tiles * self.n_tiles if stats else g
        self.split = self.BN == 64   # one 64-column unit per tile: the two warps of a quadrant take turns at tiles

    def per_cta(self):
        return self.items // self.grid, -(-self.items // self.grid)

    def stat_rows(self):
        return self.grid // self.n_tiles * (8 if self.split else 4) * (2 if self.pair else 1)

    def row_pixels(self):
        """[m_tiles, 128] flat output pixel of every tile row ((n * h + y) * w + x), -1 outside the tensor."""
        dev = "cuda"
        b1, b2, b3 = self.box
        t1, t2, _ = self.tiles
        m = torch.arange(self.m_tiles, device=dev)[:, None]
        r = torch.arange(128, device=dev)[None, :]
        p1 = (m % t1) * b1 + r % b1
        p2 = (m // t1 % t2) * b2 + r // b1 % b2
        p3 = (m // (t1 * t2)) * b3 + r // (b1 * b2)
        d1, d2, d3 = self.dims
        ok = (p1 < d1) & (p2 < d2) & (p3 < d3)
        return torch.where(ok, (p3 * d2 + p2) * d1 + p1, torch.full_like(p1, -1))

    def expected_rows(self, plane0, plane1):
        """fp64 partial-statistics rows [T, 2, N] that the epilogue warps should write: each (CTA, quadrant[, warp]) row sums
        the stored rows of exactly the tiles that CTA ran.  plane0 / plane1: fp64 [pixels, N] per-element terms."""
        T = self.stat_rows()
        out = torch.zeros(T, 2, self.N, dtype=F64, device="cuda")
        pix = self.row_pixels()                                   # [m, 128]
        quad = torch.arange(128, device="cuda")[None, :] // 32
        m = torch.arange(self.m_tiles, device="cuda")[:, None]
        for nt in range(self.n_tiles):
            if self.pair:
                item = (m // 2) * self.n_tiles + nt
                unit, it = item % self.grid, item // self.grid
                grp = (unit // self.n_tiles) * 2 + (m % 2)
            else:
                item = m * self.n_tiles + nt
                unit, it = item % self.grid, item // self.grid
                grp = unit // self.n_tiles
            srow = (grp * 4 + quad) * 2 + (it % 2) if self.split else grp * 4 + quad
            srow = srow.expand_as(pix)
            ok = pix >= 0
            c0, c1 = nt * self.BN, min(self.N, (nt + 1) * self.BN)
            src = pix[ok]
            dst = srow[ok]
            out[:, 0, c0:c1].index_add_(0, dst, plane0[src, c0:c1])
            out[:, 1, c0:c1].index_add_(0, dst, plane1[src, c0:c1])
        return out


def _check_stat_rows(what, geom, stats, plane0, plane1):
    """Row by row: each partial row against what its CTA's tiles should sum to (2^-18 of the absolute-value sums)."""
    assert stats.shape == (geom.stat_rows(), 2, geom.N), (stats.shape, geom.stat_rows())
    ref = geom.expected_rows(plane0, plane1)
    absr = geom.expected_rows(plane0.abs(), plane1.abs())
    _check(what + " partial rows", stats, ref, absr, U_F32, c=C_SUM)


# ------------------------------------------------------------------------------------------------- convolution references
def _conv_fwd64(x, w, k, s, chunk=8):
    """fp64 (conv(x, w), conv(|x|, |w|)) NHWC for bf16 x [B,H,W,C] and w [O,C,k,k], padding k // 2, via unfold + matmul."""
    B, H, W, C = x.shape
    O = w.shape[0]
    pad = k // 2
    Ho, Wo = (H + 2 * pad - k) // s + 1, (W + 2 * pad - k) // s + 1
    wm = w.double().reshape(O, -1)
    wa = wm.abs()
    ref = torch.empty(B, Ho, Wo, O, dtype=F64, device=x.device)
    S = torch.empty_like(ref)
    for b0 in range(0, B, chunk):
        xc = x[b0:b0 + chunk].double().permute(0, 3, 1, 2)
        cols = F.unfold(xc, k, padding=pad, stride=s)             # [b, C*k*k, L], k index = (c, kh, kw)
        n = xc.shape[0]
        ref[b0:b0 + n] = (wm @ cols).view(n, O, Ho, Wo).permute(0, 2, 3, 1)
        S[b0:b0 + n] = (wa @ cols.abs()).view(n, O, Ho, Wo).permute(0, 2, 3, 1)
    return ref, S


def _conv_dgrad64(dy, w, k, s, hw, chunk=8):
    """fp64 data gradient (and its absolute-value version) of conv(x, w) for dy [B,Ho,Wo,O]: fold(W^T dy), the exact adjoint."""
    B, Ho, Wo, O = dy.shape
    H, W = hw
    C = w.shape[1]
    pad = k // 2
    wt = w.double().reshape(O, -1).t()
    wta = wt.abs()
    ref = torch.empty(B, H, W, C, dtype=F64, device=dy.device)
    S = torch.empty_like(ref)
    for b0 in range(0, B, chunk):
        d = dy[b0:b0 + chunk].double().permute(0, 3, 1, 2).reshape(-1, O, Ho * Wo)
        n = d.shape[0]
        ref[b0:b0 + n] = F.fold(wt @ d, (H, W), k, padding=pad, stride=s).permute(0, 2, 3, 1)
        S[b0:b0 + n] = F.fold(wta @ d.abs(), (H, W), k, padding=pad, stride=s).permute(0, 2, 3, 1)
    return ref, S


def _bn_coeffs(ops, C, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    co = ops.BnCoeffs(C, "cuda")
    co.mean.copy_(torch.randn(C, device="cuda", generator=g) * 0.2)
    co.invstd.copy_(torch.rand(C, device="cuda", generator=g) + 0.5)
    gamma = torch.rand(C, device="cuda", generator=g) + 0.5
    co.scale.copy_(gamma * co.invstd)
    co.shift.copy_(torch.randn(C, device="cuda", generator=g) * 0.3 - co.mean * co.scale)
    return co


def _relu_mask64(xraw, scale, shift):
    """relu'(x * scale + shift) in fp64, and the positions whose pre-activation lies within fp32 rounding of zero."""
    x = xraw.double()
    t = x * scale.double() + shift.double()
    amb = t.abs() <= 2.0 ** -22 * ((x * scale.double()).abs() + shift.double().abs())
    return t > 0, amb


# ================================================================================================= A. conv_gemm_kernel, generic
def test_conv1x1_block64_fwd_stats_tiles_in_turns():
    """conv_gemm_kernel<64, kEpiStats>: 1x1 256->64 (layer1 conv1, bs 32, 784 tiles on 148 CTAs); the two warps of a quadrant
    take turns at tiles and write separate partial rows, each checked against the tiles it stored."""
    ops = _ops()
    B, H, W, Cin, Cout = 32, 56, 56, 256, 64
    x = _rand(B, H, W, Cin, seed=1)
    w = _rand(Cout, Cin, 1, 1, scale=Cin ** -0.5, seed=2)
    wp = ops.pack_weight(w.float())
    geom = _Geom((B * H * W, 1, 1), Cout, stats=True)
    assert geom.split
    _items("conv 1x1 256->64 fwd+stats", *geom.per_cta())
    y, st = ops.conv2d_fwd(x, wp, 1, 1, want_stats=True)
    y2, st2 = ops.conv2d_fwd(x, wp, 1, 1, want_stats=True)
    _same("conv 1x1 fwd", (y, st), (y2, st2))
    ref, S = _mm64(x.view(-1, Cin), w.view(Cout, Cin))
    _check("y", y.view(-1, Cout), ref, S, U_BF16)
    yv = y.view(-1, Cout).double()
    _check_stat_rows("stats", geom, st, yv, yv * yv)

    # one production-count statistics buffer (hundreds of partial rows) through bn_finalize, against fp64
    T = st.shape[0]
    assert T >= 500, T
    n = yv.shape[0]
    g = torch.Generator(device="cuda").manual_seed(3)
    gamma = torch.rand(Cout, device="cuda", generator=g) + 0.5
    beta = torch.randn(Cout, device="cuda", generator=g) * 0.1
    rm0 = torch.randn(Cout, device="cuda", generator=g) * 0.1
    rv0 = torch.rand(Cout, device="cuda", generator=g) + 0.5
    rm, rv = rm0.clone(), rv0.clone()
    nbt = torch.zeros((), dtype=torch.int64, device="cuda")
    co = ops.bn_finalize(st, n, gamma, beta, 1e-5, 0.1, rm, rv, nbt)
    s1, s2 = yv.sum(0), (yv * yv).sum(0)
    a1, a2 = yv.abs().sum(0), s2
    mean = s1 / n
    var = s2 / n - mean * mean
    # partial sums are good to 2^-18 of their absolute sums: propagate through mean / var / invstd
    e_mean = C_SUM * a1 / n
    e_var = C_SUM * (a2 + 2 * mean.abs() * a1) / n
    invstd = (var + 1e-5).rsqrt()
    # (c = 1: the second argument after the reference is the whole absolute error allowance)
    _check("bn mean", co.mean, mean, e_mean, U_F32, c=1.0)
    _check("bn invstd", co.invstd, invstd, 0.5 * invstd * e_var / (var + 1e-5), 2 * U_F32, c=1.0)
    _check("running_mean", rm, 0.9 * rm0.double() + 0.1 * mean, 0.1 * e_mean + 2 * U_F32 * rm0.double().abs(), U_F32, c=1.0)
    _check("running_var", rv, 0.9 * rv0.double() + 0.1 * var * n / (n - 1),
           0.1 * e_var * n / (n - 1) + 2 * U_F32 * rv0.double().abs(), U_F32, c=1.0)
    assert int(nbt) == 1


def test_conv3x3_block64_dgrad_bn_mask_tiles_in_turns():
    """conv_gemm_kernel<64, kEpiBnMask> (the resident-weight tap64 kernel does not take it): 3x3 64->64 dgrad of layer1 at
    bs 32 with the fused BatchNorm-backward reduce; spatial boxes with a partial last box (the row-map path)."""
    ops = _ops()
    B, H, W, C = 32, 56, 56, 64
    w = _rand(C, C, 3, 3, scale=(9 * C) ** -0.5, seed=3)
    wd = ops.pack_weight(w.float(), mode=1)
    dy = _rand(B, H, W, C, seed=4)
    c = _rand(B, H, W, C, seed=5)
    co = _bn_coeffs(ops, C, 6)
    geom = _Geom((W, H, B), C, stats=True)
    assert geom.split
    _items("conv 3x3 64->64 dgrad + bn mask", *geom.per_cta())
    dz, st = ops.conv2d_dgrad(dy, wd, (H, W), 3, 1, bn_mask=(c, co))
    dz2, st2 = ops.conv2d_dgrad(dy, wd, (H, W), 3, 1, bn_mask=(c, co))
    _same("dgrad bn_mask", (dz, st), (dz2, st2))
    ref, S = _conv_dgrad64(dy, w, 3, 1, (H, W))
    alive, amb = _relu_mask64(c, co.scale, co.shift)
    n_amb = int(amb.sum())
    print(f"  mask positions within fp32 rounding of zero: {n_amb}")
    assert n_amb < 1e-4 * amb.numel()
    _check("dz", dz, ref * alive, S * alive, U_BF16, keep=~amb)
    dzv = dz.view(-1, C).double()
    _check_stat_rows("bn-backward sums", geom, st, dzv, dzv * c.view(-1, C).double())


def test_conv3x3_block128_stride2_fwd_stats_and_dgrad():
    """conv_gemm_kernel<128>: 3x3 128->128 stride 2 (layer2 conv2, bs 80): forward with statistics (phase-view taps) and the
    data gradient as four phase launches, each with several tiles per CTA."""
    ops = _ops()
    B, H, W, C = 80, 56, 56, 128
    Ho, Wo = 28, 28
    x = _rand(B, H, W, C, seed=7)
    w = _rand(C, C, 3, 3, scale=(9 * C) ** -0.5, seed=8)
    geom = _Geom((Wo, Ho, B), C, stats=True)
    _items("conv 3x3/2 128->128 fwd+stats", *geom.per_cta())
    # every dgrad phase launch writes a (28 x 28 x B) view
    gd = _Geom((W // 2, H // 2, B), C, stats=False)
    _items("conv 3x3/2 128->128 dgrad (each of 4 phases)", *gd.per_cta())
    wp = ops.pack_weight(w.float())
    y, st = ops.conv2d_fwd(x, wp, 3, 2, want_stats=True)
    y2, st2 = ops.conv2d_fwd(x, wp, 3, 2, want_stats=True)
    _same("conv 3x3/2 fwd", (y, st), (y2, st2))
    ref, S = _conv_fwd64(x, w, 3, 2)
    _check("y", y, ref, S, U_BF16)
    yv = y.view(-1, C).double()
    _check_stat_rows("stats", geom, st, yv, yv * yv)
    del ref, S
    dy = _rand(B, Ho, Wo, C, seed=9)
    wd = ops.pack_weight(w.float(), mode=1)
    dx = ops.conv2d_dgrad(dy, wd, (H, W), 3, 2)
    _same("conv 3x3/2 dgrad", (dx,), (ops.conv2d_dgrad(dy, wd, (H, W), 3, 2),))
    ref, S = _conv_dgrad64(dy, w, 3, 2, (H, W))
    _check("dx", dx, ref, S, U_BF16)


def test_conv1x1_block256_fwd_stats_affine_and_partial_n():
    """conv_gemm_kernel<256>: 1x1 512->2048 (layer4 conv3, bs 160 = 7840 pixels: a partial last pixel tile) with statistics
    (n_tiles = 8, grid 144), the same layer in eval mode (kEpiAffine + residual + ReLU), and a 2048 -> 1000 1x1 whose last
    channel block is partial on every lap."""
    ops = _ops()
    P, Cin, Cout = 160 * 49, 512, 2048
    x = _rand(160, 7, 7, Cin, seed=10)
    w = _rand(Cout, Cin, 1, 1, scale=Cin ** -0.5, seed=11)
    wp = ops.pack_weight(w.float())
    geom = _Geom((P, 1, 1), Cout, stats=True)
    assert geom.grid == 144 and P % 128 != 0
    _items("conv 1x1 512->2048 fwd+stats", *geom.per_cta())
    y, st = ops.conv2d_fwd(x, wp, 1, 1, want_stats=True)
    _same("conv 1x1 512->2048", (y, st), ops.conv2d_fwd(x, wp, 1, 1, want_stats=True))
    ref, S = _mm64(x.view(P, Cin), w.view(Cout, Cin))
    _check("y", y.view(P, Cout), ref, S, U_BF16)
    yv = y.view(P, Cout).double()
    _check_stat_rows("stats", geom, st, yv, yv * yv)

    ga = _Geom((P, 1, 1), Cout, stats=False)
    _items("conv 1x1 512->2048 eval affine+residual", *ga.per_cta())
    co = _bn_coeffs(ops, Cout, 12)
    res = _rand(160, 7, 7, Cout, seed=13)
    ya = ops.conv2d_bn_act(x, wp, co, 1, 1, relu=True, residual=res)
    _same("conv bn_act", (ya,), (ops.conv2d_bn_act(x, wp, co, 1, 1, relu=True, residual=res),))
    sc, sh = co.scale.double(), co.shift.double()
    r64 = res.view(P, Cout).double()
    _check("y eval", ya.view(P, Cout), (ref * sc + sh + r64).clamp_min(0), S * sc.abs() + sh.abs() + r64.abs(), U_BF16)
    del ref, S, yv

    Pn, K, N = 112 * 128 + 77, 2048, 1000
    a = _rand(Pn, 1, 1, K, seed=14)
    wn = _rand(N, K, 1, 1, scale=K ** -0.5, seed=15)
    gn = _Geom((Pn, 1, 1), N, stats=False)
    assert N % gn.BN != 0
    _items("conv 1x1 2048->1000 (partial channel block)", *gn.per_cta())
    wnp = ops.pack_weight(wn.float())
    yn, _ = ops.conv2d_fwd(a, wnp, 1, 1)
    _same("conv 2048->1000", (yn,), (ops.conv2d_fwd(a, wnp, 1, 1)[0],))
    ref, S = _mm64(a.view(Pn, K), wn.view(N, K))
    _check("y", yn.view(Pn, N), ref, S, U_BF16)


# ================================================================================================= B. CTA-pair GEMM (ops.gemm)
# ViT-B/16 linear layers (D = 768) at 19323 token rows: 151 pixel tiles (odd: the last pair's peer tile is a phantom past the
# tensor, reached on a later lap), and the ConvNeXt pwconv2 epilogue at C = 384 on 221 pixel tiles (also odd).
_R, _R384 = 128 * 151 - 5, 128 * 221 - 5


def _pair_inputs(name):
    d, h = 768, 3072
    seed = sum(map(ord, name))
    if name == "qkv":
        return dict(a=_rand(_R, d, seed=seed), w=_rand(3 * d, d, scale=d ** -0.5, seed=seed + 1),
                    bias=_rand(3 * d, seed=seed + 2, dtype=torch.float32))
    if name in ("proj", "fc2"):
        k = d if name == "proj" else h
        return dict(a=_rand(_R, k, seed=seed), w=_rand(d, k, scale=k ** -0.5, seed=seed + 1),
                    bias=_rand(d, seed=seed + 2, dtype=torch.float32), residual=_rand(_R, d, seed=seed + 3, dtype=torch.float32))
    if name in ("pwconv2_384", "pwconv2_768"):
        C = 384 if name.endswith("384") else 768
        rows = _R384 if C == 384 else _R
        return dict(a=_rand(rows, 4 * C, seed=seed), w=_rand(C, 4 * C, scale=(4 * C) ** -0.5, seed=seed + 1),
                    bias=_rand(C, seed=seed + 2, dtype=torch.float32),
                    colscale=_rand(C, scale=0.1, seed=seed + 3, dtype=torch.float32),
                    residual=_rand(rows, C, seed=seed + 4, dtype=torch.float32))
    if name == "fc1":
        return dict(a=_rand(_R, d, seed=seed), w=_rand(h, d, scale=d ** -0.5, seed=seed + 1),
                    bias=_rand(h, scale=0.5, seed=seed + 2, dtype=torch.float32))
    if name == "fc1_dgrad":   # dx of fc1 = dpre @ W1: N = 768, K = 3072
        return dict(a=_rand(_R, h, seed=seed), w=_rand(d, h, scale=h ** -0.5, seed=seed + 1))
    if name == "fc2_dgrad":   # dpre of fc1 = (dy @ W2) * GELU'(pre), with the column sums (= fc1 bias gradient)
        pre = _rand(_R, h, scale=1.5, seed=seed + 2).double()
        gelu_grad = (0.5 * (1 + torch.erf(pre / math.sqrt(2))) + pre * torch.exp(-0.5 * pre * pre) / math.sqrt(2 * math.pi))
        return dict(a=_rand(_R, d, seed=seed), w=_rand(h, d, scale=d ** -0.5, seed=seed + 1), aux_in=gelu_grad.to(BF16))
    raise KeyError(name)


_PAIR_CASES = ["qkv", "proj", "fc2", "pwconv2_384", "pwconv2_768", "fc1", "fc1_dgrad", "fc2_dgrad"]


def _pair_run(name, t):
    ops = _ops()
    if name == "qkv":
        return ops.gemm(t["a"], t["w"], bias=t["bias"])[:1]
    if name in ("proj", "fc2"):
        return ops.gemm(t["a"], t["w"], bias=t["bias"], residual=t["residual"], out_f32=True)[:1]
    if name.startswith("pwconv2"):
        return ops.gemm(t["a"], t["w"], bias=t["bias"], colscale=t["colscale"], residual=t["residual"], out_f32=True)[:1]
    if name == "fc1":
        return ops.gemm(t["a"], t["w"], bias=t["bias"], act=2, aux_out=True)
    if name == "fc1_dgrad":
        return ops.gemm(t["a"], t["w"])[:1]
    if name == "fc2_dgrad":
        out, _, st = ops.gemm(t["a"], t["w"], act=3, aux_in=t["aux_in"], want_stats=True)
        return out, st
    raise KeyError(name)


def _gelu64(x):
    return x * 0.5 * (1 + torch.erf(x / math.sqrt(2)))


def _gelu_grad64(x):
    return 0.5 * (1 + torch.erf(x / math.sqrt(2))) + x * torch.exp(-0.5 * x * x) / math.sqrt(2 * math.pi)


@pytest.mark.parametrize("name", _PAIR_CASES)
def test_cta_pair_gemm_many_items(name):
    """conv_gemm_kernel<256, EPI, true> through ops.gemm (N > 128, pair switch on): ViT-B/16 / ConvNeXt linear layers with
    3+ work items per CTA pair and an odd pixel-tile count, against fp64; fc2_dgrad also runs the pair statistics path."""
    t = _pair_inputs(name)
    a, w = t["a"], t["w"]
    rows, N = a.shape[0], w.shape[0]
    stats = name == "fc2_dgrad"
    geom = _Geom((rows, 1, 1), N, stats=stats, pair=True)
    assert geom.m_tiles % 2 == 1, geom.m_tiles
    if stats:   # the host runs the pair kernel only when it writes exactly the single-CTA kernel's partial rows
        single = _Geom((rows, 1, 1), N, stats=True)
        assert 2 * geom.grid == single.grid, (geom.grid, single.grid)
    _items(f"pair gemm {name} ({rows}x{a.shape[1]} -> {N})", *geom.per_cta())
    outs = _pair_run(name, t)
    _same(f"pair gemm {name}", outs, _pair_run(name, t))
    acc, S = _mm64(a, w)
    if name == "qkv":
        b = t["bias"].double()
        _check("out", outs[0], acc + b, S + b.abs(), U_BF16)
    elif name in ("proj", "fc2"):
        b, r = t["bias"].double(), t["residual"].double()
        _check("out", outs[0], acc + b + r, S + b.abs() + r.abs(), U_F32)
    elif name.startswith("pwconv2"):
        b, g, r = t["bias"].double(), t["colscale"].double(), t["residual"].double()
        _check("out", outs[0], (acc + b) * g + r, (S + b.abs()) * g.abs() + r.abs(), U_F32)
    elif name == "fc1":
        pre = acc + t["bias"].double()
        Sp = S + t["bias"].double().abs()
        floor = 2.0 ** -21 * (1 + pre.abs())   # A&S erf and the approximate rcp / ex2 of the epilogue
        _check("gelu(pre)", outs[0], _gelu64(pre), 1.13 * Sp, U_BF16, floor=floor)
        _check("gelu'(pre)", outs[1], _gelu_grad64(pre), 0.8 * Sp, U_BF16, floor=floor)
    elif name == "fc1_dgrad":
        _check("out", outs[0], acc, S, U_BF16)
    else:
        g = t["aux_in"].double()
        _check("out", outs[0], acc * g, S * g.abs(), U_BF16)
        ov = outs[0].double()
        _check_stat_rows("column sums", geom, outs[1], ov, ov * ov)


def test_cta_pair_gemm_bit_exact_against_single_cta(tmp_path):
    """The pair kernel and the single-CTA kernel (B200_GEMM_PAIR=0, read once per process: a child process) give the same
    bits on the cases above; the partial statistics rows are laid out differently and must agree in their column totals."""
    env = dict(os.environ, B200_GEMM_PAIR="0")
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.abspath(__file__), str(tmp_path)]
    r = subprocess.run(cmd, env=env, timeout=900, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    for name in _PAIR_CASES:
        single = torch.load(tmp_path / f"{name}.pt", map_location="cuda")
        pair = _pair_run(name, _pair_inputs(name))
        if name == "fc2_dgrad":
            assert torch.equal(pair[0], single[0]), f"{name}: pair and single-CTA outputs differ"
            tp, ts = pair[1].double().sum(0), single[1].double().sum(0)
            ab = pair[1].double().abs().sum(0)
            assert bool(((tp - ts).abs() <= C_SUM * ab).all()), f"{name}: column totals differ"
        else:
            for i, (p, s) in enumerate(zip(pair, single)):
                assert torch.equal(p, s), f"{name}: output {i} differs between the pair and the single-CTA kernel"
        print(f"  {name}: pair == single-CTA")
        (tmp_path / f"{name}.pt").unlink()


# ================================================================================================= C. wgrad_gemm_kernel
def test_wgrad_vit_qkv_more_items_than_sms():
    """wgrad_gemm_kernel<256, bias>: ViT-B/16 qkv at bs 512 (100864 tokens): 18 x 3 tiles x the planner's splits gives
    more items than SMs (the other ViT / ResNet weight gradients are planned into one wave); weights and bias against fp64."""
    ops = _ops()
    lib = _lib()
    R, K, N = 512 * 197, 768, 2304
    x = _rand(R, 1, 1, K, seed=20)
    dy = _rand(R, 1, 1, N, seed=21)
    splits = lib.b200_conv2d_wgrad_splits(R, 1, 1, K, N, 1, 1)
    items = (N + 127) // 128 * ((K + 255) // 256) * splits   # 128 x 256 tiles (abi_conv.cu plan_wgrad_geom)
    sms = _sms()
    grid = min(items, sms)
    _items(f"wgrad qkv ({splits} splits, {items} items)", items // grid, -(-items // grid), need=2)
    bias = torch.empty(N, device="cuda")
    dw = ops.conv2d_wgrad(dy, x, 1, 1, bias_out=bias)
    bias2 = torch.empty(N, device="cuda")
    _same("wgrad qkv", (dw, bias), (ops.conv2d_wgrad(dy, x, 1, 1, bias_out=bias2), bias2))
    ref = torch.zeros(N, K, dtype=F64, device="cuda")
    S = torch.zeros_like(ref)
    bref = torch.zeros(N, dtype=F64, device="cuda")
    babs = torch.zeros_like(bref)
    for r0 in range(0, R, 1 << 14):
        d = dy.view(R, N)[r0:r0 + (1 << 14)].double()
        a = x.view(R, K)[r0:r0 + (1 << 14)].double()
        ref += d.t() @ a
        S += d.abs().t() @ a.abs()
        bref += d.sum(0)
        babs += d.abs().sum(0)
    _check("dw", dw.view(N, K), ref, S, U_F32)
    _check("bias", bias, bref, babs, U_F32, c=C_SUM)


# ================================================================================================= D. conv1x1_stream_kernel
# (K, bottleneck batch, spatial): pixels a multiple of 128 and at least two laps of the A ring per CTA
_STREAM = [(64, 50, 56), (128, 56, 28), (256, 96, 14)]


def _stream_per_cta(P, N):
    m_tiles, n_tiles = P // 128, N // 256
    grid = min(m_tiles * n_tiles, _sms()) // n_tiles * n_tiles
    step = grid // n_tiles
    return m_tiles // step, -(-m_tiles // step)


@pytest.mark.parametrize("K,B,hw", _STREAM)
def test_conv1x1_stream_many_items(K, B, hw):
    """conv1x1_stream_kernel<K/64, kStreamBnRelu | kStreamMask>: the bottleneck conv3 forward (relu(bn(conv) + identity)) and
    the masked conv1 dgrad with per-CTA column sums, 3+ tiles per CTA and two laps of the A ring (4 / 2 / 3 stages)."""
    ops = _ops()
    N = 4 * K
    P = B * hw * hw
    assert P % 128 == 0
    least, most = _stream_per_cta(P, N)
    stages, kb_per_item = {64: (4, 1), 128: (2, 1), 256: (3, 4)}[K]
    assert least * kb_per_item >= 2 * stages, "fewer than two laps of the A ring"
    _items(f"stream K={K} N={N} ({P} pixels)", least, most)
    x = _rand(P, K, seed=30 + K)
    w = _rand(N, K, scale=K ** -0.5, seed=31 + K)
    co = _bn_coeffs(ops, N, 32 + K)
    res = _rand(P, N, seed=33 + K)
    y = ops.conv1x1_bn_act(x, w, co, res)
    _same("stream bn_relu", (y,), (ops.conv1x1_bn_act(x, w, co, res),))
    acc, S = _mm64(x, w)
    sc, sh, r = co.scale.double(), co.shift.double(), res.double()
    _check("relu(bn(conv) + identity)", y, (acc * sc + sh + r).clamp_min(0), S * sc.abs() + sh.abs() + r.abs(), U_BF16)
    del acc, S
    # dgrad of conv1 (Cin = N, Cout = K): dz = (mask > 0) * (dy @ W + residual)
    dy = _rand(P, K, seed=34 + K)
    w1 = _rand(K, N, scale=K ** -0.5, seed=35 + K)        # conv1 weight [Cout = K, Cin = N]
    wd = w1.t().contiguous()                               # pack_weight(mode=1) of a 1x1 conv: [Cin][Cout]
    mask = torch.relu(_rand(P, N, seed=36 + K))
    dz, st = ops.conv1x1_dgrad_masked(dy, wd, res, mask)
    dz2, st2 = ops.conv1x1_dgrad_masked(dy, wd, res, mask)
    _same("stream mask", (dz, st), (dz2, st2))
    acc, S = _mm64(dy, wd)
    alive = mask > 0
    _check("masked dgrad", dz, (acc + r) * alive, (S + r.abs()) * alive, U_BF16)
    d64 = dz.double()
    _check("column sums", st[:, 0].double().sum(0), d64.sum(0), d64.abs().sum(0), U_F32, c=C_SUM)
    assert float(st[:, 1].abs().max()) == 0.0


# ================================================================================================= E. window attention
def _window_partition(x, ws):
    B, H, W, C = x.shape
    return x.view(B, H // ws, ws, W // ws, ws, C).permute(0, 1, 3, 2, 4, 5).contiguous().view(-1, ws, ws, C)


def _window_reverse(w, ws, H, W):
    B = int(w.shape[0] / (H * W / ws / ws))
    return w.view(B, H // ws, W // ws, ws, ws, -1).permute(0, 1, 3, 2, 4, 5).contiguous().view(B, H, W, -1)


def _rel_index():
    coords = torch.stack(torch.meshgrid([torch.arange(7), torch.arange(7)], indexing="ij")).flatten(1)
    rel = (coords[:, :, None] - coords[:, None, :]).permute(1, 2, 0).contiguous()
    rel[:, :, 0] += 6
    rel[:, :, 1] += 6
    rel[:, :, 0] *= 13
    return rel.sum(-1)


def _shift_mask(H, W, shift):
    img = torch.zeros(1, H, W, 1)
    cnt = 0
    for h in (slice(0, -7), slice(-7, -shift), slice(-shift, None)):
        for w in (slice(0, -7), slice(-7, -shift), slice(-shift, None)):
            img[:, h, w, :] = cnt
            cnt += 1
    mw = _window_partition(img, 7).view(-1, 49)
    m = mw.unsqueeze(1) - mw.unsqueeze(2)
    return m.masked_fill(m != 0, -100.0).masked_fill(m == 0, 0.0)


def _to_windows(t, nparts, nH, shift):
    """[B,H,W,nparts*nH*32] -> [nparts, B*nW, nH, 49, 32] in the (rolled) window order of the kernels."""
    if shift > 0:
        t = torch.roll(t, shifts=(-shift, -shift), dims=(1, 2))
    return _window_partition(t, 7).view(-1, 49, nparts, nH, 32).permute(2, 0, 3, 1, 4)


def _from_windows(t, B, H, W, shift):
    """inverse of _to_windows: [nparts, B*nW, nH, 49, 32] -> [B,H,W,nparts*nH*32]."""
    nparts, BnW, nH = t.shape[:3]
    x = _window_reverse(t.permute(1, 3, 0, 2, 4).reshape(BnW, 7, 7, -1), 7, H, W)
    if shift > 0:
        x = torch.roll(x, shifts=(shift, shift), dims=(1, 2))
    return x


def _wattn_ref64(qkv, out_k, dout, nH, table, index, mask, shift, scale):
    """fp64 roll -> partition -> biased, masked softmax attention -> reverse -> roll, forward and backward, with
    absolute-value companions for the error bounds.  The backward's delta uses the kernel's own bf16 output (its operand)."""
    B, H, W, _ = qkv.shape
    q, k, v = _to_windows(qkv.double(), 3, nH, shift)
    bias = table.double()[index.view(-1)].view(49, 49, nH).permute(2, 0, 1)
    s = q @ k.transpose(-2, -1) * scale + bias
    if mask is not None:
        nW = mask.shape[0]
        s = (s.view(-1, nW, nH, 49, 49) + mask.double()[None, :, None]).view(-1, nH, 49, 49)
    lse = torch.logsumexp(s, -1)
    P = torch.exp(s - lse[..., None])
    o = P @ v
    So = P @ v.abs()
    do = _to_windows(dout.double(), 1, nH, shift)[0]
    ok = _to_windows(out_k.double(), 1, nH, shift)[0]
    dP = do @ v.transpose(-2, -1)
    D = (do * ok).sum(-1, keepdim=True)
    dS = P * (dP - D)
    AdS = P * (do.abs() @ v.abs().transpose(-2, -1) + D.abs())
    dq, dk, dv = dS @ k * scale, dS.transpose(-2, -1) @ q * scale, P.transpose(-2, -1) @ do
    Sq, Sk, Sv = AdS @ k.abs() * scale, AdS.transpose(-2, -1) @ q.abs() * scale, P.transpose(-2, -1) @ do.abs()
    smax = s.abs().amax(-1)
    out = _from_windows(o[None], B, H, W, shift)
    Sout = _from_windows(So[None], B, H, W, shift)
    dqkv = _from_windows(torch.stack([dq, dk, dv]), B, H, W, shift)
    Sdqkv = _from_windows(torch.stack([Sq, Sk, Sv]), B, H, W, shift)
    dtab = torch.zeros(169, nH, dtype=F64, device=qkv.device)
    Stab = torch.zeros_like(dtab)
    dtab.index_add_(0, index.view(-1), dS.sum(0).permute(1, 2, 0).reshape(49 * 49, nH))
    Stab.index_add_(0, index.view(-1), AdS.sum(0).permute(1, 2, 0).reshape(49 * 49, nH))
    return out, Sout, lse, smax, dqkv, Sdqkv, dtab, Stab


# (B, H, W, nH, shift): Swin-T stage 1 with and without shift, stages 2 / 3 with shift, and an odd window count (21x21 maps:
# 9 windows, B = 99) whose last pair's second half-stage holds data left from an earlier step
_WATTN = [(32, 56, 56, 3, 0), (32, 56, 56, 3, 3), (32, 28, 28, 6, 3), (64, 14, 14, 12, 3), (99, 21, 21, 3, 3)]


@pytest.mark.parametrize("B,H,W,nH,shift", _WATTN)
def test_window_attention_many_steps(B, H, W, nH, shift):
    """wattn_fwd_kernel / wattn_bwd_kernel: (B*nW + 1) // 2 window pairs over SMs // nH CTAs per head, at least two laps of
    the 4-stage operand ring; out, lse, dqkv and the relative-position-table gradient against fp64."""
    ops = _ops()
    nW = (H // 7) * (W // 7)
    pairs = (B * nW + 1) // 2
    per_head = max(_sms() // nH, 1)
    per_head = min(per_head, pairs)
    least, most = pairs // per_head, -(-pairs // per_head)
    assert least >= 2 * 4, "fewer than two laps of the operand ring"
    _items(f"window attention B={B} {H}x{W} nH={nH} shift={shift} ({B * nW} windows)", least, most)
    C = nH * 32
    scale = 32 ** -0.5
    qkv = _rand(B, H, W, 3 * C, seed=40 + nH)
    table = _rand(169, nH, scale=0.5, seed=41, dtype=torch.float32)
    index = _rel_index().cuda()
    mask = _shift_mask(H, W, shift).cuda() if shift > 0 else None
    tab = ops.window_bias_gather(table, index, nH, mask)
    out, lse = ops.window_attention_fwd(qkv, nH, tab, shift, scale)
    _same("window attention fwd", (out, lse), ops.window_attention_fwd(qkv, nH, tab, shift, scale))
    dout = _rand(B, H, W, C, seed=42)
    dqkv, dbias = ops.window_attention_bwd(qkv, out, dout, tab, lse, nH, shift, scale)
    dqkv2, dbias2 = ops.window_attention_bwd(qkv, out, dout, tab, lse, nH, shift, scale)
    _same("window attention dqkv", (dqkv,), (dqkv2,))
    o, So, lse_ref, smax, dq, Sdq, dtab, Stab = _wattn_ref64(qkv, out, dout, nH, table, index, mask, shift, scale)
    _check("out", out, o, So, U_BF16, c=C_ATTN)
    l2 = 1.0 / math.log(2.0)
    # lse is the log2 of the sum of the bf16-rounded exponentials that multiply V (each within 2^-8 of its value): a floor of
    # 2^-8 log2(e) on top of the fp32 score arithmetic
    _check("lse (log2)", lse.view(-1, nH, 49), lse_ref * l2, (lse_ref.abs() + smax + 1) * l2, U_F32, floor=U_BF16 * l2)
    _check("dqkv", dqkv, dq, Sdq, U_BF16, c=C_ATTN)
    for i, db in enumerate((dbias, dbias2)):   # (the table gradient is accumulated in no fixed order)
        dt = ops.window_bias_scatter(db, index, torch.zeros_like(table))
        _check(f"table gradient (call {i + 1})", dt, dtab, Stab, U_F32, c=C_ATTN)


# ================================================================================================= F. row-loop kernels
def _ln_bwd_ref64(dy, x, mean, rstd, gamma):
    x64, dy64, g = x.double(), dy.double(), gamma.double()
    xh = (x64 - mean.double()[:, None]) * rstd.double()[:, None]
    gd = dy64 * g
    a = gd.mean(1, keepdim=True)
    b = (gd * xh).mean(1, keepdim=True)
    r = rstd.double()[:, None]
    dx = r * (gd - a - xh * b)
    Sdx = r * (gd.abs() + gd.abs().mean(1, keepdim=True) + xh.abs() * (gd * xh).abs().mean(1, keepdim=True))
    return dx, Sdx, (dy64 * xh).sum(0), (dy64 * xh).abs().sum(0), dy64.sum(0), dy64.abs().sum(0)


@pytest.mark.parametrize("C,rows,x_f32", [(768, 64 * 197, True), (768, 64 * 197, False), (96, 14 * 3136, True),
                                          (96, 14 * 3136, False)])
def test_layernorm_bwd_grid_stride(C, rows, x_f32):
    """layernorm_bwd2_kernel: grid min(3 * SMs, rows / 8) x 8 warps, 32 / LPR rows per warp step (C = 96: 4 packed rows);
    3+ loop iterations per warp feed the shared dgamma / dbeta accumulators."""
    ops = _ops()
    lib = _lib()
    nblk = lib.b200_layernorm_bwd_blocks(rows, C)
    rpw = 1 if C > 256 else (32 // 16 if C > 128 else 32 // 8)
    step = nblk * 8 * rpw
    _items(f"layernorm_bwd C={C} rows={rows} x {'fp32' if x_f32 else 'bf16'}", rows // step, -(-rows // step))
    x = _rand(rows, C, scale=2.0, seed=50, dtype=torch.float32 if x_f32 else BF16) + 0.3
    x = x if x_f32 else x.to(BF16)
    gamma = _rand(C, seed=51, dtype=torch.float32) * 0.5 + 1
    beta = _rand(C, seed=52, dtype=torch.float32)
    _, mean, rstd = ops.layernorm_fwd(x, gamma, beta, 1e-6)
    dy = _rand(rows, C, seed=53)
    outs = ops.layernorm_bwd(dy, x, mean, rstd, gamma)
    _same("layernorm_bwd", outs, ops.layernorm_bwd(dy, x, mean, rstd, gamma))
    dx, Sdx, dg, Sdg, db, Sdb = _ln_bwd_ref64(dy, x, mean, rstd, gamma)
    _check("dx", outs[0], dx, Sdx, U_BF16)
    _check("dgamma", outs[1], dg, Sdg, U_F32)
    _check("dbeta", outs[2], db, Sdb, U_F32)


def test_patch_merge_ln_bwd_grid_stride():
    """patch_merge_ln_bwd_kernel at Swin-T stage 1 (bs 14: 10976 merged rows, one row per warp step, 3+ steps per warp)."""
    ops = _ops()
    lib = _lib()
    B, H, W, C = 14, 56, 56, 96
    rows = B * (H // 2) * (W // 2)
    step = lib.b200_patch_merge_ln_bwd_blocks(rows) * 8
    _items(f"patch_merge_ln_bwd rows={rows}", rows // step, -(-rows // step))
    x = _rand(B, H, W, C, scale=2.0, seed=60, dtype=torch.float32) + 0.3
    gamma = _rand(4 * C, seed=61, dtype=torch.float32) * 0.5 + 1
    beta = _rand(4 * C, seed=62, dtype=torch.float32)
    _, mean, rstd = ops.patch_merge_ln_fwd(x, gamma, beta, 1e-5)
    dy = _rand(rows, 4 * C, seed=63)
    outs = ops.patch_merge_ln_bwd(dy, x, mean, rstd, gamma)
    _same("patch_merge_ln_bwd", outs, ops.patch_merge_ln_bwd(dy, x, mean, rstd, gamma))
    cat = torch.cat([x[:, 0::2, 0::2], x[:, 1::2, 0::2], x[:, 0::2, 1::2], x[:, 1::2, 1::2]], -1).reshape(rows, 4 * C)
    dxc, Sdxc, dg, Sdg, db, Sdb = _ln_bwd_ref64(dy, cat, mean, rstd, gamma)

    def uncat(t):
        t = t.view(B, H // 2, W // 2, 4, C)
        o = torch.empty(B, H, W, C, dtype=t.dtype, device=t.device)
        o[:, 0::2, 0::2], o[:, 1::2, 0::2], o[:, 0::2, 1::2], o[:, 1::2, 1::2] = t[:, :, :, 0], t[:, :, :, 1], t[:, :, :, 2], t[:, :, :, 3]
        return o

    _check("dx", outs[0], uncat(dxc), uncat(Sdxc), U_BF16)
    _check("dgamma", outs[1], dg, Sdg, U_F32)
    _check("dbeta", outs[2], db, Sdb, U_F32)


def test_bn_backward_multi_iteration():
    """bn_bwd_reduce_kernel / bn_bwd_apply_kernel at ResNet-50 layer1 (C = 64, bs 160: 501760 rows): each thread's
    four-rows-in-flight loop runs 3+ iterations; dgamma / dbeta / dx against fp64."""
    ops = _ops()
    lib = _lib()
    B, H, W, C = 160, 56, 56, 64
    rows = B * H * W
    nblk = lib.b200_bn_bwd_blocks(rows, C)
    rpi = 256 // (C // 8)
    rpb = -(-rows // nblk)
    rpb = -(-rpb // rpi) * rpi
    _items(f"bn_backward rows={rows} ({nblk} blocks of {rpb} rows)", rpb // (4 * rpi), -(-rpb // (4 * rpi)))
    x = (_rand(B, H, W, C, scale=1.5, seed=70).float() + 0.3).to(BF16)
    g = _rand(B, H, W, C, seed=71)
    co = _bn_coeffs(ops, C, 72)
    outs = ops.bn_backward(g, x, co, relu=True)[:3]
    _same("bn_backward", outs, ops.bn_backward(g, x, co, relu=True)[:3])
    x64, g64 = x.view(rows, C).double(), g.view(rows, C).double()
    alive, amb = _relu_mask64(x.view(rows, C), co.scale, co.shift)
    n_amb = int(amb.sum())
    print(f"  mask positions within fp32 rounding of zero: {n_amb}")
    assert n_amb < 1e-4 * amb.numel()
    dz = g64 * alive
    mean, inv, sc = co.mean.double(), co.invstd.double(), co.scale.double()
    # an ambiguous mask position may flip a term of the sums: its |g|, |g x| widen their bounds
    slack0 = (g64.abs() * amb).sum(0)
    slack1 = ((g64 * x64).abs() * amb).sum(0)
    s0, s1 = dz.sum(0), (dz * x64).sum(0)
    a0, a1 = dz.abs().sum(0) + slack0 / C_GEMM, (dz * x64).abs().sum(0) + slack1 / C_GEMM
    dbeta = s0
    dgamma = inv * (s1 - mean * s0)
    _check("dbeta", outs[2], dbeta, a0, U_F32)
    _check("dgamma", outs[1], dgamma, inv * (a1 + mean.abs() * a0), U_F32)
    xh = (x64 - mean) * inv
    m1, m2 = dbeta / rows, dgamma / rows
    dx = sc * (dz - m1 - xh * m2)
    # (the kernel evaluates dx = a dz - b x + c in fp32: the last term bounds that rounding, 2^-20 of its terms after c)
    Sdx = sc.abs() * (a0 / rows + xh.abs() * inv * (a1 + mean.abs() * a0) / rows
                      + 2.0 ** -4 * (dz.abs() + m1.abs() + (x64.abs() + mean.abs()) * inv * m2.abs()))
    _check("dx", outs[0].view(rows, C), dx, Sdx, U_BF16, keep=~amb)


# ------------------------------------------------------------------------------------------------- child process (pair off)
if __name__ == "__main__":
    # python test_gpu_persistent_schedules.py OUTDIR: run the pair-GEMM cases (with whatever B200_GEMM_PAIR says) and save
    # their outputs under OUTDIR for test_cta_pair_gemm_bit_exact_against_single_cta
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    outdir = sys.argv[1]
    for _name in _PAIR_CASES:
        torch.save([t.cpu() for t in _pair_run(_name, _pair_inputs(_name))], os.path.join(outdir, f"{_name}.pt"))
    torch.cuda.synchronize()
