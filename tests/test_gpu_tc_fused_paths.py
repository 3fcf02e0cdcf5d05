"""The tensor-core path as the benchmark runs it: 1-term fp16 operands with hi-only producers, the fused epilogues of
conv2d_tc (residuals, split-K finishing pass, blocked output), the deferred split-K ConvLSTM gate GEMM, every
lstm_gates_kernel instantiation and batch-slice operand views.

Reference and bound.  `ref64` is the same operation in float64 on the CPU, computed from the operands the kernel actually
multiplies: the fp16 planes it is handed and the fp16 weight matrices of PackedConvTC (1 term: hi*hi; 3 terms:
hi*hi + lo*hi + hi*lo).  Every fp16 x fp16 product is exact in fp32, so the kernel differs from ref64 only through its fp32
accumulation and epilogue.  Per element:

    |got - ref64| <= c * 2^-22 * S + 2^-22 * |ref64|,    S = conv(|x|, |w|) + |bias| + |residual|   (float64)

c = (K chunks of the GEMM: taps x 32/64-channel chunks) + (split count) + 4.  Each K chunk is a short run of MMAs into
the fp32 TMEM accumulator whose magnitude never exceeds S: allowing two fp32 ulps (2^-22) of S per chunk, per reduction of
a split and per epilogue add (bias, residual, the two halves of the concatenated three-term form, one spare) bounds the
accumulation; the 2^-22 |ref64| term is the final rounding.  Every test prints the largest err / bound it saw.

Exact checks where the arithmetic is the same: the fp16 planes are fp16_rn(out_f32) (and fp16_rn(out_f32 - hi)), the
blocked planes are the same halves re-blocked, split-K results repeat bit for bit.  The tests at the end of the file run
on the CPU: each feeds one of the comparison helpers a deliberately wrong reference and requires it to fail."""
import contextlib
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from dvmvs import _native as N
from dvmvs import _ops as ops

DEV = "cuda"
D = N.SRC_DIRECT
U = 2.0 ** -22            # two fp32 ulps: the unit of the accumulation bound
EPS32 = 2.0 ** -24        # fp32 unit roundoff


# ------------------------------------------------------------------------------------------------ fixtures
@pytest.fixture
def tc_mode():
    """Selects the tensor-core backend with `terms`-term operands everywhere (no family policy) and restores the previous
    configuration afterwards.  terms=1 is the benchmarked configuration: lo_planes_needed() is False, producers write
    hi planes only."""
    saved = (ops.conv_backend(), ops._TC_TERMS_BASE, ops._TC_STRIDE2, ops.precision_policy())

    def select(terms):
        ops.set_conv_backend("tc", terms=terms, stride2=True)
        ops.set_precision_policy(None)
        assert ops.lo_planes_needed() == (terms == 3)

    try:
        yield select
    finally:
        ops.set_conv_backend(saved[0], terms=saved[1], stride2=saved[2])
        ops.set_precision_policy(saved[3])


@contextlib.contextmanager
def nan_filled_outputs():
    """For the duration of one call, every float16 / float32 tensor torch.empty / torch.empty_like return is NaN-filled
    (_ops allocates every output that way; the split-K workspace is torch.zeros and unaffected).  A NaN left in an output
    afterwards is an element the kernel never wrote."""
    real_empty, real_like = torch.empty, torch.empty_like

    def fill(t):
        if t.dtype in (torch.float16, torch.float32):
            t.fill_(float("nan"))
        return t

    torch.empty = lambda *a, **k: fill(real_empty(*a, **k))
    torch.empty_like = lambda *a, **k: fill(real_like(*a, **k))
    try:
        yield
    finally:
        torch.empty, torch.empty_like = real_empty, real_like


def _rand(key, shape, scale=1.0):
    seed = sum(ord(ch) * (i + 1) for i, ch in enumerate(key)) % (2 ** 31)
    return torch.from_numpy(np.random.RandomState(seed).randn(*shape).astype(np.float32) * np.float32(scale))


def _nhwc(x_nchw):
    return x_nchw.permute(0, 2, 3, 1).contiguous()


# ------------------------------------------------------------------------------------------------ comparison helpers
def assert_within(got, ref, S, c, label):
    """|got - ref| <= c * 2^-22 * S + 2^-22 * |ref| element-wise (float64); prints and returns the largest err / bound."""
    got = got.detach().to("cpu", torch.float64)
    assert got.shape == ref.shape, (label, tuple(got.shape), tuple(ref.shape))
    assert torch.isfinite(got).all(), "%s: non-finite output elements" % label
    err = (got - ref).abs()
    bound = c * U * S + U * ref.abs()
    ratio = torch.where(bound > 0, err / torch.where(bound > 0, bound, torch.ones_like(bound)),
                        torch.where(err > 0, torch.full_like(err, float("inf")), torch.zeros_like(err)))
    r = float(ratio.max())
    print("%s: max err/bound = %.3g (c = %d)" % (label, r, c))
    assert r <= 1.0, "%s: max err/bound = %.3g at %s" % (label, r, np.unravel_index(int(ratio.argmax()), tuple(ratio.shape)))
    return r


def assert_all_written(t, label):
    """No element of a NaN-prefilled output may still be NaN."""
    bad = torch.isnan(t)
    assert not bool(bad.any()), "%s: %d unwritten element(s), first at %s" % (
        label, int(bad.sum()), tuple(int(i) for i in bad.nonzero()[0].tolist()))


def bits(t):
    return t.contiguous().view(torch.int16 if t.element_size() == 2 else torch.int32)


def assert_same_bits(a, b, label):
    assert a.shape == b.shape and a.dtype == b.dtype, label
    assert torch.equal(bits(a), bits(b)), "%s: %d elements differ" % (label, int((bits(a) != bits(b)).sum()))


def assert_planes_exact(f32, planes, hi_only, label):
    """planes[0] == fp16_rn(f32); planes[1] == fp16_rn(f32 - hi) or, hi-only, never written (still NaN)."""
    hi = f32.to(torch.float16)
    assert_same_bits(planes[0], hi, label + " hi plane")
    if hi_only:
        assert bool(torch.isnan(planes[1]).all()), "%s: hi-only launch wrote the lo plane" % label
    else:
        assert_same_bits(planes[1], (f32 - hi.float()).to(torch.float16), label + " lo plane")


def reblock(planes):
    """(2,B,H,W,C) -> (2,B,C/8,H,W,8), the operand layout of conv_halo_kernel"""
    two, B, H, W, C = planes.shape
    return planes.reshape(two, B, H, W, C // 8, 8).permute(0, 1, 4, 2, 3, 5)


# ------------------------------------------------------------------------------------------------ float64 references
def tc_weights(ptc, w2d):
    """PackedConvTC matrix [rows][K] (K = tap-major, then source, then zero-padded 32/64-channel chunks) -> one float64
    (Cout, Cs_i, k, k) conv weight per source."""
    k, cout = ptc.ksize, ptc.cout
    w = w2d[:cout].to("cpu", torch.float64).reshape(cout, k * k, ptc.k_per_tap)
    out, off = [], 0
    for cs in ptc.src_stored:
        kc, nch = ops.tc_chunking(cs)
        out.append(w[:, :, off:off + cs].reshape(cout, k, k, cs).permute(0, 3, 1, 2))
        off += nch * kc
    return out


def tc_chunks(ptc):
    return ptc.ksize * ptc.ksize * sum(ops.tc_chunking(cs)[1] for cs in ptc.src_stored)


def conv_terms64(planes, whi, wlo, terms, stride, drop_lo_hi=False):
    """sum over sources of hi*hi (+ lo*hi + hi*lo) in float64 -> (value, sum of |products|), both NCHW.
    planes: per source a (2,B,H,W,Cs) fp16 tensor or (hi, lo) pair; whi / wlo: per source (Cout,Cs,k,k) float64."""
    acc, S = 0, 0
    for p, wh, wl in zip(planes, whi, wlo):
        xh = p[0].to("cpu", torch.float64).permute(0, 3, 1, 2)
        prods = [(xh, wh)]
        if terms == 3:
            xl = p[1].to("cpu", torch.float64).permute(0, 3, 1, 2)
            prods += ([] if drop_lo_hi else [(xl, wh)]) + [(xh, wl)]
        pad = (wh.shape[-1] - 1) // 2
        for x, w in prods:
            acc = acc + F.conv2d(x, w, None, stride, pad)
            S = S + F.conv2d(x.abs(), w.abs(), None, stride, pad)
    return acc, S


def nearest_up(res_nhwc, Hout, Wout, row_shift=0):
    """F.interpolate(size=(Hout, Wout), mode="nearest") of an NHWC residual (the reference FPN's form), float64 NCHW.
    row_shift != 0 builds a wrong reference for the sensitivity test."""
    r = res_nhwc.to("cpu", torch.float64).permute(0, 3, 1, 2)
    if row_shift == 0:
        return F.interpolate(r, size=(Hout, Wout), mode="nearest")
    Hr = r.shape[2]
    ry = torch.clamp(torch.arange(Hout) * Hr // Hout + row_shift, 0, Hr - 1)
    rx = torch.arange(Wout) * r.shape[3] // Wout
    return r[:, :, ry][:, :, :, rx]


def epilogue64(acc, S, bias, residual, residual_mode, act, row_shift=0):
    """bias / residual / activation of the kernel epilogue in float64; returns NHWC (value, S)."""
    if bias is not None:
        b = bias.to("cpu", torch.float64).view(1, -1, 1, 1)
        acc, S = acc + b, S + b.abs()
    if residual_mode != N.RES_NONE:
        r = (residual.to("cpu", torch.float64).permute(0, 3, 1, 2) if residual_mode == N.RES_SAME else
             nearest_up(residual, acc.shape[2], acc.shape[3], row_shift))
        acc, S = acc + r, S + r.abs()
    if act == N.ACT_RELU:
        acc = acc.clamp_min(0)          # 1-Lipschitz: the pre-activation bound carries over
    return acc.permute(0, 2, 3, 1), S.permute(0, 2, 3, 1)


def cell(gates, c, ln_dims=(1, 2)):
    """MVSLayernormConvLSTMCell's gate epilogue (reference convlstm.py:45-59) on NHWC tensors in their own dtype: gates
    (B,h,w,4C) in order i, f, o, g; LayerNorm without affine over (h, w), eps 1e-5; CELU(alpha=1).
    Returns h_next, c_next and the intermediates the error propagation needs."""
    C = c.shape[-1]
    ai, af, ao, ag = gates.split(C, dim=-1)
    i, f, o = torch.sigmoid(ai), torch.sigmoid(af), torch.sigmoid(ao)

    def ln(x):
        mu = x.mean(ln_dims, keepdim=True)
        sd = torch.sqrt(((x - mu) ** 2).mean(ln_dims, keepdim=True) + 1e-5)
        return (x - mu) / sd, sd

    g, sd_g = ln(ag)
    G = F.celu(g)
    cp = f * c + i * G
    cn, sd_c = ln(cp)
    h = o * F.celu(cn)
    return h, cn, dict(i=i, o=o, c=c, g=g, sd_g=sd_g, G=G, cn=cn, sd_c=sd_c)


def cell_bound(gates64, c64, delta, hw):
    """Float64 cell and a per-element bound on the kernel's h_next / c_next, given a per-element bound `delta` on the gate
    pre-activations it summed.  Propagation (first order, made safe by the max over the LayerNorm group):
      sigmoid' <= 1/4; celu is 1-Lipschitz;
      LayerNorm over n positions with every input off by <= d:  |dy| <= (2 d + |y| d) / (sd - d)
        (the mean moves by <= d, the standard deviation by <= the RMS of the centred perturbation <= d);
    plus the fp32 evaluation of the cell itself: each LayerNorm statistic is a sum of hw values (at most hw + 13 rounded
    adds, sequential within a thread, then lanes and warps) and the transcendental functions are accurate to a few ulps;
    e32 = 4 (hw + 64) 2^-24 per stage at unit scale."""
    h, cn, t = cell(gates64, c64)
    C = c64.shape[-1]
    di, df, do, dg = delta.split(C, dim=-1)
    e32 = 4.0 * (hw + 64) * EPS32
    Dg = dg.amax((1, 2), keepdim=True)
    assert bool((t["sd_g"] > 4 * Dg).all()), "gate bound too loose for the LayerNorm of cc_g (near-constant channel)"
    dG = (2 * Dg + t["g"].abs() * Dg) / (t["sd_g"] - Dg) + e32 * (1 + t["g"].abs())
    dcp = 0.25 * df * t["c"].abs() + 0.25 * di * (t["G"].abs() + dG) + t["i"] * dG + e32 * (1 + t["G"].abs() + t["c"].abs())
    Dc = dcp.amax((1, 2), keepdim=True)
    assert bool((t["sd_c"] > 4 * Dc).all()), "state bound too loose for the second LayerNorm"
    dcn = (2 * Dc + cn.abs() * Dc) / (t["sd_c"] - Dc) + e32 * (1 + cn.abs())
    dh = 0.25 * do * (F.celu(cn).abs() + dcn) + t["o"] * dcn + e32 * (1 + h.abs())
    return h, cn, dh, dcn


def assert_cell_within(got_h, got_c, ref_h, ref_c, bound_h, bound_c, label):
    """|got - ref| <= bound per element for h_next and c_next; prints the largest err / bound."""
    worst = 0.0
    for name, got, ref, bnd in (("h", got_h, ref_h, bound_h), ("c", got_c, ref_c, bound_c)):
        got = got.detach().to("cpu", torch.float64)
        assert torch.isfinite(got).all(), "%s/%s: non-finite output" % (label, name)
        r = float(((got - ref).abs() / bnd).max())
        worst = max(worst, r)
        assert r <= 1.0, "%s/%s: max err/bound = %.3g" % (label, name, r)
    print("%s: max err/bound = %.3g" % (label, worst))
    return worst


def lstm_variant(B, C, h, w):
    """The lstm_gates_kernel<PPW, CPB> instantiation dvmvs_lstm_gates_parts launches (mirror of its host dispatch,
    csrc/conv.cu): narrow blocks of 8 channels while B*C/32 < 74 and hw <= 512, else 32-channel blocks; None = refused."""
    hw = h * w
    if B * (C // 32) < 74 and hw <= 8 * 4 * 16:
        ppw = -(-hw // 32)
        return "<2,8>" if ppw <= 2 else ("<4,8>" if ppw <= 4 else "<16,8>")
    ppw = -(-hw // 8)
    if ppw > 64:
        return None
    return "<2,32>" if ppw <= 2 else ("<8,32>" if ppw <= 8 else ("<16,32>" if ppw <= 16 else "<64,32>"))


def tc_ksplit(B, Hin, Win, Cout, k, stride, block_n, allow_split=True):
    """The split count dvmvs_conv2d_tc chooses for this launch (asked from the library)."""
    d = N.ConvTcDesc()
    d.B, d.Hin, d.Win, d.Cout, d.ksize, d.stride, d.block_n = B, Hin, Win, Cout, k, stride, block_n
    d.allow_split = 1 if allow_split else 0
    d.workspace, d.workspace_bytes = ops.workspace(torch.device(DEV, torch.cuda.current_device())).data_ptr(), ops.WORKSPACE_BYTES
    return int(N.lib().dvmvs_conv2d_tc_ksplit(ctypes.byref(d)))


# ------------------------------------------------------------------------------------------------ B. conv2d_tc fused epilogues
TCF_CASES = [
    # name, B, Hin, Win, [(src channels, x2 upsampled)], Cout, k, stride, act, block_n, residual (mode, Hr, Wr), blk_out, splits
    ("mnas_expand_c16_n48", 2, 20, 24, [(16, False)], 48, 1, 1, N.ACT_RELU, 64, None, False, False),
    ("mnas_project_c72_n24_res", 2, 20, 24, [(72, False)], 24, 1, 1, N.ACT_NONE, 32, (N.RES_SAME, 20, 24), False, False),
    ("mnas_c80_n80_res", 2, 10, 12, [(80, False)], 80, 1, 1, N.ACT_NONE, 64, (N.RES_SAME, 10, 12), False, False),
    ("mnas_k3s2_odd_c24_n40", 2, 15, 17, [(24, False)], 40, 3, 2, N.ACT_RELU, 32, None, False, True),
    ("mnas_k5s2_odd_c40_n80", 2, 13, 11, [(40, False)], 80, 5, 2, N.ACT_RELU, 64, None, False, True),
    ("mnas_k3_c96_n96_res_blk", 2, 6, 7, [(96, False)], 96, 3, 1, N.ACT_NONE, 64, (N.RES_SAME, 6, 7), True, True),
    ("fpn_lateral_up_odd", 2, 15, 13, [(40, False)], 32, 1, 1, N.ACT_NONE, 32, (N.RES_NEAREST_UP, 8, 7), False, False),
    ("fpn_lateral_up_even", 1, 16, 20, [(96, False)], 32, 1, 1, N.ACT_NONE, 32, (N.RES_NEAREST_UP, 8, 10), True, False),
    ("k3_up_res_split", 1, 9, 11, [(24, False)], 32, 3, 1, N.ACT_NONE, 32, (N.RES_NEAREST_UP, 5, 6), False, True),
    ("upsampled_src_concat", 1, 32, 40, [(32, True), (16, False)], 32, 3, 1, N.ACT_RELU, 32, None, False, True),
    ("blk_64x64_k1", 1, 64, 64, [(32, False)], 32, 1, 1, N.ACT_RELU, 32, None, True, False),
    ("blk_64x64_k3_c24_n40_res", 1, 64, 64, [(24, False)], 40, 3, 1, N.ACT_RELU, 32, (N.RES_SAME, 64, 64), True, True),
    ("large_no_split_c64", 2, 64, 80, [(64, False)], 64, 3, 1, N.ACT_RELU, 64, None, True, False),
]


def _tc_case_inputs(case):
    name, B, H, W, srcs, Cout, k, stride, act, block_n, res, use_blk, splits = case
    cin = sum(c for c, _ in srcs)
    xs = [_rand("%s/x%d" % (name, i), (B, c, H // 2, W // 2) if up else (B, c, H, W)) for i, (c, up) in enumerate(srcs)]
    w = _rand(name + "/w", (Cout, cin, k, k), (2.0 / (cin * k * k)) ** 0.5)
    bias = _rand(name + "/b", (Cout,), 0.1)
    pc = ops.PackedConv(w, bias, None, stride=stride, act=act)
    residual = _nhwc(_rand(name + "/r", (B, Cout, res[1], res[2]))) if res is not None else None
    return xs, pc, residual


def _check_upsampled_planes(planes, x_nchw, label):
    """split_planes(upsample=True) against a float64 x2 bilinear (align_corners) interpolation: the fp32 sample position
    is off by <= 2 * 2^-24 * H (resp. W) pixels, which moves the value by <= 2 max|x| per pixel; ~6 products / sums round;
    hi + lo keeps 22 bits."""
    up = F.interpolate(x_nchw.double(), scale_factor=2, mode="bilinear", align_corners=True).permute(0, 2, 3, 1)
    C = up.shape[3]
    got = planes[0, ..., :C].double().cpu() + planes[1, ..., :C].double().cpu()
    tol = (8 + 4 * (x_nchw.shape[2] + x_nchw.shape[3])) * EPS32 * float(x_nchw.abs().max()) + 2.0 ** -21 * up.abs()
    assert bool(((got - up).abs() <= tol).all()), label
    assert not bool(planes[:, ..., C:].any()), label + ": padding channels not zero"


@pytest.mark.gpu
@pytest.mark.parametrize("allow_split", [False, True], ids=["nosplit", "split"])
@pytest.mark.parametrize("terms", [1, 3])
@pytest.mark.parametrize("case", TCF_CASES, ids=[c[0] for c in TCF_CASES])
def test_conv2d_tc_fused_epilogue_vs_ref64(tc_mode, case, terms, allow_split):
    """conv2d_tc with its fused epilogue (bias, RES_SAME / RES_NEAREST_UP residual, ReLU; fp32 + fp16 planes + blocked
    planes; split-K finishing pass) per element against ref64.  Outputs are NaN-prefilled: a partial n-tile, a ragged pixel
    tile or a padding channel left unwritten fails.  terms=1 runs hi-only with NaN lo planes on every input (a 1-term
    kernel must not read them) and must be bit-identical to the run with zero lo planes."""
    name, B, H, W, srcs, Cout, k, stride, act, block_n, res, use_blk, splits = case
    tc_mode(terms)
    hi_only = terms == 1
    xs, pc, residual = _tc_case_inputs(case)
    ptc = ops.PackedConvTC(pc, [c for c, _ in srcs], DEV)
    mode = res[0] if res is not None else N.RES_NONE
    res_dev = residual.to(DEV) if residual is not None else None

    with nan_filled_outputs():
        planes = [ops.split_planes(ops.to_nhwc(x.to(DEV)), upsample=up) for x, (c, up) in zip(xs, srcs)]
    for p, x, (c, up) in zip(planes, xs, srcs):
        assert_all_written(p, name + " split_planes")
        if up:
            _check_upsampled_planes(p, x, name)

    ksplit = tc_ksplit(B, H, W, Cout, k, stride, block_n, allow_split)
    assert (ksplit > 1) == (allow_split and splits), (name, ksplit)

    Hout, Wout = (H + 2 * ((k - 1) // 2) - k) // stride + 1, (W + 2 * ((k - 1) // 2) - k) // stride + 1
    sentinel = torch.tensor(-1234.0, dtype=torch.float16)

    def launch(src):
        blk = None
        if use_blk:
            blk = torch.full((2, B, Cout // 8, Hout, Wout, 8), float(sentinel), dtype=torch.float16, device=DEV)
        with nan_filled_outputs():
            f32, pl = ops.conv2d_tc(src, ptc, residual=res_dev, residual_mode=mode, terms=terms, block_n=block_n,
                                    allow_split=allow_split, blk_out=blk)
        return f32, pl, blk

    if hi_only:
        nan_lo = [p.clone() for p in planes]
        zero_lo = [p.clone() for p in planes]
        for a, z in zip(nan_lo, zero_lo):
            a[1].fill_(float("nan"))
            z[1].zero_()
        f32, pl, blk = launch(nan_lo)
        f32_z, pl_z, blk_z = launch(zero_lo)
        assert_same_bits(f32, f32_z, name + " NaN vs zero lo planes")
        assert_same_bits(pl[0], pl_z[0], name + " NaN vs zero lo planes (hi plane)")
    else:
        f32, pl, blk = launch(planes)
    assert_all_written(f32, name + " out_f32")
    assert_planes_exact(f32, pl, hi_only, name)
    if use_blk:
        assert_same_bits(blk[0], reblock(pl)[0], name + " blk_out hi")
        if hi_only:
            assert bool((bits(blk[1]) == bits(sentinel)).all()), name + ": hi-only launch wrote the blk_out lo half"
        else:
            assert_same_bits(blk[1], reblock(pl)[1], name + " blk_out lo")
    if ksplit > 1:
        again = launch(nan_lo if hi_only else planes)
        assert_same_bits(again[0], f32, name + " split-K repeat")
        assert_same_bits(again[1][0], pl[0], name + " split-K repeat (hi plane)")

    whi, wlo = tc_weights(ptc, ptc.w_hi), tc_weights(ptc, ptc.w_lo)
    acc, S = conv_terms64(planes, whi, wlo, terms, stride)
    ref, S = epilogue64(acc, S, pc.bias, residual, mode, act)
    c = tc_chunks(ptc) + ksplit + 4
    assert_within(f32, ref, S, c, "%s terms=%d ksplit=%d" % (name, terms, ksplit))


@pytest.mark.gpu
def test_nearest_up_residual_index_rule_matches_interpolate(tc_mode):
    """RES_NEAREST_UP picks residual pixel floor(o * Hr / Hout): with a 1x1 zero-weight convolution the output IS the
    residual as read, which must equal F.interpolate(size=..., mode="nearest") for out = 2 in - 1, 2 in and odd ratios."""
    tc_mode(1)
    for (Hr, Wr), (H, W) in (((8, 7), (15, 13)), ((5, 6), (10, 12)), ((3, 5), (7, 11)), ((4, 4), (9, 16))):
        pc = ops.PackedConv(torch.zeros(32, 16, 1, 1), None, None, stride=1, act=N.ACT_NONE)
        ptc = ops.PackedConvTC(pc, [16], DEV)
        res = _rand("nn/%d%d" % (Hr, Wr), (2, 32, Hr, Wr))
        x = ops.split_planes(ops.to_nhwc(_rand("nnx", (2, 16, H, W)).to(DEV)))
        out, _ = ops.conv2d_tc([x], ptc, residual=_nhwc(res).to(DEV), residual_mode=N.RES_NEAREST_UP, terms=1, allow_split=False)
        want = F.interpolate(res, size=(H, W), mode="nearest").permute(0, 2, 3, 1)
        assert torch.equal(out.cpu(), want), ((Hr, Wr), (H, W))


# ------------------------------------------------------------------------------------------------ A. halo and sweep: lo planes unread, outputs written
HALO_NAN_CASES = [
    # name, B, H, W, [(channels, upsampled)], Cout, k, residual
    ("k3_c32_res", 2, 64, 64, [(32, False)], 32, 3, True),
    ("k5_refine_like", 1, 64, 64, [(32, True), (1, True), (3, False)], 32, 5, False),
    ("k3_ragged_c24_n40", 1, 20, 12, [(24, False)], 40, 3, False),
    ("k5_c64_n128", 1, 32, 40, [(64, False)], 128, 5, False),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", HALO_NAN_CASES, ids=[c[0] for c in HALO_NAN_CASES])
def test_conv2d_halo_hi_only_reads_no_lo_plane(tc_mode, case):
    """1-term conv2d_halo in hi-only mode: NaN lo planes on the input give finite outputs bit-identical to zero lo planes;
    every hi output element is written and no lo plane is (NaN-prefilled outputs); f32 within the ref64 bound."""
    name, B, H, W, srcs, Cout, k, use_res = case
    tc_mode(1)
    xs = [_rand("halo/%s/x%d" % (name, i), (B, c, H // 2, W // 2) if up else (B, c, H, W)) for i, (c, up) in enumerate(srcs)]
    cin = sum(c for c, _ in srcs)
    w = _rand("halo/%s/w" % name, (Cout, cin, k, k), (2.0 / (cin * k * k)) ** 0.5)
    bias = _rand("halo/%s/b" % name, (Cout,), 0.1)
    pc = ops.PackedConv(w, bias, None, stride=1, act=N.ACT_RELU)
    ph = ops.PackedConvHalo(pc, [c for c, _ in srcs], DEV, concat_padded=True)
    res = _nhwc(_rand("halo/%s/r" % name, (B, Cout, H, W))) if use_res else None
    with nan_filled_outputs():
        blk = ops.split_blocked([(ops.to_nhwc(x.to(DEV)), up) for x, (c, up) in zip(xs, srcs)])
    assert_all_written(blk, name + " split_blocked")
    runs = []
    for lo in ("nan", "zero"):
        b = blk.clone()
        b[1].fill_(float("nan")) if lo == "nan" else b[1].zero_()
        with nan_filled_outputs():
            runs.append(ops.conv2d_halo([b], ph, residual=res.to(DEV) if use_res else None, terms=1, want_f32=True,
                                        want_blk=True, want_nhwc=True))
    (f32, oblk, onhwc), (f32_z, oblk_z, onhwc_z) = runs
    assert_all_written(f32, name + " out_f32")
    assert_same_bits(f32, f32_z, name + " NaN vs zero lo planes")
    assert_same_bits(oblk[0], oblk_z[0], name + " NaN vs zero lo planes (blk hi)")
    assert_planes_exact(f32, onhwc, True, name + " nhwc")
    assert_same_bits(oblk[0], reblock(onhwc)[0], name + " blk hi")
    assert bool(torch.isnan(oblk[1]).all()), name + ": hi-only launch wrote the blocked lo plane"
    # ref64 from the operands: the blocked hi planes (channel c of source i at its 8-aligned offset) and fp16(weights)
    x_hi = blk[0].to("cpu", torch.float64)                                   # (B, C8, H, W, 8)
    x_hi = x_hi.permute(0, 1, 4, 2, 3).reshape(B, -1, H, W)
    wpad = torch.zeros(Cout, x_hi.shape[1], k, k, dtype=torch.float64)
    src_off, dst_off = 0, 0
    for c, _ in srcs:
        wpad[:, dst_off:dst_off + c] = w[:, src_off:src_off + c].half().double()
        src_off, dst_off = src_off + c, dst_off + (c + 7) // 8 * 8
    acc = F.conv2d(x_hi, wpad, None, 1, (k - 1) // 2)
    S = F.conv2d(x_hi.abs(), wpad.abs(), None, 1, (k - 1) // 2)
    ref, S = epilogue64(acc, S, pc.bias, res, N.RES_SAME if use_res else N.RES_NONE, N.ACT_RELU)
    assert_within(f32, ref, S, ph.n_groups * k * k + 4, "halo " + name)


@pytest.mark.gpu
def test_plane_sweep_tc_one_term_reads_no_lo_plane(tc_mode, cases, synth):
    """plane_sweep_tc(terms=1) handed (hi, NaN lo) pairs: finite and bit-identical to (hi, zero lo)."""
    tc_mode(1)
    c = cases.PLANE_SWEEP_CASES["dot_small"]
    inp = cases.plane_sweep_inputs(synth, c)
    cu = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(DEV)
    feats = [ops.split_planes(ops.to_nhwc(cu(x))) for x in [inp["image1"]] + list(inp["image2s"])]
    outs = []
    for fill in (float("nan"), 0.0):
        pairs = [(p[0], torch.full_like(p[1], fill)) for p in feats]
        with nan_filled_outputs():
            outs.append(ops.plane_sweep_tc(pairs[0], pairs[1:], cu(inp["pose1"]), [cu(p) for p in inp["pose2s"]], cu(inp["K"]),
                                           c["min_depth"], c["max_depth"], c["D"], terms=1))
    assert_all_written(outs[0], "plane_sweep_tc")
    assert_same_bits(outs[0], outs[1], "plane_sweep_tc NaN vs zero lo planes")


@pytest.mark.gpu
def test_split_producers_write_every_element(tc_mode):
    """split_planes / concat_planes / split_blocked fill every element including the zero padding channels, and the
    direct (not upsampled) halves are exact: hi = fp16_rn(x), lo = fp16_rn(x - hi)."""
    tc_mode(1)
    x20 = _rand("sp/x20", (2, 20, 9, 13))
    x1 = _rand("sp/x1", (2, 1, 9, 13))
    x3 = _rand("sp/x3", (2, 3, 18, 26))
    with nan_filled_outputs():
        p20 = ops.split_planes(ops.to_nhwc(x20.to(DEV)))
        p20u = ops.split_planes(ops.to_nhwc(x20.to(DEV)), upsample=True)
        cat = ops.concat_planes([(ops.to_nhwc(x20.to(DEV)), True), (ops.to_nhwc(x1.to(DEV)), True), (ops.to_nhwc(x3.to(DEV)), False)])
        blk = ops.split_blocked([(ops.to_nhwc(x20.to(DEV)), True), (ops.to_nhwc(x1.to(DEV)), True), (ops.to_nhwc(x3.to(DEV)), False)])
    for t, label in ((p20, "split_planes"), (p20u, "split_planes(up)"), (cat, "concat_planes"), (blk, "split_blocked")):
        assert_all_written(t, label)
    x = _nhwc(x20).to(DEV)
    assert_planes_exact(x, torch.stack([p20[0, ..., :20], p20[1, ..., :20]]), False, "split_planes")
    assert not bool(p20[..., 20:].any())
    _check_upsampled_planes(p20u, x20, "split_planes(up)")
    # concat_planes: channels [0,20) x20 (x2), [20,21) x1 (x2), [21,24) x3
    assert_same_bits(cat[..., :20], p20u[..., :20], "concat_planes source 0")
    _check_upsampled_planes(cat[..., 20:21], x1, "concat_planes source 1")
    assert_planes_exact(_nhwc(x3).to(DEV), torch.stack([cat[0, ..., 21:24], cat[1, ..., 21:24]]), False, "concat_planes source 2")
    # split_blocked: every source starts on an 8-channel block: [0,24) x20 (x2), [24,32) x1 (x2), [32,40) x3
    blk_nhwc = blk.permute(0, 1, 3, 4, 2, 5).reshape(2, 2, 18, 26, -1)
    _check_upsampled_planes(blk_nhwc[..., 0:24], x20, "split_blocked source 0")
    _check_upsampled_planes(blk_nhwc[..., 24:32], x1, "split_blocked source 1")
    assert not bool(blk_nhwc[..., 35:40].any()), "split_blocked padding"
    assert_planes_exact(_nhwc(x3).to(DEV), torch.stack([blk_nhwc[0, ..., 32:35], blk_nhwc[1, ..., 32:35]]), False, "split_blocked source 2")


# ------------------------------------------------------------------------------------------------ C. deferred split-K ConvLSTM gates
@pytest.mark.gpu
@pytest.mark.parametrize("hw", [(8, 8), (8, 10)], ids=["8x8", "8x10"])
def test_deferred_split_k_lstm_gates(tc_mode, hw):
    """The fusionnet bottleneck cell (hidden 512, 3x3): conv_x for the input half, conv_h.run_deferred for the split-K hidden
    half and lstm_gates(parts=, addend=) as its finishing pass must be bit-identical to the two-launch path with the same
    split count (conv2d_tc(residual=gx, RES_SAME) -> finish -> lstm_gates(gates, c)); both sum the partials in split order,
    then add the addend.  Both match the float64 cell within the bound propagated from the gate bound.  The weights give
    gates of unit scale, so no LayerNorm channel has near-zero variance."""
    from dvmvs.convlstm import MVSLayernormConvLSTMCell
    tc_mode(1)
    h_, w_ = hw
    C = 512
    cellm = MVSLayernormConvLSTMCell(C, C, (3, 3), torch.celu)
    with torch.no_grad():
        cellm.conv.weight.copy_(_rand("lstm/w", (4 * C, 2 * C, 3, 3), (1.0 / (2 * C * 9)) ** 0.5))
    cellm = cellm.to(DEV).eval()
    conv_x, conv_h = cellm.packed()
    x, h, c = (_nhwc(_rand("lstm/" + n, (1, C, h_, w_))).to(DEV) for n in ("x", "h", "c"))
    xa, ha = ops.Act(x), ops.Act(h)
    gx = conv_x.run([(xa, D)], want_planes=False)
    expect = tc_ksplit(1, h_, w_, 4 * C, 3, 1, 128)
    assert expect > 1
    with nan_filled_outputs():
        deferred = conv_h.run_deferred([(ha, D)])
        assert deferred is not None and deferred[0] == "parts"
        ws, off, n_parts, stride = deferred[1]
        assert n_parts == expect and stride == h_ * w_ * 4 * C
        h_f, c_f = ops.lstm_gates(None, c, parts=deferred[1], addend=gx.f32)
        gates = conv_h.run([(ha, D)], residual=gx, residual_mode=N.RES_SAME, want_planes=False)
        h_u, c_u = ops.lstm_gates(gates.f32, c)
    for t, n in ((h_f, "h fused"), (c_f, "c fused"), (gates.f32, "gates"), (h_u, "h"), (c_u, "c")):
        assert_all_written(t, n)
    assert_same_bits(h_f, h_u, "h_next fused vs two-launch")
    assert_same_bits(c_f, c_u, "c_next fused vs two-launch")

    ptc = conv_h._ptc
    acc, S = conv_terms64([ha.planes], tc_weights(ptc, ptc.w_hi), tc_weights(ptc, ptc.w_lo), 1, 1)
    g64, S = epilogue64(acc, S, None, gx.f32, N.RES_SAME, N.ACT_NONE)
    cgate = tc_chunks(ptc) + n_parts + 4
    assert_within(gates.f32, g64, S, cgate, "lstm gates %dx%d ksplit=%d" % (h_, w_, n_parts))
    delta = cgate * U * S + U * g64.abs()
    ref_h, ref_c, bh, bc = cell_bound(g64, c.double().cpu(), delta, h_ * w_)
    assert_cell_within(h_f, c_f, ref_h, ref_c, bh, bc, "lstm cell %dx%d" % (h_, w_))


# ------------------------------------------------------------------------------------------------ D. every lstm_gates_kernel instantiation
LSTM_SHAPES = [
    # variant, (B, C, h, w)
    ("<2,8>", (1, 512, 4, 5)),
    ("<2,8>", (1, 512, 8, 8)),          # hw 64
    ("<2,8>", (1, 2336, 2, 3)),         # B*C/32 = 73
    ("<4,8>", (2, 64, 8, 10)),
    ("<4,8>", (1, 512, 5, 13)),         # hw 65
    ("<4,8>", (1, 512, 8, 16)),         # hw 128
    ("<16,8>", (1, 512, 16, 20)),
    ("<16,8>", (1, 64, 13, 39)),        # ragged
    ("<16,8>", (1, 512, 3, 43)),        # hw 129
    ("<16,8>", (1, 64, 16, 32)),        # hw 512
    ("<2,32>", (5, 512, 3, 5)),
    ("<2,32>", (2, 1184, 2, 3)),        # B*C/32 = 74
    ("<8,32>", (5, 512, 8, 8)),
    ("<8,32>", (5, 512, 1, 17)),        # hw 17
    ("<16,32>", (5, 512, 8, 10)),
    ("<16,32>", (5, 512, 8, 16)),       # hw 128
    ("<64,32>", (5, 512, 16, 20)),
    ("<64,32>", (5, 512, 3, 43)),       # hw 129
    ("<64,32>", (5, 512, 16, 32)),      # hw 512
]
LSTM_REFUSED = [(5, 512, 16, 33), (1, 64, 19, 27)]         # hw > 512: wide (and narrow-sized, which falls through to wide)


@pytest.mark.gpu
@pytest.mark.parametrize("variant,shape", LSTM_SHAPES, ids=["%s-%dx%dx%dx%d" % ((v,) + s) for v, s in LSTM_SHAPES])
def test_lstm_gates_parts_every_variant(variant, shape):
    """dvmvs_lstm_gates_parts with 1 or 3 partial sums, with and without addend, parts spaced wider than the minimum (the
    gaps hold NaN: a read outside the parts shows up) vs the float64 cell."""
    assert lstm_variant(*shape) == variant
    B, C, h, w = shape
    hw = h * w
    n = B * hw * 4 * C
    c = _nhwc(_rand("lg/c/%s" % (shape,), (B, C, h, w))).to(DEV)
    for n_parts in (1, 3):
        for with_addend in (False, True):
            stride = n + 96
            parts = [_rand("lg/p%d/%s" % (k, shape), (B, h, w, 4 * C), (1.0 / (n_parts + with_addend)) ** 0.5) for k in range(n_parts)]
            ws = torch.full((n_parts * stride,), float("nan"), dtype=torch.float32, device=DEV)
            for k, p in enumerate(parts):
                ws[k * stride:k * stride + n] = p.reshape(-1).to(DEV)
            addend = _rand("lg/a/%s" % (shape,), (B, h, w, 4 * C), (1.0 / (n_parts + 1)) ** 0.5) if with_addend else None
            with nan_filled_outputs():
                h_out, c_out = ops.lstm_gates(None, c, parts=(ws, 0, n_parts, stride), addend=addend.to(DEV) if with_addend else None)
            assert_all_written(h_out, "h_out")
            assert_all_written(c_out, "c_out")
            terms = parts + ([addend] if with_addend else [])
            g64 = sum(t.double() for t in terms)
            delta = (len(terms) + 1) * EPS32 * sum(t.double().abs() for t in terms)
            ref_h, ref_c, bh, bc = cell_bound(g64, c.double().cpu(), delta, hw)
            assert_cell_within(h_out, c_out, ref_h, ref_c, bh, bc, "lstm_gates %s %s parts=%d addend=%d" % (variant, shape, n_parts, with_addend))


@pytest.mark.gpu
@pytest.mark.parametrize("shape", LSTM_REFUSED)
def test_lstm_gates_refuses_maps_over_512_positions(shape):
    """More than 512 positions: RuntimeError before any launch (the outputs keep their sentinel)."""
    assert lstm_variant(*shape) is None
    B, C, h, w = shape
    gates = torch.zeros(B, h, w, 4 * C, device=DEV)
    c = torch.zeros(B, h, w, C, device=DEV)
    h_out = torch.full_like(c, 7.0)
    c_out = torch.full_like(c, 7.0)
    launches = N.launch_count()
    with pytest.raises(RuntimeError):
        N.check(N.lib().dvmvs_lstm_gates_parts(gates.data_ptr(), 1, 0, None, c.data_ptr(), h_out.data_ptr(), c_out.data_ptr(), B, h, w, C,
                                               ops._stream()), "lstm_gates_parts")
    torch.cuda.synchronize()
    assert N.launch_count() == launches
    assert bool((h_out == 7.0).all()) and bool((c_out == 7.0).all())


# ------------------------------------------------------------------------------------------------ E. batch-slice operand views
def _producers(terms):
    """tc producer: 1x1 16->32 at 64x64 (emits pair planes + blocked planes); halo producer: 3x3 32->32 on its output."""
    tc = ops.ConvLayer(ops.PackedConv(_rand("bs/w1", (32, 16, 1, 1), 0.35).to(DEV), _rand("bs/b1", (32,), 0.1).to(DEV), act=N.ACT_RELU))
    halo = ops.ConvLayer(ops.PackedConv(_rand("bs/w2", (32, 32, 3, 3), 0.08).to(DEV), _rand("bs/b2", (32,), 0.1).to(DEV), act=N.ACT_RELU))
    return tc, halo


@pytest.mark.gpu
@pytest.mark.parametrize("producer", ["tc", "halo"])
def test_batch_slice_views_feed_consumers_like_contiguous_copies(tc_mode, cases, synth, producer):
    """1-term hi-only: B = 4 activations produced by a real tc / halo layer; the entries outside [1, 3) are NaN.
    batch_slice(t, 1, 3) hands its strided hi / blocked views to a conv2d_tc consumer, a conv2d_halo consumer and
    plane_sweep_tc; each result is bit-identical to the same consumer on .contiguous() copies."""
    tc_mode(1)
    tc, halo = _producers(1)
    x = ops.Act(_nhwc(_rand("bs/x", (4, 16, 64, 64))).to(DEV))
    with nan_filled_outputs():
        a = tc.run([(x, D)])
        if producer == "halo":
            assert halo.path(64, 64) == "halo"
            a = halo.run([(a, D)])
    assert a.planes is not None and a.blk is not None
    for t in (a.f32.unsqueeze(0), a.planes, a.blk):
        t[:, 0].fill_(float("nan"))
        t[:, 3].fill_(float("nan"))
    t = ops.act_to_api(a)
    s = ops.batch_slice(t, 1, 3)
    va = ops.to_act(s)
    assert va.planes is not None and va.blk is not None and not va.planes.is_contiguous()
    assert va.planes[0].data_ptr() == a.planes[0, 1].data_ptr() and va.blk[0].data_ptr() == a.blk[0, 1].data_ptr()
    ca = ops.Act(va.f32.contiguous(), va.planes.contiguous(), va.blk.contiguous())

    consumer_tc = ops.ConvLayer(ops.PackedConv(_rand("bs/w3", (32, 32, 1, 1), 0.25).to(DEV), None, act=N.ACT_NONE))
    consumer_halo = ops.ConvLayer(ops.PackedConv(_rand("bs/w4", (32, 32, 5, 5), 0.05).to(DEV), None, act=N.ACT_RELU))
    assert consumer_tc.path(64, 64) == "tc" and consumer_halo.path(64, 64) == "halo"
    for layer, label in ((consumer_tc, "conv2d_tc"), (consumer_halo, "conv2d_halo")):
        got, want = layer.run([(va, D)]), layer.run([(ca, D)])
        assert_all_written(got.f32, label)
        assert_same_bits(got.f32, want.f32, label + " on batch-slice views")
        assert_same_bits(got.planes[0], want.planes[0], label + " on batch-slice views (hi plane)")
        assert_same_bits(got.blk[0], want.blk[0], label + " on batch-slice views (blocked hi)")

    # plane sweep over 32-channel 24x40 features of the same producer, poses / K of the golden 'dot_small' case (B = 2)
    c = cases.PLANE_SWEEP_CASES["dot_small"]
    inp = cases.plane_sweep_inputs(synth, c)
    cu = lambda arr: torch.from_numpy(np.ascontiguousarray(arr)).to(DEV)
    feats = []
    for m in range(3):
        xm = ops.Act(_nhwc(_rand("bs/sweep%d" % m, (4, 16, c["h"], c["w"]))).to(DEV))
        with nan_filled_outputs():
            fm = tc.run([(xm, D)])
        for pl in (fm.planes[:, 0], fm.planes[:, 3]):
            pl.fill_(float("nan"))
        feats.append(ops.to_act(ops.batch_slice(ops.act_to_api(fm), 1, 3)))
    pairs = [ops.act_pair(f) for f in feats]
    copies = [(hi.clone(), lo.clone()) for hi, lo in pairs]
    poses = (cu(inp["pose1"]), [cu(p) for p in inp["pose2s"]], cu(inp["K"]))
    got = ops.plane_sweep_tc(pairs[0], pairs[1:], *poses, c["min_depth"], c["max_depth"], c["D"], terms=1)
    want = ops.plane_sweep_tc(copies[0], copies[1:], *poses, c["min_depth"], c["max_depth"], c["D"], terms=1)
    assert torch.isfinite(got).all()
    assert_same_bits(got, want, "plane_sweep_tc on batch-slice views")


@pytest.mark.gpu
def test_batch_slice_attaches_no_stacked_views_with_three_terms(tc_mode):
    """3-term configuration: the kernels locate the lo plane at +B*H*W*C from the hi plane, so batch_slice attaches only the
    (hi, lo) pair, never the stacked planes / blocked views."""
    tc_mode(3)
    tc, _ = _producers(3)
    a = tc.run([(ops.Act(_nhwc(_rand("bs3/x", (4, 16, 64, 64))).to(DEV)), D)])
    assert a.planes is not None and a.blk is not None
    s = ops.batch_slice(ops.act_to_api(a), 1, 3)
    va = ops.to_act(s)
    assert va.planes is None and va.blk is None
    assert va.pair is not None and va.pair[1].data_ptr() == a.planes[1, 1].data_ptr()


# ------------------------------------------------------------------------------------------------ F. sensitivity (CPU)
def _cpu_tc_case(name, B, H, W, cin, Cout, k, terms, res=None):
    """CPU stand-in for a kernel run: fp16 (hi, lo) planes, PackedConvTC weights, and the product evaluated in float32 (an
    fp32-accumulating convolution of the same operands), with the fp32 epilogue."""
    x = _nhwc(_rand(name + "/x", (B, cin, H, W)))
    hi = x.half()
    planes = [torch.stack([hi, (x - hi.float()).half()])]
    w = _rand(name + "/w", (Cout, cin, k, k), (2.0 / (cin * k * k)) ** 0.5)
    bias = _rand(name + "/b", (Cout,), 0.1)
    pc = ops.PackedConv(w, bias, None, stride=1, act=N.ACT_NONE)
    ptc = ops.PackedConvTC(pc, [cin], "cpu")
    whi, wlo = tc_weights(ptc, ptc.w_hi), tc_weights(ptc, ptc.w_lo)
    xs = planes[0].float().permute(0, 1, 4, 2, 3)
    pad = (k - 1) // 2
    got = F.conv2d(xs[0], whi[0].float(), None, 1, pad)
    if terms == 3:
        got = got + F.conv2d(xs[1], whi[0].float(), None, 1, pad) + F.conv2d(xs[0], wlo[0].float(), None, 1, pad)
    got = got + pc.bias.view(1, -1, 1, 1)
    mode, residual = N.RES_NONE, None
    if res is not None:
        mode, residual = N.RES_NEAREST_UP, _nhwc(_rand(name + "/r", (B, Cout) + res))
        got = got + F.interpolate(residual.permute(0, 3, 1, 2), size=(H, W), mode="nearest")
    return planes, ptc, whi, wlo, pc, residual, mode, got.permute(0, 2, 3, 1)


def test_sensitivity_dropped_k_chunk():
    planes, ptc, whi, wlo, pc, res, mode, got = _cpu_tc_case("sens/chunk", 1, 8, 10, 96, 32, 3, 1)
    c = tc_chunks(ptc) + 1 + 4
    acc, S = conv_terms64(planes, whi, wlo, 1, 1)
    assert_within(got, *epilogue64(acc, S, pc.bias, res, mode, N.ACT_NONE), c, "sensitivity: correct reference")
    bad = [w.clone() for w in whi]
    bad[0][:, 32:64, 1, 2] = 0                          # tap (1, 2), second of its three 32-channel chunks
    acc, S = conv_terms64(planes, bad, wlo, 1, 1)
    with pytest.raises(AssertionError):
        assert_within(got, *epilogue64(acc, S, pc.bias, res, mode, N.ACT_NONE), c, "sensitivity: dropped K chunk")


def test_sensitivity_lo_hi_term_omitted():
    planes, ptc, whi, wlo, pc, res, mode, got = _cpu_tc_case("sens/lohi", 1, 8, 10, 64, 32, 3, 3)
    c = tc_chunks(ptc) + 1 + 4
    acc, S = conv_terms64(planes, whi, wlo, 3, 1)
    assert_within(got, *epilogue64(acc, S, pc.bias, res, mode, N.ACT_NONE), c, "sensitivity: correct reference")
    acc, S = conv_terms64(planes, whi, wlo, 3, 1, drop_lo_hi=True)
    with pytest.raises(AssertionError):
        assert_within(got, *epilogue64(acc, S, pc.bias, res, mode, N.ACT_NONE), c, "sensitivity: lo*hi omitted")


def test_sensitivity_residual_row_off_by_one():
    planes, ptc, whi, wlo, pc, res, mode, got = _cpu_tc_case("sens/res", 2, 15, 13, 40, 32, 1, 1, res=(8, 7))
    c = tc_chunks(ptc) + 1 + 4
    acc, S = conv_terms64(planes, whi, wlo, 1, 1)
    assert_within(got, *epilogue64(acc, S, pc.bias, res, mode, N.ACT_NONE), c, "sensitivity: correct reference")
    with pytest.raises(AssertionError):
        assert_within(got, *epilogue64(acc, S, pc.bias, res, mode, N.ACT_NONE, row_shift=1), c, "sensitivity: residual row + 1")


def _cpu_gate_case(B, C, h, w, n_parts):
    parts = [_rand("sens/p%d" % k, (B, h, w, 4 * C), (1.0 / n_parts) ** 0.5) for k in range(n_parts)]
    c = _nhwc(_rand("sens/c", (B, C, h, w)))
    g32 = parts[0].clone()
    for p in parts[1:]:
        g32 = g32 + p
    got_h, got_c, _ = cell(g32, c)                       # the cell evaluated in float32, as the kernel does
    return parts, c, got_h, got_c


def test_sensitivity_one_split_missing():
    parts, c, got_h, got_c = _cpu_gate_case(1, 64, 8, 10, 3)
    delta = (len(parts) + 1) * EPS32 * sum(p.double().abs() for p in parts)
    ref = cell_bound(sum(p.double() for p in parts), c.double(), delta, 80)
    assert_cell_within(got_h, got_c, *ref, "sensitivity: correct reference")
    bad = cell_bound(sum(p.double() for p in parts[:-1]), c.double(), delta, 80)
    with pytest.raises(AssertionError):
        assert_cell_within(got_h, got_c, *bad, "sensitivity: one split missing")


def test_sensitivity_layernorm_over_channels():
    parts, c, got_h, got_c = _cpu_gate_case(1, 64, 8, 10, 1)
    delta = 2 * EPS32 * parts[0].double().abs()
    ref_h, ref_c, bh, bc = cell_bound(parts[0].double(), c.double(), delta, 80)
    assert_cell_within(got_h, got_c, ref_h, ref_c, bh, bc, "sensitivity: correct reference")
    bad_h, bad_c, _ = cell(parts[0].double(), c.double(), ln_dims=(3,))
    with pytest.raises(AssertionError):
        assert_cell_within(got_h, got_c, bad_h, bad_c, bh, bc, "sensitivity: LayerNorm over channels")


def test_sensitivity_one_unwritten_element():
    out = torch.full((2, 2, 5, 7, 40), float("nan"), dtype=torch.float16)
    out[0] = 1.0
    out[1] = 0.5
    assert_all_written(out, "sensitivity: fully written")
    out[0, 1, 4, 6, 39] = float("nan")
    with pytest.raises(AssertionError):
        assert_all_written(out, "sensitivity: one unwritten element")
    f32 = _rand("sens/f32", (2, 5, 7, 40))
    planes = torch.stack([f32.half(), torch.full_like(f32, float("nan")).half()])
    assert_planes_exact(f32, planes, True, "sensitivity: hi-only planes")
    planes[1, 0, 0, 0, 0] = 0.0                           # one stray lo write
    with pytest.raises(AssertionError):
        assert_planes_exact(f32, planes, True, "sensitivity: stray lo write")


def test_lstm_variant_mirror_covers_every_instantiation():
    """The dispatch mirror names each of the seven lstm_gates_kernel instantiations for at least one table shape, and every
    table shape for the variant the table says."""
    for variant, shape in LSTM_SHAPES:
        assert lstm_variant(*shape) == variant, (variant, shape)
    assert {v for v, _ in LSTM_SHAPES} == {"<2,8>", "<4,8>", "<16,8>", "<2,32>", "<8,32>", "<16,32>", "<64,32>"}
    for shape in LSTM_REFUSED:
        assert lstm_variant(*shape) is None
