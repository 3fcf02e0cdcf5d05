"""GPU parity tests: the sm_100a kernels, reached through the reference-facing Python API (which binds the C ABI),
against (a) golden vectors generated from the unmodified reference, (b) the CPU oracle on seeded inputs, and
(c) the reference's shipped end-to-end golden predictions.  Tolerances: geometry / convs are fp32 on both sides
-> <= 2e-5 of the tensor's max magnitude; end-to-end <= 1e-3 relative L1 on inverse depth (BASELINE.json)."""
import numpy as np
import pytest
import torch

from tests import helpers, scene_fixture
from tests.helpers import T, rel_err

pytestmark = pytest.mark.gpu

DEV = "cuda"
REPO_DIR = __import__("os").path.dirname(__import__("os").path.dirname(__import__("os").path.abspath(__file__)))


def _cuda(x):
    return T(np.ascontiguousarray(x)).to(DEV)


# ------------------------------------------------------------------------------------------------ plane sweep
@pytest.mark.parametrize("layout", ["nchw", "channels_last"])
def test_plane_sweep_vs_reference_golden(synth, cases, golden_ops, layout):
    from dvmvs.utils import cost_volume_fusion, get_warp_grid_for_cost_volume_calculation
    for name, c in cases.PLANE_SWEEP_CASES.items():
        inp = cases.plane_sweep_inputs(synth, c)
        conv = (lambda t: t.contiguous(memory_format=torch.channels_last)) if layout == "channels_last" else (lambda t: t)
        grid = get_warp_grid_for_cost_volume_calculation(c["w"], c["h"], DEV)
        out = cost_volume_fusion(conv(_cuda(inp["image1"])), [conv(_cuda(x)) for x in inp["image2s"]], _cuda(inp["pose1"]),
                                 [_cuda(p) for p in inp["pose2s"]], _cuda(inp["K"]), grid, c["min_depth"], c["max_depth"], c["D"],
                                 DEV, c["dot"])
        assert tuple(out.shape) == (c["B"], c["D"], c["h"], c["w"])
        err = rel_err(out.cpu().numpy(), golden_ops["plane_sweep/" + name])
        assert err <= 2e-5, "plane_sweep/%s (%s): %.3e" % (name, layout, err)


def test_plane_sweep_fast_path_equals_generic_path(synth, cases):
    from dvmvs import _ops as ops
    c = cases.PLANE_SWEEP_CASES["dot_m3"]
    inp = cases.plane_sweep_inputs(synth, c)
    ref = ops.to_nhwc(_cuda(inp["image1"]))
    meas = [ops.to_nhwc(_cuda(x)) for x in inp["image2s"]]
    args = (ref, meas, _cuda(inp["pose1"]), [_cuda(p) for p in inp["pose2s"]], _cuda(inp["K"]), c["min_depth"], c["max_depth"], c["D"])
    for dot in (True, False):
        fast = ops.plane_sweep(*args, dot_product=dot)
        gen = ops.plane_sweep(*args, dot_product=dot, force_generic=True)
        assert rel_err(fast.cpu().numpy(), gen.cpu().numpy()) <= 1e-5


@pytest.mark.skipif(__import__("os").environ.get("DVMVS_SWEEP_FP16") != "1",
                    reason="experimental fp16-feature plane sweep: opt-in (DVMVS_SWEEP_FP16=1), not yet measured on hardware")
def test_plane_sweep_fp16_features_vs_fp32_kernel(synth, cases):
    """plane_sweep_c32_h16_kernel (16-bit measurement features, one 128-byte pair load per bilinear row) against the fp32
    kernel fed the SAME fp16-rounded features (<= 2e-5: same arithmetic up to summation order) and against the unrounded
    features (<= 2e-3: the rounding itself), including the wide-baseline case with taps off every image edge."""
    from dvmvs import _ops as ops
    for name in ("dot_small", "dot_c1", "dot_m3", "dot_wide", "dot_ident"):
        c = cases.PLANE_SWEEP_CASES[name]
        inp = cases.plane_sweep_inputs(synth, c)
        ref = ops.to_nhwc(_cuda(inp["image1"]))
        meas = [ops.to_nhwc(_cuda(x)) for x in inp["image2s"]]
        hi = [m.to(torch.float16).contiguous() for m in meas]
        args = (_cuda(inp["pose1"]), [_cuda(p) for p in inp["pose2s"]], _cuda(inp["K"]), c["min_depth"], c["max_depth"], c["D"])
        got = ops.plane_sweep_h16(ref, hi, *args).cpu().numpy()
        same_inputs = ops.plane_sweep(ref, [t.float() for t in hi], *args).cpu().numpy()
        exact = ops.plane_sweep(ref, meas, *args).cpu().numpy()
        assert rel_err(got, same_inputs) <= 2e-5, name
        assert rel_err(got, exact) <= 2e-3, name


@pytest.mark.parametrize("terms,tol", [(3, 2e-5), (1, 2e-3)])
def test_plane_sweep_tensor_core_form_vs_reference_golden(synth, cases, golden_ops, terms, tol):
    """plane_sweep_tc_kernel (band correlation on tcgen05 + scalar interpolation) against the golden vectors of the unmodified
    reference, every dot-product case: small / single-frame / three frames with rotation / wide baseline with samples off
    every edge and behind the camera (direct path) / identity pose.  terms=3 (fp16 (hi, lo) pairs) is held to the fp32
    tolerance of the gather kernel; terms=1 carries the rounding of the features to fp16 (<= 2e-3 of the cost volume's
    magnitude; <= 1.3e-6 on the final inverse depth, profiles/r01_feature_fp16_probe_cpu.jsonl)."""
    from dvmvs import _ops as ops
    for name, c in cases.PLANE_SWEEP_CASES.items():
        if not c["dot"] or c["C"] != 32:
            continue
        inp = cases.plane_sweep_inputs(synth, c)
        ref = ops.split_planes(ops.to_nhwc(_cuda(inp["image1"])))
        meas = [ops.split_planes(ops.to_nhwc(_cuda(x))) for x in inp["image2s"]]
        out = ops.plane_sweep_tc(ref, meas, _cuda(inp["pose1"]), [_cuda(p) for p in inp["pose2s"]], _cuda(inp["K"]), c["min_depth"],
                                 c["max_depth"], c["D"], terms=terms)
        got = out.permute(0, 3, 1, 2).cpu().numpy()
        err = rel_err(got, golden_ops["plane_sweep/" + name])
        assert np.isfinite(got).all() and err <= tol, "plane_sweep_tc/%s terms=%d: %.3e" % (name, terms, err)


@pytest.mark.parametrize("qcap", [512, 64])
def test_plane_sweep_tensor_core_form_full_size_and_band_capacity(synth, qcap):
    """BASELINE configs 2 / 3 shapes and a batch of clips with different poses against the fp32 gather kernel; qcap=64
    forces tiny chunks and the direct path for planes whose band does not fit (same results either way)."""
    import subprocess, sys, json, os
    code = r"""
import sys, json, numpy as np, torch
sys.path[:0] = [%r, %r]
import synth_data as synth
from dvmvs import _ops as ops
res = []
for (B, h, w, D, M) in ((1, 128, 128, 64, 2), (1, 128, 160, 96, 4), (3, 64, 96, 64, 2)):
    g = torch.Generator().manual_seed(D + B)
    f1 = (torch.randn(B, h, w, 32, generator=g) * 4).cuda()
    f2 = [(torch.randn(B, h, w, 32, generator=g) * 4).cuda() for _ in range(M)]
    K = torch.from_numpy(synth.intrinsics(2 * h, 2 * w))[None].repeat(B, 1, 1).cuda(); K[:, 0:2, :] /= 2.0
    pose1 = torch.stack([torch.from_numpy(synth.camera_pose(M + 3 * b)) for b in range(B)]).cuda()
    pose2 = [torch.stack([torch.from_numpy(synth.camera_pose(M + 3 * b - k * (1 + b))) for b in range(B)]).cuda() for k in range(1, M + 1)]
    base = ops.plane_sweep(f1, f2, pose1, pose2, K, 0.25, 20.0, D, True)
    got = ops.plane_sweep_tc(ops.split_planes(f1), [ops.split_planes(t) for t in f2], pose1, pose2, K, 0.25, 20.0, D, terms=3)
    res.append(float((got - base).abs().max() / base.abs().max()))
print(json.dumps(res))
""" % (REPO_DIR, os.path.join(REPO_DIR, "deep-video-mvs_b200"))
    env = dict(os.environ, DVMVS_SWEEP_QCAP=str(qcap))        # read once per process by the library
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    errs = json.loads(out.stdout.strip().splitlines()[-1])
    assert all(e <= 2e-5 for e in errs), errs


def test_calculate_cost_volume_by_warping_is_single_frame_fusion(oracle, synth, cases):
    from dvmvs.utils import calculate_cost_volume_by_warping
    c = cases.PLANE_SWEEP_CASES["dot_c1"]
    inp = cases.plane_sweep_inputs(synth, c)
    out = calculate_cost_volume_by_warping(_cuda(inp["image1"]), _cuda(inp["image2s"][0]), _cuda(inp["pose1"]),
                                           _cuda(inp["pose2s"][0]), _cuda(inp["K"]), None, c["min_depth"], c["max_depth"],
                                           c["D"], DEV, True)
    gold = oracle.calculate_cost_volume_by_warping(T(inp["image1"]), T(inp["image2s"][0]), T(inp["pose1"]), T(inp["pose2s"][0]),
                                                   T(inp["K"]), oracle.get_warp_grid_for_cost_volume_calculation(c["w"], c["h"]),
                                                   c["min_depth"], c["max_depth"], c["D"], "cpu", True)
    assert rel_err(out.cpu().numpy(), gold.numpy()) <= 2e-5


def test_plane_sweep_full_size_configs_vs_oracle(oracle, synth):
    """BASELINE.json configs 2 and 3 shapes (128x128 D=64 M=2; 128x160 D=96 M=4) with the synthetic-clip geometry."""
    from dvmvs.utils import cost_volume_fusion
    for (h, w, D, M) in ((128, 128, 64, 2), (128, 160, 96, 4)):
        f1 = synth.tensor("full/ref", (1, 32, h, w), seed=D, scale=4.0)
        f2s = [synth.tensor("full/m%d" % m, (1, 32, h, w), seed=D, scale=4.0) for m in range(M)]
        pose1 = synth.camera_pose(M)[None]
        pose2s = [synth.camera_pose(M - k)[None] for k in range(1, M + 1)]
        K = synth.intrinsics(2 * h, 2 * w)[None].copy()
        K[:, 0:2, :] /= 2.0
        out = cost_volume_fusion(_cuda(f1), [_cuda(x) for x in f2s], _cuda(pose1), [_cuda(p) for p in pose2s], _cuda(K), None,
                                 0.25, 20.0, D, DEV, True)
        gold = oracle.cost_volume_fusion(T(f1), [T(x) for x in f2s], T(pose1), [T(p) for p in pose2s], T(K),
                                         oracle.get_warp_grid_for_cost_volume_calculation(w, h), 0.25, 20.0, D, "cpu", True)
        assert rel_err(out.cpu().numpy(), gold.numpy()) <= 1e-4, (h, w, D, M)


def test_plane_sweep_linearity_and_frame_permutation(synth, cases):
    """Size-independent properties: the cost volume is linear in the reference features and invariant to the order
    of the measurement frames (up to fp32 summation order)."""
    from dvmvs.utils import cost_volume_fusion
    c = cases.PLANE_SWEEP_CASES["dot_m3"]
    inp = cases.plane_sweep_inputs(synth, c)
    f1, f2s = _cuda(inp["image1"]), [_cuda(x) for x in inp["image2s"]]
    p1, p2s, K = _cuda(inp["pose1"]), [_cuda(p) for p in inp["pose2s"]], _cuda(inp["K"])
    a = cost_volume_fusion(f1, f2s, p1, p2s, K, None, 0.25, 20.0, c["D"], DEV, True)
    b = cost_volume_fusion(2.0 * f1, f2s, p1, p2s, K, None, 0.25, 20.0, c["D"], DEV, True)
    assert rel_err(b.cpu().numpy(), 2.0 * a.cpu().numpy()) <= 1e-6
    p = cost_volume_fusion(f1, f2s[::-1], p1, p2s[::-1], K, None, 0.25, 20.0, c["D"], DEV, True)
    assert rel_err(p.cpu().numpy(), a.cpu().numpy()) <= 1e-5


# ------------------------------------------------------------------------------------------------ hidden warp / re-projection
def test_hidden_warp_vs_reference_golden(synth, cases, golden_ops):
    from dvmvs.utils import warp_frame_depth
    for name, c in cases.HIDDEN_WARP_CASES.items():
        inp = cases.hidden_warp_inputs(synth, c)
        out = warp_frame_depth(_cuda(inp["image_src"]), _cuda(inp["depth_dst"]), _cuda(inp["trans"]), _cuda(inp["K"]))
        err = rel_err(out.cpu().numpy(), golden_ops["hidden_warp/" + name])
        assert err <= 2e-5, "hidden_warp/%s: %.3e" % (name, err)


def test_reprojection_vs_reference_golden(synth, cases, golden_ops):
    from dvmvs.utils import get_non_differentiable_rectangle_depth_estimation
    for name, c in cases.REPROJECT_CASES.items():
        inp = cases.reproject_inputs(synth, c)
        out = get_non_differentiable_rectangle_depth_estimation(_cuda(inp["reference_pose"]), _cuda(inp["measurement_pose"]),
                                                                _cuda(inp["previous_depth"]), _cuda(inp["full_K"]),
                                                                _cuda(inp["half_K"]), c["W"], c["H"]).cpu().numpy()
        gold = golden_ops["reproject/" + name]
        assert out.shape == gold.shape
        differ = np.abs(out - gold) > 1e-5 * np.maximum(1.0, np.abs(gold))
        # a differing pixel would be a rounding tie of the scatter target (a source point 1e-7 from a .5 pixel boundary landing in
        # the neighbouring cell under fp32 re-association).  Measured on B200 (round 2): 0 of 16 384 (c2) and 0 of 2 048 (batch)
        # half-resolution pixels differ -- the bound is two tie flips per case, not a ratio that could hide dozens.
        print("reproject/%s: %d of %d half-resolution pixels differ from the reference golden" % (name, int(differ.sum()), differ.size))
        assert int(differ.sum()) <= 2, "reproject/%s: %d of %d pixels differ" % (name, int(differ.sum()), differ.size)


def test_reprojection_is_idempotent_under_identity(synth):
    """Identity motion: every half-res pixel (i, j) receives the source points that round onto it; the winner is the
    farthest of them -> max-pool structure, checked against a direct numpy evaluation."""
    from dvmvs.utils import get_non_differentiable_rectangle_depth_estimation
    H, W = 64, 96
    depth = (1.0 + np.abs(synth.tensor("idem", (1, 1, H, W), seed=3))).astype(np.float32)
    K = synth.intrinsics(H, W)[None]
    hK = K.copy()
    hK[:, 0:2, :] /= 2.0
    eye = np.eye(4, dtype=np.float32)[None]
    out = get_non_differentiable_rectangle_depth_estimation(_cuda(eye), _cuda(eye), _cuda(depth), _cuda(K), _cuda(hK), W, H).cpu().numpy()
    assert out.shape == (1, 1, H // 2, W // 2)
    assert out.max() <= depth.max() + 1e-6 and out.min() >= 0.0
    assert (out > 0).mean() > 0.9


# ------------------------------------------------------------------------------------------------ conv kernels vs torch fp32 (CPU)
CONV_CASES = [
    # B, Hin, Win, [src channels], [src modes], Cout, k, stride, act, residual
    (1, 16, 24, [32], [0], 32, 3, 1, 1, 0),
    (2, 17, 23, [3], [0], 32, 3, 2, 1, 0),            # stem-like, odd size, Cin=3
    (1, 32, 32, [32, 64], [0, 0], 32, 5, 1, 1, 0),    # aggregator0-like concat
    (1, 16, 16, [32], [0], 64, 5, 2, 1, 0),
    (1, 8, 10, [512, 512], [0, 0], 96, 3, 1, 0, 0),   # small spatial, deep K -> split-K path
    (1, 8, 8, [192], [0], 40, 1, 1, 0, 1),            # 1x1 + same-size residual (MnasNet)
    (1, 16, 16, [24], [0], 32, 1, 1, 0, 2),           # 1x1 + nearest-up residual (FPN)
    (1, 16, 16, [16, 16, 1], [0, 0, 1], 16, 3, 1, 1, 0),   # decoder concat with upsampled 1-channel depth
    (1, 32, 32, [64], [1], 32, 3, 1, 1, 0),           # up-convolution: x2 bilinear fused
    (1, 32, 32, [32, 1, 3], [1, 1, 0], 32, 5, 1, 1, 0),    # refine.0-like
    (1, 12, 20, [64], [0], 1, 3, 1, 2, 0),            # depth head (sigmoid + aux depth)
    (1, 9, 7, [20], [0], 1, 3, 1, 2, 0),              # head fallback (Cin not a multiple of 32)
    (1, 16, 16, [1152], [0], 192, 1, 1, 0, 0),        # deep 1x1
    (1, 8, 8, [8], [0], 24, 1, 2, 0, 0),
]


@pytest.mark.parametrize("case", CONV_CASES)
def test_conv2d_vs_torch_fp32(synth, case):
    import torch.nn.functional as F
    from dvmvs import _native as N
    from dvmvs import _ops as ops
    B, Hin, Win, chans, modes, Cout, k, stride, act, res = case
    key = "conv/" + "_".join(str(v) for v in (B, Hin, Win, Cout, k, stride, act, res) + tuple(chans))
    srcs_cpu, full = [], []
    for i, (cs, mode) in enumerate(zip(chans, modes)):
        f = 2 if mode == 1 else 1
        x = T(synth.tensor(key + "/x%d" % i, (B, cs, Hin // f, Win // f), seed=1))
        srcs_cpu.append(x)
        full.append(F.interpolate(x, scale_factor=2, mode="bilinear", align_corners=True) if mode == 1 else x)
    cin = sum(chans)
    w = T(synth.tensor(key + "/w", (Cout, cin, k, k), seed=2, scale=(2.0 / (cin * k * k)) ** 0.5))
    bias = T(synth.tensor(key + "/b", (Cout,), seed=3, scale=0.1))
    ref = F.conv2d(torch.cat(full, 1), w, bias, stride, (k - 1) // 2)
    Hout, Wout = ref.shape[-2:]
    residual = None
    if res == 1:
        residual = T(synth.tensor(key + "/r", (B, Cout, Hout, Wout), seed=4))
        ref = ref + residual
    elif res == 2:
        residual = T(synth.tensor(key + "/r", (B, Cout, Hout // 2, Wout // 2), seed=4))
        ref = ref + F.interpolate(residual, size=(Hout, Wout), mode="nearest")
    ref = {0: ref, 1: F.relu(ref), 2: torch.sigmoid(ref)}[act]
    conv = torch.nn.Conv2d(cin, Cout, k, bias=True)
    pc = ops.PackedConv(w, bias, None, stride=stride, act=act)
    pc.weight, pc.bias = pc.weight.to(DEV), pc.bias.to(DEV)
    aux = (3.95, 0.05) if act == 2 else None
    out = ops.conv2d([(ops.to_nhwc(x.to(DEV)), m) for x, m in zip(srcs_cpu, modes)], pc,
                     residual=None if residual is None else ops.to_nhwc(residual.to(DEV)),
                     residual_mode={0: N.RES_NONE, 1: N.RES_SAME, 2: N.RES_NEAREST_UP}[res], aux=aux)
    if aux is not None:
        out, aux_out = out
        assert rel_err(ops.to_api(aux_out).cpu().numpy(), (1.0 / (3.95 * ref + 0.05)).numpy()) <= 2e-5
    assert rel_err(ops.to_api(out).cpu().numpy(), ref.numpy()) <= 2e-5, case
    del conv


@pytest.mark.parametrize("case", [(1, 16, 16, 32, 3, 1), (2, 17, 15, 48, 5, 2), (1, 8, 8, 1152, 5, 1), (1, 32, 32, 72, 3, 2)])
def test_dwconv_vs_torch_fp32(synth, case):
    import torch.nn.functional as F
    from dvmvs import _ops as ops
    B, H, W, C, k, stride = case
    x = T(synth.tensor("dw/x%d" % C, (B, C, H, W), seed=1))
    conv = torch.nn.Conv2d(C, C, k, padding=k // 2, stride=stride, groups=C, bias=False)
    bn = torch.nn.BatchNorm2d(C).eval()
    sd = synth.make_state_dict({"weight": (C,), "bias": (C,), "running_mean": (C,), "running_var": (C,)}, seed=5)
    with torch.no_grad():
        conv.weight.copy_(T(synth.tensor("dw/w%d" % C, (C, 1, k, k), seed=2, scale=0.3)))
        for kk in sd:
            getattr(bn, kk).copy_(T(sd[kk]))
        ref = F.relu(bn(conv(x)))
    pd = ops.PackedDepthwise(conv.weight, bn, stride)
    pd.weight, pd.bias = pd.weight.to(DEV), pd.bias.to(DEV)
    out = ops.dwconv2d(ops.to_nhwc(x.to(DEV)), pd)
    assert rel_err(ops.to_api(out).cpu().numpy(), ref.numpy()) <= 2e-5
    if C % 8 == 0:
        out2, planes = ops.dwconv2d(ops.to_nhwc(x.to(DEV)), pd, want_f32=True, want_planes=True)
        assert torch.equal(out2, out)
        assert rel_err((planes[0].float() + planes[1].float()).cpu().numpy(), out.cpu().numpy()) <= 2e-6


def test_layout_roundtrip_and_upsample(synth):
    import torch.nn.functional as F
    from dvmvs import _ops as ops
    x = T(synth.tensor("lay", (2, 37, 9, 13), seed=1)).to(DEV)
    nhwc = ops.to_nhwc(x)
    assert torch.equal(nhwc, x.permute(0, 2, 3, 1))
    assert torch.equal(ops.to_nchw_contiguous(nhwc), x)
    up = ops.to_api(ops.upsample2x(nhwc)).cpu()
    assert rel_err(up.numpy(), F.interpolate(x.cpu(), scale_factor=2, mode="bilinear", align_corners=True).numpy()) <= 1e-6


# ------------------------------------------------------------------------------------------------ ConvLSTM cell
def test_lstm_cell_vs_reference_golden(synth, cases, golden_ops):
    from dvmvs.convlstm import MVSLayernormConvLSTMCell
    for name, c in cases.LSTM_CASES.items():
        inp = cases.lstm_inputs(synth, c)
        cell = MVSLayernormConvLSTMCell(512, 512, (3, 3), activation_function=torch.celu)
        cell.load_state_dict({"conv.weight": T(inp["weight"])})
        cell.to(DEV).eval()
        h, cc = cell(_cuda(inp["x"]), [_cuda(inp["h"]), _cuda(inp["c"])], _cuda(inp["previous_pose"]) if c["warp"] else None,
                     _cuda(inp["current_pose"]), _cuda(inp["depth"]), _cuda(inp["K"]))
        assert rel_err(h.cpu().numpy(), golden_ops["lstm/%s/h" % name]) <= 1e-4, name
        assert rel_err(cc.cpu().numpy(), golden_ops["lstm/%s/c" % name]) <= 1e-4, name


# ------------------------------------------------------------------------------------------------ whole modules
def test_modules_vs_reference_golden(oracle, synth, cases, golden_modules):
    c = cases.MODULE_CASE
    w = helpers.oracle_weights(oracle, synth, c["seed"])
    mods = helpers.build_product_modules(w)
    inp = cases.module_inputs(synth, c)
    image = _cuda(inp["image"])
    with torch.no_grad():
        l = mods["fe"](image)
        for i, x in enumerate(l):
            assert rel_err(x.cpu().numpy(), golden_modules["fe/%d" % i]) <= 5e-5, "fe/%d" % i
        f = mods["fpn"](*l)
        for i, x in enumerate(f):
            assert rel_err(x.cpu().numpy(), golden_modules["fpn/%d" % i]) <= 5e-5, "fpn/%d" % i
        enc = mods["cve"](*f, _cuda(inp["cost_volume"]))
        for i, x in enumerate(enc):
            assert rel_err(x.cpu().numpy(), golden_modules["cve/%d" % i]) <= 1e-4, "cve/%d" % i
        h0, c0 = mods["lstm"](enc[4], None, None, _cuda(inp["pose0"]), _cuda(inp["depth_est"]), _cuda(inp["lstm_K"]))
        h1, c1 = mods["lstm"](enc[4], (h0, c0), _cuda(inp["pose0"]), _cuda(inp["pose1"]), _cuda(inp["depth_est"]), _cuda(inp["lstm_K"]))
        for k, v in (("h0", h0), ("c0", c0), ("h1", h1), ("c1", c1)):
            assert rel_err(v.cpu().numpy(), golden_modules["lstm/" + k]) <= 2e-4, "lstm/" + k
        dec = mods["cvd"](image, enc[0], enc[1], enc[2], enc[3], h1)
        for i, x in enumerate(dec):
            e = oracle.rel_l1_inverse_depth(x.cpu().numpy(), golden_modules["cvd/%d" % i])
            assert e <= 1e-4, "cvd/%d: %.3e" % (i, e)


def test_outputs_are_fresh_fp32_tensors_and_inputs_untouched(oracle, synth, cases):
    c = cases.MODULE_CASE
    mods = helpers.build_product_modules(helpers.oracle_weights(oracle, synth, c["seed"]))
    image = _cuda(cases.module_inputs(synth, c)["image"])
    keep = image.clone()
    a = mods["fe"](image)
    b = mods["fe"](image)
    assert torch.equal(image, keep)
    for x, y in zip(a, b):
        assert x.dtype == torch.float32 and x.is_cuda and x.data_ptr() != y.data_ptr()
        assert torch.equal(x, y)          # deterministic


# ------------------------------------------------------------------------------------------------ end to end
def test_fusionnet_end_to_end_vs_shipped_golden():
    """Shipped fusionnet weights + fixture scene 000 (320x256, D=64, M<=3, recurrent state carried) against the
    reference's shipped predictions: <= 1e-3 relative L1 on inverse depth per frame."""
    w = scene_fixture.load_shipped_weights("fusionnet")
    if w is None:
        pytest.skip("the original project's shipped weights are not in tests/golden/_ref_data (python tools/fetch_fixtures.py <deep-video-mvs checkout>)")
    mods = helpers.build_product_modules(w)
    frames, full_K, gold = scene_fixture.load_scene()
    state = helpers.ProductState()
    from oracle import dvmvs_oracle as oracle
    errs = []
    with torch.no_grad():
        for i, fr in enumerate(frames):
            pred, state = helpers.product_fusionnet_step(mods, state, _cuda(fr["reference_image"])[None], _cuda(fr["reference_pose"])[None],
                                                         [_cuda(x)[None] for x in fr["measurement_images"]],
                                                         [_cuda(p)[None] for p in fr["measurement_poses"]], _cuda(full_K)[None])
            errs.append(oracle.rel_l1_inverse_depth(pred[0].cpu().numpy(), gold[i]))
    print("rel-L1(inverse depth) vs shipped golden per frame:", ["%.2e" % e for e in errs])
    assert max(errs) <= 1e-3, errs


@pytest.mark.parametrize("cfg", [("c2", 256, 256, 64, 2, False), ("c3", 256, 320, 96, 4, False), ("c1", 128, 128, 32, 1, True)])
def test_baseline_configs_vs_oracle(oracle, synth, cfg):
    """BASELINE.json configs 1-3 on the synthetic posed stream (SURVEY.md 8d), synthetic weights shared by both sides,
    3 recurrent keyframes: <= 1e-3 relative L1 on inverse depth (the north-star tolerance)."""
    name, H, W, D, M, pairnet = cfg
    w = helpers.oracle_weights(oracle, synth, 7, n_depth_levels=D)
    mods = helpers.build_product_modules(w, n_depth_levels=D, pairnet=pairnet)
    clip = synth.make_clip(0, 3, H, W, M)
    K = T(clip["K"])[None]
    st_o, st_p = oracle.FusionnetState(), helpers.ProductState()
    with torch.no_grad():
        for ref_i, meas_i in clip["frames"]:
            ri, rp = T(clip["images"][ref_i])[None], T(clip["poses"][ref_i])[None]
            mi, mp = [T(clip["images"][j])[None] for j in meas_i], [T(clip["poses"][j])[None] for j in meas_i]
            if pairnet:
                gold = oracle.pairnet_step(w, ri, rp, mi, mp, K, n_depth_levels=D)
            else:
                gold, st_o = oracle.fusionnet_step(w, st_o, ri, rp, mi, mp, K, n_depth_levels=D)
            pred, st_p = helpers.product_fusionnet_step(mods, st_p, ri.to(DEV), rp.to(DEV), [x.to(DEV) for x in mi],
                                                        [p.to(DEV) for p in mp], K.to(DEV), n_depth_levels=D)
            e = oracle.rel_l1_inverse_depth(pred.cpu().numpy(), gold.numpy())
            assert e <= 1e-3, "%s frame ref=%d: %.3e" % (name, ref_i, e)


def test_pipeline_keyframe_and_cuda_graph_engine_match_script_sequence(oracle, synth):
    """dvmvs.pipeline.keyframe (features batched over the M+1 images) and the CUDA-graph engine reproduce the
    reference script's call sequence bit-for-bit / to fp32 round-off over 4 recurrent keyframes."""
    from dvmvs import pipeline
    H, W, D, M = 64, 96, 64, 2
    w = helpers.oracle_weights(oracle, synth, 11, n_depth_levels=D)
    mods = helpers.build_product_modules(w, n_depth_levels=D)
    clip = synth.make_clip(5, 6, H, W, M)
    K = _cuda(clip["K"])[None]
    st_a, st_b = helpers.ProductState(), pipeline.KeyframeState()
    eng = pipeline.GraphedFusionnet(mods, batch=1, height=H, width=W, n_measurement_frames=M, n_depth_levels=D)
    pipes = [pipeline.PipelinedFusionnet(mods, batch=1, height=H, width=W, n_measurement_frames=M, n_depth_levels=D, n_stages=ns)
             for ns in (2, 3, 4, 5)]
    expected, piped = [], [[] for _ in pipes]
    with torch.no_grad():
        for ref_i, meas_i in clip["frames"]:
            args = (_cuda(clip["images"][ref_i])[None], _cuda(clip["poses"][ref_i])[None], [_cuda(clip["images"][j])[None] for j in meas_i],
                    [_cuda(clip["poses"][j])[None] for j in meas_i], K)
            a, st_a = helpers.product_fusionnet_step(mods, st_a, *args, n_depth_levels=D)
            b, st_b = pipeline.keyframe(mods, st_b, *args, n_depth_levels=D)
            c = eng.step(*args)
            assert oracle.rel_l1_inverse_depth(b.cpu().numpy(), a.cpu().numpy()) <= 1e-6
            assert oracle.rel_l1_inverse_depth(c.cpu().numpy(), a.cpu().numpy()) <= 1e-6
            expected.append(a.cpu().numpy())
            for pi, pipe in enumerate(pipes):    # asynchronous: later keyframes' early stages overlap this one's recurrent stage
                out = torch.empty((1, H, W), dtype=torch.float32, device=DEV)
                pipe.submit(*args, out=out)
                piped[pi].append(out)
        for pipe in pipes:
            pipe.synchronize()
    for pi in range(len(pipes)):
        for e, got in zip(expected, piped[pi]):
            assert oracle.rel_l1_inverse_depth(got.cpu().numpy(), e) <= 1e-6, "pipeline with %d stages" % (pi + 2)


@pytest.mark.parametrize("backend,terms,tol", [("fp32", 3, 1e-5), ("tc", 3, 1e-5), ("tc", 1, 1e-4)])
def test_feature_cache_reproduces_recomputed_features(oracle, synth, backend, terms, tol):
    """SURVEY 8 row f1: measurement features taken from the feature cache (keyed by frame id) instead of re-running
    FeatureExtractor + FeatureShrinker give the script sequence's depths -- eager keyframe() and the pipelined engine,
    cold cache (misses computed from the images), steady state (all hits, no measurement images passed) and FIFO
    eviction with the smallest legal capacity."""
    from dvmvs import pipeline
    from dvmvs import _ops as ops
    H, W, D, M = 64, 96, 64, 2
    w = helpers.oracle_weights(oracle, synth, 13, n_depth_levels=D)
    old_backend = ops.conv_backend()
    ops.set_conv_backend(backend, terms=terms, stride2=True)        # tc / 1 term: a different FeatureExtractor batch changes the split-K
    mods = helpers.build_product_modules(w, n_depth_levels=D)      # summation order, and a 1-ulp fp32 difference can flip an fp16 operand
    clip = synth.make_clip(9, 7, H, W, M)
    K = _cuda(clip["K"])[None]
    st_a, st_b = helpers.ProductState(), pipeline.KeyframeState()
    cache = pipeline.FeatureCache(capacity=M + 1)
    pipes = [pipeline.PipelinedFusionnet(mods, batch=1, height=H, width=W, n_measurement_frames=M, n_depth_levels=D, n_stages=ns,
                                         feature_cache=cap) for ns, cap in ((3, 8), (5, M + 1))]
    expected, piped = [], [[] for _ in pipes]
    with torch.no_grad():
        for t, (ref_i, meas_i) in enumerate(clip["frames"]):
            args = (_cuda(clip["images"][ref_i])[None], _cuda(clip["poses"][ref_i])[None], [_cuda(clip["images"][j])[None] for j in meas_i],
                    [_cuda(clip["poses"][j])[None] for j in meas_i], K)
            a, st_a = helpers.product_fusionnet_step(mods, st_a, *args, n_depth_levels=D)
            b, st_b = pipeline.keyframe(mods, st_b, *args, n_depth_levels=D, cache=cache, reference_id=ref_i, measurement_ids=meas_i)
            assert oracle.rel_l1_inverse_depth(b.cpu().numpy(), a.cpu().numpy()) <= tol
            expected.append(a.cpu().numpy())
            for pi, pipe in enumerate(pipes):
                out = torch.empty((1, H, W), dtype=torch.float32, device=DEV)
                # steady state: every measurement frame was a reference frame before -> no images needed at all
                images = args[2] if t == 0 else [None] * M
                pipe.submit(args[0], args[1], images, args[3], K, out=out, reference_id=ref_i, measurement_ids=meas_i)
                piped[pi].append(out)
        for pipe in pipes:
            pipe.synchronize()
    assert cache.misses == M and cache.hits == M * (len(clip["frames"]) - 1)
    for pi, pipe in enumerate(pipes):
        assert pipe.cache.misses == M and pipe.cache.hits == M * (len(clip["frames"]) - 1)
        for e, got in zip(expected, piped[pi]):
            assert oracle.rel_l1_inverse_depth(got.cpu().numpy(), e) <= tol, "cached pipeline %d" % pi
    # a miss without an image is an error, as is a cache-less engine handed ids
    with pytest.raises(ValueError):
        pipes[0].submit(args[0], args[1], [None] * M, args[3], K, reference_id=10 ** 6, measurement_ids=[10 ** 6 + 1, 10 ** 6 + 2])
    ops.set_conv_backend(old_backend, terms=3)


def test_online_engine_reproduces_shipped_golden_with_keyframe_buffer_and_feature_cache():
    """fusionnet/run-testing-online.py's loop as dvmvs.pipeline.OnlineFusionnet: every frame of fixture scene 000 (pose only
    for the ones that never become keyframes) goes through the from-scratch KeyframeBuffer; the keyframes it selects, with
    the measurement frames it picks (3, as in the shipped run), through the shipped fusionnet weights with measurement
    features from the feature cache.  The first 10 predictions match the reference's shipped golden predictions, and only
    the buffer's very first frame misses the cache."""
    import os
    from dvmvs import pipeline
    from oracle import dvmvs_oracle as oracle
    w = scene_fixture.load_shipped_weights("fusionnet")
    if w is None:
        pytest.skip("the original project's shipped weights are not in tests/golden/_ref_data (python tools/fetch_fixtures.py <deep-video-mvs checkout>)")
    gold_dir = os.path.join(scene_fixture.REPO, "tests", "golden", "keyframes")
    poses = np.load(os.path.join(gold_dir, "poses_000.npy"))
    names = open(os.path.join(gold_dir, "image_names_000.txt")).read().split()
    _, full_K, gold = scene_fixture.load_scene()
    mods = helpers.build_product_modules(w)
    calls = []

    def preprocess(name):
        calls.append(name)
        img, _, _ = scene_fixture.preprocess_rgb(os.path.join(scene_fixture.SCENE, "images", name), 320, 256)
        return _cuda(img)[None]

    online = pipeline.OnlineFusionnet(mods, T(full_K), preprocess, n_measurement_frames=3)
    preds = []
    for pose, name in zip(poses, names):
        out = online.push(pose, name)
        if out is not None:
            preds.append(out[0].cpu().numpy())
            if len(preds) == len(gold):
                break
    assert len(preds) == len(gold) == 10
    errs = [oracle.rel_l1_inverse_depth(p, g) for p, g in zip(preds, gold)]
    assert max(errs) <= 1e-3, errs
    assert online.cache.misses == 1 and online.cache.hits == 2 + 3 * 8      # keyframe 1: one miss; keyframe 2: 2 hits; then 3 each
    assert len(calls) == 10 + 1                                                        # each keyframe once + the first frame


# ------------------------------------------------------------------------------------------------ tcgen05 backend
TC_CASES = [
    # name, B, H, W, [src real channels], Cout, k, stride, act, block_n, terms, tol
    ("k1_c64", 1, 16, 16, [64], 32, 1, 1, 0, 32, 3, 2e-5),
    ("k3_c32_n64", 1, 32, 32, [32], 64, 3, 1, 1, 64, 3, 2e-5),
    ("k5_concat", 1, 64, 64, [32, 64], 32, 5, 1, 1, 32, 3, 5e-5),
    ("k3_odd_batched", 2, 24, 40, [32, 128], 128, 3, 1, 1, 128, 3, 5e-5),
    ("k3_lstm_like", 1, 8, 10, [512, 512], 96, 3, 1, 0, 32, 3, 1e-4),
    ("k3_decoder_concat", 1, 16, 16, [128, 128, 1], 128, 3, 1, 1, 64, 3, 5e-5),
    ("k5_refine_like", 1, 32, 32, [32, 1, 3], 32, 5, 1, 1, 32, 3, 5e-5),
    ("k3_stride2", 1, 32, 32, [64], 128, 3, 2, 1, 64, 3, 2e-5),
    ("k5_stride2", 1, 64, 64, [32], 64, 5, 2, 1, 64, 3, 2e-5),
    ("k3_plain_fp16", 1, 32, 32, [64], 64, 3, 1, 1, 64, 1, 2e-3),
]


@pytest.mark.parametrize("case", TC_CASES, ids=[c[0] for c in TC_CASES])
def test_conv2d_tc_vs_fp32_kernel_and_torch(synth, case):
    """tcgen05 implicit GEMM (TMA-fed, TMEM accumulators, fp16-pair operands) vs torch fp32 on the CPU and vs the fp32
    CUDA-core kernel; also the deterministic split-K variant and the fp16-pair output planes."""
    import torch.nn.functional as F
    from dvmvs import _native as N
    from dvmvs import _ops as ops
    name, B, H, W, chans, Cout, k, stride, act, block_n, terms, tol = case
    cin = sum(chans)
    xs = [T(synth.tensor("tc/%s/x%d" % (name, i), (B, c, H, W), seed=1)) for i, c in enumerate(chans)]
    w = T(synth.tensor("tc/%s/w" % name, (Cout, cin, k, k), seed=2, scale=(2.0 / (cin * k * k)) ** 0.5))
    bias = T(synth.tensor("tc/%s/b" % name, (Cout,), seed=3, scale=0.1))
    ref = F.conv2d(torch.cat(xs, 1), w, bias, stride, (k - 1) // 2)
    ref = F.relu(ref) if act == 1 else ref
    pc = ops.PackedConv(w, bias, None, stride=stride, act=act)
    ptc = ops.PackedConvTC(pc, chans, DEV)
    pc.weight, pc.bias = pc.weight.to(DEV), pc.bias.to(DEV)
    x_dev = [ops.to_nhwc(x.to(DEV)) for x in xs]
    fp32 = ops.conv2d([(x, N.SRC_DIRECT) for x in x_dev], pc)
    planes = [ops.split_planes(x) for x in x_dev]
    out, out_planes = ops.conv2d_tc(planes, ptc, terms=terms, block_n=block_n, allow_split=False)
    out_split, _ = ops.conv2d_tc(planes, ptc, terms=terms, block_n=block_n, allow_split=True)
    again, _ = ops.conv2d_tc(planes, ptc, terms=terms, block_n=block_n, allow_split=True)
    assert torch.equal(out_split, again)                                     # split-K reduction is deterministic
    for got in (out, out_split, out_planes[0].float() + out_planes[1].float()):
        assert rel_err(ops.to_api(got).cpu().numpy(), ref.numpy()) <= tol, name
        assert rel_err(got.cpu().numpy(), fp32.cpu().numpy()) <= tol, name


# operand precision of the tensor path: (terms, bound on rel-L1 inverse depth).  3 = fp16 (hi, lo) pairs, measured ~1e-6
# (synthetic) / ~1e-5 (shipped weights); 1 = plain fp16 operands with fp32 accumulation -- what bench.py runs -- measured
# 4e-5 / 1.1e-4 (profiles/r01_terms_probe.jsonl).  The north-star budget is 1e-3; the bounds below keep a 3x margin.
TC_PRECISIONS = [(3, 1e-4), (1, 3.3e-4)]


@pytest.mark.parametrize("cfg", [("c2", 256, 256, 64, 2, 3), ("c2", 256, 256, 64, 2, 1), ("c3", 256, 320, 96, 4, 1),
                                 ("tiny", 64, 96, 64, 2, 3)])        # tiny: 2x3 bottleneck maps through the TMA / split-K paths
def test_fusionnet_tensor_core_backend_vs_oracle(oracle, synth, cfg):
    """BASELINE configs 2 / 3 through the modules with the tcgen05 backend (stride-2 convs included) vs the CPU oracle."""
    from dvmvs import _ops as ops
    from dvmvs import pipeline
    name, H, W, D, M, terms = cfg
    bound = dict(TC_PRECISIONS)[terms] if name == "c2" else 1e-3      # c2 was measured (3x margin kept); c3: the budget itself
    w = helpers.oracle_weights(oracle, synth, 7, n_depth_levels=D)
    clip = synth.make_clip(0, 3, H, W, M)
    K = T(clip["K"])[None]
    old = ops.conv_backend()
    ops.set_conv_backend("tc", terms=terms, stride2=True)
    try:
        mods = helpers.build_product_modules(w, n_depth_levels=D)
        st_o, st_p = oracle.FusionnetState(), pipeline.KeyframeState()
        with torch.no_grad():
            for ref_i, meas_i in clip["frames"]:
                ri, rp = T(clip["images"][ref_i])[None], T(clip["poses"][ref_i])[None]
                mi, mp = [T(clip["images"][j])[None] for j in meas_i], [T(clip["poses"][j])[None] for j in meas_i]
                gold, st_o = oracle.fusionnet_step(w, st_o, ri, rp, mi, mp, K, n_depth_levels=D)
                pred, st_p = pipeline.keyframe(mods, st_p, ri.to(DEV), rp.to(DEV), [x.to(DEV) for x in mi], [p.to(DEV) for p in mp],
                                               K.to(DEV), n_depth_levels=D)
                e = oracle.rel_l1_inverse_depth(pred.cpu().numpy(), gold.numpy())
                assert e <= bound, "tc backend %s terms=%d, frame ref=%d: %.3e" % (name, terms, ref_i, e)
    finally:
        ops.set_conv_backend(old, terms=3)


@pytest.mark.parametrize("terms,bound", TC_PRECISIONS)
def test_fusionnet_shipped_weights_tensor_core_backend_vs_shipped_golden(terms, bound):
    w = scene_fixture.load_shipped_weights("fusionnet")
    if w is None:
        pytest.skip("the original project's shipped weights are not in tests/golden/_ref_data (python tools/fetch_fixtures.py <deep-video-mvs checkout>)")
    from dvmvs import _ops as ops
    from oracle import dvmvs_oracle as oracle
    old = ops.conv_backend()
    ops.set_conv_backend("tc", terms=terms, stride2=True)
    try:
        mods = helpers.build_product_modules(w)
        frames, full_K, gold = scene_fixture.load_scene()
        state = helpers.ProductState()
        errs = []
        with torch.no_grad():
            for i, fr in enumerate(frames):
                pred, state = helpers.product_fusionnet_step(mods, state, _cuda(fr["reference_image"])[None], _cuda(fr["reference_pose"])[None],
                                                             [_cuda(x)[None] for x in fr["measurement_images"]],
                                                             [_cuda(p)[None] for p in fr["measurement_poses"]], _cuda(full_K)[None])
                errs.append(oracle.rel_l1_inverse_depth(pred[0].cpu().numpy(), gold[i]))
        print("tc backend terms=%d rel-L1(inverse depth) vs shipped golden per frame:" % terms, ["%.2e" % e for e in errs])
        assert max(errs) <= bound, errs
    finally:
        ops.set_conv_backend(old, terms=3)


def _bench_frames(synth, clips, t, H, W, M):
    """Batched device tensors for keyframe t of `clips` (what bench.py's stack_frame builds)."""
    ref = np.stack([c["images"][c["frames"][t][0]] for c in clips])
    rpose = np.stack([c["poses"][c["frames"][t][0]] for c in clips])
    meas = [np.stack([c["images"][c["frames"][t][1][m]] for c in clips]) for m in range(M)]
    mpose = [np.stack([c["poses"][c["frames"][t][1][m]] for c in clips]) for m in range(M)]
    K = np.stack([c["K"] for c in clips])
    return _cuda(ref), _cuda(rpose), [_cuda(x) for x in meas], [_cuda(x) for x in mpose], _cuda(K)


_BENCH_GOLD = {}


def _bench_engine(pipeline, kind, mods, **kw):
    """bench.py's engines: --lookahead 4 (default) = LookaheadFusionnet, --lookahead 0 = PipelinedFusionnet(n_stages=5)."""
    if kind == "lookahead4":
        return pipeline.LookaheadFusionnet(mods, lookahead=4, **kw)
    return pipeline.PipelinedFusionnet(mods, n_stages=5, **kw)


@pytest.mark.parametrize("engine", ["lookahead4", "pipelined5"])
@pytest.mark.parametrize("n_clips,n_frames", [(1, 105), (2, 6), (8, 3)])
def test_benchmarked_configuration_vs_oracle(oracle, synth, n_clips, n_frames, engine):
    """EXACTLY what bench.py times: LookaheadFusionnet(lookahead=4) (bench default) / PipelinedFusionnet(n_stages=5) on the tcgen05 backend with fp16 operands (terms=1), config
    c2 (256x256, 64 planes, 2 measurement frames), bench.py's seeded weights (seed 7) and clips (seed 1000 * rank + c), slots
    re-used with the recurrent state carried -- against the CPU oracle run clip by clip.  (1, 105) is the bench's whole horizon
    (--warmup 5 --steps 100 keyframes of clip 0); n_clips > 1 = the `batched` operating point and what every rank of the
    scaling run does."""
    from dvmvs import _ops as ops
    from dvmvs import pipeline
    H, W, D, M = 256, 256, 64, 2
    w = helpers.oracle_weights(oracle, synth, 7, n_depth_levels=D)
    clips = [synth.make_clip(c, n_frames, H, W, M) for c in range(n_clips)]
    old = ops.conv_backend()
    ops.set_conv_backend("tc", terms=1, stride2=True)
    try:
        mods = helpers.build_product_modules(w, n_depth_levels=D)
        pipe = _bench_engine(pipeline, engine, mods, batch=n_clips, height=H, width=W, n_measurement_frames=M, n_depth_levels=D)
        outs = []
        with torch.no_grad():
            pipe.prime(*_bench_frames(synth, clips, 0, H, W, M))
            for t in range(n_frames):
                out = torch.empty((n_clips, H, W), dtype=torch.float32, device=DEV)
                pipe.submit(*_bench_frames(synth, clips, t, H, W, M), out=out)
                outs.append(out)
            pipe.synchronize()
        worst = 0.0
        golds = _BENCH_GOLD.get((n_clips, n_frames))          # the oracle's answer does not depend on the engine: computed once
        if golds is None:
            golds = {}
            with torch.no_grad():
                for c, clip in enumerate(clips):
                    st = oracle.FusionnetState()
                    K = T(clip["K"])[None]
                    for t, (ref_i, meas_i) in enumerate(clip["frames"]):
                        gold, st = oracle.fusionnet_step(w, st, T(clip["images"][ref_i])[None], T(clip["poses"][ref_i])[None],
                                                         [T(clip["images"][j])[None] for j in meas_i], [T(clip["poses"][j])[None] for j in meas_i],
                                                         K, n_depth_levels=D)
                        golds[(c, t)] = gold.numpy()
            _BENCH_GOLD[(n_clips, n_frames)] = golds
        for c in range(n_clips):
            for t in range(n_frames):
                e = oracle.rel_l1_inverse_depth(outs[t][c:c + 1].cpu().numpy(), golds[(c, t)])
                worst = max(worst, e)
                assert e <= 3.3e-4, "clip %d keyframe %d: %.3e" % (c, t, e)
        print("benchmarked configuration (%s), %d clip(s) x %d keyframes: worst rel-L1(inverse depth) vs oracle %.2e" % (engine, n_clips, n_frames, worst))
    finally:
        ops.set_conv_backend(old, terms=3)


@pytest.mark.parametrize("engine", ["lookahead4", "pipelined5"])
def test_benchmarked_configuration_shipped_weights_vs_shipped_golden(engine):
    """The bench engines (lookahead 4 / 5-stage pipeline, tcgen05, fp16 operands) with the reference's shipped fusionnet weights on the
    fixture scene (320x256, 64 planes, 1..3 measurement frames as the index file says) vs the reference's shipped golden."""
    w = scene_fixture.load_shipped_weights("fusionnet")
    if w is None:
        pytest.skip("the original project's shipped weights are not in tests/golden/_ref_data (python tools/fetch_fixtures.py <deep-video-mvs checkout>)")
    from dvmvs import _ops as ops
    from dvmvs import pipeline
    from oracle import dvmvs_oracle as oracle
    old = ops.conv_backend()
    ops.set_conv_backend("tc", terms=1, stride2=True)
    try:
        mods = helpers.build_product_modules(w)
        frames, full_K, gold = scene_fixture.load_scene()
        M = len(frames[-1]["measurement_images"])
        steady = [i for i, fr in enumerate(frames) if len(fr["measurement_images"]) == M]      # the engine is built for a fixed M
        H, W = frames[0]["reference_image"].shape[-2:]
        pipe = _bench_engine(pipeline, engine, mods, batch=1, height=H, width=W, n_measurement_frames=M)
        state = helpers.ProductState()
        errs = []
        with torch.no_grad():
            args = lambda fr: (_cuda(fr["reference_image"])[None], _cuda(fr["reference_pose"])[None], [_cuda(x)[None] for x in fr["measurement_images"]],
                               [_cuda(p)[None] for p in fr["measurement_poses"]], _cuda(full_K)[None])
            pipe.prime(*args(frames[steady[0]]))
            # the first keyframes of the clip have fewer measurement frames: script sequence for those, then hand the state over
            for i in range(steady[0]):
                pred, state = helpers.product_fusionnet_step(mods, state, *args(frames[i]))
                errs.append(oracle.rel_l1_inverse_depth(pred[0].cpu().numpy(), gold[i]))
            if steady[0] > 0:
                pipe.load_state(state.lstm_state, state.previous_depth, state.previous_pose)
            outs = []
            for i in steady:
                out = torch.empty((1, H, W), dtype=torch.float32, device=DEV)
                pipe.submit(*args(frames[i]), out=out)
                outs.append((i, out))
            pipe.synchronize()
        for i, out in outs:
            errs.append(oracle.rel_l1_inverse_depth(out[0].cpu().numpy(), gold[i]))
        print("bench engine (%s) + shipped weights vs shipped golden:" % engine, ["%.2e" % e for e in errs])
        assert max(errs) <= 3.3e-4, errs
    finally:
        ops.set_conv_backend(old, terms=3)


def test_bench_dumps_the_last_timed_keyframe_of_both_arms(tmp_path):
    """bench.py --dump-outputs: the GPU arm (benchmarked configuration) and the reference arm (the CPU oracle) each write the depth of
    their last timed keyframe of clip 0, with the same seeded weights and frames; the two dumps agree within the bound of
    test_benchmarked_configuration_vs_oracle, and both runs report the requested number of timed steps."""
    import json, os, subprocess, sys
    from oracle import dvmvs_oracle as oracle
    arms = {"ours": ["--backend", "tc", "--tc-terms", "1", "--extras", "0", "--cpu-frames", "0", "--gpu-eager", "0"], "reference": []}
    for impl, extra in arms.items():
        run = subprocess.run([sys.executable, os.path.join(REPO_DIR, "bench.py"), "--impl", impl, "--steps", "2", "--warmup", "3", *extra,
                              "--dump-outputs", str(tmp_path / impl)], capture_output=True, text=True, timeout=900)
        assert run.returncode == 0, run.stderr[-3000:]
        rec = json.loads(run.stdout.strip().splitlines()[-1])
        assert rec["steps"] == 2 and rec.get("steps_run", 2) == 2, rec
    ours, ref = (np.load(str(tmp_path / impl / "depth.npy")) for impl in arms)
    assert ours.shape == ref.shape == (1, 256, 256) and ours.dtype == ref.dtype == np.float32
    e = oracle.rel_l1_inverse_depth(ours, ref)
    print("bench dumps, GPU arm vs reference arm: rel-L1(inverse depth) %.2e" % e)
    assert e <= 3.3e-4, e


@pytest.mark.parametrize("backend,terms,bound", [("fp32", 3, 1e-5), ("tc", 3, 1e-5), ("tc", 1, 1e-4)])
def test_lookahead_engine_matches_eager_keyframe(oracle, synth, backend, terms, bound):
    """LookaheadFusionnet (trunk, pyramid, plane sweep and encoder batched over groups of 3 consecutive keyframes; recurrent stage
    per keyframe on batch slices) against eager keyframe() on the same backend: two clips back to back with a reset() in the
    middle of a group and an incomplete last group.  Not bit for bit: the split-K choice of a few convolutions depends on the
    batch, so sums are re-associated (fp32 / 3-term: round-off; 1-term: a few fp16 operand roundings flip)."""
    from dvmvs import _ops as ops
    from dvmvs import pipeline
    H, W, D, M = 64, 96, 64, 2
    w = helpers.oracle_weights(oracle, synth, 11, n_depth_levels=D)
    old = ops.conv_backend()
    ops.set_conv_backend(backend, terms=terms, stride2=True)
    try:
        mods = helpers.build_product_modules(w, n_depth_levels=D)
        eng = pipeline.LookaheadFusionnet(mods, batch=1, height=H, width=W, n_measurement_frames=M, n_depth_levels=D, lookahead=3, n_groups=2)
        clips = [synth.make_clip(5, 7, H, W, M), synth.make_clip(6, 4, H, W, M)]
        expected, got = [], []
        with torch.no_grad():
            first = clips[0]["frames"][0]
            eng.prime(_cuda(clips[0]["images"][first[0]])[None], _cuda(clips[0]["poses"][first[0]])[None],
                      [_cuda(clips[0]["images"][j])[None] for j in first[1]], [_cuda(clips[0]["poses"][j])[None] for j in first[1]], _cuda(clips[0]["K"])[None])
            for clip in clips:
                K = _cuda(clip["K"])[None]
                st = pipeline.KeyframeState()
                eng.reset()
                for ref_i, meas_i in clip["frames"]:
                    a = (_cuda(clip["images"][ref_i])[None], _cuda(clip["poses"][ref_i])[None], [_cuda(clip["images"][j])[None] for j in meas_i],
                         [_cuda(clip["poses"][j])[None] for j in meas_i], K)
                    pred, st = pipeline.keyframe(mods, st, *a, n_depth_levels=D)
                    expected.append(pred.clone())
                    out = torch.empty((1, H, W), dtype=torch.float32, device=DEV)
                    t = eng.submit(*a, out=out)
                    got.append((t, out))
            eng.synchronize()
        errs = [float((o - e).abs().sum() / e.abs().sum()) for (t, o), e in zip(got, expected)]
        print("lookahead engine vs eager keyframe (%s, %d terms): rel-L1 per keyframe" % (backend, terms), ["%.1e" % e for e in errs])
        assert max(errs) <= bound, errs
        assert torch.equal(eng.depth_of(got[-1][0]), got[-1][1])
        assert eng.kernels_per_keyframe > 0
    finally:
        ops.set_conv_backend(old, terms=3)


@pytest.mark.parametrize("backend,terms", [("tc", 1), ("tc", 3)])
def test_engines_match_eager_keyframe_on_the_tensor_core_backend(oracle, synth, backend, terms):
    """GraphedFusionnet and PipelinedFusionnet (2..5 stages, multi-stream, per-stream split-K scratch, PDL, operand planes
    crossing stage boundaries) against eager keyframe() on the SAME backend, different inputs every keyframe: the kernels are
    deterministic, so the engines must reproduce the eager results bit for bit."""
    from dvmvs import _ops as ops
    from dvmvs import pipeline
    H, W, D, M = 64, 96, 64, 2
    w = helpers.oracle_weights(oracle, synth, 11, n_depth_levels=D)
    old = ops.conv_backend()
    ops.set_conv_backend(backend, terms=terms, stride2=True)
    try:
        mods = helpers.build_product_modules(w, n_depth_levels=D)
        clip = synth.make_clip(5, 7, H, W, M)
        K = _cuda(clip["K"])[None]
        st = pipeline.KeyframeState()
        eng = pipeline.GraphedFusionnet(mods, batch=1, height=H, width=W, n_measurement_frames=M, n_depth_levels=D)
        pipes = [pipeline.PipelinedFusionnet(mods, batch=1, height=H, width=W, n_measurement_frames=M, n_depth_levels=D, n_stages=ns)
                 for ns in (2, 3, 5)]
        expected, graphed, piped = [], [], [[] for _ in pipes]
        with torch.no_grad():
            for ref_i, meas_i in clip["frames"]:
                args = (_cuda(clip["images"][ref_i])[None], _cuda(clip["poses"][ref_i])[None], [_cuda(clip["images"][j])[None] for j in meas_i],
                        [_cuda(clip["poses"][j])[None] for j in meas_i], K)
                a, st = pipeline.keyframe(mods, st, *args, n_depth_levels=D)
                expected.append(a.clone())
                graphed.append(eng.step(*args).clone())
                for pi, pipe in enumerate(pipes):
                    out = torch.empty((1, H, W), dtype=torch.float32, device=DEV)
                    pipe.submit(*args, out=out)
                    piped[pi].append(out)
            for pipe in pipes:
                pipe.synchronize()
        for t, e in enumerate(expected):
            assert torch.equal(graphed[t], e), "graph engine, keyframe %d: max diff %.3e" % (t, float((graphed[t] - e).abs().max()))
            for pi in range(len(pipes)):
                assert torch.equal(piped[pi][t], e), "pipeline %d, keyframe %d: max diff %.3e" % (pi, t, float((piped[pi][t] - e).abs().max()))
    finally:
        ops.set_conv_backend(old, terms=3)


HALO_CASES = [
    # name, B, H, W, [(channels, upsampled)], Cout, k, residual, terms, tol
    ("k3_c32", 1, 40, 48, [(32, False)], 32, 3, False, 3, 2e-5),
    ("k5_c32", 1, 64, 64, [(32, False)], 32, 5, False, 3, 5e-5),
    ("k5_concat_96", 1, 64, 64, [(32, False), (64, False)], 32, 5, False, 3, 5e-5),
    ("k5_refine_like", 1, 64, 64, [(32, True), (1, True), (3, False)], 32, 5, False, 3, 5e-5),
    ("k3_c64_n64", 2, 32, 32, [(64, False)], 64, 3, True, 3, 5e-5),
    ("k3_ragged", 1, 20, 12, [(24, False)], 40, 3, False, 3, 5e-5),
    ("k5_c64_n128", 1, 32, 40, [(64, False)], 128, 5, False, 3, 5e-5),
    ("k3_plain_fp16", 1, 32, 32, [(32, False)], 32, 3, False, 1, 2e-3),
]


@pytest.mark.parametrize("case", HALO_CASES, ids=[c[0] for c in HALO_CASES])
def test_conv2d_halo_vs_torch_fp32(synth, case):
    """Blocked-layout halo implicit GEMM (one TMA halo load per channel group, taps = descriptor offsets) vs torch fp32."""
    import torch.nn.functional as F
    from dvmvs import _native as N
    from dvmvs import _ops as ops
    name, B, H, W, srcs, Cout, k, use_res, terms, tol = case
    xs, full = [], []
    for i, (c, up) in enumerate(srcs):
        f = 2 if up else 1
        x = T(synth.tensor("halo/%s/x%d" % (name, i), (B, c, H // f, W // f), seed=1))
        xs.append(x)
        full.append(F.interpolate(x, scale_factor=2, mode="bilinear", align_corners=True) if up else x)
    cin = sum(c for c, _ in srcs)
    w = T(synth.tensor("halo/%s/w" % name, (Cout, cin, k, k), seed=2, scale=(2.0 / (cin * k * k)) ** 0.5))
    bias = T(synth.tensor("halo/%s/b" % name, (Cout,), seed=3, scale=0.1))
    ref = F.conv2d(torch.cat(full, 1), w, bias, 1, (k - 1) // 2)
    res = T(synth.tensor("halo/%s/r" % name, (B, Cout, H, W), seed=4)) if use_res else None
    if res is not None:
        ref = ref + res
    ref = F.relu(ref)
    pc = ops.PackedConv(w, bias, None, stride=1, act=N.ACT_RELU)
    ph = ops.PackedConvHalo(pc, [c for c, _ in srcs], DEV, concat_padded=True)
    blk = ops.split_blocked([(ops.to_nhwc(x.to(DEV)), up) for x, (c, up) in zip(xs, srcs)])
    f32, oblk, onhwc = ops.conv2d_halo([blk], ph, residual=None if res is None else ops.to_nhwc(res.to(DEV)), terms=terms,
                                       want_f32=True, want_blk=True, want_nhwc=True)
    assert rel_err(ops.to_api(f32).cpu().numpy(), ref.numpy()) <= tol, name
    nh = onhwc[0].float() + onhwc[1].float()
    assert rel_err(ops.to_api(nh).cpu().numpy(), ref.numpy()) <= max(tol, 1e-5), name
    bl = (oblk[0].float() + oblk[1].float()).permute(0, 1, 4, 2, 3).reshape(B, Cout, H, W)     # (B,C8,H,W,8) -> (B,C,H,W)
    assert rel_err(bl.cpu().numpy(), ref.numpy()) <= max(tol, 1e-5), name


# ------------------------------------------------------------------------------------------------ device pre-processing (f2)
PREP_CASES = [  # name, in_h, in_w, out_h, out_w, distortion_crop, perform_crop
    ("hololens_480x640_to_256x256_crop", 480, 640, 256, 256, 0, True),
    ("fixture_540x960_to_256x320_crop", 540, 960, 256, 320, 0, True),
    ("tall_640x480_to_256x320_crop10", 640, 480, 256, 320, 10, True),
    ("no_crop_downscale", 480, 640, 256, 320, 0, False),
    ("upscale_96x128_to_256x320", 96, 128, 256, 320, 0, False),
    ("identity_64x96", 64, 96, 64, 96, 0, False),
    ("odd_ratio_231x317_to_64x96", 231, 317, 64, 96, 3, True),
]


@pytest.mark.parametrize("case", PREP_CASES, ids=[c[0] for c in PREP_CASES])
def test_device_preprocessing_vs_cv2_host_path(case):
    """PreprocessImage.apply_rgb_cuda (one kernel on the decoded uint8 frame) against the reference's host sequence
    load_image -> PreprocessImage.apply_rgb -> transpose (dataset_loader.py:260-263,322-334, run-testing.py:122-127), which
    this package's host methods reproduce with the same cv2 calls.  fp32 both sides; OpenCV's SIMD path may fuse one
    multiply-add, so the bound is a few ulp of a 0..255 value after normalisation."""
    import cv2
    from dvmvs.dataset_loader import PreprocessImage
    _, in_h, in_w, out_h, out_w, dcrop, crop = case
    rng = np.random.default_rng(in_h * 1000 + in_w)
    bgr = rng.integers(0, 256, size=(in_h, in_w, 3), dtype=np.uint8)
    bgr[: in_h // 2] = cv2.GaussianBlur(bgr[: in_h // 2], (9, 9), 3.0)          # smooth half + noise half
    K = np.array([[0.9 * in_w, 0, in_w / 2], [0, 0.9 * in_w, in_h / 2], [0, 0, 1]])
    pre = PreprocessImage(K=K, old_width=in_w, old_height=in_h, new_width=out_w, new_height=out_h, distortion_crop=dcrop, perform_crop=crop)
    scale, mean, std = 255.0, [0.485, 0.456, 0.406], [0.229, 0.224, 0.225]
    rgb_f32 = cv2.cvtColor(bgr.astype(np.float32), cv2.COLOR_BGR2RGB)           # == load_image
    got_u8 = pre.apply_rgb_cuda(torch.from_numpy(bgr).to(DEV), scale, mean, std)
    got_f32 = pre.apply_rgb_cuda(torch.from_numpy(rgb_f32).to(DEV), scale, mean, std)
    raw = pre.apply_rgb_cuda(torch.from_numpy(bgr).to(DEV), scale, mean, std, normalize_colors=False)
    assert tuple(got_u8.shape) == (1, 3, out_h, out_w) and got_u8.dtype == torch.float32

    def host(normalize):
        return np.transpose(pre.apply_rgb(image=rgb_f32, scale_rgb=scale, mean_rgb=mean, std_rgb=std, normalize_colors=normalize), (2, 0, 1))[None]

    # (1) OpenCV's own INTER_LINEAR float path (the algorithm restated in csrc/preprocess.cu): equal to rounding
    use_ipp = cv2.ipp.useIPP()
    cv2.ipp.setUseIPP(False)
    try:
        want, want_raw = host(True), host(False)
    finally:
        cv2.ipp.setUseIPP(use_ipp)
    for got in (got_u8, got_f32):
        assert np.abs(got.cpu().numpy() - want).max() <= 2e-6 * 4.5            # |normalised value| <= ~2.7
    assert np.abs(raw.cpu().numpy() - want_raw).max() <= 6.2e-5                 # 2 ulp at 255
    # (2) this image's cv2 build dispatches float resizes to Intel IPP, whose interpolation coefficients are rounded
    # differently (measured <= 0.009 on the 0..255 scale for white-noise images, 0 for dyadic scale factors): same bound
    want_ipp = host(True)
    assert np.abs(got_u8.cpu().numpy() - want_ipp).max() <= 0.02 / 255.0 / 0.224


def test_device_preprocessing_feeds_the_network_like_the_host_path(oracle, synth):
    """End to end: a keyframe computed from device-preprocessed frames equals the one from host-preprocessed frames."""
    import cv2
    from dvmvs import pipeline
    from dvmvs.dataset_loader import PreprocessImage
    H, W, D, M = 64, 96, 64, 2
    w = helpers.oracle_weights(oracle, synth, 3, n_depth_levels=D)
    mods = helpers.build_product_modules(w, n_depth_levels=D)
    clip = synth.make_clip(2, 1, H, W, M)
    rng = np.random.default_rng(5)
    frames = [cv2.GaussianBlur(rng.integers(0, 256, size=(240, 320, 3), dtype=np.uint8), (7, 7), 2.0) for _ in range(M + 1)]
    K0 = np.array([[290.0, 0, 160], [0, 290.0, 120], [0, 0, 1]])
    pre = PreprocessImage(K=K0, old_width=320, old_height=240, new_width=W, new_height=H, distortion_crop=0, perform_crop=True)
    scale, mean, std = 255.0, [0.485, 0.456, 0.406], [0.229, 0.224, 0.225]
    host = [_cuda(np.transpose(pre.apply_rgb(cv2.cvtColor(f.astype(np.float32), cv2.COLOR_BGR2RGB), scale, mean, std), (2, 0, 1)))[None] for f in frames]
    dev = [pre.apply_rgb_cuda(torch.from_numpy(f).to(DEV), scale, mean, std) for f in frames]
    K = _cuda(pre.get_updated_intrinsics().astype(np.float32))[None]
    ref_i, meas_i = clip["frames"][0]
    poses = [_cuda(clip["poses"][i])[None] for i in [ref_i] + list(meas_i)]
    with torch.no_grad():
        a, _ = pipeline.keyframe(mods, pipeline.KeyframeState(), host[0], poses[0], host[1:], poses[1:], K, n_depth_levels=D)
        b, _ = pipeline.keyframe(mods, pipeline.KeyframeState(), dev[0], poses[0], dev[1:], poses[1:], K, n_depth_levels=D)
    assert oracle.rel_l1_inverse_depth(b.cpu().numpy(), a.cpu().numpy()) <= 1e-4     # host side may use IPP's coefficients (see above)
