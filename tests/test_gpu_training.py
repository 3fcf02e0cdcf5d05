"""GPU parity tests of the training-step ops (SURVEY section 8 row f3): the hand-written backward kernels, reached through
dvmvs.training / dvmvs.utils (ctypes over the C ABI), against
 (a) gradients of the unmodified reference under autograd (tests/golden/training.npz),
 (b) torch autograd through the CPU oracle on seeded inputs, and
 (c) size-independent properties at BASELINE.json's full sizes: the adjoint identity <g, J d> == <J^T g, d> (the cost volume
     is linear in each feature map, so J d is one forward launch) and linearity of the backward in the upstream gradient.
Tolerances: fp32 on both sides; scatter-adds use fp32 atomics (order not fixed) -> <= 5e-5 of the tensor's max magnitude."""
import os

import numpy as np
import pytest
import torch

from tests.helpers import T, rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda"
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _cuda(x):
    return T(np.ascontiguousarray(x)).to(DEV)


@pytest.fixture(scope="module")
def golden_training():
    from oracle import npz_parts
    return npz_parts.load(os.path.join(REPO, "tests", "golden", "training.npz"))


# ------------------------------------------------------------------------------------------------ plane sweep
@pytest.mark.parametrize("layout", ["nchw", "channels_last"])
def test_plane_sweep_backward_vs_reference_golden(synth, cases, golden_training, layout):
    """cost_volume_fusion routes to the differentiable op when a feature map requires grad (as run-training.py:231 does)."""
    from dvmvs.utils import cost_volume_fusion
    conv = (lambda t: t.contiguous(memory_format=torch.channels_last)) if layout == "channels_last" else (lambda t: t)
    for name in cases.SWEEP_GRAD_CASES:
        c = cases.PLANE_SWEEP_CASES[name]
        inp = cases.plane_sweep_inputs(synth, c)
        f1 = conv(_cuda(inp["image1"])).requires_grad_(True)
        f2s = [conv(_cuda(x)).requires_grad_(True) for x in inp["image2s"]]
        cost = cost_volume_fusion(f1, f2s, _cuda(inp["pose1"]), [_cuda(p) for p in inp["pose2s"]], _cuda(inp["K"]), None, c["min_depth"],
                                  c["max_depth"], c["D"], DEV, True)
        assert cost.requires_grad and tuple(cost.shape) == (c["B"], c["D"], c["h"], c["w"])
        cost.backward(conv(_cuda(cases.upstream(synth, "sweep/" + name, tuple(cost.shape), c["seed"]))))
        err = rel_err(f1.grad.cpu().numpy(), golden_training["sweep/%s/g_image1" % name])
        assert err <= 5e-5, "sweep/%s/g_image1 (%s): %.3e" % (name, layout, err)
        for m, t in enumerate(f2s):
            err = rel_err(t.grad.cpu().numpy(), golden_training["sweep/%s/g_image2_%d" % (name, m)])
            assert err <= 5e-5, "sweep/%s/g_image2_%d (%s): %.3e" % (name, m, layout, err)


def test_plane_sweep_backward_same_tensor_twice_and_partial_grads(synth, cases, oracle):
    """The same measurement tensor used for two frames accumulates both gradients; inputs that do not require grad get none."""
    from dvmvs.training import plane_sweep_cost_volume
    c = cases.PLANE_SWEEP_CASES["dot_small"]
    inp = cases.plane_sweep_inputs(synth, c)
    g = cases.upstream(synth, "sweep/twice", (c["B"], c["D"], c["h"], c["w"]), 3)
    f1 = _cuda(inp["image1"])
    f2 = _cuda(inp["image2s"][0]).requires_grad_(True)
    poses = [_cuda(p) for p in inp["pose2s"]]
    cost = plane_sweep_cost_volume(f1, [f2, f2], _cuda(inp["pose1"]), poses, _cuda(inp["K"]), c["min_depth"], c["max_depth"], c["D"])
    cost.backward(_cuda(g))
    assert f1.grad is None
    o1 = T(inp["image1"])
    o2 = T(inp["image2s"][0]).requires_grad_(True)
    grid = oracle.get_warp_grid_for_cost_volume_calculation(c["w"], c["h"])
    oc = oracle.cost_volume_fusion(o1, [o2, o2], T(inp["pose1"]), [T(p) for p in inp["pose2s"]], T(inp["K"]), grid, c["min_depth"],
                                   c["max_depth"], c["D"], "cpu", True)
    oc.backward(T(g))
    assert rel_err(f2.grad.cpu().numpy(), o2.grad.numpy()) <= 5e-5


def test_plane_sweep_backward_full_size_adjoint_identity_and_linearity(synth):
    """BASELINE.json configs 2 / 3 shapes.  cost(f1, f2s) is bilinear, so with J the Jacobian w.r.t. one argument,
    J d == cost with that argument replaced by d; the backward kernel must satisfy <g, J d> == <J^T g, d>."""
    from dvmvs.training import plane_sweep_cost_volume
    for (h, w, D, M) in ((128, 128, 64, 2), (128, 160, 96, 4)):
        f1 = _cuda(synth.tensor("adj/ref", (1, 32, h, w), seed=D, scale=2.0)).requires_grad_(True)
        f2s = [_cuda(synth.tensor("adj/m%d" % m, (1, 32, h, w), seed=D, scale=2.0)).requires_grad_(True) for m in range(M)]
        pose1 = _cuda(synth.camera_pose(M)[None])
        pose2s = [_cuda(synth.camera_pose(M - k)[None]) for k in range(1, M + 1)]
        K = synth.intrinsics(2 * h, 2 * w)[None].copy()
        K[:, 0:2, :] /= 2.0
        K = _cuda(K)
        g = _cuda(synth.tensor("adj/g", (1, D, h, w), seed=D))
        cost = plane_sweep_cost_volume(f1, f2s, pose1, pose2s, K, 0.25, 20.0, D)
        cost.backward(g)
        with torch.no_grad():
            d1 = _cuda(synth.tensor("adj/d1", (1, 32, h, w), seed=D))
            lhs = float((g.double() * plane_sweep_cost_volume(d1, [t.detach() for t in f2s], pose1, pose2s, K, 0.25, 20.0, D).double()).sum())
            rhs = float((f1.grad.double() * d1.double()).sum())
            assert abs(lhs - rhs) <= 2e-5 * max(abs(lhs), abs(rhs), 1.0), ("ref", h, w, lhs, rhs)
            for m in range(M):
                d2 = _cuda(synth.tensor("adj/d2_%d" % m, (1, 32, h, w), seed=D))
                probe = [torch.zeros_like(d2) for _ in range(M)]
                probe[m] = d2
                lhs = float((g.double() * plane_sweep_cost_volume(f1.detach(), probe, pose1, pose2s, K, 0.25, 20.0, D).double()).sum())
                rhs = float((f2s[m].grad.double() * d2.double()).sum())
                assert abs(lhs - rhs) <= 2e-5 * max(abs(lhs), abs(rhs), 1.0), ("meas", m, h, w, lhs, rhs)
        # linearity in the upstream gradient
        ga = f1.grad.clone()
        f1.grad = None
        cost2 = plane_sweep_cost_volume(f1, [t.detach() for t in f2s], pose1, pose2s, K, 0.25, 20.0, D)
        cost2.backward(-2.0 * g)
        assert rel_err(f1.grad.cpu().numpy(), (-2.0 * ga).cpu().numpy()) <= 1e-6


# ------------------------------------------------------------------------------------------------ hidden-state warp
def test_hidden_warp_backward_vs_reference_golden(synth, cases, golden_training):
    from dvmvs.utils import warp_frame_depth
    for name in cases.HIDDEN_WARP_GRAD_CASES:
        c = cases.HIDDEN_WARP_CASES[name]
        inp = cases.hidden_warp_inputs(synth, c)
        src = _cuda(inp["image_src"]).requires_grad_(True)
        res = warp_frame_depth(src, _cuda(inp["depth_dst"]), _cuda(inp["trans"]), _cuda(inp["K"]))
        res.backward(_cuda(cases.upstream(synth, "warp/" + name, tuple(res.shape), c["seed"])))
        err = rel_err(src.grad.cpu().numpy(), golden_training["warp/%s/g_image_src" % name])
        assert err <= 5e-5, "warp/%s: %.3e" % (name, err)


def test_recurrent_cell_gradients_vs_reference_golden(synth, cases, golden_training):
    """The ConvLSTM cell of convlstm.py:26-59 assembled from the differentiable ops (warp + mask -> torch conv2d for the gate
    convolution -> gate epilogue) reproduces the reference cell's input gradients, including the reference's quirk that
    its mask (a .data write) does not act on the gradient."""
    from dvmvs.training import lstm_gate_epilogue, warp_hidden_state
    torch.backends.cudnn.allow_tf32 = False          # the caller's convolution must be fp32 for a 2e-4 comparison
    torch.backends.cuda.matmul.allow_tf32 = False
    for name in cases.LSTM_GRAD_CASES:
        c = cases.LSTM_CASES[name]
        inp = cases.lstm_inputs(synth, c)
        x, h, cc = (_cuda(inp[k]).requires_grad_(True) for k in ("x", "h", "c"))
        hw = h
        if c["warp"]:
            hw = warp_hidden_state(h, _cuda(inp["depth"]), _cuda(inp["previous_pose"]), _cuda(inp["current_pose"]), _cuda(inp["K"]), 0.01)
        combined = torch.nn.functional.conv2d(torch.cat([x, hw], dim=1), _cuda(inp["weight"]), None, 1, 1)
        hn, cn = lstm_gate_epilogue(combined, cc)
        torch.autograd.backward([hn, cn], [_cuda(cases.upstream(synth, "lstm/%s/h" % name, tuple(hn.shape), c["seed"])),
                                           _cuda(cases.upstream(synth, "lstm/%s/c" % name, tuple(cn.shape), c["seed"]))])
        for key, t in (("g_x", x), ("g_h", h), ("g_c", cc)):
            err = rel_err(t.grad.cpu().numpy(), golden_training["lstm/%s/%s" % (name, key)])
            assert err <= 2e-4, "lstm/%s/%s: %.3e" % (name, key, err)      # torch's cuDNN conv in the middle: TF32 off, fp32 round-off


# ------------------------------------------------------------------------------------------------ gate epilogue
@pytest.mark.parametrize("shape", [(1, 512, 8, 8), (2, 64, 8, 10), (1, 32, 2, 2), (3, 96, 1, 3), (1, 512, 8, 16)])
def test_lstm_gate_epilogue_backward_vs_oracle_autograd(oracle, synth, shape):
    from dvmvs.training import lstm_gate_epilogue
    B, C, h, w = shape
    cc_np = synth.tensor("gates/cc", (B, 4 * C, h, w), seed=C + h, scale=1.5)
    c_np = synth.tensor("gates/c", (B, C, h, w), seed=C + h)
    gh_np = synth.tensor("gates/gh", (B, C, h, w), seed=C + h)
    gc_np = synth.tensor("gates/gc", (B, C, h, w), seed=C + h)
    a, b = _cuda(cc_np).requires_grad_(True), _cuda(c_np).requires_grad_(True)
    hn, cn = lstm_gate_epilogue(a, b)
    torch.autograd.backward([hn, cn], [_cuda(gh_np), _cuda(gc_np)])
    oa, ob = T(cc_np).requires_grad_(True), T(c_np).requires_grad_(True)
    ohn, ocn = oracle.lstm_gate_epilogue(oa, ob)
    torch.autograd.backward([ohn, ocn], [T(gh_np), T(gc_np)])
    assert rel_err(hn.detach().cpu().numpy(), ohn.detach().numpy()) <= 2e-5
    assert rel_err(a.grad.cpu().numpy(), oa.grad.numpy()) <= 5e-5
    assert rel_err(b.grad.cpu().numpy(), ob.grad.numpy()) <= 5e-5
    # only h used downstream (last timestep): grad_c is zero
    a.grad = b.grad = None
    hn, cn = lstm_gate_epilogue(a, b)
    hn.backward(_cuda(gh_np))
    oa.grad = ob.grad = None
    ohn, ocn = oracle.lstm_gate_epilogue(oa, ob)
    ohn.backward(T(gh_np))
    assert rel_err(a.grad.cpu().numpy(), oa.grad.numpy()) <= 5e-5


# ------------------------------------------------------------------------------------------------ loss
def test_multi_scale_loss_vs_reference_golden(synth, cases, golden_training):
    from dvmvs.training import multi_scale_depth_loss
    c = cases.LOSS_CASE
    inp = cases.loss_inputs(synth, c)
    gt = _cuda(inp["groundtruth"])
    for loss_type in cases.LOSS_TYPES:
        preds = [_cuda(p).requires_grad_(True) for p in inp["predictions"]]
        loss, sums = multi_scale_depth_loss(preds, c["weights"], gt, loss_type)
        (3.0 * loss).backward()                                   # a non-trivial upstream gradient
        gold_sums = golden_training["loss/%s/sums" % loss_type]
        assert abs(float(loss) - float(golden_training["loss/%s/loss" % loss_type])) <= 1e-5 * abs(float(loss))
        assert np.array_equal(sums[:, 4].cpu().numpy(), gold_sums[:, 4].astype(np.float32))        # valid counts: exact
        assert rel_err(sums.cpu().numpy(), gold_sums) <= 1e-5
        for j, p in enumerate(preds):
            err = rel_err(p.grad.cpu().numpy(), 3.0 * golden_training["loss/%s/g_pred_%d" % (loss_type, j)])
            assert err <= 2e-6, "loss/%s/g_pred_%d: %.3e" % (loss_type, j, err)


def test_multi_scale_loss_full_size_properties(synth):
    """c2 training size (256x256, five scales): the gradient is zero exactly on the invalid pixels and the loss is the
    weight-linear combination of its per-scale parts."""
    from dvmvs.training import multi_scale_depth_loss
    B, H, W = 2, 256, 256
    gt_np = (0.5 + 3.0 * np.abs(synth.tensor("lossfull/gt", (B, H, W), seed=1))).astype(np.float32)
    gt_np[:, ::7, :] = 0.0
    gt = _cuda(gt_np)
    preds = [_cuda((0.4 + np.abs(synth.tensor("lossfull/p%d" % k, (B, H // s, W // s), seed=1))).astype(np.float32)).requires_grad_(True)
             for k, s in enumerate((16, 8, 4, 2, 1))]
    loss, sums = multi_scale_depth_loss(preds, [1, 1, 1, 1, 1], gt, "L1-inv")
    loss.backward()
    full = preds[4].grad
    assert bool((full[gt == 0] == 0).all()) and bool((full[gt != 0] != 0).all())
    parts = [float(multi_scale_depth_loss([p.detach()], [1.0], gt, "L1-inv")[0]) for p in preds]
    assert abs(float(loss) - sum(parts)) <= 1e-5 * abs(float(loss))
