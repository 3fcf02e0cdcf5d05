"""CPU-only checks of the host side: the C-ABI library loads and exports every symbol include/dvmvs_b200.h declares,
argument validation works without a GPU, the drop-in modules carry the reference's state-dict contract, and the
geometry prologue (run on the host through a test hook) matches numpy."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from tests import scene_fixture

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from dvmvs import _native as N
    header = open(os.path.join(REPO, "include", "dvmvs_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = sorted(set(re.findall(r"\b(dvmvs_[a-z0-9_]+)\s*\(", header)))
    assert declared, "no declarations parsed"
    lib = N.lib()
    for sym in declared:
        assert hasattr(lib, sym), "libdvmvs_sm100.so does not export %s" % sym
    assert sorted(N.EXPORTED_SYMBOLS) == declared
    assert lib.dvmvs_abi_version() == N.ABI_VERSION == 6


def test_binding_argtypes_match_header_prototypes():
    """Every prototype of include/dvmvs_b200.h against the ctypes binding: same number of parameters, and each parameter's C
    class (pointer / int / long long / float / double) maps to the ctypes type the binding declares.  A drifted argtypes list
    passes garbage in registers without any error."""
    import ctypes
    from dvmvs import _native as N
    header = open(os.path.join(REPO, "include", "dvmvs_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    lib = N.lib()
    protos = re.findall(r"\b(?:int|const char\*)\s+(dvmvs_[a-z0-9_]+)\s*\(([^)]*)\)\s*;", header)
    assert len(protos) >= 30

    def c_class(param):
        param = param.strip()
        if param in ("void", ""):
            return None
        if "*" in param or "dvmvs_stream_t" in param:
            return "ptr"
        base = re.sub(r"\b(const|unsigned|signed)\b", "", param).split()
        kinds = {"int": "int", "float": "float", "double": "double"}
        if "long" in base:
            return "longlong"
        return kinds[base[0]]

    ok = {"ptr": (ctypes.c_void_p, ctypes.c_char_p), "int": (ctypes.c_int, ctypes.c_uint), "longlong": (ctypes.c_longlong, ctypes.c_ulonglong, ctypes.c_size_t),
          "float": (ctypes.c_float,), "double": (ctypes.c_double,)}
    checked = 0
    for name, params in protos:
        want = [c for c in (c_class(q) for q in params.split(",")) if c is not None]
        fn = getattr(lib, name)
        if fn.argtypes is None:
            assert not want or name in ("dvmvs_abi_version", "dvmvs_kernel_launch_count", "dvmvs_last_error_string"), \
                "%s takes %d arguments but the binding declares no argtypes" % (name, len(want))
            continue
        assert len(fn.argtypes) == len(want), "%s: header has %d parameters, binding declares %d" % (name, len(want), len(fn.argtypes))
        for i, (kind, at) in enumerate(zip(want, fn.argtypes)):
            is_ptr = isinstance(at, type) and (issubclass(at, ctypes._Pointer) or at in ok["ptr"])
            assert (kind == "ptr" and is_ptr) or (kind != "ptr" and at in ok[kind]), "%s parameter %d: header %s, binding %s" % (name, i, kind, at)
        checked += 1
    assert checked >= 25, checked


def test_desc_structs_match_header_field_order():
    """The ctypes mirrors must list exactly the fields of the C structs, in order (a mismatch corrupts memory)."""
    from dvmvs import _native as N
    header = open(os.path.join(REPO, "include", "dvmvs_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    for cname, mirror in (("dvmvs_conv_desc", N.ConvDesc), ("dvmvs_conv_tc_desc", N.ConvTcDesc), ("dvmvs_conv_halo_desc", N.ConvHaloDesc)):
        end = header.index("} %s;" % cname)
        start = header.rindex("typedef struct {", 0, end)
        body = header[start + len("typedef struct {"):end]
        names = re.findall(r"[\s\*]([A-Za-z_][A-Za-z0-9_]*)(?:\[3\])?\s*[;,]", body)
        assert names == [f[0] for f in mirror._fields_], (cname, names, [f[0] for f in mirror._fields_])
        # ctypes silently accepts assignments to unknown attributes: make sure every mirror forbids them in tests
        obj = mirror()
        for f in names:
            getattr(obj, f)


def test_argument_validation_without_gpu():
    from dvmvs import _native as N
    lib = N.lib()
    rc = lib.dvmvs_plane_sweep_fused(None, None, None, None, None, None, 1, 32, 8, 8, 4, 1, 0.25, 20.0, 0, None)
    assert rc == -1 and b"null" in lib.dvmvs_last_error_string()
    d = N.ConvDesc()
    d.n_src = 7
    assert lib.dvmvs_conv2d(ctypes.byref(d), None) == -1
    assert lib.dvmvs_dwconv2d(None, None, None, None, None, 1, 8, 8, 6, 3, 1, 0, None) == -1
    assert lib.dvmvs_lstm_gates(None, None, None, None, 1, 8, 8, 512, None) == -1


def test_ops_refuse_cpu_tensors_loudly():
    from dvmvs.fusionnet.model import FeatureExtractor
    from dvmvs.utils import cost_volume_fusion, warp_frame_depth
    x = torch.zeros(1, 32, 8, 8)
    with pytest.raises(RuntimeError):
        cost_volume_fusion(x, [x], torch.eye(4)[None], [torch.eye(4)[None]], torch.eye(3)[None], None, 0.25, 20.0, 8, "cpu", True)
    with pytest.raises(TypeError):
        warp_frame_depth(None, x, x, x)
    with pytest.raises(ValueError):
        warp_frame_depth(x, x, torch.eye(4)[None], torch.eye(3)[None])      # depth must be (B,1,H,W)
    fe = FeatureExtractor().eval()
    with pytest.raises(RuntimeError):
        fe(torch.zeros(1, 3, 64, 64))                                       # CPU module / tensor: no fallback
    with pytest.raises(RuntimeError):
        FeatureExtractor()(torch.zeros(1, 3, 64, 64))                       # training mode: inference only


def test_state_dict_contract(oracle):
    from dvmvs.fusionnet import model as fm
    from dvmvs.pairnet import model as pm
    shapes = oracle.state_dict_shapes(64)
    for tag, cls in (("fe", fm.FeatureExtractor), ("fpn", fm.FeatureShrinker), ("cve", fm.CostVolumeEncoder),
                     ("lstm", fm.LSTMFusion), ("cvd", fm.CostVolumeDecoder)):
        sd = cls().state_dict()
        assert list(sd.keys()) == list(shapes[tag].keys()), tag
        assert all(tuple(sd[k].shape) == tuple(shapes[tag][k]) for k in sd), tag
    assert not hasattr(pm, "LSTMFusion")
    for net in ("fusionnet", "pairnet"):
        w = scene_fixture.load_shipped_weights(net)
        if w is None:
            continue
        mod = fm if net == "fusionnet" else pm
        classes = {"fe": mod.FeatureExtractor, "fpn": mod.FeatureShrinker, "cve": mod.CostVolumeEncoder,
                   "cvd": mod.CostVolumeDecoder}
        if net == "fusionnet":
            classes["lstm"] = mod.LSTMFusion
        for tag, cls in classes.items():
            cls().load_state_dict(w[tag], strict=True)


def test_bn_folding_matches_conv_bn(synth):
    from dvmvs import _ops as ops
    conv = torch.nn.Conv2d(8, 12, 3, padding=1, bias=False)
    bn = torch.nn.BatchNorm2d(12).eval()
    sd = synth.make_state_dict({"weight": (12,), "bias": (12,), "running_mean": (12,), "running_var": (12,)}, seed=9)
    with torch.no_grad():
        for k, v in sd.items():
            getattr(bn, k).copy_(torch.from_numpy(v))
        pc = ops.PackedConv(conv.weight, None, bn)
        x = torch.randn(1, 8, 6, 6)
        ref = bn(conv(x))
        w = pc.weight.permute(3, 2, 0, 1)        # [k][k][Cin][Cout] -> (Cout, Cin, k, k)
        got = torch.nn.functional.conv2d(x, w, pc.bias, 1, 1)
    assert float((ref - got).abs().max()) < 1e-5


def test_geometry_prologue_on_host_matches_numpy(synth):
    from dvmvs import _native as N
    lib = N.lib()
    fp = ctypes.POINTER(ctypes.c_float)
    lib.dvmvs_host_sweep_geometry.argtypes = [fp, fp, fp, ctypes.c_float, ctypes.c_float, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                              ctypes.c_int, ctypes.c_float, ctypes.c_float, fp, fp]
    p1, p2 = synth.camera_pose(3), synth.camera_pose(1)
    K = synth.intrinsics(256, 256).copy()
    K[0:2] /= 2
    out, xy = np.zeros(12, np.float32), np.zeros(2, np.float32)
    f = lambda a: a.ctypes.data_as(fp)
    for (u, v, d) in ((0, 0, 0), (17, 90, 31), (127, 127, 63)):
        assert lib.dvmvs_host_sweep_geometry(f(p1), f(p2), f(K), u, v, 128, 128, d, 64, 0.25, 20.0, f(out), f(xy)) == 0
        E = np.linalg.inv(p2.astype(np.float64)) @ p1
        G = K @ E[:3, :3] @ np.linalg.inv(K.astype(np.float64))
        Kt = K @ E[:3, 3]
        assert np.abs(out[:9].reshape(3, 3) - G).max() < 1e-4 and np.abs(out[9:] - Kt).max() < 1e-4
        q = G @ np.array([u, v, 1.0]) + Kt * (1 / 20.0 + d * (1 / 0.25 - 1 / 20.0) / 63)
        assert abs(xy[0] - q[0] / (q[2] + 1e-8) * 127 / 128) < 2e-3 and abs(xy[1] - q[1] / (q[2] + 1e-8) * 127 / 128) < 2e-3


def test_device_preprocessing_refuses_host_tensors_and_bad_shapes():
    """apply_rgb_cuda is the device path only: CPU tensors / wrong shapes raise instead of silently falling back."""
    import numpy as np
    import torch
    from dvmvs.dataset_loader import PreprocessImage
    pre = PreprocessImage(K=np.eye(3), old_width=64, old_height=48, new_width=32, new_height=32, distortion_crop=0, perform_crop=True)
    assert (pre.crop_x, pre.crop_y) == (8, 0)
    with pytest.raises(RuntimeError, match="CUDA"):
        pre.apply_rgb_cuda(torch.zeros(48, 64, 3, dtype=torch.uint8), 255.0, [0, 0, 0], [1, 1, 1])


def test_feature_cache_ring_semantics():
    """Row f1 host logic (no kernels involved): FIFO eviction at capacity, re-store of a live id keeps its slot, lookups
    return channels_last views of the ring entries, counters."""
    from dvmvs.pipeline import FeatureCache
    cache = FeatureCache(capacity=3)
    feats = {i: torch.full((1, 32, 4, 6), float(i)).contiguous(memory_format=torch.channels_last) for i in range(5)}
    assert cache.lookup(0) is None and cache.misses == 1
    for i in range(3):
        cache.store(i, feats[i])
    assert all(i in cache for i in range(3))
    got = cache.lookup(1)
    assert got.shape == (1, 32, 4, 6) and got.is_contiguous(memory_format=torch.channels_last) and float(got.mean()) == 1.0
    slot_of_1 = cache._index[1]
    cache.store(1, feats[4])                      # same id again: same slot, new content, nobody evicted
    assert cache._index[1] == slot_of_1 and float(cache.lookup(1).mean()) == 4.0 and 0 in cache and 2 in cache
    cache.store(3, feats[3])                      # capacity reached: the oldest entry (id 0) goes
    assert 0 not in cache and 1 in cache and 2 in cache and 3 in cache
    cache.store(4, feats[4])
    assert 1 not in cache and float(cache.lookup(3).mean()) == 3.0
    assert cache.hits == 3 and cache.misses == 1
    cache.clear()
    assert 3 not in cache and cache.lookup(3) is None
    with pytest.raises(ValueError):
        FeatureCache(0)


def test_precision_policy_parsing_and_scoping():
    from dvmvs import _ops as ops
    try:
        ops.set_precision_policy("fe=1, fpn=1,cvd=3")
        assert ops.precision_policy() == {"fe": 1, "fpn": 1, "cvd": 3}
        seen = []

        @ops.family_terms("fe")
        def inner():
            seen.append(ops._TC_TERMS)
            raise KeyError("x")

        before = ops._TC_TERMS
        with pytest.raises(KeyError):
            inner()
        assert seen == [1] and ops._TC_TERMS == before          # restored even when the forward raises
        with pytest.raises(ValueError):
            ops.set_precision_policy({"fe": 2})
        with pytest.raises(ValueError):
            ops.set_precision_policy({"decoder": 1})
    finally:
        ops.set_precision_policy(None)
    assert ops.precision_policy() == {}


@pytest.mark.parametrize("n_measurement_frames", [1, 2, 3])
def test_keyframe_buffer_regenerates_the_shipped_index_files(n_measurement_frames):
    """dvmvs.keyframe_buffer.KeyframeBuffer, driven the way simulate_keyframe_buffer.py:21-47 drives the reference's, over the
    373 poses of fixture scene 000 reproduces the reference's shipped selection files line for line (which frames become
    keyframes, which measurement frames are picked, and in which order)."""
    from dvmvs.config import Config
    from dvmvs.keyframe_buffer import KeyframeBuffer
    gold_dir = os.path.join(REPO, "tests", "golden", "keyframes")
    poses = np.load(os.path.join(gold_dir, "poses_000.npy"))
    names = open(os.path.join(gold_dir, "image_names_000.txt")).read().split()
    buf = KeyframeBuffer(buffer_size=Config.test_keyframe_buffer_size, keyframe_pose_distance=Config.test_keyframe_pose_distance,
                         optimal_t_score=Config.test_optimal_t_measure, optimal_R_score=Config.test_optimal_R_measure,
                         store_return_indices=True)
    lines, id_of_index = [], {}
    for i, pose in enumerate(poses):
        response = buf.try_new_keyframe(pose, None, index=i)
        if response in (0, 1):
            id_of_index[i] = buf.last_frame_id
        if response == 3:
            lines.append("TRACKING LOST")
        elif response == 1:
            frames, ids = buf.get_best_measurement_frames(n_measurement_frames, with_ids=True)
            assert ids == [id_of_index[f[2]] for f in frames]            # the ids name the frames that were handed out
            lines.append(" ".join([names[i]] + [names[f[2]] for f in frames]))
    gold = open(os.path.join(gold_dir, "keyframe+hololens-dataset+000+nmeas+%d" % n_measurement_frames)).read().splitlines()
    assert len(lines) == len(gold) == 286
    assert lines == gold


def test_keyframe_buffer_response_codes_and_tracking_loss():
    from dvmvs.keyframe_buffer import KeyframeBuffer, SimpleBuffer
    eye = np.eye(4)
    moved = np.eye(4)
    moved[0, 3] = 0.2
    bad = np.full((4, 4), np.nan)
    buf = KeyframeBuffer(4, 0.1, 0.15, 0.0, store_return_indices=False)
    assert buf.try_new_keyframe(bad, "x") == 5 and buf.last_frame_id is None
    assert buf.try_new_keyframe(eye, "a") == 0 and buf.last_frame_id == 0
    assert buf.try_new_keyframe(eye, "b") == 2                       # no motion
    assert buf.try_new_keyframe(moved, "c") == 1 and buf.last_frame_id == 1
    (pose, image), = buf.get_best_measurement_frames(3)              # only one candidate: n is clipped
    assert image == "a" and np.array_equal(pose, eye)
    for k in range(30):
        assert buf.try_new_keyframe(bad, None) == 5
    assert buf.try_new_keyframe(bad, None) == 3 and len(buf.buffer) == 0
    assert buf.try_new_keyframe(bad, None) == 4
    assert buf.try_new_keyframe(eye, "d") == 0 and buf.last_frame_id == 2      # ids keep counting across a loss
    with pytest.raises(ValueError):
        KeyframeBuffer(4, 0.1, 0.15, 0.0, store_return_indices=True).try_new_keyframe(eye, None)
    sb = SimpleBuffer(2, store_return_indices=True)
    assert [sb.try_new_keyframe(eye, None, index=k) for k in range(4)] == [0, 1, 1, 1]
    frames, ids = sb.get_measurement_frames(with_ids=True)
    assert [f[2] for f in frames] == [1, 2] and ids == [1, 2]


def test_pixel_pair_formulation_of_the_fp16_sweep_equals_zero_padded_bilinear(oracle):
    """The experimental fp16-feature sweep kernel (plane_sweep_c32_h16_kernel) fetches, per bilinear ROW, the in-image pixel
    pair (xa, xa+1), xa = clamp(x0, 0, w-2), and moves the two tap weights onto its members (0 for a tap outside the image).
    This restates that rule in numpy (same expressions as sweep_phase_a_h16) and checks it against grid_sample-style
    zero-padded bilinear sampling (the oracle's bilinear_sample_zeros), including positions off every edge."""
    rng = np.random.RandomState(0)
    h, w, C = 7, 9, 4
    img = rng.randn(1, C, h, w).astype(np.float32)
    xs = np.concatenate([rng.uniform(-1.5, w + 0.5, 400), [-1.0, -0.999, 0.0, w - 1.0, w - 1.001, w - 0.5, 3.0, -0.5]]).astype(np.float32)
    ys = np.concatenate([rng.uniform(-1.5, h + 0.5, 400), [2.0, -0.5, h - 1.0, h - 0.25, 0.0, -1.0, h - 1.0, -0.999]]).astype(np.float32)
    want = oracle.bilinear_sample_zeros(torch.from_numpy(img), torch.from_numpy(xs).reshape(1, 1, -1), torch.from_numpy(ys).reshape(1, 1, -1)).numpy()[0, :, 0]
    got = np.zeros((C, xs.size), dtype=np.float64)
    for i, (x, y) in enumerate(zip(xs, ys)):
        if not (x > -1.0 and x < w and y > -1.0 and y < h):
            continue
        x0, y0 = int(np.floor(x)), int(np.floor(y))
        fx, fy = x - np.floor(x), y - np.floor(y)
        gx, gy = (np.floor(x) + 1.0) - x, (np.floor(y) + 1.0) - y
        xa = min(max(x0, 0), w - 2)
        wl = gx if x0 == xa else (fx if x0 + 1 == xa else 0.0)
        wr = fx if x0 + 1 == xa + 1 else (gx if x0 == xa + 1 else 0.0)
        rows = ((max(y0, 0), gy if y0 >= 0 else 0.0), (min(y0 + 1, h - 1), fy if y0 + 1 < h else 0.0))
        for yy, wy in rows:
            got[:, i] += wy * (wl * img[0, :, yy, xa] + wr * img[0, :, yy, xa + 1])
    assert np.abs(got - want).max() <= 1e-5


def test_bench_output_dump_is_float32_in_clip_order_and_capped(tmp_path, monkeypatch):
    import bench
    depth = np.arange(5 * 4 * 6, dtype=np.float64).reshape(5, 4, 6)
    bench.dump_outputs(str(tmp_path / "all"), depth)
    got = np.load(str(tmp_path / "all" / "depth.npy"))
    assert got.dtype == np.float32 and np.array_equal(got, depth)
    # above the size limit: the same seeded sample of whole clips every time, in clip order
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 4096 + 2 * depth[0].size * 4)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), depth)
    a, b = np.load(str(tmp_path / "a" / "depth.npy")), np.load(str(tmp_path / "b" / "depth.npy"))
    assert a.shape == (2, 4, 6) and np.array_equal(a, b)
    rows = [int(r[0, 0]) // depth[0].size for r in a]
    assert rows == sorted(rows) and all(np.array_equal(r, depth[i]) for r, i in zip(a, rows))
