"""Benchmark of the plane-sweep depth-inference hot path (BASELINE.json metric: fusionnet depth frames/sec at
256x256 with 64 planes; warp+correlate HBM GB/s vs peak).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--clips B] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one fusionnet keyframe (config c2: 256x256, D=64, 2 measurement frames, recurrent state carried, hidden-
state warp on) for each of the B independent clips a rank holds (B=1 = BASELINE.json configs[1]); clips are sharded
across ranks with no data-path collective (weak scaling: per-GPU work fixed).  One JSON line is printed by rank 0:
  value      frames/s, all ranks, inputs resident in HBM, timed with CUDA events (L2 flushed between steps)
  e2e        same metric through the reference-facing modules with HOST (pinned) inputs and a host read of the depth
  roofline   the fused plane-sweep kernel timed alone against the measured HBM peak (MEASURED_PEAKS.json)
  cpu_baseline  the oracle (CPU restatement of the reference) on the box's host cores, bounded sample
`--impl reference` times that CPU path alone (the reference is pure PyTorch-CPU; there is nothing to pip-install).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
for _p in (REPO, os.path.join(REPO, "deep-video-mvs_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

H, W, D, M = 256, 256, 64, 2
WORKLOAD = "fusionnet inference 256x256, 64 planes, 2 measurement frames, batch=%d clip(s)/GPU (BASELINE.json configs[1])"
SWEEP_BYTES_PER_CLIP = ((1 + M) * 32 + D) * (H // 2) * (W // 2) * 4        # SURVEY.md 8(d): 10,485,760 B at c2
CONV_FLOP_PER_KEYFRAME = 30.0e9                                             # SURVEY.md 8(a) / App. B: 2 x 15.0 GMAC at c2
# dram__bytes_read.sum + dram__bytes_write.sum PER CLIP of the sweep kernel from the committed ncu --set full capture named in
# SWEEP_TRAFFIC_SOURCE (a profiler run cannot happen inside a timed bench; tools/summarize_ncu.py writes the summary)
SWEEP_TRAFFIC_FILE = os.path.join(REPO, "profiles", "r02_sweep_tc_traffic.json")


def sweep_traffic_per_clip(n_clips=1):
    try:
        with open(SWEEP_TRAFFIC_FILE) as fh:
            d = json.load(fh)
        by = d.get("by_clips", {})
        if by:
            k = min(by, key=lambda c: abs(int(c) - n_clips))
            return (by[k]["dram_bytes_read"] + by[k]["dram_bytes_write"]) / float(k), d.get("source", "") + " (capture at %s clips)" % k
        return float(d["dram_bytes_per_clip"]), d.get("source", os.path.basename(SWEEP_TRAFFIC_FILE))
    except Exception:  # noqa: BLE001
        return None, None


def workload_config(n_clips, weights_desc):
    """The workload-defining part of the JSON line: identical for the GPU arm and the reference arm."""
    return {"workload": WORKLOAD % n_clips, "clips_per_gpu": n_clips, "height": H, "width": W, "planes": D, "measurement_frames": M,
            "weights": weights_desc, "inputs": "synthetic posed RGB stream (synth_data.make_clip, clip seed = global clip index)",
            "gpu_l2": "no flush between timed steps: the per-step working set (138 MB of weights + activations, fresh input frames every step) "
                      "exceeds the 126 MB L2 and the steps run back to back through the pipelined engine"}


SHIPPED_FILES = ["0_feature_extractor", "1_feature_pyramid", "2_encoder", "3_lstm_fusion", "4_decoder"]
TAGS = ["fe", "fpn", "cve", "lstm", "cvd"]


def load_weights(which="auto"):
    """tag -> state dict.  The reference's shipped fusionnet weights when they travelled with the snapshot (D = 64 is what
    they were trained for; tests/golden/_ref_data, fetched by tools/fetch_fixtures.py), else seeded He-scaled random weights
    of the same architecture (synth_data.make_state_dict, seed 7)."""
    d = os.path.join(REPO, "tests", "golden", "_ref_data", "weights", "fusionnet")
    if which in ("auto", "shipped") and all(os.path.isfile(os.path.join(d, f)) for f in SHIPPED_FILES):
        return ({tag: torch.load(os.path.join(d, f), map_location="cpu", weights_only=True) for tag, f in zip(TAGS, SHIPPED_FILES)},
                "reference's shipped fusionnet weights (dvmvs/fusionnet/weights)")
    if which == "shipped":
        raise RuntimeError("shipped weights not found under %s" % d)
    return None, "random-init (seeded, He-scaled) reference architecture"


def cpus_of_gpu(index):
    """Logical CPUs NVML reports as local to GPU `index` (its NUMA node), or None."""
    try:
        import pynvml as nv
        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(index)
        n = os.cpu_count() or 64
        words = nv.nvmlDeviceGetCpuAffinity(h, (n + 63) // 64)
        cpus = [w * 64 + b for w, word in enumerate(words) for b in range(64) if (int(word) >> b) & 1]
        return [c for c in cpus if c < n] or None
    except Exception:  # noqa: BLE001
        return None


def physical_core_cpus():
    """One logical CPU per physical core, socket by socket (Linux sysfs); falls back to all logical CPUs."""
    seen, out = set(), []
    n = os.cpu_count() or 1
    try:
        allowed = sorted(os.sched_getaffinity(0))
    except Exception:  # noqa: BLE001
        allowed = list(range(n))
    for c in allowed:
        base = "/sys/devices/system/cpu/cpu%d/topology/" % c
        try:
            key = (int(open(base + "physical_package_id").read()), int(open(base + "core_id").read()))
        except Exception:  # noqa: BLE001
            key = (0, c)
        if key not in seen:
            seen.add(key)
            out.append((key, c))
    out.sort()
    return [c for _, c in out]


def measured_peaks():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        with open(path) as fh:
            return json.load(fh), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback (B200_PROFILING.md)"


def log(msg):
    print("[bench] " + msg, file=sys.stderr, flush=True)


DUMP_LIMIT_BYTES = 64 * 10 ** 6


def dump_outputs(out_dir, depth):
    """Writes the depth maps (clips, H, W) of the timed path's last step, in clip order, as out_dir/depth.npy (float32), so that
    two builds run with the same arguments can be compared output for output.  When all clips together exceed 64 MB, a fixed
    seeded sample of whole clips is written instead, still in clip order."""
    depth = np.ascontiguousarray(depth, dtype=np.float32)
    keep = max(1, (DUMP_LIMIT_BYTES - 4096) // depth[0].nbytes)      # 4 KiB left for the .npy header
    if len(depth) > keep:
        depth = depth[np.sort(np.random.RandomState(0).choice(len(depth), keep, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    path = os.path.join(out_dir, "depth.npy")
    np.save(path, depth)
    log("wrote %s %s" % (path, tuple(depth.shape)))


class ClockSampler(threading.Thread):
    """SM clock / throttle reasons during the timed region via NVML in-process (no fork of a CUDA process)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag, self.max_mhz = index, [], threading.Event(), None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            bits = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown if hasattr(nv, "nvmlClocksEventReasonHwSlowdown") else 0x8,
                    "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
            while not self.stop_flag.is_set():
                mhz = float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                try:
                    r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))
                except Exception:
                    r = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                self.samples.append((mhz, [n for n, b in bits.items() if r & b]))
                self.stop_flag.wait(0.004)
        except Exception as e:  # noqa: BLE001
            self.samples.append((None, ["nvml unavailable: %s" % e]))

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=5)
        mhz = sorted(m for m, _ in self.samples if m is not None)
        reasons = sorted({r for _, rs in self.samples for r in rs})
        return {"sm_mhz": mhz[len(mhz) // 2] if mhz else None, "sm_max_mhz": self.max_mhz, "reasons": reasons,
                "samples": len(self.samples)}


# ---------------------------------------------------------------------------------------------------- workload
def make_inputs(n_clips, n_frames, rank):
    import synth_data as synth
    clips = [synth.make_clip(100000 + 1000 * rank + c, n_frames, H, W, M) for c in range(n_clips)]
    return clips


def stack_frame(clips, t):
    """Batched tensors (numpy) for keyframe t of every clip of this rank."""
    ref = np.stack([c["images"][c["frames"][t][0]] for c in clips])
    rpose = np.stack([c["poses"][c["frames"][t][0]] for c in clips])
    meas = [np.stack([c["images"][c["frames"][t][1][m]] for c in clips]) for m in range(M)]
    mpose = [np.stack([c["poses"][c["frames"][t][1][m]] for c in clips]) for m in range(M)]
    K = np.stack([c["K"] for c in clips])
    return ref, rpose, meas, mpose, K


def run_ours(args, rank, world, local_rank):
    import torch.distributed as dist
    import synth_data as synth
    from dvmvs import _native
    from dvmvs.fusionnet.model import CostVolumeDecoder, CostVolumeEncoder, FeatureExtractor, FeatureShrinker, LSTMFusion
    from dvmvs.utils import cost_volume_fusion
    from dvmvs import pipeline
    from dvmvs import _ops as ops
    ops.set_conv_backend(args.backend, terms=args.tc_terms, stride2=True)

    from dvmvs import sharding
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    # the host thread that enqueues this rank's work stays on the cores of its GPU's NUMA node
    numa_cpus = cpus_of_gpu(local_rank) if args.pin else None
    if numa_cpus:
        try:
            os.sched_setaffinity(0, numa_cpus)
        except Exception:  # noqa: BLE001
            numa_cpus = None
    B = args.clips
    n_frames = args.warmup + args.steps
    my_clips = sharding.clips_of_rank(B * world, rank, world)          # clip ids of this rank (round-robin over ranks)
    clips = [synth.make_clip(c, n_frames, H, W, M) for c in my_clips]

    shipped, weights_desc = load_weights(args.weights)
    mods = {"fe": FeatureExtractor(), "fpn": FeatureShrinker(), "cve": CostVolumeEncoder(), "lstm": LSTMFusion(), "cvd": CostVolumeDecoder()}
    for tag, m in mods.items():
        if shipped is not None:
            m.load_state_dict(shipped[tag], strict=True)
        else:
            shapes = {k: tuple(v.shape) for k, v in m.state_dict().items()}
            m.load_state_dict({k: torch.from_numpy(v) for k, v in synth.make_state_dict(shapes, seed=7).items()}, strict=True)
        m.to(dev).eval()

    log("modules built; staging %d frames" % n_frames)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)     # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()

    # ---------------- device-resident arm
    frames_dev = []
    for t in range(n_frames):
        ref, rpose, meas, mpose, K = stack_frame(clips, t)
        frames_dev.append((torch.from_numpy(ref).to(dev), torch.from_numpy(rpose).to(dev), [torch.from_numpy(x).to(dev) for x in meas],
                           [torch.from_numpy(p).to(dev) for p in mpose], torch.from_numpy(K).to(dev)))
    state = pipeline.KeyframeState()
    engine = pipeline.GraphedFusionnet(mods, batch=B, height=H, width=W, n_measurement_frames=M, n_depth_levels=D) if args.mode == "graph" else None

    def dev_step(t, state):
        if engine is not None:
            return engine.step(*frames_dev[t]), state
        return pipeline.keyframe(mods, state, *frames_dev[t], n_depth_levels=D)

    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    sampler = ClockSampler(local_rank)
    pipe = None
    engine_check = None
    if args.mode == "pipeline":
        def make_engine(mods_, batch_, h_=H, w_=W, m_=M, d_=D):
            if args.lookahead > 0:
                return pipeline.LookaheadFusionnet(mods_, batch=batch_, height=h_, width=w_, n_measurement_frames=m_, n_depth_levels=d_, lookahead=args.lookahead)
            return pipeline.PipelinedFusionnet(mods_, batch=batch_, height=h_, width=w_, n_measurement_frames=m_, n_depth_levels=d_, n_stages=args.stages)
        pipe = make_engine(mods, B)
        pred = torch.empty((B, H, W), dtype=torch.float32, device=dev)
        with torch.no_grad():
            pipe.prime(*frames_dev[0])            # one-off graph captures, outside warm-up and timing
            # the engine must reproduce the module call sequence: first keyframe (no recurrent state) through both
            pipe.submit(*frames_dev[0], out=pred)
            pipe.synchronize()
            eager0, _ = pipeline.keyframe(mods, pipeline.KeyframeState(), *frames_dev[0], n_depth_levels=D)
            engine_check = float((pred - eager0).abs().sum() / eager0.abs().sum())
            # PipelinedFusionnet reproduces the module sequence bit for bit; LookaheadFusionnet re-associates a few split-K sums (batch)
            assert engine_check <= (1e-4 if args.lookahead > 0 else 0.0) + 1e-7, "engine deviates from the eager module sequence: rel-L1 %g" % engine_check
            pipe.reset()
            for t in range(args.warmup):
                pipe.submit(*frames_dev[t], out=pred)
            pipe.synchronize()
            torch.cuda.synchronize()
            barrier()
            sampler.start()
            if os.environ.get("DVMVS_PROFILE") == "1":
                torch.cuda.profiler.start()
            p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            wall0 = time.perf_counter()
            p0.record(pipe.stream_a)
            for i in range(args.steps):
                pipe.submit(*frames_dev[args.warmup + i], out=pred)
            pipe.flush()                            # lookahead engine: launch an incomplete last group inside the timed region
            wall_enq = time.perf_counter()          # host side done enqueueing (the device may still be far behind)
            p1.record(pipe.stream_b)
            pipe.synchronize()
            torch.cuda.synchronize()
            wall1 = time.perf_counter()
            if os.environ.get("DVMVS_PROFILE") == "1":
                torch.cuda.profiler.stop()
            barrier()
        dev_ms_total = p0.elapsed_time(p1)
        launches = pipe.kernels_per_keyframe * args.steps
    else:
      with torch.no_grad():
        for t in range(args.warmup):
            _, state = dev_step(t, state)
        torch.cuda.synchronize()
        barrier()
        sampler.start()
        launches0 = _native.launch_count()
        if os.environ.get("DVMVS_PROFILE") == "1":
            torch.cuda.profiler.start()
        wall0 = time.perf_counter()
        for i in range(args.steps):
            flush.zero_()
            ev[i][0].record()
            pred, state = dev_step(args.warmup + i, state)
            ev[i][1].record()
        torch.cuda.synchronize()
        wall1 = time.perf_counter()
        if os.environ.get("DVMVS_PROFILE") == "1":
            torch.cuda.profiler.stop()
        barrier()
      launches = _native.launch_count() - launches0
      if engine is not None:
        launches = engine.kernels_per_replay[True] * args.steps
      dev_ms_total = sum(a.elapsed_time(b) for a, b in ev)
    log("device-resident arm done")
    clocks = sampler.summary()
    dev_ms = dev_ms_total
    assert bool(torch.isfinite(pred).all()), "non-finite depth"
    # the depth maps of the timed path's last step, copied before the other arms reuse the engines' buffers
    last_depth = pred.detach().float().reshape(B, H, W).clone()

    # ---------------- end-to-end arm: pinned host inputs -> modules -> host depth, copies inside the timed region
    frames_host = []
    for t in range(n_frames):
        ref, rpose, meas, mpose, K = stack_frame(clips, t)
        frames_host.append(tuple(torch.from_numpy(np.ascontiguousarray(a)).pin_memory() for a in (ref, rpose, *meas, *mpose, K)))
    h2d_bytes = sum(a.numel() * 4 for a in frames_host[0])
    out_host = torch.empty((B, H, W), dtype=torch.float32).pin_memory()
    d2h_bytes = out_host.numel() * 4
    state = pipeline.KeyframeState()
    if engine is not None:
        engine.reset()

    if pipe is not None:
        pipe.reset()

    def e2e_step(t, state):
        fh = frames_host[t]
        if pipe is not None:            # H2D on the feature stream, D2H of the depth on the recurrent stream
            pipe.submit(fh[0], fh[1], fh[2:2 + M], fh[2 + M:2 + 2 * M], fh[2 + 2 * M], out=out_host)
            return state
        if engine is not None:          # H2D copies into the graph's static buffers happen inside step()
            pred = engine.step(fh[0], fh[1], fh[2:2 + M], fh[2 + M:2 + 2 * M], fh[2 + 2 * M])
        else:
            hs = [a.to(dev, non_blocking=True) for a in fh]
            ref, rpose, meas, mpose, K = hs[0], hs[1], hs[2:2 + M], hs[2 + M:2 + 2 * M], hs[2 + 2 * M]
            pred, state = pipeline.keyframe(mods, state, ref, rpose, meas, mpose, K, n_depth_levels=D)
        out_host.copy_(pred, non_blocking=True)
        return state

    with torch.no_grad():
        for t in range(args.warmup):
            state = e2e_step(t, state)
        if pipe is not None:
            pipe.synchronize()
        torch.cuda.synchronize()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(pipe.stream_a if pipe is not None else torch.cuda.current_stream())
        for i in range(args.steps):
            state = e2e_step(args.warmup + i, state)
        if pipe is not None:
            pipe.flush()
        e1.record(pipe.stream_b if pipe is not None else torch.cuda.current_stream())
        if pipe is not None:
            pipe.synchronize()
        torch.cuda.synchronize()
        barrier()
    e2e_ms = e0.elapsed_time(e1)
    log("e2e arm done")

    # ---------------- roofline of the dominant geometric kernel: the fused plane sweep the engine runs, timed alone
    from dvmvs import _ops as ops
    ref, rpose, meas, mpose, K = frames_dev[0]

    def time_sweep(nb):
        """CUDA-event time of one sweep launch over nb clips (L2 flushed between launches) + its error vs the fp32 gather kernel."""
        g = torch.Generator(device="cpu").manual_seed(nb)
        f1 = (torch.randn(nb, H // 2, W // 2, 32, generator=g) * 4).to(dev)
        f2 = [(torch.randn(nb, H // 2, W // 2, 32, generator=g) * 4).to(dev) for _ in range(M)]
        rp = rpose[:1].repeat(nb, 1, 1)
        mp = [p_[:1].repeat(nb, 1, 1) for p_ in mpose]
        hk = K[:1].repeat(nb, 1, 1).clone()
        hk[:, 0:2, :] /= 2.0
        use_tc = ops.sweep_uses_tc(True, 32, D, M)
        if use_tc:
            p1, p2 = ops.split_planes(f1), [ops.split_planes(t) for t in f2]
            run = lambda: ops.plane_sweep_tc(p1, p2, rp, mp, hk, 0.25, 20.0, D, terms=ops.sweep_terms())
        else:
            run = lambda: ops.plane_sweep(f1, f2, rp, mp, hk, 0.25, 20.0, D, True)
        base = ops.plane_sweep(f1, f2, rp, mp, hk, 0.25, 20.0, D, True)
        err = float((run() - base).abs().max() / base.abs().max())
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(20)]
        for _ in range(3):
            run()
        for a, b in evs:
            flush.zero_()
            a.record()
            run()
            b.record()
        torch.cuda.synchronize()
        return float(np.median([a.elapsed_time(b) for a, b in evs])), err, ("plane_sweep_tc_kernel<%d>" % ops.sweep_terms()) if use_tc else "plane_sweep_c32_kernel"

    # the launch the timed region issues: the lookahead engine sweeps a whole group (lookahead x B clips) per launch
    sweep_nb = B * (args.lookahead if (args.mode == "pipeline" and args.lookahead > 0) else 1)
    sweep_ms, sweep_err, sweep_kernel = time_sweep(sweep_nb)
    sweep_points = {}
    for nb in (B, 8, 32):
        if nb != sweep_nb and (args.extras or nb == B) and ("clips_%d" % nb) not in sweep_points:
            ms_nb, _, _ = time_sweep(nb)
            sweep_points["clips_%d" % nb] = {"ms_per_launch": ms_nb, "achieved_GBps": SWEEP_BYTES_PER_CLIP * nb / (ms_nb * 1e-3) / 1e9}
    log("roofline arm done: plane sweep %.3f ms" % sweep_ms)

    # ---------------- extra operating points (reported next to the headline, SURVEY.md 8d): strictly sequential latency
    # of one keyframe (CUDA graph, no inter-keyframe overlap) and batched throughput (EXTRA_B clips per GPU)
    extras = {}
    if args.extras:
        with torch.no_grad():
            eng = pipeline.GraphedFusionnet(mods, batch=B, height=H, width=W, n_measurement_frames=M, n_depth_levels=D)
            for t in range(4):
                eng.step(*frames_dev[t])
            lat = []
            for t in range(4, min(n_frames, 16)):
                flush.zero_()
                a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                eng.step(*frames_dev[t])
                b_.record()
                torch.cuda.synchronize()
                lat.append(a.elapsed_time(b_))
            extras["sequential_latency_ms_per_keyframe"] = float(np.median(lat)) if lat else None
            del eng
            for EB in sorted({int(v) for v in str(args.extra_clips).split(",") if int(v) > B}):
                clips_b = make_inputs(EB, 12, rank)
                fb = []
                for t in range(12):
                    ref, rpose, meas, mpose, K = stack_frame(clips_b, t)
                    fb.append((torch.from_numpy(ref).to(dev), torch.from_numpy(rpose).to(dev), [torch.from_numpy(x).to(dev) for x in meas],
                               [torch.from_numpy(p_).to(dev) for p_ in mpose], torch.from_numpy(K).to(dev)))
                pb = pipeline.PipelinedFusionnet(mods, batch=EB, height=H, width=W, n_measurement_frames=M, n_depth_levels=D, n_stages=args.stages)
                outb = torch.empty((EB, H, W), dtype=torch.float32, device=dev)
                pb.prime(*fb[0])
                for t in range(4):
                    pb.submit(*fb[t], out=outb)
                pb.synchronize()
                q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                q0.record(pb.stream_a)
                for t in range(4, 12):
                    pb.submit(*fb[t], out=outb)
                q1.record(pb.stream_b)
                pb.synchronize()
                torch.cuda.synchronize()
                ms = q0.elapsed_time(q1)
                fps_b = EB * 8 / (ms * 1e-3)
                extras["batched_%d" % EB] = {"clips_per_gpu": EB, "frames_per_s_per_gpu": fps_b, "ms_per_step": ms / 8,
                                             "conv_TFLOPs_algorithmic": fps_b * CONV_FLOP_PER_KEYFRAME / 1e12,
                                             "finite": bool(torch.isfinite(outb).all())}
                del pb, fb, outb
                torch.cuda.empty_cache()
            # the reference script's own call sequence (module forward()s one by one, M + 1 separate feature passes, host launches)
            st_s = pipeline.KeyframeState()
            lat_s = []
            for t in range(min(n_frames, 14)):
                a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                w0 = time.perf_counter()
                a.record()
                _, st_s = pipeline.keyframe(mods, st_s, *frames_dev[t], n_depth_levels=D, batch_features=False)
                b_.record()
                torch.cuda.synchronize()
                if t >= 4:
                    lat_s.append((a.elapsed_time(b_), (time.perf_counter() - w0) * 1e3))
            extras["script_sequence"] = {"ms_per_keyframe_device": float(np.median([x[0] for x in lat_s])),
                                         "ms_per_keyframe_wall": float(np.median([x[1] for x in lat_s])),
                                         "note": "run-testing.py:153-202 call sequence through the drop-in modules (M + 1 separate feature passes, eleven module / utils calls per keyframe, "
                                                 "each replaying its own auto-captured CUDA graph: dvmvs/_base.py)"}
            # SURVEY 8 row f4: the predicted depth maps fused into a TSDF volume (the reference's run-tsdf-reconstruction.py),
            # 4 cm voxels over an 8 x 6.4 x 4.8 m room, frames at the network's resolution; device-resident and from host arrays
            try:
                from dvmvs.tsdf import TSDFVolume
                rng_t = np.random.RandomState(5)
                vol_t = TSDFVolume(np.array([[-4.0, 4.0], [-3.2, 3.2], [0.0, 4.8]]), 0.04, device=dev)
                K_t = np.array([[0.78 * W, 0, W / 2.0], [0, 0.78 * W, H / 2.0], [0, 0, 1.0]])
                fr_t = []
                for i in range(16):
                    yy, xx = np.mgrid[0:H, 0:W]
                    dep = (2.0 + 0.8 * np.sin(xx / 40.0 + i) * np.cos(yy / 30.0)).astype(np.float32)
                    col = rng_t.randint(0, 256, size=(H, W, 3)).astype(np.uint8)
                    pose_t = np.eye(4)
                    pose_t[:3, 3] = [0.05 * i, -0.02 * i, 0.01 * i]
                    fr_t.append((col, dep, pose_t))
                dev_t = [(torch.from_numpy(c).to(dev), torch.from_numpy(d_).to(dev), p_) for c, d_, p_ in fr_t]
                for c, d_, p_ in fr_t[:4] + dev_t[:4]:
                    vol_t.integrate(c, d_, K_t, p_)
                torch.cuda.synchronize()
                t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0.record()
                for _ in range(4):
                    for c, d_, p_ in dev_t:
                        vol_t.integrate(c, d_, K_t, p_)
                t1.record()
                torch.cuda.synchronize()
                w0 = time.perf_counter()
                for _ in range(4):
                    for c, d_, p_ in fr_t:
                        vol_t.integrate(c, d_, K_t, p_)
                torch.cuda.synchronize()
                extras["tsdf_fusion"] = {"voxels": int(np.prod(vol_t._vol_dim)), "frame": [H, W],
                                         "frames_per_s_resident": 64.0 / (t0.elapsed_time(t1) * 1e-3),
                                         "frames_per_s_host_frames": 64.0 / (time.perf_counter() - w0),
                                         "note": "dvmvs.tsdf.TSDFVolume.integrate (one launch per frame, bit-identical to the reference's CPU path; tests/test_tsdf.py)"}
                del vol_t, dev_t
            except Exception as e:  # noqa: BLE001
                extras["tsdf_fusion"] = {"error": repr(e)}
            # BASELINE.json configs[2]: 320x256, 96 planes, 4 measurement frames (its own module set: aggregator0 has D+32 inputs)
            if args.mode == "pipeline":
                from dvmvs.config import Config as _Config
                H3, W3, D3, M3 = 256, 320, 96, 4
                saved_levels = _Config.train_n_depth_levels
                _Config.train_n_depth_levels = D3
                try:
                    mods3 = {"fe": FeatureExtractor(), "fpn": FeatureShrinker(), "cve": CostVolumeEncoder(), "lstm": LSTMFusion(), "cvd": CostVolumeDecoder()}
                finally:
                    _Config.train_n_depth_levels = saved_levels
                for tag, m in mods3.items():
                    shapes = {k: tuple(v.shape) for k, v in m.state_dict().items()}
                    m.load_state_dict({k: torch.from_numpy(v) for k, v in synth.make_state_dict(shapes, seed=7).items()}, strict=True)
                    m.to(dev).eval()
                clip3 = synth.make_clip(7000 + rank, 16, H3, W3, M3)
                f3 = []
                for ref_i, meas_i in clip3["frames"]:
                    up = lambda a: torch.from_numpy(np.ascontiguousarray(a))[None].to(dev)
                    f3.append((up(clip3["images"][ref_i]), up(clip3["poses"][ref_i]), [up(clip3["images"][j]) for j in meas_i],
                               [up(clip3["poses"][j]) for j in meas_i], up(clip3["K"])))
                p3 = make_engine(mods3, 1, H3, W3, M3, D3)
                out3 = torch.empty((1, H3, W3), dtype=torch.float32, device=dev)
                p3.prime(*f3[0])
                for t in range(4):
                    p3.submit(*f3[t], out=out3)
                p3.synchronize()
                torch.cuda.synchronize()
                r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                r0.record(p3.stream_a)
                for t in range(4, 16):
                    p3.submit(*f3[t], out=out3)
                p3.flush()
                r1.record(p3.stream_b)
                p3.synchronize()
                torch.cuda.synchronize()
                ms = r0.elapsed_time(r1)
                extras["config_c3_320x256_96planes_4frames"] = {"frames_per_s_per_gpu": 12 / (ms * 1e-3), "ms_per_step": ms / 12,
                                                                "finite": bool(torch.isfinite(out3).all())}
                del p3, mods3, f3
            # the same stream through PipelinedFusionnet (5 stages, one keyframe per stage launch, results available keyframe by
            # keyframe): what the headline engine's batching of the state-independent stages over time buys
            if args.mode == "pipeline" and args.lookahead > 0:
                pn = pipeline.PipelinedFusionnet(mods, batch=B, height=H, width=W, n_measurement_frames=M, n_depth_levels=D, n_stages=args.stages)
                outn = torch.empty((B, H, W), dtype=torch.float32, device=dev)
                pn.prime(*frames_dev[0])
                for t in range(args.warmup):
                    pn.submit(*frames_dev[t], out=outn)
                pn.synchronize()
                torch.cuda.synchronize()
                n0, n1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                n0.record(pn.stream_a)
                for t in range(args.warmup, n_frames):
                    pn.submit(*frames_dev[t], out=outn)
                n1.record(pn.stream_b)
                pn.synchronize()
                torch.cuda.synchronize()
                ms_n = n0.elapsed_time(n1) / args.steps
                extras["pipelined_%d_stages_no_lookahead" % args.stages] = {
                    "frames_per_s_per_gpu": B * 1e3 / ms_n, "ms_per_step": ms_n, "launches_per_keyframe": pn.kernels_per_keyframe,
                    "rel_l1_inverse_depth_vs_headline_last_keyframe": float(((1.0 / outn) - (1.0 / pred)).abs().sum() / (1.0 / pred).abs().sum())}
                del pn
            # the other operand precision of the tensor path (fp16 (hi, lo) pairs, three products: ~fp32 accuracy)
            if args.backend == "tc" and args.mode == "pipeline":
                other = 3 if args.tc_terms == 1 else 1
                ops.set_conv_backend("tc", terms=other, stride2=True)
                po = make_engine(mods, B)
                outo = torch.empty((B, H, W), dtype=torch.float32, device=dev)
                po.prime(*frames_dev[0])
                for t in range(args.warmup):
                    po.submit(*frames_dev[t], out=outo)
                po.synchronize()
                torch.cuda.synchronize()
                o0, o1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                o0.record(po.stream_a)
                for t in range(args.warmup, n_frames):
                    po.submit(*frames_dev[t], out=outo)
                po.flush()
                o1.record(po.stream_b)
                po.synchronize()
                torch.cuda.synchronize()
                ms = o0.elapsed_time(o1)
                d = (1.0 / outo - 1.0 / pred).abs().sum() / (1.0 / outo).abs().sum()
                extras["operands_%s" % ("fp16_pairs_3_terms" if other == 3 else "fp16_1_term")] = {
                    "frames_per_s_per_gpu": B * args.steps / (ms * 1e-3), "ms_per_step": ms / args.steps,
                    "rel_l1_inverse_depth_between_the_two_precisions_last_keyframe": float(d)}
                del po
                ops.set_conv_backend("tc", terms=args.tc_terms, stride2=True)
            # SURVEY 8 row f1: measurement features from the feature cache (every measurement frame of the synthetic stream
            # was the reference frame of an earlier keyframe).  Reported beside the headline, never as it: the headline
            # recomputes FeatureExtractor + FeatureShrinker for all M+1 images like the reference does.
            ids = clips[0]["frames"]
            pc = pipeline.PipelinedFusionnet(mods, batch=B, height=H, width=W, n_measurement_frames=M, n_depth_levels=D,
                                             n_stages=args.stages, feature_cache=max(8, M + 1))
            outc = torch.empty((B, H, W), dtype=torch.float32, device=dev)
            pc.prime(*frames_dev[0])
            for t in range(args.warmup):
                pc.submit(*frames_dev[t], out=outc, reference_id=ids[t][0], measurement_ids=ids[t][1])
            pc.synchronize()
            torch.cuda.synchronize()
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            h0, m0 = pc.cache.hits, pc.cache.misses
            c0.record(pc.stream_a)
            for t in range(args.warmup, n_frames):
                pc.submit(*frames_dev[t], out=outc, reference_id=ids[t][0], measurement_ids=ids[t][1])
            c1.record(pc.stream_b)
            pc.synchronize()
            torch.cuda.synchronize()
            ms = c0.elapsed_time(c1)
            extras["feature_cache"] = {"frames_per_s_per_gpu": B * args.steps / (ms * 1e-3), "ms_per_step": ms / args.steps,
                                       "hits": pc.cache.hits - h0, "misses": pc.cache.misses - m0,
                                       "rel_l1_inverse_depth_vs_headline_last_keyframe": (float((1.0 / outc - 1.0 / pred).abs().sum() / (1.0 / pred).abs().sum())
                                                                                           if args.mode == "pipeline" else None),
                                       "note": "different FeatureExtractor batch (1 vs M + 1) => different split-K summation order; with fp16 operands a "
                                               "1-ulp fp32 difference can flip an operand's rounding, so the two engines agree to ~3e-5, not bit for bit "
                                               "(both are <= 4.5e-5 from the oracle: tools/cache_probe.py)"}
            del pc
        log("extra operating points done")

    # ---------------- max over ranks
    t = torch.tensor([dev_ms, e2e_ms], dtype=torch.float64, device=dev)
    lt = torch.tensor([float(launches)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(lt, op=dist.ReduceOp.SUM)
    dev_ms, e2e_ms = float(t[0]), float(t[1])
    total_frames = B * args.steps * world
    peaks, peak_src = measured_peaks()
    achieved = SWEEP_BYTES_PER_CLIP * sweep_nb / (sweep_ms * 1e-3) / 1e9
    traffic_per_clip, traffic_src = sweep_traffic_per_clip(sweep_nb)
    fps = total_frames / (dev_ms * 1e-3)
    tensor_peak = peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"])
    conv_tf = fps / world * CONV_FLOP_PER_KEYFRAME / 1e12          # per GPU
    dtype = "f32" if args.backend == "fp32" else ("f16+f32acc" if args.tc_terms == 1 else "f16x2+f32acc")
    # final depth maps of every clip on every rank (clip order): the trivial gather of independent clips, outside the timed region
    gathered = sharding.gather_clip_results({c: last_depth[i] for i, c in enumerate(my_clips)}, B * world, device=dev)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, torch.stack(gathered).cpu().numpy())
    result = {
        "metric": "fusionnet depth frames/sec @256x256x64planes", "value": fps, "unit": "frames/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": dtype, "data": "synthetic",
        "config": (workload_config(B, weights_desc) if args.mode == "pipeline" else
                   dict(workload_config(B, weights_desc), gpu_l2="flushed (256 MiB write) between timed steps")),
        "engine": {"mode": args.mode + ((" (LookaheadFusionnet: trunk, pyramid, plane sweep and encoder batched over groups of %d consecutive keyframes, "
                                          "recurrent stage per keyframe; 5 streams)" % args.lookahead) if (args.mode == "pipeline" and args.lookahead > 0)
                                         else (" (%d stages)" % args.stages if args.mode == "pipeline" else "")),
                   "conv_backend": args.backend + ("" if args.backend == "fp32" else (" (tcgen05, fp16 operands, fp32 accumulate)" if args.tc_terms == 1
                                                                                         else " (tcgen05, fp16-pair operands x3 terms, fp32 accumulate)")),
                   "plane_sweep": sweep_kernel,
                   "parity": "this exact configuration is held to <= 3.3e-4 rel-L1 on inverse depth vs the oracle / the shipped golden by "
                             "tests/test_gpu_parity.py::test_benchmarked_configuration_* (budget 1e-3)",
                   "engine_vs_eager_modules_rel_l1_first_keyframe": engine_check,
                   "l2": ("per-step working set (weights 138 MB + activations) exceeds the 126 MB L2; steps run back to back (pipelined)"
                          if args.mode == "pipeline" else "flushed (256 MiB write) between timed steps"),
                   "parallelism": "clip-sharded x%d (dvmvs.sharding, round-robin), no data-path collective" % world,
                   "host_thread_pinned_to_gpu_numa_cpus": len(numa_cpus) if numa_cpus else 0,
                   "host_loop_wall_ms_per_step": (wall1 - wall0) * 1e3 / args.steps,
                   "host_enqueue_ms_per_step": ((wall_enq - wall0) * 1e3 / args.steps) if args.mode == "pipeline" else None,
                   "gathered_depth_checksum": float(sum(float(t.double().sum()) for t in gathered))},
        "clocks": clocks,
        "e2e": {"value": total_frames / (e2e_ms * 1e-3), "unit": "frames/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes},
        "gpu_launches": int(lt[0]),
        "operating_points": extras,
        "roofline": {"kernel": sweep_kernel, "bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                     "frac": achieved / peaks["hbm_gbs"], "traffic": (traffic_per_clip * sweep_nb) if traffic_per_clip else None,
                     "traffic_source": traffic_src, "peak_source": peak_src, "ms_per_launch": sweep_ms,
                     "algorithmic_bytes_per_launch": SWEEP_BYTES_PER_CLIP * sweep_nb, "clips_per_launch": sweep_nb,
                     "rel_err_vs_fp32_gather_kernel": sweep_err,
                     "other_batches": {k: dict(v, frac=v["achieved_GBps"] / peaks["hbm_gbs"]) for k, v in sweep_points.items()},
                     "note": "correlate-then-interpolate on tcgen05: bound by shared-memory traffic and issue slots of the look-ups, not by HBM "
                             "(64 FLOP per algorithmic byte; DESIGN.md section 6)"},
        "roofline_conv": {"bound": "tensor", "achieved": conv_tf, "peak": tensor_peak, "unit": "TFLOP/s", "frac": conv_tf / tensor_peak,
                          "algorithmic_flop_per_keyframe": CONV_FLOP_PER_KEYFRAME, "peak_source": peak_src + " (sustained bf16)",
                          "batched": {k: {"achieved": v["conv_TFLOPs_algorithmic"], "frac": v["conv_TFLOPs_algorithmic"] / tensor_peak}
                                      for k, v in extras.items() if k.startswith("batched_")},
                          "note": "whole conv stack of a keyframe (2 x MACs of SURVEY App. B) over the CUDA-event time of the pipelined step; "
                                  "algorithmic FLOPs (1-term products)"},
    }
    return result


# ---------------------------------------------------------------------------------------------------- CPU arms
def oracle_inputs(n_frames, weights_which="auto"):
    """Weights (same choice as the GPU arm) and one c2 clip for the oracle-based baselines."""
    import synth_data as synth
    from oracle import dvmvs_oracle as oracle
    w, desc = load_weights(weights_which)
    if w is None:
        shapes = oracle.state_dict_shapes(D)
        w = {tag: {k: torch.from_numpy(v) for k, v in synth.make_state_dict(shapes[tag], seed=7).items()} for tag in shapes}
    clip = synth.make_clip(0, n_frames, H, W, M)
    return oracle, w, desc, clip


def oracle_frames(oracle, w, clip, first, count, device="cpu", state=None):
    """Runs `count` recurrent keyframes of the clip starting at `first`; returns (seconds per frame list, state)."""
    K = torch.from_numpy(clip["K"])[None].to(device)
    st = state if state is not None else oracle.FusionnetState()
    times = []
    up = lambda a: torch.from_numpy(a)[None].to(device)
    with torch.no_grad():
        for ref_i, meas_i in clip["frames"][first:first + count]:
            if device != "cpu":
                torch.cuda.synchronize()
            t0 = time.perf_counter()
            _, st = oracle.fusionnet_step(w, st, up(clip["images"][ref_i]), up(clip["poses"][ref_i]), [up(clip["images"][j]) for j in meas_i],
                                          [up(clip["poses"][j]) for j in meas_i], K, n_depth_levels=D)
            if device != "cpu":
                torch.cuda.synchronize()
            times.append(time.perf_counter() - t0)
    return times, st


def best_thread_count(oracle, w, clip):
    """The reference's PyTorch-CPU path scales poorly past one socket and collapses when SMT siblings spin in OpenMP barriers
    (round 1: 0.78 frames/s with 64 threads on one box, 3.76 on another).  Try {8, 16, 32, physical cores} threads, each pinned to
    that many physical cores (socket 0 first), on one keyframe after a warm-up keyframe; keep the fastest."""
    cores = physical_core_cpus()
    cand = sorted({n for n in (8, 16, 32, len(cores)) if 1 <= n <= len(cores)}) or [len(cores)]
    trials = {}
    for n in cand:
        try:
            os.sched_setaffinity(0, cores[:n])
        except Exception:  # noqa: BLE001
            pass
        torch.set_num_threads(n)
        t, _ = oracle_frames(oracle, w, clip, 0, 2)
        trials[n] = t[1]
        log("cpu threads %d: %.2f s per keyframe" % (n, t[1]))
        if t[1] > min(trials.values()):          # past the knee: more threads only add OpenMP barrier cost (64 threads: 1.2 - 60 s per keyframe)
            break
    best = min(trials, key=trials.get)
    try:
        os.sched_setaffinity(0, cores[:best])
    except Exception:  # noqa: BLE001
        pass
    torch.set_num_threads(best)
    return best, {str(k): round(v, 3) for k, v in trials.items()}, len(cores)


def cpu_baseline(n_frames, weights_which="auto", budget_s=40.0, warmup=1):
    """The oracle (restatement of the reference's PyTorch-CPU path) on the host cores: up to n_frames recurrent keyframes of ONE
    c2 clip after `warmup` untimed keyframes, stopping early once budget_s is spent (budget_s=None: all n_frames).  Returns the
    record and the depth map (1, H, W) of the last timed keyframe."""
    saved_aff = None
    try:
        saved_aff = os.sched_getaffinity(0)
    except Exception:  # noqa: BLE001
        pass
    saved_threads = torch.get_num_threads()
    oracle, w, desc, clip = oracle_inputs(warmup + n_frames, weights_which)
    threads, trials, n_phys = best_thread_count(oracle, w, clip)
    log("cpu baseline: oracle on %d threads, %d warm-up + up to %d frames" % (threads, warmup, n_frames))
    _, st = oracle_frames(oracle, w, clip, 0, warmup)      # untimed: they build the recurrent state the timed keyframes start from
    times = []
    for t in range(warmup, warmup + n_frames):
        dt, st = oracle_frames(oracle, w, clip, t, 1, state=st)
        times += dt
        if budget_s is not None and sum(times) > budget_s and len(times) >= 2:
            break
    out = {"value": len(times) / sum(times), "unit": "frames/s", "cores": threads, "kind": "port", "frames_run": len(times),
           "thread_trials_s_per_keyframe": trials, "physical_cores": n_phys, "weights": desc,
           "sample": "%d recurrent keyframes of one c2 clip (256x256, D=64, M=2) after %d warm-up, torch %s CPU, %d threads pinned to %d physical cores"
                     % (len(times), warmup, torch.__version__, threads, threads)}
    try:        # SURVEY 8(d): the reference's cost_volume_fusion alone, beside the GPU kernel's roofline entry (never fatal)
        g = torch.Generator().manual_seed(0)
        f1 = torch.randn(1, 32, H // 2, W // 2, generator=g) * 4
        f2 = [torch.randn(1, 32, H // 2, W // 2, generator=g) * 4 for _ in range(M)]
        ref_i, meas_i = clip["frames"][0]
        half_K = torch.from_numpy(clip["K"])[None].clone()
        half_K[:, 0:2, :] /= 2.0
        grid = oracle.get_warp_grid_for_cost_volume_calculation(W // 2, H // 2)
        poses = [torch.from_numpy(clip["poses"][j])[None] for j in meas_i]
        sw = []
        with torch.no_grad():
            for _ in range(3):
                t0 = time.perf_counter()
                oracle.cost_volume_fusion(f1, f2, torch.from_numpy(clip["poses"][ref_i])[None], poses, half_K, grid, 0.25, 20.0, D, "cpu", True)
                sw.append(time.perf_counter() - t0)
        best = min(sw[1:])
        out["plane_sweep"] = {"ms_per_cost_volume": best * 1e3, "algorithmic_GBps": SWEEP_BYTES_PER_CLIP / best / 1e9,
                              "sample": "cost_volume_fusion of one c2 clip (128x128x32 features, D=64, M=2), best of 2 after 1 warm-up"}
    except Exception as e:  # noqa: BLE001
        out["plane_sweep"] = {"error": str(e)[:200]}
    if saved_aff is not None:
        try:
            os.sched_setaffinity(0, saved_aff)
        except Exception:  # noqa: BLE001
            pass
    torch.set_num_threads(saved_threads)
    return out, st.previous_depth.reshape(1, H, W).numpy()


def gpu_eager_baseline(n_frames=6, weights_which="auto"):
    """SURVEY 8(d)'s second baseline: the reference algorithm as plain PyTorch eager ON THE B200 (the oracle port moved to
    cuda: cuDNN convolutions, the D x M Python plane loop with its ~20 element-wise launches per plane, the host round trip
    in the depth re-projection) -- what a user gets from the reference today on this GPU.  CUDA-event time per keyframe."""
    try:
        oracle, w, desc, clip = oracle_inputs(n_frames + 2, weights_which)
        dev = "cuda"
        wd = {tag: {k: v.to(dev) for k, v in sd.items()} for tag, sd in w.items()}
        _, st = oracle_frames(oracle, wd, clip, 0, 2, device=dev)
        evs = []
        K = torch.from_numpy(clip["K"])[None].to(dev)
        up = lambda a: torch.from_numpy(a)[None].to(dev)
        with torch.no_grad():
            for ref_i, meas_i in clip["frames"][2:2 + n_frames]:
                args_ = (up(clip["images"][ref_i]), up(clip["poses"][ref_i]), [up(clip["images"][j]) for j in meas_i], [up(clip["poses"][j]) for j in meas_i])
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                _, st = oracle.fusionnet_step(wd, st, *args_, K, n_depth_levels=D)
                b.record()
                torch.cuda.synchronize()
                evs.append(a.elapsed_time(b))
        ms = float(np.median(evs))
        return {"value": 1e3 / ms, "unit": "frames/s", "ms_per_keyframe": ms, "kind": "port on cuda (torch eager / cuDNN, fp32, TF32 off)",
                "frames_run": len(evs), "weights": desc}
    except Exception as e:  # noqa: BLE001
        return {"error": str(e)[:300]}


def run_reference(args):
    """The reference's own CPU implementation of the path (oracle port: the reference is pure PyTorch, nothing compiles), all the
    host threads it can use (best of a small thread sweep), on the GPU arm's workload and clip: the warm-up keyframes untimed, then
    exactly `steps` timed keyframes."""
    # torchrun exports OMP_NUM_THREADS=1 to its workers: rank 0 is the only rank doing work here, give it the machine back
    os.environ.pop("OMP_NUM_THREADS", None)
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    t0 = time.perf_counter()
    base, last_depth = cpu_baseline(args.steps, args.weights, budget_s=None, warmup=args.warmup)
    wall = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last_depth)
    fps = base["value"]
    cfg = workload_config(1, base["weights"])
    return {"impl": "reference", "metric": "fusionnet depth frames/sec @256x256x64planes", "value": fps, "unit": "frames/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "steps_run": base["frames_run"], "ms_per_step": 1e3 / fps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
            "engine": {"mode": "reference's own PyTorch-CPU path (oracle port; the reference has no compiled code)", "wall_s": wall},
            "cpu_baseline": base, "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)       # ~60 ms timed region: enough for a dozen in-region clock samples
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--clips", type=int, default=1, help="independent clips per GPU (batched through the modules)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default=os.environ.get("DVMVS_BENCH_MODE", "pipeline"), choices=["pipeline", "graph", "eager"],
                    help="pipeline (default): CUDA graphs, keyframe t+1's feature stage overlapped with keyframe t's recurrent "
                         "stage on a second stream; graph: one CUDA graph per keyframe, strictly sequential; eager: one host "
                         "launch per kernel")
    ap.add_argument("--backend", default=os.environ.get("DVMVS_CONV_BACKEND", "tc"), choices=["tc", "fp32"])
    ap.add_argument("--tc-terms", type=int, default=1, choices=[1, 3],
                    help="operand precision of the tcgen05 convolutions: 1 = fp16 operands, fp32 accumulate (default; measured "
                         "<= 1.1e-4 rel-L1 on inverse depth, budget 1e-3); 3 = fp16 (hi, lo) pairs, three products (~1e-6)")
    ap.add_argument("--stages", type=int, default=5, choices=[2, 3, 4, 5], help="pipeline depth of --mode pipeline (with --lookahead 0)")
    ap.add_argument("--lookahead", type=int, default=4,
                    help="--mode pipeline: keyframes per group of LookaheadFusionnet (state-independent stages batched over consecutive "
                         "keyframes; every keyframe still gets all its feature passes); 0 = PipelinedFusionnet(--stages)")
    ap.add_argument("--extras", type=int, default=1, help="also measure sequential latency and batched throughput (0 to skip)")
    ap.add_argument("--extra-clips", default="8,32", help="clips per GPU of the batched operating points (comma separated)")
    ap.add_argument("--cpu-frames", type=int, default=6, help="frames of the bounded CPU-baseline sample")
    ap.add_argument("--weights", default="synthetic", choices=["auto", "shipped", "synthetic"],
                    help="synthetic (default): seeded He-scaled weights of the reference architecture -- the configuration the parity tests "
                         "pin over the bench's full 105-keyframe horizon.  shipped / auto: the reference's shipped fusionnet weights "
                         "(tests/golden/_ref_data): same kernels and shapes, i.e. the same speed, but on the synthetic NOISE clips the trained "
                         "network is ill-conditioned -- fp16 operands drift to 6e-3 rel-L1 after ~90 recurrent keyframes there (3-term: 9e-5) "
                         "while staying at 1.1e-4 over 72 keyframes of the real fixture scene (profiles/r02_drift_*.json, DESIGN.md section 6)")
    ap.add_argument("--pin", type=int, default=1, help="pin each rank's host thread to the CPUs local to its GPU (NVML affinity)")
    ap.add_argument("--gpu-eager", type=int, default=1, help="also time the reference algorithm as PyTorch eager on the GPU (0 to skip)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write the depth maps of the last timed step of every clip to DIR/depth.npy (float32; "
                         "a seeded sample of whole clips above 64 MB); --impl reference writes its one clip the same way")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(3, args.warmup)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        if rank == 0:
            print(json.dumps(run_reference(args)))
        return 0

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py: no CUDA device -- the product path has no CPU fallback (use --impl reference for the CPU arm)")
    if world > 1:
        import torch.distributed as dist
        # stdout carries exactly one JSON line (rank 0): NCCL prints its "NCCL version ..." banner with a bare printf when the
        # first communicator is created, so file descriptor 1 points at stderr while that happens
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local_rank))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
    result = run_ours(args, rank, world, local_rank)
    if rank == 0:
        if args.gpu_eager and world == 1:
            result["gpu_eager_baseline"] = gpu_eager_baseline(6, args.weights)
        if args.cpu_frames > 0 and world == 1:          # the CPU baseline is an N = 1 entry (the other ranks would idle through it)
            os.environ.pop("OMP_NUM_THREADS", None)
            try:
                os.sched_setaffinity(0, range(os.cpu_count() or 1))      # the GPU arm pinned this process to one NUMA node
            except Exception:  # noqa: BLE001
                pass
            torch.set_num_threads(max(1, os.cpu_count() or 1))
            result["cpu_baseline"], _ = cpu_baseline(args.cpu_frames, args.weights)
        print(json.dumps(result))
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
