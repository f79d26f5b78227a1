#!/usr/bin/env python3
"""bench.py -- ORB extract+match throughput on synthetic KITTI-shaped stereo frames.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--frames F] [--impl ours|reference]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

One step = one batch of F consecutive stereo frames (1241x376, 8 levels, scale 1.2, 2000 features) through
the hot path, BASELINE.json configs[1] as SURVEY.md §8d defines it: extract(left) + extract(right) + StereoMatch
(the keyframe path of the reference pipeline, src/pipeline.cpp:243-249) + the tracker's ProjectionMatch of the
previous frame's stereo-triangulated keypoints into the frame (StereoFrame::GetDepth, identity motion prior, r = 50).
  value : whole-job stereo frames/s with inputs resident in HBM (sfe_stereo_sequence_dev), timed
          with CUDA events on the extractor's own stream, max over ranks.
  e2e   : the same metric through the host entry point (sfe_stereo_sequence): pinned host images in,
          host keypoints/descriptors/stereo indices/track indices out, copies inside the timed region.
  roofline     : the dominant kernel's algorithmic bytes / its CUDA-event time, vs the measured HBM peak.
  cpu_baseline : the CPU oracle (port of the reference) on a bounded sample, host cores stated.
--impl reference times the reference's own CPU code alone (oracle/_ref: src/orb_extractor.cpp, matcher.cpp, camera.cpp
compiled unmodified against stand-in third-party headers; the C port when that prebuilt library is absent), all host
threads, same metric/config.
Frames are sharded across GPUs with no data-path collective (weak scaling: F frames per GPU).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W, H = 1241, 376
SEQ_LEN, SEQ_STEP = 16, 4  # a batch is made of 16-frame sequences: the camera slides 4 px per frame over one synthetic scene
PYR_PIXELS = 1_444_097   # sum of level sizes (SURVEY.md §8)
B_IMG = 466_616 + PYR_PIXELS + 2000 * 60          # algorithmic bytes per image extraction
B_FRAME = 2 * B_IMG + 4 * 2000                     # per stereo frame
WORKLOAD = ("kitti_stereo_frontend: extract L + extract R + StereoMatch + ProjectionMatch(previous frame's stereo points, r=50), "
            "1241x376, 8 levels, 1.2, 2000 feats")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--frames", type=int, default=128, help="stereo frames per step per GPU")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-frames", type=int, default=0, help="stereo frames in the CPU sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--e2e-threads", type=int, default=2, help="host threads (one handle each) issuing the e2e calls")
    ap.add_argument("--knn-rows", type=int, default=10_000_000, help="rows of the descriptor map of the Hamming leg (0 = skip)")
    ap.add_argument("--proj-points", type=int, default=500_000, help="map points of the ProjectionMatch leg (0 = skip)")
    ap.add_argument("--clock-period", type=float, default=0.05, help="seconds between NVML clock samples (0 = no sampling)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    return args


def make_frames(n):
    """n consecutive stereo frames: 16-frame sequences over scenes 0, 1, 2, ... (synth.stereo_sequence)."""
    from slam_toolkit_b200 import synth
    Ls, Rs = [], []
    for s in range((n + SEQ_LEN - 1) // SEQ_LEN):
        l, r = synth.stereo_sequence(s, min(SEQ_LEN, n - s * SEQ_LEN), SEQ_STEP)
        Ls.append(l)
        Rs.append(r)
    return np.concatenate(Ls), np.concatenate(Rs)


def dump_outputs(path, d_out, F, cap, n_frames=32):
    """What the caller of sfe_stereo_sequence_dev receives from one step, for a fixed sample of its frames
    (default_rng(0); 32 of 128 frames are about 27 MB): keypoint fields, descriptor bytes, keypoint counts, stereo and
    tracking indices and distances, one DIR/<name>.npy each, float32 (every value is exact in it).  Slots past a frame's
    keypoint count hold no result and are written as 0."""
    from slam_toolkit_b200 import api
    frames = np.sort(np.random.default_rng(0).choice(F, min(F, n_frames), replace=False))
    n = {s: d_out[f"n_{s}"].download((F,), np.int32)[frames] for s in "lr"}
    valid = {s: np.arange(cap)[None, :] < n[s][:, None] for s in "lr"}
    arrays = {"frames": frames, "n_l": n["l"], "n_r": n["r"]}
    for s in "lr":
        kps = d_out[f"kps_{s}"].download((F, cap), api.KP_DTYPE)[frames]
        for field in api.KP_DTYPE.names:
            arrays[f"kps_{s}_{field}"] = np.where(valid[s], kps[field], 0)
        arrays[f"desc_{s}"] = np.where(valid[s][..., None], d_out[f"desc_{s}"].download((F, cap, 32), np.uint8)[frames], 0)
    for k in ("stereo_idx", "stereo_dist", "track_idx", "track_dist"):     # per left keypoint
        arrays[k] = np.where(valid["l"], d_out[k].download((F, cap), np.int32)[frames], 0)
    arrays = {k: a.astype(np.float32) for k, a in arrays.items()}
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, f"{k}.npy"), a)


def track_params():
    from slam_toolkit_b200 import api, synth
    cam = api.Camera.make(synth.KITTI_FX, synth.KITTI_FY, synth.KITTI_CX, synth.KITTI_CY, (0, 0, 0, 0), W, H)
    return api.TrackParams.make(cam, synth.KITTI_BASELINE, None, 50.0)


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons sampled DURING the timed regions (B200_PROFILING.md): NVML every 50 ms,
    `nvidia-smi --query-gpu` every 200 ms when the NVML binding is unavailable.  Rank 0 alone samples, for every GPU of
    the job: NVML queries from several processes at once serialise against the other ranks' CUDA calls in the driver
    (measured: 8 ranks polling at 50 Hz cut the end-to-end figure fivefold)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, devices, period=0.05):
        super().__init__(daemon=True)
        self.devices, self.sm, self.reasons, self.sm_max, self.stop_flag, self.source = list(devices), [], set(), None, False, None
        self.period, self.active = period, False   # samples are kept only while a timed region is running
        self.once = threading.Event()              # one extra sample on request (before / after the end-to-end region)
        self.once_done = threading.Event()

    def _nvml_loop(self):
        import pynvml as N
        N.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        handles = []
        for d in self.devices:
            idx = d
            if vis:
                try:
                    idx = int(vis.split(",")[d])
                except (ValueError, IndexError):
                    pass
            handles.append(N.nvmlDeviceGetHandleByIndex(idx))
        self.sm_max = float(N.nvmlDeviceGetMaxClockInfo(handles[0], N.NVML_CLOCK_SM))
        bits = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
        get_reasons = getattr(N, "nvmlDeviceGetCurrentClocksEventReasons", None) or N.nvmlDeviceGetCurrentClocksThrottleReasons
        self.source = "nvml"
        last = 0.0
        while not self.stop_flag:
            due = self.active and time.perf_counter() - last >= self.period
            if (due or self.once.is_set()) and self.period > 0:
                last = time.perf_counter()
                for h in handles:
                    self.sm.append(float(N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM)))
                    r = int(get_reasons(h))
                    for name, bit in bits.items():
                        if r & bit:
                            self.reasons.add(name)
                if self.once.is_set():
                    self.once.clear()
                    self.once_done.set()
            time.sleep(0.005)

    def _smi_loop(self):
        self.source = "nvidia-smi"
        while not self.stop_flag:
            if not self.active or self.period <= 0:
                time.sleep(0.01)
                continue
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.devices[0])],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                r = [c.strip() for c in out.split(",")]
                if len(r) >= 9:
                    self.sm.append(float(r[1]))
                    self.sm_max = float(r[2])
                    for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                        if v.lower().startswith("active"):
                            self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.2)

    def sample_once(self):
        """One sample now (blocking); used around regions where periodic NVML polling would perturb the measurement."""
        if not self.devices or self.period <= 0 or self.source != "nvml":
            return
        self.once_done.clear()
        self.once.set()
        self.once_done.wait(timeout=2)

    def run(self):
        if not self.devices:
            return
        try:
            self._nvml_loop()
        except Exception:
            self._smi_loop()

    def summary(self):
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.sm_max, "reasons": ["no clock samples"], "samples": 0}
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2], "sm_min_mhz": sm[0], "sm_max_mhz": self.sm_max, "reasons": sorted(self.reasons),
                "samples": len(sm), "source": self.source}


def cpu_impl():
    """("reference", module) when oracle/_ref/libslamref.so -- the reference's own src/orb_extractor.cpp + src/matcher.cpp +
    src/camera.cpp compiled unmodified, prebuilt in the authoring container -- is present, else ("port", the C oracle)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_c
    oracle_c.build()
    try:
        import ref_c
        if ref_c.available():
            ref_c.lib()
            return "reference", ref_c, oracle_c
    except Exception:
        pass
    return "port", oracle_c, oracle_c


def cpu_sample(frames, threads, impl=None):
    kind, mod, oracle_c = impl or cpu_impl()
    from slam_toolkit_b200 import synth
    L, R = make_frames(frames)
    cam = oracle_c.make_camera(synth.KITTI_FX, synth.KITTI_FY, synth.KITTI_CX, synth.KITTI_CY, [0, 0, 0, 0], W, H)
    t0 = time.perf_counter()
    matches, kps, tracked = mod.stereo_sequence(L, R, threads, cam, synth.KITTI_BASELINE, 50.0)
    dt = time.perf_counter() - t0
    return frames / dt, dt, matches + tracked, kps


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path (oracle/_ref: its sources compiled unmodified
    against stand-in third-party headers; the C oracle port when that library is absent), all host threads, one frame per
    thread, rank 0 only.  One step = a bounded sample of the workload: its size is chosen from a warm-up measurement so that
    the K steps take about a minute."""
    if rank != 0:
        return
    impl = cpu_impl()
    cores = os.cpu_count() or 1
    est_fps, _, _, _ = cpu_sample(max(cores, 4), cores, impl)          # also the warm-up (pages in the library)
    for _ in range(max(min(args.warmup, 2) - 1, 0)):
        est_fps, _, _, _ = cpu_sample(max(cores, 4), cores, impl)
    frames = args.cpu_frames or int(min(max(60.0 * est_fps / max(args.steps, 1), cores), 4 * cores))
    times = []
    tot_matches = 0
    for _ in range(args.steps):
        fps, dt, matches, _ = cpu_sample(frames, cores, impl)
        times.append(dt)
        tot_matches += matches
    total = sum(times)
    value = frames * args.steps / total
    what = ("the reference's own orb_extractor.cpp / matcher.cpp / camera.cpp (oracle/_ref, -O1)" if impl[0] == "reference"
            else "C port of the reference path (oracle/orb_oracle.c)")
    line = {"impl": "reference", "metric": "orb_extract_match_stereo_frames_per_s", "value": value, "unit": "frames/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": WORKLOAD, "frames_per_step_per_gpu": args.frames, "cpu_sample_frames_per_step": frames},
            "cpu_baseline": {"value": value, "unit": "frames/s", "cores": cores, "kind": impl[0],
                             "sample": f"{frames} synthetic stereo frames per step, {args.steps} steps, one frame per thread; {what}"},
            "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "matches_per_s": tot_matches / total, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def latency_leg(api, dev, left, right, calls=400):
    """The reference-shaped call: ONE stereo pair per call, host buffers in and out, synchronous (what Frame::Frame +
    ExtractRightKeypoints + StereoMatch cost a caller that does not batch; src/frame.cpp:47,388, src/pipeline.cpp:248).
    Median and mean wall time per call of sfe_stereo_frames(1 pair) with pinned and with pageable buffers, rank 0 only."""
    out = {}
    ex = api.ORBextractor(2000, 1.2, 8, 20, 7, device=dev, max_images=2)
    for kind in ("pinned", "pageable"):
        if kind == "pinned":
            pl, pr = api.PinnedArray(left.shape, np.uint8), api.PinnedArray(right.shape, np.uint8)
            pl.array[:], pr.array[:] = left, right
            a, b = pl.array[None], pr.array[None]
        else:
            a, b = left[None].copy(), right[None].copy()
        res = ex.alloc_stereo_out(1, pinned=kind == "pinned")
        for _ in range(20):
            ex.stereo_frames(a, b, res)
        ts = np.empty(calls)
        for i in range(calls):
            t0 = time.perf_counter()
            ex.stereo_frames(a, b, res)
            ts[i] = time.perf_counter() - t0
        out[f"stereo_pair_{kind}_median"] = float(np.median(ts) * 1e6)
        out[f"stereo_pair_{kind}_mean"] = float(ts.mean() * 1e6)
    out["what"] = ("sfe_stereo_frames(1 pair): upload 2 x 1241x376, extract L + R, StereoMatch, download, synchronous; CUDA graph of "
                   "programmatically serialized kernels, results stored into pinned arrays by one kernel")
    return out


def _max_over_ranks(dist, dev, values):
    if dist is None:
        return list(values)
    import torch
    t = torch.tensor(list(values), dtype=torch.float64, device=f"cuda:{dev}")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return t.tolist()


def _event_ms(api, m, dev, fn, reps, barrier):
    """reps calls of fn queued back to back on the matcher's stream, timed with CUDA events on that stream"""
    fn()
    m.wait()
    e0, e1 = api.Event(dev), api.Event(dev)
    barrier()
    e0.record(m)
    for _ in range(reps):
        fn()
    e1.record(m)
    m.wait()
    return e0.elapsed_ms(e1) / reps


def hamming_leg(args, dev, rank, world, dist):
    """BASELINE config 4 beside the headline, as SURVEY §8d states it: brute-force Hamming top-2 of Q queries against the
    10 M-row map `default_rng(1234)`, queries = map rows picked by `default_rng(5678)` with bit flips (a fifth of them
    hard enough to fail the ratio test).  Rows are sharded over the ranks; the exchange is the library's own step
    (sfe_knn2_sharded: every rank's merge kernel stores its top-2 keys into every peer's inbox over NVLink peer memory,
    the final merge waits on flags) -- resident queries, no host round trip, timed with CUDA events on the matcher's stream,
    max over ranks.  Q = 2000 is `popc`-bound (SURVEY §8d); Q in {1, 2, 4} stream the map once: those are the
    GB/s-vs-HBM figures.  At world > 1 rank 0 also runs the UNSHARDED query on its own GPU and compares every value."""
    from slam_toolkit_b200 import api, sharding, synth
    rows = args.knn_rows
    a, b = sharding.block(rows, world, rank)
    db = synth.knn_database(rows, seed=1234)                       # the same on every rank; each keeps its block resident
    queries, _ = synth.knn_queries(db, 2000, seed=5678, hard_fraction=0.2)
    m = api.Matcher(dev)
    sd = sharding.ShardedDatabase(m, db[a:b], rows)
    d_q = api.DeviceBuffer(queries.nbytes, dev).upload(queries)
    d_o = api.DeviceBuffer(2000 * 16, dev)

    def barrier():
        if dist is not None:
            dist.barrier()
    out_ms = {}
    for nq, reps in ((2000, 5), (1, 50), (2, 50), (4, 50)):
        out_ms[nq] = _event_ms(api, m, dev, lambda: sd.knn2_dev(d_q.ptr, nq, d_o.ptr), reps, barrier)
    sd.knn2_dev(d_q.ptr, 2000, d_o.ptr)
    m.wait()
    out = d_o.download((2000, 4), np.int32)
    sd.comm.status()
    equal = None
    if world > 1 and rank == 0:                                   # the unsharded map fits one GPU (320 MB)
        whole = m.create_db(db)
        equal = bool(np.array_equal(m.knn2(whole, queries), out))
        del whole
    ms = _max_over_ranks(dist, dev, [out_ms[2000], out_ms[1], out_ms[2], out_ms[4]])
    res = {"map_rows": rows, "map": "default_rng(1234), queries default_rng(5678) rows + flips (SURVEY §8d config 4)",
           "sharding": f"{world} row shard(s); exchange = peer-memory stores + flags inside the merge kernels (sfe_knn2_sharded)",
           "q2000_ms_per_batch": ms[0], "q2000_pair_distances_per_s": 2000 * rows / (ms[0] / 1e3),
           "q2000_algorithmic_gbs": (32 * rows + 48 * 2000) / (ms[0] / 1e3) / 1e9,
           "accepted_ratio_test": float((2 * out[:, 1] < out[:, 3]).mean())}
    for i, nq in ((1, 1), (2, 2), (3, 4)):
        res[f"q{nq}_stream_ms"] = ms[i]
        res[f"q{nq}_stream_gbs"] = (32 * rows + 48 * nq) / (ms[i] / 1e3) / 1e9
    if world > 1:
        res["sharded_equals_unsharded"] = equal
    return res


def projection_leg(args, dev, rank, world, dist, kps, desc):
    """BASELINE config 5 beside the headline: ProjectionMatch (r = 50 px, identity pose as an SE3Quat) of a local map of N
    points against one resident frame; map points sharded over the ranks, exchange inside the library
    (sfe_projection_match_sharded).  Timed with CUDA events on the matcher's stream, max over ranks.
    Algorithmic bytes per call (SURVEY §8d): N * (24 + 32) + M * (8 + 32) + 8 * M."""
    from slam_toolkit_b200 import api, sharding, synth
    n, m_kps = args.proj_points, len(kps)
    xy = np.stack([kps["x"], kps["y"]], axis=1).astype(np.float64)
    xw, mpd = synth.projection_scene(xy, desc, n, seed=99)
    a, b = sharding.block(n, world, rank)
    cam = api.Camera.make(synth.KITTI_FX, synth.KITTI_FY, synth.KITTI_CX, synth.KITTI_CY, (0, 0, 0, 0), W, H)
    m = api.Matcher(dev)
    frame = api.Frame(m, kps, desc, cam)
    lm = sharding.ShardedLocalMap(m, xw[a:b], mpd[a:b], n)
    d_q, d_d = api.DeviceBuffer(m_kps * 4, dev), api.DeviceBuffer(m_kps * 4, dev)
    Tcw = np.array([0, 0, 0, 1, 0, 0, 0], np.float64)

    def barrier():
        if dist is not None:
            dist.barrier()
    ms = _event_ms(api, m, dev, lambda: lm.projection_match_dev(frame, Tcw, 50.0, d_q.ptr, d_d.ptr), 20, barrier)
    lm.projection_match_dev(frame, Tcw, 50.0, d_q.ptr, d_d.ptr)
    m.wait()
    got_q, got_d = d_q.download((m_kps,), np.int32), d_d.download((m_kps,), np.int32)
    lm.comm.status()
    equal, single_ms = None, None
    if world > 1 and rank == 0:
        want_q, want_d = frame.ProjectionMatch(xw, mpd, None, Tcw, 50.0)
        equal = bool(np.array_equal(want_q, got_q) and np.array_equal(want_d, got_d))
    ms, = _max_over_ranks(dist, dev, [ms])
    alg = n * 56 + m_kps * 48
    res = {"map_points": n, "frame_keypoints": m_kps, "radius_px": 50.0, "ms_per_call": ms,
           "map_points_per_s": n / (ms / 1e3), "algorithmic_gbs": alg / (ms / 1e3) / 1e9,
           "keypoints_matched": int((got_q >= 0).sum()),
           "sharding": f"{world} map-point shard(s); exchange = peer-memory stores + flags (sfe_projection_match_sharded)"}
    if world > 1:
        res["sharded_equals_unsharded"] = equal
    return res


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from slam_toolkit_b200 import api
    F, K, Wm = args.frames, args.steps, max(args.warmup, 3)
    dev = local
    ex = api.ORBextractor(2000, 1.2, 8, 20, 7, device=dev, max_images=2 * F)
    cap = ex.cap
    # ---- inputs: NB rotated batches resident in HBM (NB*F*2*466 KB > L2 so no step re-reads a cached batch)
    L, R = make_frames(F)
    PITCH = api.image_pitch(W)           # resident images are pitched (cudaMallocPitch style): TMA needs 16-B multiples
    per_batch = 2 * F * PITCH * H

    def pitched(a):
        out = np.zeros((a.shape[0], H, PITCH), np.uint8)
        out[:, :, :W] = a
        return out
    NB = max(2, int(np.ceil(2.2 * 126e6 / per_batch)))
    d_left, d_right = [], []
    for b in range(NB):
        sh = (b * SEQ_LEN) % F       # rotated by whole sequences: consecutive frames stay consecutive
        d_left.append(api.DeviceBuffer(F * PITCH * H, dev).upload(pitched(np.roll(L, sh, axis=0))))
        d_right.append(api.DeviceBuffer(F * PITCH * H, dev).upload(pitched(np.roll(R, sh, axis=0))))
    spec = {"kps_l": 28 * cap * F, "desc_l": 32 * cap * F, "n_l": 4 * F, "kps_r": 28 * cap * F, "desc_r": 32 * cap * F,
            "n_r": 4 * F, "stereo_idx": 4 * cap * F, "stereo_dist": 4 * cap * F, "track_idx": 4 * cap * F,
            "track_dist": 4 * cap * F}
    tp = track_params()
    d_out = {k: api.DeviceBuffer(v, dev) for k, v in spec.items()}
    ptrs = {k: b.ptr for k, b in d_out.items()}

    def barrier():
        if dist is not None:
            dist.barrier()

    def step_resident(i):
        ex.stereo_sequence_dev(d_left[i % NB].ptr, d_right[i % NB].ptr, F, W, H, ptrs, tp, pitch=PITCH)

    sampler = ClockSampler(range(world) if rank == 0 else [], args.clock_period if rank == 0 else 0)
    sampler.start()                      # NVML initialises here, outside the timed regions
    for i in range(Wm):
        step_resident(i)
    # per-stage CUDA-event times: a few synchronous profiled steps outside the timed region
    ex.set_profiling(True)
    for i in range(min(K, 10)):
        step_resident(i)
    stage_ms, calls = ex.stage_ms()
    ex.set_profiling(False)
    # timed region: K batches queued back to back on the extractor's stream (asynchronous _dev calls), one wait
    ex.set_async(True)
    for i in range(2):
        step_resident(i)
    ex.wait()
    l0 = ex.launches()
    ev0, ev1 = api.Event(dev), api.Event(dev)
    barrier()
    sampler.active = True
    ev0.record(ex)
    for i in range(K):
        step_resident(Wm + i)
    ev1.record(ex)
    ex.wait()
    sampler.active = False
    ms = ev0.elapsed_ms(ev1)
    if args.dump_outputs and rank == 0:     # before the extract-only leg below reuses the output buffers
        dump_outputs(args.dump_outputs, d_out, F, cap)
    barrier()
    launches = ex.launches() - l0
    # BASELINE config 3 beside the headline: extraction only (sfe_extract_batch_dev) of the same resident images, 2F
    # independent frames per step (two calls of F), sharded over the ranks like the headline
    def step_extract(i):
        for d in (d_left[i % NB], d_right[i % NB]):
            api._check(api.lib().sfe_extract_batch_dev(ex.h, api._p(d.ptr), PITCH * H, F, W, H, PITCH, api._p(ptrs["kps_l"]),
                                                       api._p(ptrs["desc_l"]), cap, api._p(ptrs["n_l"])))
    KX = max(K // 4, 5)
    for i in range(3):
        step_extract(i)
    ex.wait()
    ev2, ev3 = api.Event(dev), api.Event(dev)
    barrier()
    ev2.record(ex)
    for i in range(KX):
        step_extract(3 + i)
    ev3.record(ex)
    ex.wait()
    ms_x = ev2.elapsed_ms(ev3) / KX
    barrier()
    ex.set_async(False)
    n_stereo = int((d_out["stereo_idx"].download((F, cap), np.int32) >= 0).sum())
    n_track = int((d_out["track_idx"].download((F, cap), np.int32) >= 0).sum())
    n_match = n_stereo + n_track
    n_kps = int(d_out["n_l"].download((F,), np.int32).sum() + d_out["n_r"].download((F,), np.int32).sum())

    # ---- e2e: pinned host images -> host results through the public host entry point (sfe_stereo_sequence), synchronous
    # calls.  T host threads, one extractor handle each (handles are per-thread objects, include/sfe.h), issue calls back to
    # back, so one call's pipeline fill / drain overlaps the other's steady state; T = 1 is reported beside it.  The
    # threads are started and parked on a barrier BEFORE the clock; the region runs a call count sized for >= 2.5 s.
    T = max(1, args.e2e_threads)
    wc = os.environ.get("SFE_BENCH_WC", "0") == "1"   # write-combined input pages (tools/copy_probe.py measures both)
    handles = [ex] + [api.ORBextractor(2000, 1.2, 8, 20, 7, device=dev, max_images=2 * F) for _ in range(T - 1)]
    pins = []
    for h in handles:
        pl, pr = api.PinnedArray((F, H, W), np.uint8, write_combined=wc), api.PinnedArray((F, H, W), np.uint8, write_combined=wc)
        pl.array[:], pr.array[:] = L, R
        pins.append((pl, pr, h.alloc_stereo_out(F, pinned=True, track=True)))
    out = pins[0][2]

    def timed(nthreads, calls_each):
        gate = threading.Barrier(nthreads + 1)
        done = threading.Barrier(nthreads + 1)

        def work(t):
            pl, pr, o = pins[t]
            gate.wait()
            for _ in range(calls_each):
                handles[t].stereo_sequence(pl.array, pr.array, tp, o)
            done.wait()
        ths = [threading.Thread(target=work, args=(t,)) for t in range(nthreads)]
        for th in ths:
            th.start()
        barrier()                       # every rank's threads are parked
        gate.wait()
        t0 = time.perf_counter()
        done.wait()
        dt = time.perf_counter() - t0
        for th in ths:
            th.join()
        return dt

    timed(T, max(Wm // T, 2))                                  # warm-up (the extra handles allocate their buffers here)
    est = timed(T, 4) / 4                                       # seconds per call per thread
    est, = _max_over_ranks(dist, dev, [est])
    calls_each = int(min(max(np.ceil(2.5 / max(est, 1e-4)), 4), 2000))
    # (periodic NVML polling during this region stalls the CUDA calls of the OTHER ranks inside the driver -- measured
    # 73 k -> 26 k frames/s at 2 GPUs -- so the clocks are sampled immediately before and after it instead)
    sampler.sample_once()
    e2e_s = timed(T, calls_each)
    sampler.sample_once()
    e2e_calls = T * calls_each
    calls_single = max(calls_each * T // 2, 4)
    e2e_single_s = timed(1, calls_single) if T > 1 else e2e_s
    if T == 1:
        calls_single = e2e_calls
    barrier()
    # copy-only ceiling of the same path: the bytes of one step, both directions at once, every rank at the same time
    barrier()
    ceil_h2d, ceil_d2h = api.copy_probe(dev, 2 * F * W * H, sum(v.nbytes for v in out.values()), 8, 1.5, wc)
    barrier()
    sampler.stop_flag = True
    sampler.join(timeout=2)
    hamming = hamming_leg(args, dev, rank, world, dist) if args.knn_rows > 0 else None
    projection = None
    if args.proj_points > 0:
        nl0 = int(out["n_l"][0])
        projection = projection_leg(args, dev, rank, world, dist, out["kps_l"][0, :nl0].copy(), out["desc_l"][0, :nl0].copy())
    h2d = 2 * F * W * H
    d2h = sum(v.nbytes for v in out.values())

    if dist is not None:
        import torch
        t = torch.tensor([ms, e2e_s * 1e3, e2e_single_s * 1e3, ms_x], dtype=torch.float64, device=f"cuda:{local}")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_ms, e2e_single_ms, ms_x = t.tolist()
        e2e_s, e2e_single_s = e2e_ms / 1e3, e2e_single_ms / 1e3
        t = torch.tensor([ceil_h2d, ceil_d2h], dtype=torch.float64, device=f"cuda:{local}")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        ceil_h2d, ceil_d2h = t.tolist()
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    value = world * F * K / (ms / 1e3)
    e2e = world * F * e2e_calls / e2e_s
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    # dominant kernel = stage with the largest event time; algorithmic bytes per launch in DESIGN.md §5
    alg_bytes = {"pyramid": 2 * F * (466_616 + PYR_PIXELS) / 7.0,  # per launch: 7 launches per step
                 "fast_cells": 2 * F * (PYR_PIXELS + 11_800 * 4), "quadtree": 2 * F * (11_800 * 4 + 2000 * 4),
                 "blur": 2 * F * 2 * PYR_PIXELS, "orient_describe": 2 * F * (2000 * (749 + 512) + 2000 * 60),
                 "stereo_match": F * (2 * 2000 * 40 + 2000 * 8),
                 "track": F * 2000 * (2 * 60 + 28 + 4 + 8) / 3.0}
    launches_per_step = {"pyramid": 7, "fast_cells": 1, "quadtree": 1, "blur": 1, "orient_describe": 1, "stereo_match": 1, "track": 3}
    top = max(stage_ms, key=lambda k: stage_ms[k])
    top_ms = stage_ms[top] / max(calls, 1) / launches_per_step[top]
    achieved = alg_bytes[top] / (top_ms / 1e3) / 1e9 if top_ms > 0 else 0.0
    # DRAM traffic of that kernel per launch from the committed ncu --set full capture (dram__bytes_read + write, per image
    # there, scaled to this run's images per launch); well above the algorithmic bytes would mean wasted re-reads
    traffic, traffic_src, issue = None, None, None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "dram_traffic.json")))
        units = F if top in ("stereo_match", "track") else 2 * F
        traffic = tj["kernels"][top]["dram_bytes_per_image"] * units / launches_per_step[top]
        traffic_src = tj["source"]
        # the pipe that actually binds extraction: warp instructions of the kernel (ncu smsp__inst_executed.sum of the same
        # committed capture, per image) over its live CUDA-event time, against the issue peak 4 per clk per SM at the
        # sampled SM clock
        winst = tj["kernels"][top].get("warp_instructions_per_image", 0) * units / launches_per_step[top]
        clk = (sampler.summary() or {}).get("sm_mhz") or float(peaks.get("sm_max_mhz", 1965.0))
        sms = 148
        if winst > 0 and top_ms > 0:
            issue = {"warp_instructions_per_launch": winst, "achieved_gwarp_inst_per_s": winst / (top_ms / 1e3) / 1e9,
                     "peak_gwarp_inst_per_s": 4 * sms * clk * 1e6 / 1e9, "sm_clock_mhz": clk}
            issue["frac"] = issue["achieved_gwarp_inst_per_s"] / issue["peak_gwarp_inst_per_s"]
    except Exception:
        pass
    # The dominant kernel is integer-issue bound (SURVEY.md §8d: the HBM roofline is ~30x away), so the primary entry is the
    # issue roofline -- the kernel's warp instructions (ncu smsp__inst_executed of the committed capture at this launch
    # size) over its live CUDA-event time against 4 issues / clk / SM -- and the HBM figures the contract asks for sit beside it.
    hbm = {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak, "traffic": traffic,
           "traffic_source": traffic_src, "algorithmic_bytes_per_launch": alg_bytes[top], "peak_source": peak_src,
           "whole_step_achieved": value / world * B_FRAME / 1e9, "whole_step_frac": value / world * B_FRAME / 1e9 / hbm_peak}
    if issue:
        roofline = {"bound": "issue", "kernel": top, "achieved": issue["achieved_gwarp_inst_per_s"], "peak": issue["peak_gwarp_inst_per_s"],
                    "unit": "Gwarp-inst/s", "frac": issue["frac"], "traffic": traffic, "sm_clock_mhz": issue["sm_clock_mhz"],
                    "warp_instructions_per_launch": issue["warp_instructions_per_launch"], "hbm": hbm,
                    "note": "extraction is integer-issue bound, not HBM bound: peak = 4 warp instructions / clk / SM x 148 SMs at the "
                            "sampled SM clock; `hbm` holds the algorithmic-bytes roofline of the same kernel; profiles/ holds the pipes"}
    else:
        roofline = dict(hbm, kernel=top)
    line = {"metric": "orb_extract_match_stereo_frames_per_s", "value": value, "unit": "frames/s", "n_gpus": world,
            "steps": K, "warmup": Wm, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": WORKLOAD, "frames_per_step_per_gpu": F, "l2": f"inputs rotate over {NB} resident batches ({NB * per_batch / 1e6:.0f} MB > 126 MB L2)",
                       "resident_layout": f"row pitch {PITCH} B (sfe_image_pitch)",
                       "sharding": "frames partitioned across GPUs, no collective"},
            "e2e": {"value": e2e, "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "host_threads": T, "single_thread_value": world * F * calls_single / e2e_single_s,
                    "calls_timed": world * e2e_calls, "seconds_timed": e2e_s, "input_pages": "write-combined" if wc else "pinned",
                    "h2d_ceiling_gbs": ceil_h2d, "d2h_ceiling_gbs": ceil_d2h,
                    "ceiling_frames_per_s": ceil_h2d * 1e9 / (2 * W * H), "frac_of_copy_ceiling": e2e / (ceil_h2d * 1e9 / (2 * W * H)),
                    "ceiling_note": "sfe_copy_probe: the bytes of one step, H2D + D2H at once, all ranks at once, no kernels"},
            "gpu_launches": launches,
            "clocks": sampler.summary(),
            "roofline": roofline,
            "stage_ms_per_step": {k: v / max(calls, 1) for k, v in stage_ms.items()},
            "keypoints_per_frame": n_kps / F, "matches_per_s": value * n_match / F,
            "stereo_matches_per_frame": n_stereo / F, "tracked_matches_per_frame": n_track / F,
            "extract_only": {"images_per_s": world * 2 * F / (ms_x / 1e3), "ms_per_call_of_F_images": ms_x / 2,
                             "algorithmic_gbs": world * 2 * F / (ms_x / 1e3) * B_IMG / 1e9,
                             "note": "BASELINE config 3: sfe_extract_batch_dev on resident images, no matching"}}
    if hamming is not None:
        for nq in (1, 2, 4):
            hamming[f"q{nq}_stream_frac_of_hbm_peak"] = hamming[f"q{nq}_stream_gbs"] / (world * hbm_peak)
        line["hamming"] = hamming
    if projection is not None:
        projection["frac_of_hbm_peak"] = projection["algorithmic_gbs"] / hbm_peak
        line["projection_match"] = projection
    line["latency_us"] = latency_leg(api, dev, L[0], R[0])
    if not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        impl = cpu_impl()
        frames = args.cpu_frames or (24 if impl[0] == "reference" else 32) * cores   # ~2 s per core: 10-30 s of CPU work in all
        cpu_sample(cores, cores, impl)                 # warm-up
        fps_all, dt_all, _, _ = cpu_sample(frames, cores, impl)
        fps_1, dt_1, _, _ = cpu_sample(8, 1, impl)
        line["cpu_baseline"] = {"value": fps_all, "unit": "frames/s", "cores": cores, "kind": impl[0],
                                "sample": f"{frames} synthetic stereo frames, one frame per thread ({dt_all:.1f} s)",
                                "single_thread_value": fps_1,
                                "what": ("oracle/_ref: the reference's own sources compiled unmodified (-O1; its own build uses no "
                                         "optimisation) against stand-in third-party headers" if impl[0] == "reference"
                                         else "oracle/orb_oracle.c, the C restatement")}
        if impl[0] == "reference":
            port = ("port", impl[2], impl[2])
            cpu_sample(cores, cores, port)
            line["cpu_baseline"]["port_value"] = cpu_sample(frames, cores, port)[0]
    print(json.dumps(line), flush=True)
    bad = [k for k in ("hamming", "projection_match") if line.get(k) and line[k].get("sharded_equals_unsharded") is False]
    if dist is not None:
        dist.destroy_process_group()
    if bad:
        print(f"sharded result differs from the unsharded one: {bad}", file=sys.stderr)
        sys.exit(1)


def _only_the_json_line_on_stdout(fn):
    """Libraries (NCCL prints its version banner on stdout at the first communicator) must not share stdout with the one
    JSON line: fd 1 points at stderr while the bench runs and is restored for the final print."""
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    real_print = print

    def emit(*a, **k):
        if k.get("file") in (None, sys.stdout):
            sys.stdout.flush()
            os.dup2(saved, 1)
            real_print(*a, **k)
            sys.stdout.flush()
            os.dup2(2, 1)
        else:
            real_print(*a, **k)
    globals()["print"] = emit
    try:
        fn()
    finally:
        sys.stdout.flush()
        os.dup2(saved, 1)


if __name__ == "__main__":
    _only_the_json_line_on_stdout(main)
