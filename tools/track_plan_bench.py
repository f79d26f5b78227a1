#!/usr/bin/env python3
"""Cost of the per-pair motion priors and the tracker's wide-radius retry (sfe_stereo_sequence_plan_dev) on bench.py's
workload: 128 resident KITTI-sized stereo frames per step (16-frame sequences sliding 4 px per frame over one scene each),
batches rotated over more images than L2 holds, asynchronous calls queued back to back.  Cases, alternated round by round:
  (a) sfe_stereo_sequence_dev, identity prior, radius 50 (bench.py's step);
  (b) the plan call with a prior per pair (the 4-px slide inside a scene, identity across a cut between scenes) and the
      tracker's retry (100 px below 8 matches: the cuts are matched again);
  (c) the same priors with retry_below = INT32_MAX: every pair is matched twice (the worst case).
Each round times `steps` calls per case with CUDA events on the extractor's stream; the median over rounds is reported, with
the kernel launches per step.  Prints the card's name and power limit; ends with one JSON line."""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench import H, SEQ_LEN, SEQ_STEP, W, make_frames, track_params  # noqa: E402
from bow_bench import card  # noqa: E402
from slam_toolkit_b200 import api, synth  # noqa: E402

F = 128


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20, help="calls per case per round")
    ap.add_argument("--rounds", type=int, default=10)
    args = ap.parse_args()
    if api.device_count() < 1:
        sys.exit("no CUDA device")
    print("card:", card())
    ex = api.ORBextractor(2000, 1.2, 8, 20, 7, device=0, max_images=2 * F)
    cap = ex.cap
    L, R = make_frames(F)
    pitch = api.image_pitch(W)

    def pitched(a):
        out = np.zeros((a.shape[0], H, pitch), np.uint8)
        out[:, :, :W] = a
        return out
    nb = max(2, int(np.ceil(2.2 * 126e6 / (2 * F * pitch * H))))
    # rotated by whole sequences, so the cuts between scenes stay at multiples of SEQ_LEN
    imgs = [(api.DeviceBuffer(F * pitch * H).upload(pitched(np.roll(L, b * SEQ_LEN, axis=0))),
             api.DeviceBuffer(F * pitch * H).upload(pitched(np.roll(R, b * SEQ_LEN, axis=0)))) for b in range(nb)]
    spec = {"kps_l": 28, "desc_l": 32, "n_l": 0, "kps_r": 28, "desc_r": 32, "n_r": 0, "stereo_idx": 4, "stereo_dist": 4,
            "track_idx": 4, "track_dist": 4}
    bufs = {k: api.DeviceBuffer(b * cap * F if b else 4 * F) for k, b in spec.items()}
    ptrs = {k: b.ptr for k, b in bufs.items()}
    tp = track_params()
    priors = np.stack([np.eye(4)] * F)
    for f in range(F):
        if f % SEQ_LEN:
            priors[f, 0, 3] = -SEQ_STEP * synth.KITTI_BASELINE / synth.DISPARITY
    cases = {"a_sequence_dev": {}, "b_plan_retry8": {"priors": priors, "retry_radius": 100.0, "retry_below": 8},
             "c_plan_retry_all": {"priors": priors, "retry_radius": 100.0, "retry_below": 2 ** 31 - 1}}

    def step(i, plan):
        ex.stereo_sequence_dev(imgs[i % nb][0].ptr, imgs[i % nb][1].ptr, F, W, H, ptrs, tp, pitch=pitch, **plan)

    tracked, launches = {}, {}
    ex.set_async(True)
    for name, plan in cases.items():  # warm-up: every buffer of every case allocated before the first timed call
        for i in range(3):
            step(i, plan)
        ex.wait()
        tracked[name] = int((bufs["track_idx"].download((F, cap), np.int32) >= 0).sum())
    times = {name: [] for name in cases}
    e0, e1 = api.Event(0), api.Event(0)
    for r in range(args.rounds):
        for name, plan in cases.items():
            l0 = ex.launches()
            e0.record(ex)
            for i in range(args.steps):
                step(r * args.steps + i, plan)
            e1.record(ex)
            ex.wait()
            times[name].append(e0.elapsed_ms(e1) / args.steps)
            launches[name] = (ex.launches() - l0) / args.steps
    ex.set_async(False)
    res = {"card": card(), "frames_per_step": F, "steps_per_round": args.steps, "rounds": args.rounds}
    for name in cases:
        ms = float(np.median(times[name]))
        res[name] = {"ms_per_step": round(ms, 4), "spread_ms": [round(min(times[name]), 4), round(max(times[name]), 4)],
                     "frames_per_s": round(F / ms * 1e3, 1), "launches_per_step": launches[name], "tracked": tracked[name]}
        print(f"{name:18s} {ms:.4f} ms/step (rounds {min(times[name]):.4f}..{max(times[name]):.4f})  "
              f"{F / ms * 1e3:9.1f} frames/s  {launches[name]:.0f} launches/step  {tracked[name]} tracked keypoints")
    for name in ("b_plan_retry8", "c_plan_retry_all"):
        res[name]["extra_ms_vs_a"] = round(res[name]["ms_per_step"] - res["a_sequence_dev"]["ms_per_step"], 4)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
