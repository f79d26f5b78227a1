"""bench.py's reference arm runs without a GPU: check the JSON line it prints against the bench contract
(metric / unit / config of the product arm, impl = reference, cpu_baseline, e2e with zero copy bytes)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from slam_toolkit_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--cpu-frames", "4"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "orb_extract_match_stereo_frames_per_s" and line["unit"] == "frames/s"
    assert line["higher_is_better"] is True and line["steps"] == 1 and line["value"] > 0 and line["vs_baseline"] is None
    assert line["config"]["workload"].startswith("kitti_stereo_frontend") and line["config"]["cpu_sample_frames_per_step"] == 4
    assert line["config"]["frames_per_step_per_gpu"] == 128   # the product arm's batch: same config keys on both arms
    cb = line["cpu_baseline"]
    # "reference" = oracle/_ref (the reference's own sources, prebuilt here), "port" = the C oracle when that library is absent
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == line["value"] and "sample" in cb
    if os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libslamref.so")):
        assert cb["kind"] == "reference"
    assert line["e2e"] == {"value": line["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["gpu_launches"] == 0 and line["matches_per_s"] > 0


@pytest.mark.gpu
def test_dump_outputs_is_the_last_timed_step(oracle, tmp_path):
    """--dump-outputs: float32 arrays of a sampled set of frames of the last timed step, within 64 MB.  With 16 frames per
    step (one synthetic sequence, so no batch is rotated) frame f is frame f of synth.stereo_sequence(0, 16, 4)."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "1", "--frames", "16",
                          "--knn-rows", "0", "--proj-points", "0", "--no-cpu-baseline", "--e2e-threads", "1", "--clock-period", "0",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == 3
    z = {p.stem: np.load(p) for p in tmp_path.glob("*.npy")}
    assert all(a.dtype == np.float32 for a in z.values()) and sum(a.nbytes for a in z.values()) <= 64 << 20
    assert z["frames"].tolist() == list(range(16))
    L, R = synth.stereo_sequence(0, 16, 4)
    ex = oracle.Extractor()
    for f in (0, 9):
        kd = {}
        for s, img in (("l", L[f]), ("r", R[f])):
            k, d = kd[s] = ex.extract(img)
            n = int(z[f"n_{s}"][f])
            assert n == len(k)
            for field in k.dtype.names:
                assert np.array_equal(z[f"kps_{s}_{field}"][f, :n], k[field].astype(np.float32)), (f, s, field)
            assert np.array_equal(z[f"desc_{s}"][f, :n], d) and not z[f"desc_{s}"][f, n:].any()
        si, sd = oracle.stereo_match(*kd["l"], *kd["r"])
        assert np.array_equal(z["stereo_idx"][f, :len(si)], si) and np.array_equal(z["stereo_dist"][f, :len(si)], sd)
    nl = z["n_l"].astype(int)
    for f in range(16):
        idx, dist = z["stereo_idx"][f, :nl[f]].astype(int), z["stereo_dist"][f, :nl[f]]
        ok = idx >= 0
        assert ok.sum() > 500
        dl, dr = z["desc_l"][f, :nl[f]][ok].astype(np.uint8), z["desc_r"][f][idx[ok]].astype(np.uint8)
        assert np.array_equal(np.unpackbits(dl ^ dr, axis=1).sum(1), dist[ok])


def test_reference_arm_is_silent_on_other_ranks():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""
