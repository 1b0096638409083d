"""Per-frame timing in the OMD configuration (example/omd.yaml): python profiles/time_omd.py [--frames N] [--reps R] [--out FILE]

A synthetic OMD-shaped sequence (640x480, DepthMapFactor 1000, ORBextractor.nFeatures 3000, SFMgThres 0.02, SFDsThres 0.99,
WINDOW 20 / OVERLAP 4, ChooseData 1) runs through vdo_tracker_track with UseSampleFeature 1 (sampled background keypoints, time-seeded
like the reference) and UseSampleFeature 0 (ORB keypoints) on the same frames.  The two settings alternate over R repetitions, a fresh
tracker each, so that drift of the shared machine hits both alike; one untimed run of each setting comes first (module loading and
first-touch allocations otherwise land in whichever repetition runs first).  Reported per setting: end-to-end frames/s of every repetition (host
buffers -> pose, write-back included, the first 3 frames excluded) and the per-stage host wall-clock per frame of the last repetition,
with the card's name and power limit read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from vdo_slam_b200 import capi  # noqa: E402
from vdo_slam_b200.synth import make_sequence_frame  # noqa: E402

OMD_K = np.array([618.3587036132812, 618.5924072265625, 328.9866333007812, 237.7507629394531], np.float32)
STAGES = ["upload+depth_prep", "update_mask", "frame_build(orb+static keys+object samples)", "lookups", "init_model_cam", "flow_lm_cam",
          "objects(sceneflow+classify+init+lm)", "renew_frame_info", "windowed_ba(amortised)"]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, timeout=30)
        name, power, clk = [s.strip() for s in q.stdout.strip().split(",")]
        return {"name": name, "power_limit": power, "sm_clock_max": clk}
    except Exception as e:                      # the run still needs a device: capi.Context raises without one
        return {"name": None, "error": f"nvidia-smi: {e}"}


def run(ctx, frames, use_sample, warm=3):
    tr = capi.Tracker(ctx, width=640, height=480, fx=float(OMD_K[0]), fy=float(OMD_K[1]), cx=float(OMD_K[2]), cy=float(OMD_K[3]), depth_factor=1000.0,
                      sf_mg_thres=0.02, sf_ds_thres=0.99, n_features=3000, is_kitti=0, dataset=1, window_size=20, overlap_size=4,
                      use_sample_feature=int(use_sample), sample_seed=0)
    dt, st0, n_stat = [], None, []
    for t, f in enumerate(frames):
        d, m = f["depth_raw"].copy(), f["mask"].copy()
        if t == warm:
            st0 = tr.get("stage_ms").copy()
        t0 = time.perf_counter()
        tr.track(f["gray"], d, f["flow"], m, f["obj_ids"], writeback=True)
        dt.append(time.perf_counter() - t0)
        n_stat.append(len(tr.get("mvStatKeysTmp")) // 2)
    n = len(frames) - warm
    stage = (tr.get("stage_ms") - st0) / n
    out = {"frames_per_s_e2e": n / sum(dt[warm:]), "stage_ms_per_frame": dict(zip(STAGES, [round(float(x), 4) for x in stage])),
           "static_keys_per_frame_mean": float(np.mean(n_stat)), "windowed_ba": dict(zip(["runs", "lm_iterations"], tr.get("local_ba").tolist()))}
    tr.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=60)
    ap.add_argument("--reps", type=int, default=4)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    ctx = capi.Context(0)
    info = card()
    frames = [make_sequence_frame(t, seed=0, width=640, height=480, K=OMD_K, depth_factor=1000) for t in range(a.frames)]
    for mode in (1, 0):
        run(ctx, frames[:24], mode)
    res = {1: [], 0: []}
    for r in range(a.reps):
        for mode in ((1, 0) if r % 2 == 0 else (0, 1)):
            res[mode].append(run(ctx, frames, mode))
    out = {"workload": f"synthetic OMD-shaped RGB-D sequence 640x480, {a.frames} frames (3 warm-up), 3 moving objects, example/omd.yaml values "
                       "(nFeatures 3000, SFMgThres 0.02, SFDsThres 0.99, DepthMapFactor 1000, WINDOW 20 / OVERLAP 4)",
           "card": info, "reps": a.reps, "order": "one untimed run of each setting, then alternating, a fresh tracker per repetition"}
    for mode, key in ((1, "use_sample_feature_1"), (0, "use_sample_feature_0")):
        fps = [x["frames_per_s_e2e"] for x in res[mode]]
        out[key] = {"frames_per_s_e2e": [round(v, 2) for v in fps], "frames_per_s_e2e_median": round(float(np.median(fps)), 2),
                    "stage_ms_per_frame_last_rep": res[mode][-1]["stage_ms_per_frame"], "static_keys_per_frame_mean": res[mode][-1]["static_keys_per_frame_mean"],
                    "windowed_ba": res[mode][-1]["windowed_ba"]}
    s = json.dumps(out, indent=1)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
