"""Sampled background features (UseSampleFeature: 1, the setting of example/omd.yaml): the cv::RNG restatement of the oracle against cv2,
vdo_frame_sample_static against Frame::SampleKeyPoints + the Option II filter, and the whole path in the OMD configuration against the oracle
pipeline, through the C ABI and through the host shim."""
import os
import subprocess

import numpy as np
import pytest

from oracle import sampled_features as sf

OMD_K = np.array([618.3587036132812, 618.5924072265625, 328.9866333007812, 237.7507629394531], np.float32)   # example/omd.yaml
SEEDS = [1, 12345, 1760659200, 0xFFFFFFFF, 0x9E3779B9]


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("seed", [1, 12345, 1760659200])
def test_oracle_rng_matches_cv2(seed):
    import cv2
    cv2.setRNGSeed(seed)                          # cv2 takes a C int: seeds below 2^31 only
    r = sf.CvRNG(seed)
    bounds = np.random.default_rng(seed).integers(0, 700, (5000, 2))
    m = np.zeros((1, 1), np.int32)
    for a, d in bounds:
        a, b = int(a), int(a) + 1 + int(d) % 64
        cv2.randu(m, a, b)
        assert int(m[0, 0]) == r.uniform(a, b)


@pytest.mark.parametrize("seed", [0, 1, 2 ** 31, 0xFFFFFFFF, 0x9E3779B9])
def test_oracle_rng_jump_ahead_equals_sequential(seed):
    r = sf.CvRNG(seed)
    for k in range(1, 7201):                      # a frame draws at most 2 * 9 * 400 times
        r.next()
        assert r.state == sf.CvRNG.state_after(seed, k), k
    assert sf.CvRNG(0).state == sf.CvRNG(0xFFFFFFFF).state


@pytest.mark.parametrize("rows,cols", [(480, 640), (375, 1242), (20, 20)])
def test_sample_keypoints_layout(rows, cols):
    s = sf.sample_keypoints(rows, cols, 12345)
    assert s.shape == (3000, 2) and s.dtype == np.float32
    xs, ys = cols // 20, rows // 20
    i, j = s[:, 0].astype(int) // xs, s[:, 1].astype(int) // ys
    assert (s > 0).all() and (s[:, 0] < cols).all() and (s[:, 1] < rows).all()
    cell = i * 20 + j
    assert (np.diff(cell) >= 0).all()            # cell-major
    assert (i < 20).all() and (j < 20).all()


def test_tracker_params_layout_unchanged():
    import ctypes
    from vdo_slam_b200 import capi
    assert capi.load().vdo_abi_struct_size(b"vdo_tracker_params") == ctypes.sizeof(capi.TrackerParams) == 108
    assert capi.TrackerParams.use_sample_feature.offset == 100 and capi.TrackerParams.sample_seed.offset == 104


ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHIM = os.path.join(ROOT, "tests", "shim_stub")
EXE = os.path.join(SHIM, "shim_main")

OMD_YAML = """%YAML:1.0
Camera.fx: 618.3587036132812
Camera.fy: 618.5924072265625
Camera.cx: 328.9866333007812
Camera.cy: 237.7507629394531
Camera.k1: 0.0
Camera.width: 640
Camera.height: 480
Camera.fps: 30.0
Camera.bf: 387.5744
Camera.RGB: 1
ChooseData: 1
DepthMapFactor: 1000.0
ThDepthBG: 40.0
ThDepthOBJ: 25.0
MaxTrackPointBG: 1200
MaxTrackPointOBJ: 800
SFMgThres: 0.02
SFDsThres: 0.99
WINDOW_SIZE: 20
OVERLAP_SIZE: 4
UseSampleFeature: 1
{extra}
ORBextractor.nFeatures: 3000
ORBextractor.scaleFactor: 1.2
ORBextractor.nLevels: 8
ORBextractor.iniThFAST: 20
ORBextractor.minThFAST: 7
"""


def _has_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def test_shim_accepts_use_sample_feature(tmp_path):
    subprocess.check_call(["make", "-C", SHIM, "shim_main"], stdout=subprocess.DEVNULL)
    y = tmp_path / "omd.yaml"
    y.write_text(OMD_YAML.format(extra="UseSampleFeature: 2"))
    r = subprocess.run([EXE, str(y), str(tmp_path), "1", "640", "480"], capture_output=True, text=True)
    assert r.returncode != 0 and "UseSampleFeature must be 0" in r.stderr
    if not _has_gpu():
        y.write_text(OMD_YAML.format(extra=""))
        r = subprocess.run([EXE, str(y), str(tmp_path), "1", "640", "480"], capture_output=True, text=True)
        assert r.returncode != 0 and "no CPU fallback" in r.stderr and "not supported" not in r.stderr


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("size", [(640, 480), (1242, 375)])
@pytest.mark.parametrize("seed", SEEDS + [0])
def test_sample_static_matches_oracle(seed, size):
    from vdo_slam_b200 import capi
    from vdo_slam_b200.synth import make_sequence_frame
    w, h = size
    f = make_sequence_frame(1, seed=5, width=w, height=h, K=OMD_K * np.float32([1, 1, w / 640, h / 480]), depth_factor=1000)
    ctx = capi.Context()
    fr = capi.Frame(ctx, w, h)
    fr.upload(f["gray"], f["depth_raw"], f["flow"], f["mask"])
    depth = fr.depth_prep(387.5744, 1000.0)
    g = fr.sample_static(seed, 40.0)
    raw = sf.sample_keypoints(h, w, seed)
    assert np.array_equal(g["raw"], raw)
    keys, corres, flow, dep = sf.filter_sampled(raw, f["mask"], depth, f["flow"], 40.0)
    assert 0 < len(keys) < len(raw)
    assert np.array_equal(np.stack([g["x"], g["y"]], 1), keys) and np.array_equal(np.stack([g["cx"], g["cy"]], 1), corres)
    assert np.array_equal(np.stack([g["fu"], g["fv"]], 1), flow) and np.array_equal(g["depth"], dep)


def _omd_pair(sample_seed, window=6, overlap=2):
    from vdo_slam_b200 import capi
    w, h = 640, 480
    ctx = capi.Context()
    tr = capi.Tracker(ctx, width=w, height=h, fx=float(OMD_K[0]), fy=float(OMD_K[1]), cx=float(OMD_K[2]), cy=float(OMD_K[3]), depth_factor=1000.0,
                      sf_mg_thres=0.02, sf_ds_thres=0.99, n_features=3000, is_kitti=0, dataset=1, window_size=window, overlap_size=overlap,
                      use_sample_feature=1, sample_seed=sample_seed)
    orc = sf.SampledOracleTracker(width=w, height=h, K4=OMD_K, depth_factor=1000.0, sf_mg_thres=0.02, sf_ds_thres=0.99, n_features=3000, is_kitti=False,
                        window_size=window, overlap_size=overlap, use_sample_feature=True, sample_seed=sample_seed)
    return ctx, tr, orc


@pytest.mark.gpu
@pytest.mark.parametrize("sample_seed", [0x9E3779B9, 0])
def test_tracker_omd_configuration_matches_oracle(sample_seed):
    """OMD settings (dataset 1, factor 1000, 3 000 ORB features, SFMg 0.02 / SFDs 0.99) with sampled background features; 8 frames with a
    window of 6 / overlap 2, so that the windowed BA runs at frame 5.  sample_seed 0 seeds each frame with time(NULL); the oracle replays the
    seeds the tracker reports."""
    from tests.test_tracker_gpu import _compare
    from vdo_slam_b200.synth import make_sequence_frame
    ctx, tr, orc = _omd_pair(sample_seed)
    n_stat = []
    for t in range(8):
        f = make_sequence_frame(t, seed=6, width=640, height=480, K=OMD_K, depth_factor=1000)
        d, m = f["depth_raw"].copy(), f["mask"].copy()
        T = tr.track(f["gray"], d, f["flow"], m, f["obj_ids"], writeback=True)
        used = int(tr.get("sample_seed")[0]) & 0xFFFFFFFF
        assert used == sample_seed if sample_seed else used > 0
        orc.sample_seed = used
        T_ref = orc.track(f["gray"], f["depth_raw"], f["flow"], f["mask"], f["obj_ids"])
        assert np.abs(T - T_ref).max() <= 1e-4, f"frame {t}: pose"
        assert np.array_equal(m, orc.mask) and np.array_equal(d, orc.depth), f"frame {t}: write-back"
        _compare(tr, orc, t)
        n_stat.append(len(orc.cur.statKeysTmp))
    runs, iters = tr.get("local_ba").tolist()
    assert runs == len(orc.local_ba) == 1 and iters == sum(orc.local_ba)
    assert min(n_stat) > 0


@pytest.mark.gpu
def test_shim_omd_settings_match_oracle(tmp_path):
    """example/omd.yaml's values plus SampleSeed through VDO_SLAM::System: poses and the depth / mask write-back against the oracle pipeline."""
    from vdo_slam_b200.synth import make_sequence_frame
    subprocess.check_call(["make", "-C", SHIM, "shim_main"], stdout=subprocess.DEVNULL)
    w, h, n, seed = 640, 480, 4, 1760659200
    (tmp_path / "omd.yaml").write_text(OMD_YAML.format(extra=f"SampleSeed: {seed}"))
    orc = sf.SampledOracleTracker(width=w, height=h, K4=OMD_K, depth_factor=1000.0, sf_mg_thres=0.02, sf_ds_thres=0.99, n_features=3000, is_kitti=False,
                        use_sample_feature=True, sample_seed=seed)
    ref, ref_depth, ref_mask = [], [], []
    for t in range(n):
        f = make_sequence_frame(t, seed=7, width=w, height=h, K=OMD_K, depth_factor=1000)
        b = str(tmp_path / f"f{t}")
        np.repeat(f["gray"][..., None], 3, -1).astype(np.uint8).tofile(b + ".rgb")
        f["depth_raw"].astype(np.float32).tofile(b + ".depth"); f["flow"].astype(np.float32).tofile(b + ".flow"); f["mask"].astype(np.int32).tofile(b + ".mask")
        np.array([len(f["obj_ids"])], np.int32).tofile(b + ".ngt"); np.array(f["obj_ids"], np.int32).tofile(b + ".gt")
        ref.append(orc.track(f["gray"], f["depth_raw"], f["flow"], f["mask"], f["obj_ids"]))
        ref_depth.append(orc.depth.copy()); ref_mask.append(orc.mask.copy())
    r = subprocess.run([EXE, str(tmp_path / "omd.yaml"), str(tmp_path), str(n), str(w), str(h)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    poses = [np.array(l.split()[2:], np.float32).reshape(4, 4) for l in r.stdout.splitlines() if l.startswith("POSE")]
    assert len(poses) == n
    for t in range(n):
        assert np.abs(poses[t] - ref[t]).max() <= 1e-4, t
        assert np.array_equal(np.fromfile(str(tmp_path / f"f{t}.depth_out"), np.float32).reshape(h, w), ref_depth[t])
        assert np.array_equal(np.fromfile(str(tmp_path / f"f{t}.mask_out"), np.int32).reshape(h, w), ref_mask[t])
