"""Generates the golden vectors under tests/golden/ from the CPU oracle on seeded synthetic inputs.

The reference cannot be built or imported in this image (no Eigen3 / OpenCV C++ / CSparse; SURVEY.md section 8c), it ships
no fixtures of its own, and its demo data is an external download -- so the vectors below are the ORACLE's outputs, frozen:
they pin the oracle against drift (tests/test_golden.py, CPU) and give the GPU parity tests a committed target that does not
depend on rebuilding the oracle on the GPU box.  Re-run only when the oracle is deliberately changed:
    python tests/golden/make_golden.py              # the small cases (seconds)
    python tests/golden/make_golden.py --config4    # BASELINE config 4, full LM solve (blocked oracle solver, ~10 s on 8 cores)
    python tests/golden/make_golden.py --config5    # BASELINE config 5, full LM solve (~5 min on 8 cores, 4 GB)
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import pyoracle as po                                   # noqa: E402
from vdo_slam_b200.synth import make_batch_graph, make_flow_problem  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))


CONFIG4 = dict(n_frames=200, n_objects=5, n_static=40000, n_dynamic=10000, seed=4)
CONFIG5 = dict(n_frames=1000, n_objects=50, n_static=800000, n_dynamic=200000, seed=5, obj_span=(100, 400))


def graph_fingerprint(g):
    """A few sums over the generated graph: the GPU test regenerates the graph from the seed and checks it is the same one."""
    return np.array([g["se3"].sum(), g["pt"].sum(), g["obs_z"].sum(), g["se3e_Z"].sum(), float(g["obs_cp"].astype(np.int64).sum()),
                     float(g["ter_pph"].astype(np.int64).sum())])


def big(name, cfg, pt_stride, se3_stride=None):
    """Full LM solve of a BASELINE config by the oracle (blocked direct solver, oracle/ba_block.h: the same Cholesky solve of the
    full system as oracle/ba_lm.c's scalar one, which tests/test_oracle_ba.py checks on small graphs).  Keeps: iteration count,
    chi2 / lambda history, every se3 vertex (or, with se3_stride, every se3_stride-th one, listed in se3_idx), every pt_stride-th
    point.  The strides keep each file under 1 MB."""
    g = make_batch_graph(**cfg)
    r = po.ba_optimize_blocked(g, max_iters=300, gain_threshold=1e-4, verbose=True)
    idx = np.arange(0, len(g["pt"]), pt_stride)
    se3 = {"se3": r["se3"]}
    if se3_stride:
        se3_idx = np.arange(0, len(g["se3"]), se3_stride)
        se3 = {"se3": r["se3"][se3_idx], "se3_idx": se3_idx}
    np.savez_compressed(os.path.join(HERE, name), iters=r["iters"], chi2=r["chi2"], lam=r["lam"], **se3, pt_idx=idx,
                        pt=r["pt"][idx], fingerprint=graph_fingerprint(g), trials=r["stats"]["trials"],
                        cfg=np.array(repr(cfg)), oracle_seconds=r["stats"]["t_total"])
    print(name, "iters", r["iters"], "chi2", r["chi2"][0], "->", r["chi2"][-1], "seconds", r["stats"]["t_total"])


def main():
    if "--config4" in sys.argv:
        return big("ba_config4.npz", CONFIG4, 7)
    if "--config5" in sys.argv:
        return big("ba_config5.npz", CONFIG5, 177, se3_stride=4)
    # batch LM (Optimizer::FullBatchOptimization constants): 10 frames, 1 object, 120 static + 40 dynamic tracks
    g = make_batch_graph(n_frames=10, n_objects=1, n_static=120, n_dynamic=40, seed=42)
    r = po.ba_optimize(g, max_iters=12, gain_threshold=1e-4)
    np.savez_compressed(os.path.join(HERE, "ba_small.npz"), iters=r["iters"], chi2=r["chi2"], se3=r["se3"], pt=r["pt"],
                        **{"g_" + k: v for k, v in g.items() if isinstance(v, np.ndarray)})
    # per-frame flow / pose LM (Optimizer::PoseOptimizationFlow2), both arithmetic modes, object and camera priors
    out = {}
    p = make_flow_problem(n=300, seed=7)
    for mode in (0, 1):
        for quirk in (0, 1):
            f = po.flow2(p, mode=mode, quirk=quirk)
            out[f"T_m{mode}_q{quirk}"] = f["T"]; out[f"iters_m{mode}_q{quirk}"] = f["iters"]; out[f"inlier_m{mode}_q{quirk}"] = f["inlier"]
    np.savez_compressed(os.path.join(HERE, "flow2_small.npz"), **out, **{"p_" + k: np.asarray(v) for k, v in p.items()})
    print("written:", [f for f in sorted(os.listdir(HERE)) if f.endswith(".npz")])


if __name__ == "__main__":
    main()
