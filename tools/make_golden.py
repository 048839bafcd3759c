"""Generate tests/golden/tls_small.npz: a small seeded frame + what the CPU oracle computes for it.

The reference has no golden vectors of its own and cannot be run here (DESIGN.md section 2), so these vectors
pin the ORACLE (a regression guard for the checker) and give the GPU tests a fixture that does not depend on
re-running the oracle.  Re-run this script only when the oracle is deliberately changed.

    python tools/make_golden.py            # tls_small.npz, feature_small.npz
    python tools/make_golden.py opencv     # opencv_pins.npz (needs OpenCV's Python package)
"""
import os
import sys

import numpy as np

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
from oracle import pyoracle  # noqa: E402
from tloam_b200 import synth  # noqa: E402


def main():
    cfg = synth.scaled(0.02, seed=20260924)
    T_gt = synth.se3_exp([12.0, -7.0, 0.03, 0.004, -0.006, 0.9])
    predict = T_gt @ synth.se3_exp([0.05, -0.03, 0.01, 0.004, -0.003, 0.006])
    mp = synth.make_map(cfg, T_gt)
    origin = np.rint(0.5 * (mp[0].min(0) + mp[0].max(0)))     # the library's rule: bounding box of the first cloud
    mp = [origin + (c - origin).astype(np.float32).astype(np.float64) for c in mp]   # float-representable map
    scan = synth.make_scan(cfg, T_gt, 0)
    out = {"T_gt": T_gt, "predict": predict, "origin": origin}
    for i, name in enumerate(synth.CLOUDS):
        out[f"map_{name}"] = (mp[i] - origin).astype(np.float32)     # stored relative to origin, exactly
        out[f"scan_{name}"] = scan[i]
    o = pyoracle.Oracle()                                             # reference default caps
    o.set_input_target(mp)
    o.set_input_source(scan)
    rc, T, st = o.scan_matching(predict)
    assert rc == 0
    out["pose"] = T
    out["x_init"] = np.array(st.x_init)
    out["n_outer"] = st.n_outer
    out["n_factors"] = np.array([list(st.outer[i].n_factors) for i in range(st.n_outer)])
    out["n_inner"] = np.array([st.outer[i].n_inner for i in range(st.n_outer)])
    out["termination"] = np.array([st.outer[i].termination for i in range(st.n_outer)])
    out["initial_cost"] = np.array([st.outer[i].initial_cost for i in range(st.n_outer)])
    out["final_cost"] = np.array([st.outer[i].final_cost for i in range(st.n_outer)])
    out["H0"] = np.array([list(st.outer[i].H0) for i in range(st.n_outer)]).reshape(-1, 6, 6)
    out["g0"] = np.array([list(st.outer[i].g0) for i in range(st.n_outer)])
    out["x_end"] = np.array([list(st.outer[i].x_end) for i in range(st.n_outer)])
    out["accepted"] = np.array([[st.outer[i].inner[k].accepted if k < st.outer[i].n_inner else -9 for k in range(8)]
                                for i in range(st.n_outer)])
    x = pyoracle.se3_log(predict)
    for c, name in enumerate(synth.CLOUDS):
        v, p = o.build_factors(c, x)
        out[f"valid_{name}"] = v.astype(np.uint8)
        out[f"prim_{name}"] = p
    # functor known answers at fixed inputs
    rng = np.random.default_rng(5)
    xf = np.array([0.8, 0.02, -0.4, 0.01, -0.02, 0.15])
    P, Q, A = rng.normal(0, 30, (8, 3)), rng.normal(0, 30, (8, 3)), rng.normal(0, 30, (8, 3))
    D = rng.normal(size=(8, 3))
    D /= np.linalg.norm(D, axis=1, keepdims=True)
    B = A - 0.2 * D
    W = rng.uniform(0, 1, 8)
    out.update(f_x=xf, f_p=P, f_q=Q, f_a=A, f_b=B, f_n=D, f_d=rng.normal(0, 5, 8), f_w=W)
    pp = [pyoracle.eval_point_to_point(xf, P[i], Q[i], W[i]) for i in range(8)]
    pl = [pyoracle.eval_point_to_line(xf, P[i], A[i], B[i], W[i]) for i in range(8)]
    pn = [pyoracle.eval_point_to_plane(xf, P[i], D[i], out["f_d"][i], W[i]) for i in range(8)]
    for tag, res in (("pp", pp), ("pl", pl), ("pn", pn)):
        out[f"{tag}_r"] = np.array([r[0] for r in res])
        out[f"{tag}_J"] = np.array([r[1] for r in res])
        out[f"{tag}_c"] = np.array([r[2] for r in res])
    path = os.path.join(ROOT, "tests", "golden", "tls_small.npz")
    np.savez_compressed(path, **out)
    print(path, os.path.getsize(path), "bytes; factors per outer:", out["n_factors"].tolist())
    feature_golden()


def feature_golden():
    """tests/golden/feature_small.npz: a 3000-point general cloud + what oracle/feature_oracle.cpp computes for it
    ((f)-2, featureExtract::calculatePCAInfo / extractPlanarSphere)."""
    pts = synth.general_cloud(3000, seed=20260924)
    info = pyoracle.pca_info(pts)
    lists = pyoracle.extract_planar_sphere(pts)
    out = {"points": pts, "cvr": info["cvr"], "flatness": info["flatness"], "sphericity": info["sphericity"],
           "normal": info["normal"], "num_sum": info["num_sum"], "neigh": info["neigh"].astype(np.int16)}
    for name, lst in zip(("planar_scan", "planar_submap", "sphere_scan", "sphere_submap", "sphere_candidates"), lists):
        out[name] = lst.astype(np.int32)
    path = os.path.join(ROOT, "tests", "golden", "feature_small.npz")
    np.savez_compressed(path, **out)
    print(path, os.path.getsize(path), "bytes; lists:", [len(x) for x in lists])


def opencv_golden():
    """tests/golden/opencv_pins.npz: what OpenCV answers for the inputs of the two oracle pins that restate it --
    cv2.fastAtan2 (groundRemove's angle) and exact FLANN kNN (FLANN_INDEX_KDTREE_SINGLE, the tree Open3D's
    KDTreeFlann builds).  OpenCV is needed only to make this file, not to run the tests.

        python tools/make_golden.py opencv
    """
    import cv2
    rng = np.random.default_rng(0)
    ys = np.concatenate([rng.normal(0, 20, 4000), [0.0, 0.0, 1.0, -1.0, 1e-30, -1e-30, 3.0, -3.0]]).astype(np.float32)
    xs = np.concatenate([rng.normal(0, 20, 4000), [0.0, 1.0, 0.0, 0.0, 5.0, 5.0, 1e-30, -1e-30]]).astype(np.float32)
    atan = np.array([cv2.fastAtan2(float(y), float(x)) for y, x in zip(ys, xs)], dtype=np.float32)
    rng = np.random.default_rng(5)
    pts = rng.uniform(-20, 20, (4000, 3)).astype(np.float32)
    qs = rng.uniform(-20, 20, (500, 3)).astype(np.float32)
    index = cv2.flann_Index(pts, dict(algorithm=4))
    idx, d2 = index.knnSearch(qs, 5, params=dict(checks=-1))
    out = {"atan_y": ys, "atan_x": xs, "fast_atan2": atan, "knn_points": pts, "knn_queries": qs,
           "flann_idx": idx.astype(np.int32), "flann_d2": d2.astype(np.float32), "opencv_version": cv2.__version__}
    path = os.path.join(ROOT, "tests", "golden", "opencv_pins.npz")
    np.savez_compressed(path, **out)
    print(path, os.path.getsize(path), "bytes; OpenCV", cv2.__version__)


if __name__ == "__main__":
    if sys.argv[1:] == ["opencv"]:
        opencv_golden()
    else:
        main()
