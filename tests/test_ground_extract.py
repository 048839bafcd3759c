"""(f)-4, first part: multi-region ground extraction (Segmentation::groundRemove, ref:
src/models/segmentation/segmentation.cpp:738-770 and what it calls) -- the CPU restatement against independent
implementations, and the device path bit-exact against the restatement (index lists, beams, regions, plane models)."""
import os

import numpy as np
import pytest

from tloam_b200 import synth


@pytest.fixture(scope="module")
def scan():
    return synth.raw_scan()


def test_fast_atan2_restatement_matches_opencv(oracle):
    """Against cv2.fastAtan2's answers, recorded in tests/golden/opencv_pins.npz (tools/make_golden.py opencv)."""
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "opencv_pins.npz"))
    for y, x, a in zip(g["atan_y"], g["atan_x"], g["fast_atan2"]):
        assert oracle.fast_atan2(y, x) == float(a), (y, x)


def test_section_bounds_reproduce_the_stalled_table(oracle):
    """initSections (:174-221): the `continue` at :203-206 skips the angle increment, so only the first two of the three
    section bounds exist: beams 20 and 41, h / tan(16.9 deg), h / tan(6.8 deg)."""
    b = oracle.ground_section_bounds()
    assert len(b) == 2
    assert np.isclose(b[0], 1.73 / np.tan(np.radians(16.9)), rtol=1e-6)
    assert np.isclose(b[1], 1.73 / np.tan(np.radians(6.8)), rtol=1e-6)


def numpy_ground(p, thr, bounds, plane_dis=0.3, h=1.73):
    """Independent (vectorised) restatement of the region assignment and of ONE region's 3-iteration plane fit."""
    x, y, z = p[:, 0], p[:, 1], p[:, 2]
    keep = ~(z > thr)
    th = np.degrees(np.arctan2(-y, x)) % 360.0
    q = (th // 90).astype(int)
    r = np.hypot(x, y)
    s = np.where(r < bounds[0], 0, np.where(r < bounds[1], 1, 2))
    return keep, q * 3 + s


def test_oracle_ground_extract_against_numpy(oracle, scan):
    r = oracle.ground_extract(scan)
    n = len(scan)
    # beams: number of quadrant 4 -> 1 transitions so far, saturating at 63
    x, y = scan[:, 0], scan[:, 1]
    quad = np.where((x > 0) & (y >= 0), 1, np.where((x <= 0) & (y > 0), 2, np.where((x < 0) & (y <= 0), 3, 4)))
    tr = np.concatenate([[False], (quad[1:] == 1) & (quad[:-1] == 4)])
    assert np.array_equal(r["beam"], np.minimum(np.cumsum(tr), 63))
    assert np.isclose(r["height_threshold"], scan[:, 2].mean() + 0.5, rtol=0, atol=1e-10)
    keep, reg = numpy_ground(scan, r["height_threshold"], oracle.ground_section_bounds())
    assert np.array_equal(r["region"] == 12, ~keep)
    # fastAtan2 is a 0.3-degree approximation of atan2: regions agree except within that of a quadrant boundary
    same = r["region"][keep] == reg[keep]
    assert same.mean() > 0.995
    # every point is in exactly one of: ground, object, or a skipped region
    both = np.concatenate([r["ground"], r["object"]])
    assert len(np.unique(both)) == len(both) and len(both) <= n
    # the final plane of region 0, refitted independently from the ground points it produced
    g0 = [i for i in r["ground"] if r["region"][i] == 0]
    assert g0 == sorted(g0)                                  # index order inside a region
    pl = r["planes"][0, 2]
    d = np.abs(scan[g0] @ pl[:3] + pl[3])
    assert d.max() < 0.3 and abs(np.linalg.norm(pl[:3]) - 1) < 1e-12
    # ground is (nearly) the z = -1.73 plane in this scene
    assert abs(abs(pl[2]) - 1) < 1e-3 and abs(abs(pl[3]) - 1.73) < 0.05
    assert 0.5 * n < len(r["ground"]) < 0.8 * n


def test_oracle_ground_extract_edge_cases(oracle):
    r = oracle.ground_extract(np.zeros((0, 3)))
    assert len(r["ground"]) == 0 and len(r["object"]) == 0 and r["height_threshold"] == 1.0
    # a region with <= 3 seeds is skipped entirely: its points reach neither list (ref: :665-666)
    p = np.array([[5.0, -1.0, -1.7]] * 25 + [[-5.0, 1.0, -1.7]] * 400)      # fastAtan2(-y, x): quadrant 0, then quadrant 2
    p[:, 0] += np.linspace(0, 1, len(p))
    r = oracle.ground_extract(p)
    assert set(r["region"][:25]) == {0} and not (set(range(25)) & set(np.concatenate([r["ground"], r["object"]])))
    assert len(r["ground"]) > 300


@pytest.mark.gpu
def test_gpu_ground_extract_is_bit_exact(oracle, scan):
    import tloam_b200
    reg = tloam_b200.LocalRegistration()
    for pts in (scan, scan[::3], scan[:5000], synth.raw_scan(seed=9, n_az=900), np.zeros((0, 3))):
        g = reg.ground_extract(pts)
        o = oracle.ground_extract(pts)
        assert g["height_threshold"] == o["height_threshold"]
        assert np.array_equal(g["beam"], o["beam"])
        assert np.array_equal(g["region"], o["region"])
        assert np.array_equal(g["planes"], o["planes"], equal_nan=True)
        assert np.array_equal(g["ground"], o["ground"])
        assert np.array_equal(g["object"], o["object"])
    reg.close()


@pytest.mark.gpu
def test_gpu_ground_extract_skipped_region_and_ties(oracle):
    import tloam_b200
    reg = tloam_b200.LocalRegistration()
    p = np.array([[5.0, -1.0, -1.7]] * 25 + [[-5.0, 1.0, -1.7]] * 400)       # exact z ties among the seeds
    p[:, 0] += np.linspace(0, 1, len(p))
    g, o = reg.ground_extract(p), oracle.ground_extract(p)
    for k in ("ground", "object", "beam", "region"):
        assert np.array_equal(g[k], o[k]), k
    assert np.array_equal(g["planes"], o["planes"], equal_nan=True)
    reg.close()
