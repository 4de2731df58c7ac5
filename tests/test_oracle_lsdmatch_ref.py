"""CPU tests: the line-matcher oracle against the REFERENCE's own LSDmatcher.cpp (compiled unmodified, with lineIterator.cpp, into
oracle/_ref/libref_match.so against mock Frame / KeyFrame / MapLine - oracle/ref_lsd_wrap.cpp, oracle/shim_slam/).
FrameBFMatch + lineDescriptorMAD, SearchDouble, both SearchByProjection overloads, SearchForTriangulation, Fuse:
identical match lists and counts."""
import os
import sys
import numpy as np
import pytest
import oracle
from plslam_b200 import synth

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_localmap2 import _line_fuse_problem, _args  # noqa: E402

BOUNDS = [0.0, 0.0, 640.0, 480.0]


@pytest.fixture(scope="module")
def lines():
    f0 = synth.synth_frame(640, 480, 1); f1 = synth.warp_frame(f0, 1001)
    return [oracle.line_extract(f, nfeatures=400) for f in (f0, f1)]


@pytest.mark.parametrize("th,ratio", [(50.0, 0.7), (80.0, 0.8), (30.0, 0.6)])
def test_frame_bf_match_and_mad(lines, th, ratio):
    d0, d1 = lines[0][1][:-1], lines[1][1][:-1]
    for a, b in ((d0, d1), (d1, d0), (d0[:57], d1[:33])):
        om = oracle.frame_bf_match(a, b, th, ratio)
        rm = oracle.frame_bf_match(a, b, th, ratio, impl="ref")
        assert (om >= 0).sum() > 5 and np.array_equal(om, rm)
    # heavy ties: many identical descriptors on both sides (the MAD medians sit on plateaus)
    rng = np.random.default_rng(2)
    base = rng.integers(0, 256, (12, 32), dtype=np.uint8)
    a = base[rng.integers(0, 12, 90)].copy(); b = base[rng.integers(0, 12, 70)].copy()
    a[::3, 0] ^= 1
    assert np.array_equal(oracle.frame_bf_match(a, b, th, ratio), oracle.frame_bf_match(a, b, th, ratio, impl="ref"))


@pytest.mark.parametrize("ratio", [0.7, 0.9])
def test_search_double(lines, ratio):
    d0, d1 = lines[0][1][:-1], lines[1][1][:-1]
    onm, om = oracle.search_double(d0, d1, ratio)
    rnm, rm = oracle.search_double(d0, d1, ratio, impl="ref")
    assert onm > 30 and onm == rnm and np.array_equal(om, rm)
    assert oracle.search_double(d0[:0], d1, ratio, impl="ref")[0] == 0 == oracle.search_double(d0[:0], d1, ratio)[0]


def _queries(lines, rng, jitter):
    (kl0, d0, lf0), (kl1, d1, lf1) = lines
    kl0, d0 = kl0[:-1], d0[:-1]
    proj = np.stack([kl0["startPointX"], kl0["startPointY"], kl0["endPointX"], kl0["endPointY"]], 1).astype(np.float32)
    proj += rng.normal(0, jitter, proj.shape).astype(np.float32)
    return kl0, d0, proj, rng.random(len(kl0)) < 0.85


@pytest.mark.parametrize("th", [15.0, 40.0])
def test_search_by_projection_last(lines, th):
    rng = np.random.default_rng(3)
    kl0, d0, proj, valid = _queries(lines, rng, 1.5)
    kl1, d1, lf1 = (x[:-1] for x in lines[1])
    pre = (rng.random(len(kl1)) < 0.05).astype(np.uint8)
    a = (kl1, lf1, d1, BOUNDS, valid, proj, d0, kl0["lineLength"], th)
    onm, om = oracle.line_search_by_projection_last(*a, preassigned=pre)
    rnm, rm = oracle.line_search_by_projection_last(*a, preassigned=pre, impl="ref")
    assert onm > 30 and onm == rnm and np.array_equal(om, rm)


@pytest.mark.parametrize("th", [1.0, 3.0])
def test_search_by_projection_lines(lines, th):
    rng = np.random.default_rng(5)
    kl0, d0, proj, valid = _queries(lines, rng, 1.0)
    kl1, d1, lf1 = (x[:-1] for x in lines[1])
    vc = rng.uniform(0.99, 1.0, len(kl0)).astype(np.float32)
    pre = (rng.random(len(kl1)) < 0.05).astype(np.uint8)
    a = (kl1, lf1, d1, BOUNDS, valid, proj, vc, d0)
    onm, om = oracle.line_search_by_projection_lines(*a, th, 0.7, preassigned=pre)
    rnm, rm = oracle.line_search_by_projection_lines(*a, th, 0.7, preassigned=pre, impl="ref")
    assert onm > 20 and onm == rnm and np.array_equal(om, rm)


@pytest.mark.parametrize("seed,dbl", [(1, True), (2, True), (3, False)])
def test_search_for_triangulation(seed, dbl):
    f = synth.synth_sequence(2, 640, 480, seed=seed)
    (_, d1, _), (_, d2, _) = oracle.line_extract(f[0]), oracle.line_extract(f[1])
    rng = np.random.default_rng(seed)
    ml1 = (rng.random(len(d1)) < 0.25).astype(np.uint8); ml2 = (rng.random(len(d2)) < 0.25).astype(np.uint8)
    onm, om = oracle.lsd_search_for_triangulation(d1, ml1, d2, ml2, 0.8, dbl)
    rnm, rm = oracle.lsd_search_for_triangulation(d1, ml1, d2, ml2, 0.8, dbl, impl="ref")
    assert onm > 10 and onm == rnm and np.array_equal(om, rm)


@pytest.mark.parametrize("seed,behind", [(21, None), (23, None), (22, 37)])
def test_fuse(seed, behind):
    f = _line_fuse_problem(seed, behind=behind)
    # every keyframe line gets a row in the POINT descriptor matrix here: the reference indexes that matrix with the LINE index
    # (LSDmatcher.cpp:966) and real OpenCV would fail on the rows that do not exist
    rng = np.random.default_rng(seed)
    f["pdesc"] = np.concatenate([f["pdesc"], rng.integers(0, 256, (len(f["kl"]) - len(f["pdesc"]), 32), dtype=np.uint8)])
    obi, obd, stop = oracle.lsd_fuse_search(*_args(f))
    rbi, ret = oracle.lsd_fuse_search(*_args(f), impl="ref")
    want = np.where(obd <= 50, obi, -1)             # Fuse acts on bestDist <= TH_LOW only
    assert np.array_equal(rbi, want)
    if stop == len(f["pos"]):
        assert (want >= 0).sum() > 20 and ret == (want >= 0).sum()
    else:                                            # an end point behind the camera: `return false`, whatever was fused before stays
        assert ret == 0 and (want[stop:] == -1).all()
