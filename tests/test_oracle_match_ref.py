"""CPU tests: the matcher oracle against the REFERENCE's own ORBmatcher.cc and MapPoint.cc (compiled unmodified into
oracle/_ref/libref_match.so against mock Frame / KeyFrame / Map - oracle/Makefile target `ref`, oracle/ref_match_wrap.cpp,
oracle/shim_slam/).  Same flat inputs to both (`impl="ref"` routes an oracle binding to the reference's code): match lists,
match counts and the updated vbPrevMatched must be identical."""
import os
import sys
import numpy as np
import pytest
import oracle
from plslam_b200 import synth

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_localmap2 import _mp_lists  # noqa: E402

BOUNDS = [0.0, 0.0, 640.0, 480.0]


@pytest.fixture(scope="module")
def frames():
    seq = synth.synth_sequence(3, 640, 480, seed=2)
    out = {}
    for nf in (1000, 2000):
        o = oracle.OrbOracle(nf, 1.2, 8, 20, 7)
        out[nf] = [o.extract(f) for f in seq]
    return out


def test_descriptor_distance():
    rng = np.random.default_rng(0)
    a = rng.integers(0, 256, (300, 32), dtype=np.uint8); b = rng.integers(0, 256, (300, 32), dtype=np.uint8)
    b[:20] = a[:20]; b[20:30] = ~a[20:30]
    for i in range(300):
        assert oracle.descriptor_distance(a[i], b[i]) == oracle.descriptor_distance(a[i], b[i], impl="ref")


@pytest.mark.parametrize("nf,win,ratio,ori", [(1000, 100, 0.9, True), (2000, 100, 0.9, True), (2000, 30, 0.7, False), (1000, 60, 0.8, True)])
def test_search_for_initialization(frames, nf, win, ratio, ori):
    (k1, d1), (k2, d2) = frames[nf][0], frames[nf][1]
    prev = np.stack([k1["x"], k1["y"]], 1).astype(np.float32)
    onm, om, opm = oracle.search_for_initialization(k1, d1, k2, d2, BOUNDS, prev, win, ratio, ori)
    rnm, rm, rpm = oracle.search_for_initialization(k1, d1, k2, d2, BOUNDS, prev, win, ratio, ori, impl="ref")
    assert onm > 50
    assert onm == rnm and np.array_equal(om, rm) and opm.tobytes() == rpm.tobytes()
    # the second call re-uses the updated vbPrevMatched, as Tracking::MonocularInitialization does
    k3, d3 = frames[nf][2]
    o2 = oracle.search_for_initialization(k1, d1, k3, d3, BOUNDS, opm, win, ratio, ori)
    r2 = oracle.search_for_initialization(k1, d1, k3, d3, BOUNDS, rpm, win, ratio, ori, impl="ref")
    assert o2[0] == r2[0] and np.array_equal(o2[1], r2[1]) and o2[2].tobytes() == r2[2].tobytes()


def _fake_map(k_last, rng, K):
    z = rng.uniform(1.5, 6.0, len(k_last)).astype(np.float32)
    return np.stack([(k_last["x"] - K[2]) / K[0] * z, (k_last["y"] - K[3]) / K[1] * z, z], 1).astype(np.float32)


@pytest.mark.parametrize("nf,th,seed", [(1000, 15.0, 4), (2000, 7.0, 4), (1000, 30.0, 9)])
def test_search_by_projection_last(frames, nf, th, seed):
    rng = np.random.default_rng(seed)
    (kl, dl), (kc, dc) = frames[nf][0], frames[nf][1]
    K = np.array(synth.TUM1_K, np.float32)
    X = _fake_map(kl, rng, K)
    X[:20, 2] *= -1                                  # behind the camera: invzc < 0
    valid = rng.random(len(kl)) < 0.8
    T = np.eye(4, dtype=np.float32); T[:3, 3] = [0.004, -0.003, 0.002]
    c, s = np.cos(0.002), np.sin(0.002)
    T[:3, :3] = np.array([[c, -s, 0], [s, c, 0], [0, 0, 1]], np.float32)
    sf = oracle.OrbOracle(nf, 1.2, 8, 20, 7).tables()["scale"]
    pre = (rng.random(len(kc)) < 0.05).astype(np.uint8)
    args = (kc, dc, BOUNDS, T, K, sf, valid, X, dl, kl["octave"], kl["angle"], th)
    for ori in (True, False):
        onm, om = oracle.search_by_projection_last(*args, check_ori=ori, preassigned=pre)
        rnm, rm = oracle.search_by_projection_last(*args, check_ori=ori, preassigned=pre, impl="ref")
        assert onm > 100
        assert onm == rnm and np.array_equal(om, rm)


def test_search_by_projection_points(frames):
    rng = np.random.default_rng(6)
    k, d = frames[1000][1]
    kl, dl = frames[1000][0]
    n_mp = 1500
    src = rng.integers(0, len(kl), n_mp)
    proj = np.stack([kl["x"][src], kl["y"][src]], 1).astype(np.float32) + rng.normal(0, 2.0, (n_mp, 2)).astype(np.float32)
    level = np.clip(kl["octave"][src] + rng.integers(-1, 2, n_mp), 0, 7).astype(np.int32)
    in_view = rng.random(n_mp) < 0.85
    view_cos = rng.uniform(0.99, 1.0, n_mp).astype(np.float32)
    sf = oracle.OrbOracle(1000, 1.2, 8, 20, 7).tables()["scale"]
    pre = (rng.random(len(k)) < 0.05).astype(np.uint8)
    for th in (1.0, 3.0, 5.0):
        a = (k, d, BOUNDS, sf, in_view, proj, level, view_cos, dl[src])
        onm, om = oracle.search_by_projection_points(*a, th, 0.8, preassigned=pre)
        rnm, rm = oracle.search_by_projection_points(*a, th, 0.8, preassigned=pre, impl="ref")
        assert onm > 100
        assert onm == rnm and np.array_equal(om, rm)


@pytest.mark.parametrize("seed,ori", [(5, True), (5, False), (7, True), (11, True), (12, False)])
def test_search_for_triangulation(seed, ori):
    s = synth.synth_two_view(seed)
    a, b = s["1"], s["2"]
    args = (a["keys"], a["desc"], a["has_mp"], b["keys"], b["desc"], b["has_mp"], a["fv"], b["fv"], s["F12"], s["Cw1"], b["R"], b["t"],
            s["K"], s["scale_factors"], s["level_sigma2"])
    onm, om = oracle.search_for_triangulation(*args, ori)
    rnm, rm = oracle.search_for_triangulation(*args, ori, impl="ref")
    assert onm > 200 and onm == rnm and np.array_equal(om, rm)


@pytest.mark.parametrize("seed,th", [(6, 3.0), (8, 3.0), (9, 1.0), (10, 6.0)])
def test_fuse(seed, th):
    f = synth.synth_fuse_problem(seed)
    args = (f["keys"], f["desc"], f["bounds"], f["Tcw"], f["Ow"], f["K"], f["scale_factors"], f["inv_level_sigma2"],
            f["log_scale_factor"], f["skip"], f["pos"], f["normal"], f["min_dist"], f["max_dist"], f["mp_desc"], th)
    obi, obd = oracle.fuse_search(*args)
    rbi, nfused = oracle.fuse_search(*args, impl="ref")
    # ORBmatcher::Fuse acts on a candidate only if bestDist <= TH_LOW (50): the oracle reports the search for every point
    want = np.where(obd <= 50, obi, -1)
    assert (want >= 0).sum() > 20
    assert np.array_equal(rbi, want)
    assert nfused == (want >= 0).sum()


@pytest.mark.parametrize("seed,ori,ratio", [(5, True, 0.7), (5, False, 0.7), (7, True, 0.9), (11, True, 0.6), (12, False, 0.75)])
def test_search_by_bow(seed, ori, ratio):
    s = synth.synth_two_view(seed)
    a, b = s["1"], s["2"]
    args = (a["keys"], a["desc"], a["has_mp"], b["keys"], b["desc"], a["fv"], b["fv"])
    onm, om = oracle.search_by_bow(*args, ratio, ori)
    rnm, rm = oracle.search_by_bow(*args, ratio, ori, impl="ref")
    assert onm > 100 and onm == rnm and np.array_equal(om, rm)


def test_distinctive_descriptors():
    desc, off = _mp_lists(3)
    best = oracle.distinctive_descriptors(desc, off)
    chosen = oracle.ref_distinctive_descriptors(desc, off)
    want = np.zeros((len(off) - 1, 32), np.uint8)    # no observation: the reference returns early and keeps the old (zero) descriptor
    for m in range(len(off) - 1):
        if off[m + 1] > off[m]:
            want[m] = desc[off[m] + best[m]]
    assert np.array_equal(chosen, want)


def test_predict_scale():
    rng = np.random.default_rng(1)
    n = 200000
    max_dist = rng.uniform(2.0, 12.0, n).astype(np.float32)
    dist = (max_dist / rng.uniform(0.5, 6.0, n)).astype(np.float32)
    # exact level boundaries and their fp32 neighbours: where logf / the fp32 quotient decide the level
    k = np.arange(n // 2) % 9
    edge = (max_dist[:n // 2] / (np.float32(1.2) ** k.astype(np.float32))).astype(np.float32)
    dist[:n // 2] = np.nextafter(edge, np.where(np.arange(n // 2) % 3 == 0, np.float32(0), np.where(np.arange(n // 2) % 3 == 1, np.float32(1e9), edge)).astype(np.float32))
    log_sf = np.float32(np.log(np.float32(1.2)))
    ref = oracle.ref_predict_scale(dist, max_dist, log_sf, 8)
    got = oracle.predict_scale(dist, max_dist, log_sf, 8)
    assert np.array_equal(ref, got)
    # and it is not the fp64 formula: on the boundaries the two disagree somewhere (which is why the float functions matter)
    ratio = (max_dist / dist).astype(np.float32)
    f64 = np.clip(np.ceil(np.log(ratio.astype(np.float64)) / np.float64(log_sf)), 0, 7).astype(np.int32)
    assert (f64 != got).sum() > 0


@pytest.mark.parametrize("seed,ori,ratio", [(5, True, 0.75), (7, False, 0.75), (11, True, 0.6)])
def test_search_by_bow_keyframes(seed, ori, ratio):
    s = synth.synth_two_view(seed)
    a, b = s["1"], s["2"]
    args = (a["keys"], a["desc"], 1 - a["has_mp"], b["keys"], b["desc"], 1 - b["has_mp"], a["fv"], b["fv"])
    onm, om = oracle.search_by_bow_keyframes(*args, ratio, ori)
    rnm, rm = oracle.search_by_bow_keyframes(*args, ratio, ori, impl="ref")
    assert onm > 100 and onm == rnm and np.array_equal(om, rm)


@pytest.mark.parametrize("seed,th,dist,ori", [(6, 10.0, 100, True), (8, 3.0, 64, True), (9, 10.0, 100, False), (10, 3.0, 64, False)])
def test_search_by_projection_keyframe(seed, th, dist, ori):
    from test_oracle_localmap import _reloc_args
    args, pre = _reloc_args(seed, th, dist)
    rnm, rm, ow = oracle.search_by_projection_keyframe(*args, ori, pre, impl="ref")
    a = list(args); a[4] = ow                       # the camera centre as the reference derives it from Tcw (fp32 gemm of -Rcw^T tcw)
    onm, om = oracle.search_by_projection_keyframe(*a, ori, pre)
    assert onm > 10 and onm == rnm and np.array_equal(om, rm)
    assert np.allclose(ow, args[4], rtol=0, atol=1e-5)
