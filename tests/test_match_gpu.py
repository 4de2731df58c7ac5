"""GPU parity tests: matching through the C ABI vs the CPU oracle — indices and Hamming distances bit-exact."""
import numpy as np
import pytest
import oracle
import plslam_b200 as pl
from plslam_b200 import synth

pytestmark = pytest.mark.gpu
BOUNDS = [0.0, 0.0, 640.0, 480.0]


@pytest.fixture(scope="module")
def frames():
    seq = synth.synth_sequence(3, 640, 480, seed=2)
    out = {}
    for nf in (1000, 2000):
        o = oracle.OrbOracle(nf, 1.2, 8, 20, 7)
        out[nf] = [o.extract(f) for f in seq]
    return out


def test_descriptor_distance(frames):
    rng = np.random.default_rng(0)
    a = rng.integers(0, 256, (500, 32), dtype=np.uint8); b = rng.integers(0, 256, (500, 32), dtype=np.uint8)
    b[:50] = a[:50]; b[50:60] = ~a[50:60]
    got = pl.ORBmatcher.DescriptorDistance(a, b)
    assert list(got) == [oracle.descriptor_distance(a[i], b[i]) for i in range(500)]
    assert got[0] == 0 and got[55] == 256


@pytest.mark.parametrize("nf", [1000, 2000])
def test_assign_grid(frames, nf):
    k, d = frames[nf][0]
    s, it = pl.frame_assign_grid(k, BOUNDS)
    os_, oit = oracle.assign_grid(k, BOUNDS)
    assert np.array_equal(s, os_) and np.array_equal(it, oit)
    # keypoints outside the bounds are dropped (Frame::PosInGrid)
    k2 = k.copy(); k2["x"][:50] += 700
    s, it = pl.frame_assign_grid(k2, BOUNDS)
    os_, oit = oracle.assign_grid(k2, BOUNDS)
    assert np.array_equal(s, os_) and np.array_equal(it, oit)


@pytest.mark.parametrize("nf,win,ratio,ori", [(1000, 100, 0.9, True), (2000, 100, 0.9, True), (2000, 30, 0.7, False)])
def test_search_for_initialization(frames, nf, win, ratio, ori):
    (k1, d1), (k2, d2) = frames[nf][0], frames[nf][1]
    prev = np.stack([k1["x"], k1["y"]], 1).astype(np.float32)
    nm, m, pm = pl.ORBmatcher(ratio, ori).SearchForInitialization(k1, d1, k2, d2, BOUNDS, prev, win)
    onm, om, opm = oracle.search_for_initialization(k1, d1, k2, d2, BOUNDS, prev, win, ratio, ori)
    assert onm > 50
    assert nm == onm and np.array_equal(m, om) and np.array_equal(pm, opm)
    # second call re-uses the updated vbPrevMatched like Tracking::MonocularInitialization does
    nm2, m2, _ = pl.ORBmatcher(ratio, ori).SearchForInitialization(k1, d1, frames[nf][2][0], frames[nf][2][1], BOUNDS, pm, win)
    onm2, om2, _ = oracle.search_for_initialization(k1, d1, frames[nf][2][0], frames[nf][2][1], BOUNDS, opm, win, ratio, ori)
    assert nm2 == onm2 and np.array_equal(m2, om2)


def _fake_map(k_last, rng, K):
    """3-D points whose projection with identity pose is the last frame's keypoint."""
    z = rng.uniform(1.5, 6.0, len(k_last)).astype(np.float32)
    X = np.stack([(k_last["x"] - K[2]) / K[0] * z, (k_last["y"] - K[3]) / K[1] * z, z], 1).astype(np.float32)
    return X


@pytest.mark.parametrize("nf,th", [(1000, 15.0), (2000, 7.0)])
def test_search_by_projection_last(frames, nf, th):
    rng = np.random.default_rng(4)
    (kl, dl), (kc, dc) = frames[nf][0], frames[nf][1]
    K = np.array(synth.TUM1_K, np.float32)
    X = _fake_map(kl, rng, K)
    valid = rng.random(len(kl)) < 0.8
    T = np.eye(4, dtype=np.float32); T[:3, 3] = [0.004, -0.003, 0.002]
    sf = oracle.OrbOracle(nf, 1.2, 8, 20, 7).tables()["scale"]
    pre = (rng.random(len(kc)) < 0.05).astype(np.uint8)
    args = (kc, dc, BOUNDS, T, K, sf, valid, X, dl, kl["octave"], kl["angle"], th)
    for ori in (True, False):
        nm, m = pl.ORBmatcher(0.9, ori).SearchByProjectionLast(*args, preassigned=pre)
        onm, om = oracle.search_by_projection_last(*args, check_ori=ori, preassigned=pre)
        assert onm > 100
        assert nm == onm and np.array_equal(m, om)


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
    for th in (1.0, 3.0, 5.0):
        a = (k, d, BOUNDS, sf, in_view, proj, level, view_cos, dl[src])
        nm, m = pl.ORBmatcher(0.8).SearchByProjectionPoints(*a, th=th)
        onm, om = oracle.search_by_projection_points(*a, th, 0.8)
        assert onm > 100
        assert nm == onm and np.array_equal(m, om)


def test_bf_knn_and_line_matching():
    rng = np.random.default_rng(8)
    # tie-heavy descriptors (bytes are 0x00/0xff) exercise "lower train index first"
    d1 = rng.integers(0, 2, (201, 32), dtype=np.uint8) * 255
    d2 = rng.integers(0, 2, (187, 32), dtype=np.uint8) * 255
    idx, dist = pl.LSDmatcher.knnMatch(d1, d2)
    oi, od = oracle.bf_knn2(d1, d2)
    assert np.array_equal(idx, oi) and np.array_equal(dist, od)
    # realistic: second set = noisy permutation of the first
    base = rng.integers(0, 256, (201, 32), dtype=np.uint8)
    perm = rng.permutation(201)[:180]
    d2 = base[perm].copy()
    for i in range(len(d2)):
        bits = rng.integers(0, 256, rng.integers(0, 30))
        for b in bits:
            d2[i, b // 8] ^= np.uint8(1 << (b % 8))
    for th, ratio in ((50.0, 0.7), (80.0, 0.9)):
        m = pl.LSDmatcher(ratio).FrameBFMatch(base, d2, th)
        assert np.array_equal(m, oracle.frame_bf_match(base, d2, th, ratio))
    nm, m = pl.LSDmatcher(0.7).SearchDouble(base, d2)
    onm, om = oracle.search_double(base, d2, 0.7)
    assert onm > 100 and nm == onm and np.array_equal(m, om)
    # degenerate sizes (reference reads out of bounds for <2 rows; defined as "no matches")
    for a, b in ((base[:0], d2), (base, d2[:0]), (base, d2[:1]), (base[:1], d2), (base[:2], d2[:2])):
        nm, m = pl.LSDmatcher(0.7).SearchDouble(a, b)
        onm, om = oracle.search_double(a, b, 0.7)
        assert nm == onm and np.array_equal(m, om)


def test_matchers_equal_the_reference_matcher_code(frames):
    """The CUDA matchers against the REFERENCE's own ORBmatcher.cc (compiled into oracle/_ref/libref_match.so, run on this box's CPU):
    SearchForInitialization and the two tracking searches, same inputs, identical match lists."""
    (k1, d1), (k2, d2) = frames[1000][0], frames[1000][1]
    prev = np.stack([k1["x"], k1["y"]], 1).astype(np.float32)
    nm, m, pm = pl.ORBmatcher(0.9, True).SearchForInitialization(k1, d1, k2, d2, BOUNDS, prev, 100)
    rnm, rm, rpm = oracle.search_for_initialization(k1, d1, k2, d2, BOUNDS, prev, 100, 0.9, True, impl="ref")
    assert rnm > 50 and nm == rnm and np.array_equal(m, rm) and pm.tobytes() == rpm.tobytes()
    rng = np.random.default_rng(14)
    K = np.array(synth.TUM1_K, np.float32)
    X = _fake_map(k1, rng, K)
    valid = rng.random(len(k1)) < 0.8
    T = np.eye(4, dtype=np.float32); T[:3, 3] = [0.004, -0.003, 0.002]
    sf = oracle.OrbOracle(1000, 1.2, 8, 20, 7).tables()["scale"]
    pre = (rng.random(len(k2)) < 0.05).astype(np.uint8)
    args = (k2, d2, BOUNDS, T, K, sf, valid, X, d1, k1["octave"], k1["angle"], 15.0)
    nm, m = pl.ORBmatcher(0.9, True).SearchByProjectionLast(*args, preassigned=pre)
    rnm, rm = oracle.search_by_projection_last(*args, check_ori=True, preassigned=pre, impl="ref")
    assert rnm > 100 and nm == rnm and np.array_equal(m, rm)
    n_mp = 1500
    src = rng.integers(0, len(k1), n_mp)
    proj = np.stack([k1["x"][src], k1["y"][src]], 1).astype(np.float32) + rng.normal(0, 2.0, (n_mp, 2)).astype(np.float32)
    level = np.clip(k1["octave"][src] + rng.integers(-1, 2, n_mp), 0, 7).astype(np.int32)
    a = (k2, d2, BOUNDS, sf, rng.random(n_mp) < 0.85, proj, level, rng.uniform(0.99, 1.0, n_mp).astype(np.float32), d1[src])
    nm, m = pl.ORBmatcher(0.8).SearchByProjectionPoints(*a, th=3.0)
    rnm, rm = oracle.search_by_projection_points(*a, 3.0, 0.8, impl="ref")
    assert rnm > 100 and nm == rnm and np.array_equal(m, rm)
