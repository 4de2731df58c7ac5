"""GPU parity: line grid (Frame::AssignFeaturesToGridForLine) and the two LSDmatcher::SearchByProjection variants."""
import numpy as np
import pytest
import oracle
import plslam_b200 as pl
from plslam_b200 import synth

pytestmark = pytest.mark.gpu
BOUNDS = [0.0, 0.0, 640.0, 480.0]


@pytest.fixture(scope="module")
def lines():
    f0 = synth.synth_frame(640, 480, 1); f1 = synth.warp_frame(f0, 1001)
    return [oracle.line_extract(f, nfeatures=400) for f in (f0, f1)]


def test_line_grid(lines):
    kl = lines[0][0][:-1]
    s, it = pl.frame_assign_grid_lines(kl, BOUNDS)
    os_, oit = oracle.assign_grid_lines(kl, BOUNDS)
    assert np.array_equal(s, os_) and np.array_equal(it, oit) and len(it) > len(kl)


def _queries(lines, rng, jitter):
    (kl0, d0, lf0), (kl1, d1, lf1) = lines
    kl0, d0 = kl0[:-1], d0[:-1]
    n = len(kl0)
    proj = np.stack([kl0["startPointX"], kl0["startPointY"], kl0["endPointX"], kl0["endPointY"]], 1).astype(np.float32)
    proj += rng.normal(0, jitter, proj.shape).astype(np.float32)
    valid = rng.random(n) < 0.85
    return kl0, d0, proj, valid


@pytest.mark.parametrize("th", [15.0, 40.0])
def test_search_by_projection_last(lines, th):
    rng = np.random.default_rng(3)
    kl0, d0, proj, valid = _queries(lines, rng, 1.5)
    kl1, d1, lf1 = lines[1]
    kl1, d1, lf1 = kl1[:-1], d1[:-1], lf1[:-1]
    pre = (rng.random(len(kl1)) < 0.05).astype(np.uint8)
    a = (kl1, lf1, d1, BOUNDS, valid, proj, d0, kl0["lineLength"], th)
    nm, m = pl.LSDmatcher(0.7).SearchByProjectionLast(*a, preassigned=pre)
    onm, om = oracle.line_search_by_projection_last(*a, preassigned=pre)
    assert onm > 30 and nm == onm and np.array_equal(m, om)


@pytest.mark.parametrize("th", [1.0, 3.0])
def test_search_by_projection_lines(lines, th):
    rng = np.random.default_rng(5)
    kl0, d0, proj, valid = _queries(lines, rng, 1.0)
    kl1, d1, lf1 = lines[1]
    kl1, d1, lf1 = kl1[:-1], d1[:-1], lf1[:-1]
    vc = rng.uniform(0.99, 1.0, len(kl0)).astype(np.float32)
    a = (kl1, lf1, d1, BOUNDS, valid, proj, vc, d0)
    nm, m = pl.LSDmatcher(0.7).SearchByProjectionLines(*a, th=th)
    onm, om = oracle.line_search_by_projection_lines(*a, th, 0.7)
    assert onm > 20 and nm == onm and np.array_equal(m, om)


def test_line_matchers_equal_the_reference_matcher_code(lines):
    """The CUDA line matchers against the REFERENCE's own LSDmatcher.cpp (compiled into oracle/_ref/libref_match.so, run on this box's
    CPU): SearchDouble and the two projection searches, same inputs, identical match lists."""
    d0, d1 = lines[0][1][:-1], lines[1][1][:-1]
    nm, m = pl.LSDmatcher(0.7).SearchDouble(d0, d1)
    rnm, rm = oracle.search_double(d0, d1, 0.7, impl="ref")
    assert rnm > 30 and nm == rnm and np.array_equal(m, rm)
    rng = np.random.default_rng(13)
    kl0, dd0, proj, valid = _queries(lines, rng, 1.5)
    kl1, dd1, lf1 = (x[:-1] for x in lines[1])
    pre = (rng.random(len(kl1)) < 0.05).astype(np.uint8)
    a = (kl1, lf1, dd1, BOUNDS, valid, proj, dd0, kl0["lineLength"], 15.0)
    nm, m = pl.LSDmatcher(0.7).SearchByProjectionLast(*a, preassigned=pre)
    rnm, rm = oracle.line_search_by_projection_last(*a, preassigned=pre, impl="ref")
    assert rnm > 30 and nm == rnm and np.array_equal(m, rm)
    vc = rng.uniform(0.99, 1.0, len(kl0)).astype(np.float32)
    a = (kl1, lf1, dd1, BOUNDS, valid, proj, vc, dd0)
    nm, m = pl.LSDmatcher(0.7).SearchByProjectionLines(*a, th=3.0)
    rnm, rm = oracle.line_search_by_projection_lines(*a, 3.0, 0.7, impl="ref")
    assert rnm > 20 and nm == rnm and np.array_equal(m, rm)
