"""CPU tests: the frame-glue oracle against the REFERENCE's own Frame.cc, compiled unmodified against the reference's real Frame.h into
oracle/_ref/libref_frame.so (with its ORBextractor.cc, LineExtractor.cpp, MapPoint.cc and the vendored line-descriptor sources;
oracle/ref_frame_wrap.cpp, oracle/shim_frame/).

* the monocular Frame constructor end to end (Frame.cc:193-276): undistortion map + remap, ORB on the raw image and LSD / LBD on the
  undistorted one, UndistortKeyPoints, ComputeImageBounds, AssignFeaturesToGrid / ...ForLine - every output byte-identical to the
  oracle's pipeline of the same stages;
* Frame::GetFeaturesInArea on the frame's own grid;
* Frame::isInFrustum for map points and map lines (flags, projections, predicted levels, viewing cosines)."""
import ctypes as C
import numpy as np
import pytest
import oracle
from oracle import recorded
from oracle.binding import lib, _p
from plslam_b200 import synth

NODIST = (0.0, 0.0, 0.0, 0.0, 0.0)


def _ref_in_view(name, f, *args):
    """isInFrustum of the reference -> (inview, then proj / level / viewcos of the points in view only, Ow)"""
    def run():
        r = f(*args)
        inv = r[0].astype(bool)
        return r[0], r[1][inv], r[2][inv], r[3][inv], r[4]
    return recorded.call(name, args, oracle.ref_frame_available(), run)


def _oracle_frame(img, K, D, nfeatures=1000, nlines=200, mask=None, mll=0.0):
    keys, desc = oracle.OrbOracle(nfeatures, 1.2, 8, 20, 7).extract(img)
    keysUn = oracle.undistort_keypoints(keys, K, D)
    kl, ldesc, lfunc = oracle.line_extract(oracle.undistort_remap(img, K, D), mask=mask, nfeatures=nlines, min_line_length=mll)
    bounds = oracle.image_bounds(K, D, img.shape[1], img.shape[0])
    return dict(keys=keys, keysUn=keysUn, desc=desc, keylines=kl, ldesc=ldesc, lfunc=lfunc, bounds=bounds, grid=oracle.assign_grid(keysUn, bounds),
                line_grid=oracle.assign_grid_lines(kl, bounds))


@pytest.mark.parametrize("w,h,seed,K,D,nf", [(640, 480, 1, synth.TUM1_K, synth.TUM1_DIST, 1000), (640, 480, 4, synth.TUM1_K, synth.TUM1_DIST, 2000),
                                             (752, 480, 5, synth.EUROC_K, synth.EUROC_DIST, 1000), (640, 480, 2, synth.TUM1_K, NODIST, 1000),
                                             (1241, 376, 4, (718.856, 718.856, 607.1928, 185.2157), NODIST, 2000)])
def test_frame_constructor_end_to_end(w, h, seed, K, D, nf):
    img = synth.synth_frame(w, h, seed)
    F = oracle.ref_frame_construct(img, K, D, nfeatures=nf)
    O = _oracle_frame(img, K, D, nfeatures=nf)
    assert len(F["keys"]) > 500 and len(F["keylines"]) == 201
    for k in ("keys", "keysUn", "keylines"):
        assert F[k].tobytes() == O[k].tobytes(), k
    assert np.array_equal(F["desc"], O["desc"]) and np.array_equal(F["ldesc"], O["ldesc"])
    assert F["lfunc"].tobytes() == O["lfunc"].tobytes()
    assert F["bounds"].tobytes() == O["bounds"].tobytes()
    for g in ("grid", "line_grid"):
        assert np.array_equal(F[g][0], O[g][0]) and np.array_equal(F[g][1], O[g][1]), g


def test_frame_constructor_with_mask():
    img = synth.synth_frame(640, 480, 4)     # (seed 6 has two lines of equal response, which the reference's unstable std::sort swaps)
    mask = np.zeros((480, 640), np.uint8); mask[14:465, 14:625] = 255        # masks/mask.png geometry
    F = oracle.ref_frame_construct(img, synth.TUM1_K, synth.TUM1_DIST, mask=mask)
    O = _oracle_frame(img, synth.TUM1_K, synth.TUM1_DIST, mask=mask)
    assert F["keylines"].tobytes() == O["keylines"].tobytes() and np.array_equal(F["ldesc"], O["ldesc"])
    assert np.array_equal(F["line_grid"][1], O["line_grid"][1])


def test_get_features_in_area():
    img = synth.synth_frame(640, 480, 3)
    F = oracle.ref_frame_construct(img, synth.TUM1_K, synth.TUM1_DIST)
    O = _oracle_frame(img, synth.TUM1_K, synth.TUM1_DIST)
    assert O["keysUn"].tobytes() == F["keysUn"].tobytes() and O["bounds"].tobytes() == F["bounds"].tobytes()
    keysUn, b = O["keysUn"], O["bounds"]        # the frame's own keypoints and bounds (identical bytes)
    rng = np.random.default_rng(0)
    f = lib().oracle_features_in_area
    f.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_float, C.c_float, C.c_float, C.c_int, C.c_int, C.c_void_p]
    out = np.zeros(len(keysUn), np.int32)
    for _ in range(400):
        x, y = float(rng.uniform(-40, 680)), float(rng.uniform(-40, 520))
        r = float(rng.choice([5.0, 15.0, 40.0, 100.0, 700.0]))
        lo, hi = [(-1, -1), (0, 0), (2, 4), (0, 7), (3, -1), (1, 1)][int(rng.integers(0, 6))]
        n = f(_p(keysUn), len(keysUn), _p(b), np.float32(x), np.float32(y), np.float32(r), lo, hi, _p(out))
        want = oracle.ref_frame_features_in_area(np.float32(x), np.float32(y), np.float32(r), lo, hi)
        assert n == len(want) and np.array_equal(out[:n], want), (x, y, r, lo, hi)


@pytest.mark.parametrize("seed,cosl", [(7, 0.5), (8, 0.5), (9, 0.0), (10, 0.9)])
def test_is_in_frustum_points(seed, cosl):
    v = synth.synth_map_view(seed, 6000)
    b = oracle.image_bounds(synth.TUM1_K, synth.TUM1_DIST, 640, 480)
    log_sf = float(np.float32(np.log(np.float32(1.2))))
    ref = _ref_in_view("ref_in_view_points", oracle.ref_frame_is_in_frustum_points, v["Tcw"], synth.TUM1_K, b, log_sf, 8, cosl, v["pos"], v["normal"],
                       v["min_dist"], v["max_dist"])
    got = oracle.is_in_frustum_points(v["Tcw"], ref[4], synth.TUM1_K, b, log_sf, 8, cosl, v["pos"], v["normal"], v["min_dist"], v["max_dist"])
    assert got[0].sum() > 100 and np.array_equal(got[0], ref[0])
    inv = got[0].astype(bool)
    assert got[1][inv].tobytes() == ref[1].tobytes() and np.array_equal(got[2][inv], ref[2]) and got[3][inv].tobytes() == ref[3].tobytes()
    # the camera centre the frame derives is the fp32 gemm of -Rcw^T tcw; the synthetic Ow agrees to an ulp or so
    assert np.allclose(ref[4], v["Ow"], rtol=0, atol=1e-5)


@pytest.mark.parametrize("seed,cosl", [(9, 0.5), (11, 0.5), (12, 0.0)])
def test_is_in_frustum_lines(seed, cosl):
    v = synth.synth_map_view(seed, 5000, lines=True)
    if seed == 11:
        v["min_dist"] = (v["max_dist"] / 1.2 ** 12).astype(np.float32)
    b = oracle.image_bounds(synth.TUM1_K, synth.TUM1_DIST, 640, 480)
    log_sf = float(np.float32(np.log(np.float32(1.2))))
    ref = _ref_in_view("ref_in_view_lines", oracle.ref_frame_is_in_frustum_lines, v["Tcw"], synth.TUM1_K, b, log_sf, cosl, v["pos"], v["normal"],
                       v["min_dist"], v["max_dist"])
    got = oracle.is_in_frustum_lines(v["Tcw"], ref[4], synth.TUM1_K, b, log_sf, cosl, v["pos"], v["normal"], v["min_dist"], v["max_dist"])
    assert got[0].sum() > 50 and np.array_equal(got[0], ref[0])
    inv = got[0].astype(bool)
    assert got[1][inv].tobytes() == ref[1].tobytes() and np.array_equal(got[2][inv], ref[2]) and got[3][inv].tobytes() == ref[3].tobytes()
