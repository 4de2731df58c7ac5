"""GPU parity tests: ORB extraction through the C ABI vs the CPU oracle — bit-exact (SURVEY.md §8d)."""
import os
import numpy as np
import pytest
import oracle
import plslam_b200 as pl
from plslam_b200 import synth

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(__file__), "golden")


def _assert_same(kps, desc, okps, odesc):
    assert len(kps) == len(okps)
    for f in ("x", "y", "size", "angle", "response", "octave", "class_id"):
        assert np.array_equal(kps[f], okps[f]), f
    assert np.array_equal(desc, odesc)


@pytest.mark.parametrize("w,h,seed,nf", [(640, 480, 1, 1000), (640, 480, 1, 2000), (752, 480, 5, 1000),
                                         (1241, 376, 4, 2000), (640, 480, 11, 500)])
def test_extract_matches_oracle(w, h, seed, nf):
    img = synth.synth_frame(w, h, seed)
    ex = pl.ORBextractor(nf, 1.2, 8, 20, 7, width=w, height=h)
    kps, desc = ex(img)
    o = oracle.OrbOracle(nf, 1.2, 8, 20, 7)
    okps, odesc = o.extract(img)
    # stage taps first so a failure names the stage
    for l in range(8):
        assert np.array_equal(ex.mvImagePyramid(l), o.level(l)), f"pyramid level {l}"
        c, oc = ex.debug_candidates(l), o.candidates(l)
        assert len(c) == len(oc), f"candidate count level {l}"
        for f in ("x", "y", "response"):
            assert np.array_equal(c[f], oc[f]), f"candidates {f} level {l}"
    assert np.array_equal(ex.mvImagePyramid(2, with_border=True), o.level(2, True))
    _assert_same(kps, desc, okps, odesc)


@pytest.mark.parametrize("name", ["640x480_n1000", "1241x376_n2000"])
def test_extract_matches_committed_golden(name):
    g = np.load(os.path.join(G, f"orb_oracle_{name}.npz"))
    w, h, seed, nf = [int(v) for v in g["params"]]
    kps, desc = pl.ORBextractor(nf, 1.2, 8, 20, 7, width=w, height=h)(synth.synth_frame(w, h, seed))
    assert kps.tobytes() == g["kps"].tobytes()
    assert np.array_equal(desc, g["desc"])


@pytest.mark.parametrize("name", ["640x480_n1000", "640x480_n2000", "752x480_n1000", "1241x376_n2000", "640x480_low",
                                  "640x480_noise", "640x480_sparse", "640x480_n500_s11"])
def test_extract_matches_reference_output(name):
    """CUDA path vs the REFERENCE's own ORBextractor.cc (compiled where it lies by oracle/Makefile `ref`; its outputs on the
    seeded frames are committed by tools/gen_golden_orb_ref.py because /root/reference does not exist on the GPU box)."""
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    from gen_golden_orb_ref import frame
    g = np.load(os.path.join(G, f"orb_ref_{name}.npz"))
    w, h, seed, nf, nl = [int(v) for v in g["params"]]
    img = frame(str(g["kind"]), w, h, seed)
    assert int(img.astype(np.int64).sum()) == int(g["img_sum"])
    ex = pl.ORBextractor(nf, float(g["scale_factor"]), nl, 20, 7, width=w, height=h, cell_slot_cap=256 if "noise" in name else 0)
    kps, desc = ex(img)
    assert kps.tobytes() == g["kps"].tobytes()
    assert np.array_equal(desc, g["desc"])
    assert ex.GetScaleFactors().tobytes() == g["scale"].tobytes() and ex.GetInverseScaleSigmaSquares().tobytes() == g["inv_sigma2"].tobytes()
    assert [tuple(d) for d in g["level_dims"]] == [ex.mvImagePyramid(l).shape[::-1] for l in range(nl)]


def test_extract_matches_live_reference_library():
    # the prebuilt reference library itself, run on the GPU box's CPU next to the CUDA path (fresh seeds, not in the fixtures)
    for w, h, seed, nf in [(640, 480, 21, 1000), (752, 480, 22, 1000), (1241, 376, 23, 2000)]:
        img = synth.synth_frame(w, h, seed)
        kps, desc = pl.ORBextractor(nf, 1.2, 8, 20, 7, width=w, height=h)(img)
        rk, rd = oracle.RefOrb(nf, 1.2, 8, 20, 7).extract(img)
        assert kps.tobytes() == rk.tobytes() and np.array_equal(desc, rd), (w, h, seed)


def test_tables_match_reference_ctor():
    ex = pl.ORBextractor(1000, 1.2, 8, 20, 7)
    t = oracle.OrbOracle(1000, 1.2, 8, 20, 7).tables()
    assert np.array_equal(ex.GetScaleFactors(), t["scale"])
    assert np.array_equal(ex.GetInverseScaleFactors(), t["inv_scale"])
    assert np.array_equal(ex.GetScaleSigmaSquares(), t["sigma2"])
    assert np.array_equal(ex.GetInverseScaleSigmaSquares(), t["inv_sigma2"])
    assert np.array_equal(ex.mnFeaturesPerLevel, t["per_level"])


def test_batch_equals_single_and_sequence():
    seq = synth.synth_sequence(6, 640, 480, seed=2)
    ex = pl.ORBextractor(1000, 1.2, 8, 20, 7, max_batch=6)
    kps, desc, n = ex.extract_batch(seq)
    o = oracle.OrbOracle(1000, 1.2, 8, 20, 7)
    for b in range(6):
        okps, odesc = o.extract(seq[b])
        _assert_same(kps[b, :n[b]], desc[b, :n[b]], okps, odesc)


def test_edge_cases():
    ex = pl.ORBextractor(1000, 1.2, 8, 20, 7)
    o = oracle.OrbOracle(1000, 1.2, 8, 20, 7)
    flat = np.full((480, 640), 128, np.uint8)              # no corners anywhere
    kps, desc = ex(flat)
    assert len(kps) == 0 and desc.shape == (0, 32)
    rng = np.random.default_rng(5)
    noise = rng.integers(0, 256, (480, 640), dtype=np.uint8)  # maximum candidate density
    ex2 = pl.ORBextractor(1000, 1.2, 8, 20, 7, cell_slot_cap=256)
    kps, desc = ex2(noise)
    _assert_same(kps, desc, *o.extract(noise))
    low = (synth.synth_frame(640, 480, 9) // 16 + 100).astype(np.uint8)  # only the minThFAST fallback fires
    kps, desc = ex(low)
    _assert_same(kps, desc, *o.extract(low))
    sparse = np.full((480, 640), 90, np.uint8); sparse[200:230, 300:340] = 200   # fewer candidates than quota
    kps, desc = ex(sparse)
    _assert_same(kps, desc, *o.extract(sparse))
    e, d = ex(np.zeros((0, 0), np.uint8))                   # empty image -> silent empty return (ORBextractor.cc:1046)
    assert len(e) == 0


def test_slot_capacity_overflow_is_loud():
    rng = np.random.default_rng(5)
    noise = rng.integers(0, 256, (480, 640), dtype=np.uint8)
    ex = pl.ORBextractor(1000, 1.2, 8, 20, 7, cell_slot_cap=8)
    with pytest.raises(pl.PLError, match="cell_slot_cap"):
        ex(noise)
