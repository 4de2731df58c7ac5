"""CPU tests: the ORB oracle against the REFERENCE's own ORBextractor (src/ORBextractor.cc compiled unmodified into
oracle/_ref/libref_orb.so - oracle/Makefile target `ref`, oracle/ref_orb_wrap.cpp, oracle/shim/).

(a) committed reference outputs (tests/golden/orb_ref_*.npz, tools/gen_golden_orb_ref.py): run everywhere, no reference needed;
(b) comparison against libref_orb.so (live where it is built, elsewhere its recorded outputs, oracle/recorded.py):
    keypoints and descriptors byte-identical, pyramid levels identical, constructor tables identical;
(c) how much glibc's allocation order (the pointer tie-break of ORBextractor.cc:684) moves the result.
"""
import os
import sys
import numpy as np
import pytest
import oracle
from oracle import recorded
from plslam_b200 import synth

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
from gen_golden_orb_ref import CASES, frame  # noqa: E402

G = os.path.join(os.path.dirname(__file__), "golden")


@pytest.mark.parametrize("name", sorted(CASES))
def test_oracle_equals_committed_reference_output(name):
    g = np.load(os.path.join(G, f"orb_ref_{name}.npz"))
    w, h, seed, nf, nl = [int(v) for v in g["params"]]
    img = frame(str(g["kind"]), w, h, seed)
    assert int(img.astype(np.int64).sum()) == int(g["img_sum"])  # the generator is bit-stable
    o = oracle.OrbOracle(nf, float(g["scale_factor"]), nl, 20, 7)
    kps, desc = o.extract(img)
    assert kps.tobytes() == g["kps"].tobytes()
    assert np.array_equal(desc, g["desc"])
    t = o.tables()
    for k in ("scale", "inv_scale", "sigma2", "inv_sigma2"):
        assert t[k].tobytes() == g[k].tobytes(), k
    assert [tuple(d) for d in g["level_dims"]] == [o.level_dims(l) for l in range(nl)]
    assert [int(s) for s in g["level_sums"]] == [int(o.level(l).astype(np.int64).sum()) for l in range(nl)]


@pytest.mark.parametrize("w,h,seed,nf,sf,nl", [(640, 480, 2, 1000, 1.2, 8), (640, 480, 3, 1500, 1.2, 8), (752, 480, 7, 1000, 1.2, 8),
                                               (1241, 376, 8, 2000, 1.2, 8), (320, 240, 5, 500, 1.2, 8), (640, 480, 6, 1000, 1.5, 4),
                                               (800, 600, 12, 1200, 1.1, 8), (333, 251, 13, 300, 1.2, 6)])
def test_oracle_equals_live_reference(w, h, seed, nf, sf, nl):
    img = synth.synth_frame(w, h, seed)
    r, o = oracle.RefOrb(nf, sf, nl, 20, 7), oracle.OrbOracle(nf, sf, nl, 20, 7)
    rk, rd = r.extract(img)
    ok, od = o.extract(img)
    for l in range(nl):
        assert np.array_equal(r.level(l), o.level(l)), f"pyramid level {l}"
    assert rk.tobytes() == ok.tobytes()
    assert np.array_equal(rd, od)
    rt, ot = r.tables(), o.tables()
    for k in rt:
        assert rt[k].tobytes() == ot[k].tobytes(), k


def test_reference_sequence_and_reuse():
    # one extractor object over a warped sequence (the pyramid buffers and the arena are reused between calls)
    seq = synth.synth_sequence(5, 640, 480, seed=4)
    r, o = oracle.RefOrb(1000, 1.2, 8, 20, 7), oracle.OrbOracle(1000, 1.2, 8, 20, 7)
    for b in range(5):
        rk, rd = r.extract(seq[b])
        ok, od = o.extract(seq[b])
        assert rk.tobytes() == ok.tobytes() and np.array_equal(rd, od), b
    e, d = r.extract(np.full((480, 640), 128, np.uint8))    # no corners: empty output
    assert len(e) == 0


def test_glibc_allocation_order_only_moves_ties():
    # With malloc's own address order the pair<int, ExtractorNode*> sort breaks equal-size ties differently (the C++ program does
    # not define it): the same candidates, the same per-level quota, a handful of different picks.  Recorded, not required equal.
    img = synth.synth_frame(640, 480, 1)

    def counts():
        a, _ = oracle.RefOrb(1000, 1.2, 8, 20, 7).extract(img)
        b, _ = oracle.RefOrb(1000, 1.2, 8, 20, 7, ordered_heap=False).extract(img)
        sa, sb = {x.tobytes() for x in a}, {x.tobytes() for x in b}
        return len(a), len(b), len(sa & sb), len(sa)
    na, nb, common, nsa = recorded.call("ref_allocation_order_ties", (img,), oracle.ref_orb_available(), counts)
    assert abs(na - nb) <= 8
    assert common >= 0.95 * nsa
