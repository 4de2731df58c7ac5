"""GPU parity tests: LSD + LBD line extraction through the C ABI vs the CPU oracle.
Everything is compared BYTE FOR BYTE: scaled image, seed order, Sobel pair, the LSD segment list (order and fp32
coordinates: every region is grown and fitted by one lane in the oracle's own sequential fp64 order), KeyLine records,
LBD descriptors and line equations."""
import os
import numpy as np
import pytest
import oracle
from oracle import recorded
import plslam_b200 as pl
from plslam_b200 import synth

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(__file__), "golden")


def _segments_equal(a, b):
    a = np.asarray(a, np.float32).reshape(-1, 4); b = np.asarray(b, np.float32).reshape(-1, 4)
    assert a.shape == b.shape, (a.shape, b.shape)
    assert a.tobytes() == b.tobytes(), "segment lists differ: first row %d" % int(np.nonzero((a != b).any(1))[0][0])


@pytest.mark.parametrize("spec_maxb", [0, 4])
@pytest.mark.parametrize("w,h,seed", [(640, 480, 1), (640, 480, 2), (752, 480, 5), (1241, 376, 4)])
def test_stages_match_oracle(monkeypatch, w, h, seed, spec_maxb):
    monkeypatch.setenv("PLSLAM_LSD_GROW_SPEC_MAXB", str(spec_maxb))     # 0: ordered kernel, 4: speculative kernel
    img = synth.synth_frame(w, h, seed)
    ex = pl.LINEextractor(1, 1.2, 200, 0.0, width=w, height=h)
    kl, desc, lf = ex(img)
    sc, mg, an = oracle.lsd_stages(img)
    assert np.array_equal(ex.debug_scaled(), sc), "blur + 0.8x resize"
    # seed order: defined pixels, magnitude bin descending, row-major inside a bin
    order = ex.debug_order()
    defined = (an != -1024.0)
    assert len(order) == defined.sum()
    mgf = mg.ravel(); bins = (mgf * (1023.0 / mgf[defined.ravel()].max())).astype(np.int64)
    idx = np.nonzero(defined.ravel())[0]
    ref_order = idx[np.argsort(-bins[idx], kind="stable")]
    assert np.array_equal(order, ref_order.astype(np.uint32)), "seed order"
    dx, dy = ex.debug_sobel()
    odx, ody = oracle.lbd_sobel(img)
    assert np.array_equal(dx, odx) and np.array_equal(dy, ody), "LBD Sobel pair"
    _segments_equal(ex.debug_segments(), oracle.lsd_detect(img))
    okl, odesc, olf = oracle.line_extract(img)
    assert len(kl) == len(okl)
    assert kl.tobytes() == okl.tobytes(), "KeyLine records"
    assert np.array_equal(desc, odesc), "LBD descriptors"
    assert lf.tobytes() == olf.tobytes(), "line equations"


@pytest.mark.parametrize("name", ["640x480_s1", "640x480_s2", "752x480_s5", "1241x376_s4"])
def test_extract_matches_reference_output(name):
    """CUDA path vs the reference tree's OWN line-descriptor sources (LSDDetector_custom.cpp KeyLines + binary_descriptor_custom.cpp
    LBD, compiled where they lie by oracle/Makefile `ref`; outputs committed by tools/gen_golden_line_ref.py because /root/reference
    does not exist on the GPU box): KeyLine records (libm's atan2f angle included) and LBD bytes identical."""
    g = np.load(os.path.join(G, f"line_ref_{name}.npz"))
    w, h, seed, nf = [int(v) for v in g["params"]]
    img = synth.synth_frame(w, h, seed)
    assert int(img.astype(np.int64).sum()) == int(g["img_sum"])
    kl, desc, lf = pl.LINEextractor(1, 1.2, nf, 0.0, width=w, height=h)(img)
    assert kl.tobytes() == g["top"].tobytes(), "KeyLine records vs the reference's"
    assert np.array_equal(desc, g["desc"]), "LBD descriptors vs the reference's"
    # every KeyLine of the frame, not only the selection: ask for more lines than there are (one zero record is appended then)
    n_all = len(g["keylines"])
    kl2, _, _ = pl.LINEextractor(1, 1.2, n_all + 10, 0.0, width=w, height=h)(img)
    order = np.argsort(-g["keylines"]["response"], kind="stable")
    want = g["keylines"][order].copy(); want["class_id"] = np.arange(n_all)
    assert len(kl2) == n_all + 1 and kl2[:-1].tobytes() == want.tobytes(), "all KeyLines of the frame vs the reference's"


def test_extract_matches_live_reference_library():
    # the prebuilt reference library itself on the GPU box's CPU (fresh seeds, not in the fixtures): the CUDA KeyLines through the
    # reference's LBD, and the reference's KeyLines against the CUDA ones
    for w, h, seed in [(640, 480, 31), (752, 480, 32)]:
        img = synth.synth_frame(w, h, seed)
        kl, desc, lf = pl.LINEextractor(1, 1.2, 200, 0.0, width=w, height=h)(img)

        def top_keylines():
            rk = oracle.ref_lsd_keylines(img)
            order = np.argsort(-rk["response"], kind="stable")
            want = rk[order][:201].copy(); want["class_id"] = np.arange(201)
            return want
        want = recorded.call("ref_top_keylines", (img, 200), oracle.ref_line_available(), top_keylines)
        assert kl.tobytes() == want.tobytes(), (w, h, seed)
        assert np.array_equal(desc, oracle.ref_lbd_compute(img, want)), (w, h, seed)


def test_lbd_given_oracle_keylines_is_bit_exact():
    """Descriptor stage alone: feed identical frames; every line whose record matches must have identical 32 bytes."""
    img = synth.synth_frame(640, 480, 7)
    ex = pl.LINEextractor(1, 1.2, 500, 0.0)
    kl, desc, lf = ex(img)
    okl, odesc, olf = oracle.line_extract(img, nfeatures=500)
    assert len(kl) == len(okl) and kl.tobytes() == okl.tobytes()
    assert np.array_equal(desc, odesc)
    assert lf.tobytes() == olf.tobytes()


def test_quirks_mask_batch_and_edge_cases():
    img = synth.synth_frame(640, 480, 1)
    n_seg = len(oracle.lsd_detect(img))
    ex = pl.LINEextractor(1, 1.2, n_seg + 50, 0.0)            # size <= nFeatures: one zero KeyLine appended
    kl, desc, lf = ex(img)
    assert len(kl) == n_seg + 1 and kl[-1]["lineLength"] == 0 and not desc[-1].any() and np.isnan(lf[-1]).all()
    mask = np.zeros((480, 640), np.uint8); mask[14:465, 14:625] = 255   # masks/mask.png geometry (SURVEY.md §2 row 19)
    ex2 = pl.LINEextractor(1, 1.2, 200, 0.0)
    kl, desc, lf = ex2(img, mask)
    okl, odesc, olf = oracle.line_extract(img, mask=mask)
    assert len(kl) == len(okl) and kl.tobytes() == okl.tobytes() and np.array_equal(desc, odesc)
    with pytest.raises(pl.PLError, match="Mask error"):
        ex2(img, np.zeros((10, 10), np.uint8))
    flat = np.full((480, 640), 77, np.uint8)                   # no gradients -> no segments -> 1 zero KeyLine
    kl, desc, lf = ex2(flat)
    okl, odesc, olf = oracle.line_extract(flat)
    assert len(kl) == len(okl) == 1 and kl.tobytes() == okl.tobytes()
    ex3 = pl.LINEextractor(1, 1.2, 200, 30.0)                  # min_line_length cut
    kl, _, _ = ex3(img); okl, _, _ = oracle.line_extract(img, min_line_length=30.0)
    assert len(kl) == len(okl) and kl.tobytes() == okl.tobytes()
    seq = synth.synth_sequence(4, 640, 480, seed=3)            # batch == single
    exb = pl.LINEextractor(1, 1.2, 200, 0.0, max_batch=4)
    klb, descb, lfb, nb = exb.extract_batch(seq)
    for b in range(4):
        k1, d1, l1 = ex2(seq[b])
        assert nb[b] == len(k1) and klb[b, :nb[b]].tobytes() == k1.tobytes() and np.array_equal(descb[b, :nb[b]], d1)


def test_committed_golden():
    g = np.load(os.path.join(G, "line_oracle_640x480_s1.npz"))
    kl, desc, lf = pl.LINEextractor(1, 1.2, 200, 0.0)(synth.synth_frame(640, 480, 1))
    assert len(kl) == len(g["kl"]) and kl.tobytes() == g["kl"].tobytes() and np.array_equal(desc, g["desc"])
    seg = np.load(os.path.join(G, "lsd_cv2_640x480_s1.npz"))["segments"]      # straight against cv2's own output
    _segments_equal(_last_segments(), seg)


def _last_segments():
    ex = pl.LINEextractor(1, 1.2, 200, 0.0)
    ex(synth.synth_frame(640, 480, 1))
    return ex.debug_segments()


@pytest.mark.parametrize("warps,wpf", [(1, 1), (4, 4), (64, 64), (2368, 64), (2368, 256)])
def test_grow_warps_per_frame_do_not_change_the_result(monkeypatch, warps, wpf):
    """The speculative region growing must give the sequential result whatever the number of warps (= regions in flight)
    serving a frame: 1 warp (32 tasks in flight) ... 256 warps (8192 tasks in flight, heavy stealing / re-execution)."""
    monkeypatch.setenv("PLSLAM_LSD_GROW_SPEC_MAXB", "64")        # the speculative kernel (the default is the ordered one)
    monkeypatch.setenv("PLSLAM_LSD_GROW_WARPS", str(warps))
    monkeypatch.setenv("PLSLAM_LSD_GROW_WPF", str(wpf))
    K, D = synth.TUM1_K, synth.TUM1_DIST
    img = oracle.undistort_remap(synth.synth_sequence(2, 640, 480, seed=1)[1], K, D)
    ex = pl.LINEextractor(1, 1.2, 200, 0.0)
    for rep in range(3):                     # the interleaving differs from run to run; the result must not
        kl, desc, lf = ex(img)
        _segments_equal(ex.debug_segments(), oracle.lsd_detect(img))
    okl, odesc, olf = oracle.line_extract(img)
    assert kl.tobytes() == okl.tobytes() and np.array_equal(desc, odesc)


@pytest.mark.parametrize("spec_maxb", [0, 64])
def test_grow_batches_of_odd_sizes(monkeypatch, spec_maxb):
    """Batches that do not divide the warp budget: 3 and 37 frames, each frame against the oracle (both growing kernels)."""
    monkeypatch.setenv("PLSLAM_LSD_GROW_SPEC_MAXB", str(spec_maxb))
    seq = synth.synth_sequence(37, 640, 480, seed=5)
    ex = pl.LINEextractor(1, 1.2, 200, 0.0, max_batch=37)
    for B in (3, 37):
        klb, descb, lfb, nb = ex.extract_batch(seq[:B])
        for b in range(0, B, 4):
            okl, odesc, olf = oracle.line_extract(seq[b])
            assert nb[b] == len(okl) and klb[b, :nb[b]].tobytes() == okl.tobytes() and np.array_equal(descb[b, :nb[b]], odesc), (B, b)


@pytest.mark.parametrize("spec_maxb", [0, 4])
def test_grow_degenerate_frames(monkeypatch, spec_maxb):
    """No gradient at all, pure noise (thousands of tiny regions), one long edge across the frame (one huge region);
    through both region-growing kernels (0: ordered one-warp-per-frame kernel, 4: speculative kernel for a single frame)."""
    monkeypatch.setenv("PLSLAM_LSD_GROW_SPEC_MAXB", str(spec_maxb))
    rng = np.random.Generator(np.random.PCG64(11))
    flat = np.full((480, 640), 128, np.uint8)
    noise = rng.integers(0, 256, (480, 640), dtype=np.uint8)
    edge = np.zeros((480, 640), np.uint8); edge[:, 320:] = 255
    stripes = ((np.arange(640)[None, :] // 6 + np.arange(480)[:, None] // 50) % 2 * 200 + 20).astype(np.uint8)
    ex = pl.LINEextractor(1, 1.2, 200, 0.0)
    for name, img in (("flat", flat), ("noise", noise), ("edge", edge), ("stripes", stripes)):
        kl, desc, lf = ex(img)
        _segments_equal(ex.debug_segments(), oracle.lsd_detect(img))
        okl, odesc, olf = oracle.line_extract(img)
        assert kl.tobytes() == okl.tobytes() and np.array_equal(desc, odesc), name
