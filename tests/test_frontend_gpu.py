"""GPU test of the batch front-end (the bench "step" and e2e entry point): every per-frame result equals what the CPU
oracle produces for the same frame / frame pair / pose problem."""
import numpy as np
import pytest
import oracle
import plslam_b200 as pl
from plslam_b200 import synth

pytestmark = pytest.mark.gpu


def test_frontend_batch_matches_oracle():
    B = 4
    frames = synth.synth_sequence(B, 640, 480, seed=4)
    problems = [synth.synth_pose_problem(50 + k) for k in range(B)]
    fe = pl.Frontend(640, 480, max_batch=B, lm_caps=(320, 88))
    fe.set_wrap(True)                 # frame 0 against frame B-1 of the same batch (closed loop)
    fe.set_pose_problems(problems)
    out = fe.run(frames)
    o = oracle.OrbOracle(1000, 1.2, 8, 20, 7)
    feats = []
    for b in range(B):
        okps, odesc = o.extract(frames[b])
        okl, oldesc, olf = oracle.line_extract(frames[b])
        n, nl = out["n"][b], out["nl"][b]
        assert n == len(okps) and out["kps"][b, :n].tobytes() == okps.tobytes() and np.array_equal(out["desc"][b, :n], odesc)
        assert nl == len(okl)
        assert out["keylines"][b, :nl].tobytes() == okl.tobytes() and np.array_equal(out["ldesc"][b, :nl], oldesc)
        feats.append((okps, odesc, oldesc, True))
    for b in range(B):
        pk, pd, pld, _ = feats[(b - 1) % B]
        ck, cd, cld, _ = feats[b]
        pm = np.stack([pk["x"], pk["y"]], 1).astype(np.float32)
        onm, om, _ = oracle.search_for_initialization(pk, pd, ck, cd, [0, 0, 640, 480], pm, 100, 0.9, True)
        assert out["n_pt_matches"][b] == onm and np.array_equal(out["pt_matches"][b, :len(pk)], om)
        onl, olm = oracle.search_double(pld, cld, 0.7)     # the oracle's own descriptors on both sides
        assert out["n_line_matches"][b] == onl and np.array_equal(out["line_matches"][b, :len(pld)], olm)
        p = problems[b]
        on, oT, opo, olo, oits = oracle.pose_optimization(0, p["Tcw0"], p["K"], p["pt_obs"], p["pt_inv_sigma2"], p["pt_Xw"],
                                                          p["line_func"], p["line_Xw"])
        for call in range(2):
            T = out["poses"][call, b].reshape(4, 4)
            assert np.linalg.norm(T[:3, 3] - oT[:3, 3]) <= 1e-4 * np.linalg.norm(oT[:3, 3])
            assert out["inliers"][call, b] == on
    # the device-resident path gives the same results as the host-buffer path
    import torch
    d = torch.from_numpy(frames).cuda()
    fe.run_dev(d.data_ptr(), 640, 640 * 480, B, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    dev = fe.fetch(B)
    for k in ("kps", "desc", "n", "keylines", "ldesc", "nl", "pt_matches", "n_pt_matches", "line_matches", "n_line_matches", "poses", "inliers"):
        assert dev[k].tobytes() == out[k].tobytes(), k


def test_frontend_with_distorting_camera():
    """TUM1 camera (k1 != 0): ORB on the raw frame, LSD/LBD on the undistorted frame (Frame.cc:220-225), matching on
    mvKeysUn inside ComputeImageBounds' grid (Frame.cc:233, :947-985)."""
    B = 3
    K, D = synth.TUM1_K, synth.TUM1_DIST
    frames = synth.synth_sequence(B, 640, 480, seed=6)
    problems = [synth.synth_pose_problem(70 + k) for k in range(B)]
    fe = pl.Frontend(640, 480, max_batch=B, lm_caps=(320, 88))
    fe.set_wrap(True)
    fe.set_pose_problems(problems)
    fe.set_camera(K, D)
    out = fe.run(frames)
    ku = fe.fetch_keys_un(B)
    bounds = oracle.image_bounds(K, D, 640, 480)
    o = oracle.OrbOracle(1000, 1.2, 8, 20, 7)
    feats = []
    for b in range(B):
        okps, odesc = o.extract(frames[b])
        n, nl = out["n"][b], out["nl"][b]
        assert n == len(okps) and out["kps"][b, :n].tobytes() == okps.tobytes() and np.array_equal(out["desc"][b, :n], odesc)
        oku = oracle.undistort_keypoints(okps, K, D)
        assert ku[b, :n].tobytes() == oku.tobytes()
        okl, oldesc, olf = oracle.line_extract(oracle.undistort_remap(frames[b], K, D))
        assert nl == len(okl)
        assert out["keylines"][b, :nl].tobytes() == okl.tobytes() and np.array_equal(out["ldesc"][b, :nl], oldesc)
        feats.append((oku, odesc))
    for b in range(B):
        pk, pd = feats[(b - 1) % B]
        ck, cd = feats[b]
        pm = np.stack([pk["x"], pk["y"]], 1).astype(np.float32)
        onm, om, _ = oracle.search_for_initialization(pk, pd, ck, cd, bounds, pm, 100, 0.9, True)
        assert out["n_pt_matches"][b] == onm and np.array_equal(out["pt_matches"][b, :len(pk)], om)
    # a camera without distortion is the default path
    fe.set_camera(K, (0, 0, 0, 0, 0))
    out0 = fe.run(frames)
    ref = pl.Frontend(640, 480, max_batch=B, lm_caps=(320, 88)); ref.set_wrap(True); ref.set_pose_problems(problems)
    out1 = ref.run(frames)
    for k in ("kps", "desc", "n", "keylines", "ldesc", "nl", "pt_matches", "n_pt_matches", "line_matches", "n_line_matches"):
        assert out0[k].tobytes() == out1[k].tobytes(), k
    assert fe.fetch_keys_un(B).tobytes() == out0["kps"].tobytes()


def test_frontend_streaming_submit_wait():
    """pl_frontend_submit / pl_frontend_wait (H2D, kernels, D2H of consecutive steps overlapped) return, for every step,
    exactly what the synchronous pl_frontend_run returns for that step's frames."""
    import torch
    B = 3
    seqs = [synth.synth_sequence(B, 640, 480, seed=s) for s in (4, 5, 6, 7)]
    problems = [synth.synth_pose_problem(60 + k) for k in range(B)]
    def make():
        f = pl.Frontend(640, 480, max_batch=B, lm_caps=(320, 88)); f.set_pose_problems(problems)
        f.set_camera(synth.TUM1_K, synth.TUM1_DIST)
        return f
    ref = make()      # same call history on a second handle (entries beyond the per-frame counts keep earlier contents)
    want = [{k: v.copy() for k, v in ref.run(s).items()} for s in seqs]
    fe = make()
    pins = []
    for s in seqs:
        t = torch.empty(s.shape, dtype=torch.uint8, pin_memory=True); t.numpy()[:] = s; pins.append(t)
    outs = [fe.alloc_outputs(B, pinned=True) for _ in range(2)]
    got = []
    for i, p in enumerate(pins):
        fe.submit(p.numpy(), outs[i & 1])
        fe.wait(1)
        if i >= 1:
            got.append({k: outs[(i - 1) & 1][k].copy() for k in pl.Frontend.ORDER})
    fe.wait(0)
    got.append({k: outs[(len(pins) - 1) & 1][k].copy() for k in pl.Frontend.ORDER})
    for w, g in zip(want, got):
        for k in pl.Frontend.ORDER:
            assert w[k].tobytes() == g[k].tobytes(), k


def test_frontend_large_batch_properties():
    """Size-independent properties at a batch that fills the GPU with one warp per frame (96 frames = 32 copies of a 3-frame
    cycle): every frame's results depend only on the frame and its predecessor, so each copy must reproduce the 3-frame run
    bit for bit; keylines come out ordered by response; match lists are injective."""
    B0, R = 3, 32
    base = synth.synth_sequence(B0, 640, 480, seed=8)
    problems = [synth.synth_pose_problem(80 + k) for k in range(B0)]
    small = pl.Frontend(640, 480, max_batch=B0, lm_caps=(320, 88)); small.set_wrap(True); small.set_pose_problems(problems)
    small.set_camera(synth.TUM1_K, synth.TUM1_DIST)
    ref = small.run(base)
    big = pl.Frontend(640, 480, max_batch=B0 * R, lm_caps=(320, 88)); big.set_wrap(True); big.set_pose_problems(problems * R)
    big.set_camera(synth.TUM1_K, synth.TUM1_DIST)
    out = big.run(np.tile(base, (R, 1, 1)))
    for r in range(R):
        for b in range(B0):
            i = r * B0 + b
            n, nl = ref["n"][b], ref["nl"][b]
            assert out["n"][i] == n and out["nl"][i] == nl
            assert out["kps"][i, :n].tobytes() == ref["kps"][b, :n].tobytes() and np.array_equal(out["desc"][i, :n], ref["desc"][b, :n])
            assert out["keylines"][i, :nl].tobytes() == ref["keylines"][b, :nl].tobytes()
            assert np.array_equal(out["ldesc"][i, :nl], ref["ldesc"][b, :nl])
            npv = ref["n"][(b - 1) % B0]
            assert out["n_pt_matches"][i] == ref["n_pt_matches"][b] and np.array_equal(out["pt_matches"][i, :npv], ref["pt_matches"][b, :npv])
            nlp = ref["nl"][(b - 1) % B0]
            assert out["n_line_matches"][i] == ref["n_line_matches"][b]
            assert np.array_equal(out["line_matches"][i, :nlp], ref["line_matches"][b, :nlp])
            assert np.array_equal(out["poses"][:, i], ref["poses"][:, b]) and np.array_equal(out["inliers"][:, i], ref["inliers"][:, b])
    for i in range(0, B0 * R, 7):
        nl = out["nl"][i]
        resp = out["keylines"][i, :nl]["response"]
        resp = resp[resp > 0]                                    # the reference's zero KeyLine (nfeatures+1 quirk) has response 0
        assert len(resp) >= 100 and (np.diff(resp) <= 0).all()
        prev = (i - 1) % (B0 * R)
        m = out["pt_matches"][i, :out["n"][prev]]; m = m[m >= 0]           # entries past the predecessor's count are not written
        assert len(m) == out["n_pt_matches"][i] and len(np.unique(m)) == len(m)
        lm = out["line_matches"][i, :out["nl"][prev]]; lm = lm[lm >= 0]
        assert len(lm) == out["n_line_matches"][i] and len(np.unique(lm)) == len(lm)


def test_frontend_batch_with_featureless_frame():
    """A flat frame inside a batch: zero keypoints, the reference's single zero KeyLine, no matches on either side of it; the
    neighbouring frames are unaffected (frame independence)."""
    base = synth.synth_sequence(2, 640, 480, seed=12)
    frames = np.stack([base[0], np.full((480, 640), 93, np.uint8), base[1]])
    problems = [synth.synth_pose_problem(120 + k) for k in range(3)]
    fe = pl.Frontend(640, 480, max_batch=3, lm_caps=(320, 88)); fe.set_wrap(True); fe.set_pose_problems(problems)
    out = fe.run(frames)
    o = oracle.OrbOracle(1000, 1.2, 8, 20, 7)
    assert out["n"][1] == 0 and out["nl"][1] == 1 and not out["keylines"][1, 0].tobytes().strip(b"\0")
    for b in (0, 2):
        okps, odesc = o.extract(frames[b])
        n = out["n"][b]
        assert n == len(okps) and out["kps"][b, :n].tobytes() == okps.tobytes() and np.array_equal(out["desc"][b, :n], odesc)
    assert out["n_pt_matches"][1] == 0 and out["n_pt_matches"][2] == 0          # into / out of the empty frame
    assert out["n_line_matches"][1] == 0 and out["n_line_matches"][2] == 0
    # frame 0 is matched against frame 2 (the batch's last frame): same as a two-frame run of (frame 2, frame 0)
    k2, d2 = o.extract(frames[2]); k0, d0 = o.extract(frames[0])
    pm = np.stack([k2["x"], k2["y"]], 1).astype(np.float32)
    onm, om, _ = oracle.search_for_initialization(k2, d2, k0, d0, [0, 0, 640, 480], pm, 100, 0.9, True)
    assert out["n_pt_matches"][0] == onm and np.array_equal(out["pt_matches"][0, :len(k2)], om)
    for b in range(3):
        p = problems[b]
        on, oT, *_ = oracle.pose_optimization(0, p["Tcw0"], p["K"], p["pt_obs"], p["pt_inv_sigma2"], p["pt_Xw"], p["line_func"], p["line_Xw"])
        assert out["inliers"][0, b] == on


def test_frontend_consecutive_steps_are_one_sequence():
    """Default (no wrap): the steps are consecutive batches of ONE sequence - frame 0 of a step is matched against the last
    frame of the previous step, and the very first frame has no predecessor (no matches, PL_OK)."""
    B = 2
    seq = synth.synth_sequence(2 * B, 640, 480, seed=9)
    problems = [synth.synth_pose_problem(90 + k) for k in range(B)]
    fe = pl.Frontend(640, 480, max_batch=B, lm_caps=(320, 88)); fe.set_pose_problems(problems)
    o = oracle.OrbOracle(1000, 1.2, 8, 20, 7)
    feats = [o.extract(f) for f in seq]
    lfeat = [oracle.line_extract(f)[1] for f in seq]
    outs = [{k: v.copy() for k, v in fe.run(seq[s * B:(s + 1) * B]).items()} for s in range(2)]
    assert outs[0]["n_pt_matches"][0] == 0 and outs[0]["n_line_matches"][0] == 0
    for s in range(2):
        for b in range(B):
            g = s * B + b
            if g == 0:
                continue
            pk, pd = feats[g - 1]; ck, cd = feats[g]
            pm = np.stack([pk["x"], pk["y"]], 1).astype(np.float32)
            onm, om, _ = oracle.search_for_initialization(pk, pd, ck, cd, [0, 0, 640, 480], pm, 100, 0.9, True)
            assert outs[s]["n_pt_matches"][b] == onm and np.array_equal(outs[s]["pt_matches"][b, :len(pk)], om), (s, b)
            onl, olm = oracle.search_double(lfeat[g - 1], lfeat[g], 0.7)
            assert outs[s]["n_line_matches"][b] == onl and np.array_equal(outs[s]["line_matches"][b, :len(lfeat[g - 1])], olm), (s, b)


def test_tracking_stage_matches_oracle():
    """The steady-state projection searches of the step (Tracking.cc:1345-1357, :1799, :1855) on the previous frame's features as
    the map: each search equals the CPU oracle's on the same inputs, including the 2 x th retry for frames under 20 matches."""
    B = 4
    frames = synth.synth_sequence(B, 640, 480, seed=9).copy()
    frames[2] = 127                                            # featureless: frame 3 has an empty map -> 0 matches -> retry path
    problems = [synth.synth_pose_problem(80 + k) for k in range(B)]
    for p in problems[1:]:
        p["K"] = problems[0]["K"]                              # one camera
    fe = pl.Frontend(640, 480, max_batch=B, lm_caps=(320, 88))
    fe.set_wrap(True)
    fe.set_pose_problems(problems)
    fe.set_tracking(True)
    out = fe.run(frames)
    t0, t1 = fe.fetch_tracking(B, 0), fe.fetch_tracking(B, 1)
    K = np.asarray(problems[0]["K"], np.float32)
    sf = np.cumprod(np.r_[np.float32(1), np.full(7, np.float32(1.2))]).astype(np.float32)
    bounds = [0, 0, 640, 480]
    retried = 0
    for b in range(B):
        a = (b - 1) % B
        n, npv, nl, nlp = out["n"][b], out["n"][a], out["nl"][b], out["nl"][a]
        ck, cd, pk, pd = out["kps"][b, :n], out["desc"][b, :n], out["kps"][a, :npv], out["desc"][a, :npv]
        T = np.asarray(problems[b]["Tcw0"], np.float32).reshape(4, 4)
        pos = t0["map_pos"][b, :npv]
        assert np.array_equal(t0["pt_in_view"][b], (np.arange(fe.capK) < npv).astype(np.uint8))
        if npv:                                                 # the synthetic map point projects back onto the previous keypoint
            Xc = pos.astype(np.float64) @ T[:3, :3].T.astype(np.float64) + T[:3, 3]
            uv = np.stack([Xc[:, 0] / Xc[:, 2] * K[0] + K[2], Xc[:, 1] / Xc[:, 2] * K[1] + K[3]], 1)
            assert np.abs(uv - np.stack([pk["x"], pk["y"]], 1)).max() < 2e-2 and Xc[:, 2].min() > 1.0
        valid = np.ones(npv, np.uint8)
        nm, m = oracle.search_by_projection_last(ck, cd, bounds, T, K, sf, valid, pos, pd, pk["octave"], pk["angle"], 15.0, True)
        if nm < 20:
            retried += 1
            nm, m = oracle.search_by_projection_last(ck, cd, bounds, T, K, sf, valid, pos, pd, pk["octave"], pk["angle"], 30.0, True)
        assert t0["n_pt"][b] == nm and np.array_equal(t0["pt_match"][b, :n], m)
        view = valid.copy(); view[m[m >= 0]] = 0
        assert np.array_equal(t1["pt_in_view"][b, :npv], view)
        nm2, m2 = oracle.search_by_projection_points(ck, cd, bounds, sf, view, np.stack([pk["x"], pk["y"]], 1), pk["octave"],
                                                     np.ones(npv, np.float32), pd, 1.0, 0.8, (m >= 0).astype(np.uint8))
        assert t1["n_pt"][b] == nm2 and np.array_equal(t1["pt_match"][b, :n], m2)
        # lines
        kl, lf, ld = out["keylines"][b, :nl], out["linefunc"][b, :nl], out["ldesc"][b, :nl]
        pkl, pld = out["keylines"][a, :nlp], out["ldesc"][a, :nlp]
        proj = np.stack([pkl["startPointX"], pkl["startPointY"], pkl["endPointX"], pkl["endPointY"]], 1).astype(np.float32)
        lvalid = np.ones(nlp, np.uint8)
        lnm, lm = oracle.line_search_by_projection_last(kl, lf, ld, bounds, lvalid, proj, pld, pkl["lineLength"], 15.0)
        assert t0["n_line"][b] == lnm and np.array_equal(t0["line_match"][b, :nl], lm)
        lview = lvalid.copy(); lview[lm[lm >= 0]] = 0
        lnm2, lm2 = oracle.line_search_by_projection_lines(kl, lf, ld, bounds, lview, proj, np.ones(nlp, np.float32), pld, 1.0, 0.7,
                                                           (lm >= 0).astype(np.uint8))
        assert t1["n_line"][b] == lnm2 and np.array_equal(t1["line_match"][b, :nl], lm2)
    assert retried >= 2 and t0["n_pt"].max() > 100 and t0["n_line"].max() > 20


@pytest.mark.parametrize("K,D,w,h,seed", [(synth.TUM1_K, synth.TUM1_DIST, 640, 480, 16), (synth.EUROC_K, synth.EUROC_DIST, 752, 480, 17)])
def test_frontend_equals_the_reference_frame_constructor(K, D, w, h, seed):
    """The CUDA front-end against the REFERENCE's own monocular Frame constructor (src/Frame.cc compiled with its ORBextractor,
    LINEextractor and line-descriptor sources into oracle/_ref/libref_frame.so, run on this box's CPU): keypoints, undistorted
    keypoints, ORB descriptors, keylines and LBD descriptors of every frame, byte for byte."""
    B = 3
    frames = synth.synth_sequence(B, w, h, seed=seed)
    fe = pl.Frontend(w, h, max_batch=B, lm_caps=(320, 88))
    fe.set_wrap(True)
    fe.set_pose_problems([synth.synth_pose_problem(90 + k) for k in range(B)])
    fe.set_camera(K, D)
    out = fe.run(frames)
    ku = fe.fetch_keys_un(B)
    for b in range(B):
        F = oracle.ref_frame_construct(frames[b], K, D)
        n, nl = out["n"][b], out["nl"][b]
        assert n == len(F["keys"]) and out["kps"][b, :n].tobytes() == F["keys"].tobytes(), b
        assert np.array_equal(out["desc"][b, :n], F["desc"]) and ku[b, :n].tobytes() == F["keysUn"].tobytes(), b
        assert nl == len(F["keylines"]) and out["keylines"][b, :nl].tobytes() == F["keylines"].tobytes(), b
        assert np.array_equal(out["ldesc"][b, :nl], F["ldesc"]), b
