"""Generate tests/golden/orb_ref_*.npz from the REFERENCE's own ORBextractor.

oracle/_ref/libref_orb.so is /root/reference/src/ORBextractor.cc compiled unmodified where it lies (oracle/Makefile target
`ref`; the OpenCV primitives behind oracle/shim/ are the oracle's cv2-4.13-pinned restatements, and list nodes get increasing
heap addresses so that the pointer tie-break of ORBextractor.cc:684 is reproducible).  The reference does not travel to the
GPU box, so its outputs on the seeded synthetic frames are committed here: tests/test_oracle_orb_ref.py checks the oracle
against them on CPU, tests/test_orb_gpu.py checks the CUDA path against them on the GPU.
Run from the repo root, in the container that has /root/reference:  python tools/gen_golden_orb_ref.py
"""
import os, sys
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import plslam_b200  # noqa  (synth only; no GPU needed)
from plslam_b200 import synth
import oracle

out = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def frame(kind, w, h, seed):
    if kind == "synth":
        return synth.synth_frame(w, h, seed)
    if kind == "low":      # only the minThFAST fallback fires
        return (synth.synth_frame(w, h, seed) // 16 + 100).astype(np.uint8)
    if kind == "noise":    # maximum candidate density
        return np.random.default_rng(seed).integers(0, 256, (h, w), dtype=np.uint8)
    if kind == "sparse":   # fewer candidates than the quota
        im = np.full((h, w), 90, np.uint8); im[200:230, 300:340] = 200
        return im
    raise ValueError(kind)


CASES = {"640x480_n1000": ("synth", 640, 480, 1, 1000, 1.2, 8), "640x480_n2000": ("synth", 640, 480, 1, 2000, 1.2, 8),
         "752x480_n1000": ("synth", 752, 480, 5, 1000, 1.2, 8), "1241x376_n2000": ("synth", 1241, 376, 4, 2000, 1.2, 8),
         "640x480_low": ("low", 640, 480, 9, 1000, 1.2, 8), "640x480_noise": ("noise", 640, 480, 5, 1000, 1.2, 8),
         "640x480_sparse": ("sparse", 640, 480, 0, 1000, 1.2, 8), "640x480_n500_s11": ("synth", 640, 480, 11, 500, 1.2, 8)}

if __name__ == "__main__":
    assert oracle.ref_orb_available(), "needs oracle/_ref/libref_orb.so (make -C oracle ref, where the reference tree exists)"
    for name, (kind, w, h, seed, nf, sf, nl) in CASES.items():
        im = frame(kind, w, h, seed)
        r = oracle.RefOrb(nf, sf, nl, 20, 7)
        kps, desc = r.extract(im)
        t = r.tables()
        np.savez_compressed(os.path.join(out, f"orb_ref_{name}.npz"), kps=kps, desc=desc, img_sum=np.int64(im.astype(np.int64).sum()),
                            params=np.array([w, h, seed, nf, nl]), scale_factor=np.float32(sf), kind=kind,
                            scale=t["scale"], inv_scale=t["inv_scale"], sigma2=t["sigma2"], inv_sigma2=t["inv_sigma2"],
                            level_dims=np.array([r.level(l).shape[::-1] for l in range(nl)]),
                            level_sums=np.array([int(r.level(l).astype(np.int64).sum()) for l in range(nl)]))
        print(name, len(kps))
