"""ctypes binding of oracle/liboracle.so (test infrastructure only)."""
import ctypes as C
import os
import subprocess
import numpy as np

from . import recorded as _rec

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "liboracle.so")

KP_DTYPE = np.dtype([("x", "<f4"), ("y", "<f4"), ("size", "<f4"), ("angle", "<f4"),
                     ("response", "<f4"), ("octave", "<i4"), ("class_id", "<i4")])
assert KP_DTYPE.itemsize == 28


def build(force=False):
    srcs = [os.path.join(_HERE, f) for f in os.listdir(_HERE) if f.endswith(".cpp")]
    if force or not os.path.exists(_LIB) or any(os.path.getmtime(s) > os.path.getmtime(_LIB) for s in srcs):
        subprocess.check_call(["make", "-C", _HERE, "-s"])
    return _LIB


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        # bench.py's CPU legs time the -march=native build of the same sources (oracle/Makefile target `native`)
        _lib = C.CDLL(os.environ.get("PLSLAM_ORACLE_LIB") or _LIB)
        _lib.oracle_orb_create.restype = C.c_void_p
        _lib.oracle_orb_create.argtypes = [C.c_int, C.c_float, C.c_int, C.c_int, C.c_int]
        _lib.oracle_orb_destroy.argtypes = [C.c_void_p]
        _lib.oracle_orb_extract.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                            C.c_void_p, C.c_int]
        _lib.oracle_orb_tables.argtypes = [C.c_void_p] + [C.c_void_p] * 6
        _lib.oracle_orb_level_dims.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        _lib.oracle_orb_level.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int]
        _lib.oracle_orb_blurred.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        _lib.oracle_orb_candidates.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int]
        _lib.oracle_orb_selected.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int]
        _lib.oracle_fast_atan2.restype = C.c_float
        _lib.oracle_fast_atan2.argtypes = [C.c_float, C.c_float]
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


_REF_LIB = os.path.join(_HERE, "_ref", "libref_orb.so")
_ref = None


_REF_LINE_LIB = os.path.join(_HERE, "_ref", "libref_line.so")
_ref_line = None


def ref_line_available():
    """True when oracle/_ref/libref_line.so exists: the reference tree's own line-descriptor sources
    (Thirdparty/line_descriptor/src/binary_descriptor_custom.cpp, LSDDetector_custom.cpp) compiled where they lie."""
    if os.path.isdir("/root/reference/src") and not os.path.exists(_REF_LINE_LIB):
        build()
        subprocess.call(["make", "-C", _HERE, "-s", "ref"])
    return os.path.exists(_REF_LINE_LIB)


def ref_line_lib():
    global _ref_line
    if _ref_line is None:
        lib()
        _ref_line = C.CDLL(_REF_LINE_LIB)
        _ref_line.ref_lsd_keylines.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int]
        _ref_line.ref_lbd_compute.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    return _ref_line


@_rec.entry("ref_lsd_keylines", ref_line_available, ref_only=True)
def ref_lsd_keylines(img, mask=None, scale=1, num_octaves=1):
    """LSDDetectorC::detect(image, keylines, scale, numOctaves, mask) of the reference tree itself -> KeyLine records
    in detection order (LINEextractor passes scale = (int)1.2 = 1 and one octave)."""
    img = np.ascontiguousarray(img, np.uint8)
    m = None if mask is None else np.ascontiguousarray(mask, np.uint8)
    cap = 65536
    kl = np.zeros(cap, KEYLINE_DTYPE)
    n = ref_line_lib().ref_lsd_keylines(_p(img), img.shape[1], img.shape[0], _p(m), scale, num_octaves, _p(kl), cap)
    assert 0 <= n <= cap
    return kl[:n].copy()


@_rec.entry("ref_line_extract", ref_line_available, ref_only=True)
def ref_line_extract(img, mask=None, nfeatures=200, min_line_length=0.0):
    """LINEextractor::operator() of the reference itself (src/LineExtractor.cpp) -> (keylines, descriptors, line functions).
    Only for frames with more lines than nfeatures (see oracle/ref_line_wrap.cpp)."""
    img = np.ascontiguousarray(img, np.uint8)
    cap = nfeatures + 2
    kl = np.zeros(cap, KEYLINE_DTYPE); desc = np.zeros((cap, 32), np.uint8); lf = np.zeros((cap, 3), np.float64)
    m = None if mask is None else np.ascontiguousarray(mask, np.uint8)
    f = ref_line_lib().ref_line_extract
    f.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
    n = f(_p(img), img.shape[1], img.shape[0], _p(m), nfeatures, float(min_line_length), _p(kl), _p(desc), _p(lf), cap)
    assert n >= 0, n
    return kl[:n].copy(), desc[:n].copy(), lf[:n].copy()


@_rec.entry("ref_lbd_compute", ref_line_available, ref_only=True)
def ref_lbd_compute(img, keylines, want_float=False):
    """BinaryDescriptor::compute(image, keylines, descriptors) of the reference tree itself (class_id must index the lines)."""
    img = np.ascontiguousarray(img, np.uint8); kl = np.ascontiguousarray(keylines)
    desc = np.zeros((max(len(kl), 1), 32), np.uint8)
    dv = np.zeros((max(len(kl), 1), 72), np.float32) if want_float else None
    n = ref_line_lib().ref_lbd_compute(_p(img), img.shape[1], img.shape[0], _p(kl), len(kl), _p(desc), _p(dv))
    assert n == len(kl), n
    return (desc[:len(kl)], dv[:len(kl)]) if want_float else desc[:len(kl)]


_REF_FRAME_LIB = os.path.join(_HERE, "_ref", "libref_frame.so")
_ref_frame = None


def ref_frame_available():
    """True when oracle/_ref/libref_frame.so exists: the reference's OWN src/Frame.cc against its real Frame.h, with its ORBextractor,
    LINEextractor, MapPoint and the vendored line-descriptor sources (oracle/ref_frame_wrap.cpp, oracle/shim_frame/)."""
    if os.path.isdir("/root/reference/src") and not os.path.exists(_REF_FRAME_LIB):
        build()
        subprocess.call(["make", "-C", _HERE, "-s", "ref"])
    return os.path.exists(_REF_FRAME_LIB)


def _ref_frame_lib():
    global _ref_frame
    if _ref_frame is None:
        lib()
        _ref_frame = C.CDLL(_REF_FRAME_LIB)
    return _ref_frame


_frame_key = None      # the arguments of the last ref_frame_construct: ref_frame_features_in_area answers for that frame


def ref_frame_construct(img, K, D, mask=None, nfeatures=1000, scale_factor=1.2, nlevels=8, ini_th=20, min_th=7, nlines=200, min_line_length=0.0):
    """The reference's monocular Frame constructor itself (Frame.cc:193-276) -> dict(keys, keysUn, desc, keylines, ldesc, lfunc, bounds,
    grid (start, items), line_grid (start, items)).  The frame stays alive for ref_frame_features_in_area(_line)."""
    global _frame_key
    a = (img, K, D, mask, nfeatures, scale_factor, nlevels, ini_th, min_th, nlines, min_line_length)
    _frame_key = _rec.digest("ref_frame_construct", *a)
    return _rec.call("ref_frame_construct", a, ref_frame_available(), lambda: _ref_frame_construct(*a))


def _ref_frame_construct(img, K, D, mask, nfeatures, scale_factor, nlevels, ini_th, min_th, nlines, min_line_length):
    img = np.ascontiguousarray(img, np.uint8); h, w = img.shape
    cap, capl = 2 * nfeatures + 64, nlines + 2
    counts = np.zeros(2, np.int32)
    keys = np.zeros(cap, KP_DTYPE); keysUn = np.zeros(cap, KP_DTYPE); desc = np.zeros((cap, 32), np.uint8)
    kl = np.zeros(capl, KEYLINE_DTYPE); ldesc = np.zeros((capl, 32), np.uint8); lfunc = np.zeros((capl, 3), np.float64)
    bounds = np.zeros(4, np.float32)
    gs = np.zeros(64 * 48 + 1, np.int32); gi = np.zeros(cap, np.int32)
    lcap = capl * 200
    ls = np.zeros(64 * 48 + 1, np.int32); li = np.zeros(lcap, np.int32); ln = C.c_int(0)
    m = None if mask is None else np.ascontiguousarray(mask, np.uint8)
    Kc = _f32(K); Dc = _f32(D)
    f = _ref_frame_lib().ref_frame_construct
    f.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_float, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double,
                  C.c_int, C.c_int] + [C.c_void_p] * 12 + [C.c_int, C.c_void_p]
    rc = f(_p(img), w, h, _p(m), _p(Kc), _p(Dc), nfeatures, scale_factor, nlevels, ini_th, min_th, nlines, float(min_line_length), cap, capl,
           _p(counts), _p(keys), _p(keysUn), _p(desc), _p(kl), _p(ldesc), _p(lfunc), _p(bounds), _p(gs), _p(gi), _p(ls), _p(li), lcap, C.byref(ln))
    assert rc == 0, rc
    n, nl = int(counts[0]), int(counts[1])
    return dict(keys=keys[:n].copy(), keysUn=keysUn[:n].copy(), desc=desc[:n].copy(), keylines=kl[:nl].copy(), ldesc=ldesc[:nl].copy(),
                lfunc=lfunc[:nl].copy(), bounds=bounds, grid=(gs, gi[:gs[-1]].copy()), line_grid=(ls, li[:ln.value].copy()))


def ref_frame_features_in_area(x, y, r, min_level=-1, max_level=-1):
    return _rec.call("ref_frame_features_in_area", (_frame_key, x, y, r, min_level, max_level), ref_frame_available(),
                     lambda: _ref_frame_features_in_area(x, y, r, min_level, max_level))


def _ref_frame_features_in_area(x, y, r, min_level, max_level):
    out = np.zeros(8192, np.int32)
    f = _ref_frame_lib().ref_frame_features_in_area
    f.argtypes = [C.c_float, C.c_float, C.c_float, C.c_int, C.c_int, C.c_void_p, C.c_int]
    n = f(x, y, r, min_level, max_level, _p(out), len(out))
    return out[:n].copy()


@_rec.entry("ref_frame_is_in_frustum_points", ref_frame_available, ref_only=True)
def ref_frame_is_in_frustum_points(Tcw, K, bounds, log_scale_factor, n_levels, cos_limit, pos, normal, min_dist, max_dist):
    """Frame::isInFrustum(MapPoint*) of the reference itself -> (inview, proj, level, viewcos, Ow as the frame derives it)."""
    n = len(pos)
    T = _f32(Tcw); Kc = _f32(K); b = _f32(bounds); pos = _f32(pos); normal = _f32(normal); mn = _f32(min_dist); mx = _f32(max_dist)
    inview = np.zeros(n, np.uint8); proj = np.zeros((n, 2), np.float32); level = np.zeros(n, np.int32); vc = np.zeros(n, np.float32); Ow = np.zeros(3, np.float32)
    _ref_frame_lib().ref_frame_is_in_frustum_points(_p(T), _p(Kc), _p(b), C.c_float(log_scale_factor), C.c_int(n_levels), C.c_float(cos_limit), C.c_int(n),
                                                    _p(pos), _p(normal), _p(mn), _p(mx), _p(inview), _p(proj), _p(level), _p(vc), _p(Ow))
    return inview, proj, level, vc, Ow


@_rec.entry("ref_frame_is_in_frustum_lines", ref_frame_available, ref_only=True)
def ref_frame_is_in_frustum_lines(Tcw, K, bounds, log_scale_factor, cos_limit, pos, normal, min_dist, max_dist):
    n = len(pos)
    T = _f32(Tcw); Kc = _f32(K); b = _f32(bounds); mn = _f32(min_dist); mx = _f32(max_dist)
    pos = np.ascontiguousarray(pos, np.float64); normal = np.ascontiguousarray(normal, np.float64)
    inview = np.zeros(n, np.uint8); proj = np.zeros((n, 4), np.float32); level = np.zeros(n, np.int32); vc = np.zeros(n, np.float32); Ow = np.zeros(3, np.float32)
    _ref_frame_lib().ref_frame_is_in_frustum_lines(_p(T), _p(Kc), _p(b), C.c_float(log_scale_factor), C.c_float(cos_limit), C.c_int(n), _p(pos), _p(normal),
                                                   _p(mn), _p(mx), _p(inview), _p(proj), _p(level), _p(vc), _p(Ow))
    return inview, proj, level, vc, Ow


_REF_MATCH_LIB = os.path.join(_HERE, "_ref", "libref_match.so")
_ref_match = None


def ref_match_available():
    """True when oracle/_ref/libref_match.so exists: the reference's OWN src/ORBmatcher.cc and src/MapPoint.cc compiled where they
    lie against mock Frame / KeyFrame / Map (oracle/shim_slam/, oracle/ref_match_wrap.cpp)."""
    if os.path.isdir("/root/reference/src") and not os.path.exists(_REF_MATCH_LIB):
        build()
        subprocess.call(["make", "-C", _HERE, "-s", "ref"])
    return os.path.exists(_REF_MATCH_LIB)


def _fn(name, impl):
    """the oracle's restatement (`oracle_<name>` in liboracle.so) or the reference's own code (`ref_<name>` in libref_match.so):
    same flat-array signature"""
    global _ref_match
    if impl == "oracle":
        return getattr(lib(), "oracle_" + name)
    assert impl == "ref", impl
    if _ref_match is None:
        _ref_match = C.CDLL(_REF_MATCH_LIB)
    return getattr(_ref_match, "ref_" + name)


def ref_orb_available():
    """True when oracle/_ref/libref_orb.so exists: the reference's OWN src/ORBextractor.cc compiled where it lies
    (oracle/Makefile target `ref`, oracle/ref_orb_wrap.cpp, oracle/shim/).  Built in the container that has /root/reference;
    the file travels to the GPU box with the snapshot."""
    if os.path.isdir("/root/reference/src") and not os.path.exists(_REF_LIB):
        build()
        subprocess.call(["make", "-C", _HERE, "-s", "ref"])
    return os.path.exists(_REF_LIB)


def ref_lib():
    global _ref
    if _ref is None:
        lib()   # liboracle.so first (libref_orb.so links it for the cv2-pinned image primitives)
        _ref = C.CDLL(_REF_LIB)
        _ref.ref_orb_create.restype = C.c_void_p
        _ref.ref_orb_create.argtypes = [C.c_int, C.c_float, C.c_int, C.c_int, C.c_int]
        _ref.ref_orb_destroy.argtypes = [C.c_void_p]
        _ref.ref_orb_extract.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
        _ref.ref_orb_tables.argtypes = [C.c_void_p] + [C.c_void_p] * 4
        _ref.ref_orb_level.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        _ref.ref_orb_set_bump.argtypes = [C.c_int]
    return _ref


class RefOrb:
    """The reference's ORB_SLAM2::ORBextractor itself (src/ORBextractor.cc compiled unmodified), not a restatement.
    `ordered_heap=True` (default): list nodes get increasing addresses in allocation order, which fixes the otherwise
    allocator-dependent pointer tie-break of ORBextractor.cc:684; False: glibc malloc order."""

    def __init__(self, nfeatures=1000, scale_factor=1.2, nlevels=8, ini_th=20, min_th=7, ordered_heap=True):
        self.nlevels, self.nfeatures, self.ordered_heap = nlevels, nfeatures, ordered_heap
        self.live = ref_orb_available()
        self.args = (nfeatures, scale_factor, nlevels, ini_th, min_th, ordered_heap)
        self.last = None       # the last extracted image: level() returns its pyramid
        self.h = ref_lib().ref_orb_create(nfeatures, scale_factor, nlevels, ini_th, min_th) if self.live else None

    def __del__(self):
        if getattr(self, "h", None):
            ref_lib().ref_orb_destroy(self.h)
            self.h = None

    def tables(self):
        return _rec.call("RefOrb.tables", self.args, self.live, self._tables)

    def extract(self, img):
        self.last = _rec.digest("RefOrb.image", img)
        return _rec.call("RefOrb.extract", (self.args, img), self.live, lambda: self._extract(img))

    def level(self, l):
        return _rec.call("RefOrb.level", (self.args, self.last, l), self.live, lambda: self._level(l))

    def _tables(self):
        n = self.nlevels
        sc, isc, s2, is2 = (np.zeros(n, np.float32) for _ in range(4))
        ref_lib().ref_orb_tables(self.h, _p(sc), _p(isc), _p(s2), _p(is2))
        return dict(scale=sc, inv_scale=isc, sigma2=s2, inv_sigma2=is2)

    def _extract(self, img):
        img = np.ascontiguousarray(img, np.uint8)
        cap = self.nfeatures * 2 + 64
        kps = np.zeros(cap, KP_DTYPE)
        desc = np.zeros((cap, 32), np.uint8)
        ref_lib().ref_orb_set_bump(1 if self.ordered_heap else 0)
        n = ref_lib().ref_orb_extract(self.h, _p(img), img.shape[1], img.shape[0], img.strides[0], _p(kps), _p(desc), cap)
        assert 0 <= n <= cap, n
        return kps[:n].copy(), desc[:n].copy()

    def _level(self, l):
        w, h = C.c_int(), C.c_int()
        ref_lib().ref_orb_level(self.h, l, None, C.byref(w), C.byref(h))
        out = np.zeros((h.value, w.value), np.uint8)
        ref_lib().ref_orb_level(self.h, l, _p(out), C.byref(w), C.byref(h))
        return out


class OrbOracle:
    """Restatement of ORB_SLAM2::ORBextractor (reference src/ORBextractor.cc)."""

    def __init__(self, nfeatures=1000, scale_factor=1.2, nlevels=8, ini_th=20, min_th=7):
        self.nlevels = nlevels
        self.nfeatures = nfeatures
        self.h = lib().oracle_orb_create(nfeatures, scale_factor, nlevels, ini_th, min_th)

    def __del__(self):
        if getattr(self, "h", None):
            lib().oracle_orb_destroy(self.h)
            self.h = None

    def tables(self):
        n = self.nlevels
        sc, isc, s2, is2 = (np.zeros(n, np.float32) for _ in range(4))
        per = np.zeros(n, np.int32)
        umax = np.zeros(16, np.int32)
        lib().oracle_orb_tables(self.h, _p(sc), _p(isc), _p(s2), _p(is2), _p(per), _p(umax))
        return dict(scale=sc, inv_scale=isc, sigma2=s2, inv_sigma2=is2, per_level=per, umax=umax)

    def extract(self, img):
        img = np.ascontiguousarray(img, np.uint8)
        cap = self.nfeatures * 2 + 64
        kps = np.zeros(cap, KP_DTYPE)
        desc = np.zeros((cap, 32), np.uint8)
        n = lib().oracle_orb_extract(self.h, _p(img), img.shape[1], img.shape[0], img.strides[0], _p(kps),
                                     _p(desc), cap)
        assert n >= 0
        return kps[:n].copy(), desc[:n].copy()

    def level_dims(self, l):
        w, h = C.c_int(), C.c_int()
        lib().oracle_orb_level_dims(self.h, l, C.byref(w), C.byref(h))
        return w.value, h.value

    def level(self, l, with_border=False):
        w, h = self.level_dims(l)
        if with_border:
            w, h = w + 38, h + 38
        out = np.zeros((h, w), np.uint8)
        lib().oracle_orb_level(self.h, l, _p(out), int(with_border))
        return out

    def blurred(self, l):
        w, h = self.level_dims(l)
        out = np.zeros((h, w), np.uint8)
        rc = lib().oracle_orb_blurred(self.h, l, _p(out))
        return out if rc == 0 else None

    def candidates(self, l):
        n = lib().oracle_orb_candidates(self.h, l, None, 0)
        out = np.zeros(max(n, 1), KP_DTYPE)
        lib().oracle_orb_candidates(self.h, l, _p(out), n)
        return out[:n]

    def selected(self, l):
        n = lib().oracle_orb_selected(self.h, l, None, 0)
        out = np.zeros(max(n, 1), KP_DTYPE)
        lib().oracle_orb_selected(self.h, l, _p(out), n)
        return out[:n]


def resize_linear_u8(src, dw, dh):
    src = np.ascontiguousarray(src, np.uint8)
    dst = np.zeros((dh, dw), np.uint8)
    lib().oracle_resize_linear_u8(_p(src), src.shape[1], src.shape[0], _p(dst), dw, dh)
    return dst


def blur_u8(src, ksize):
    src = np.ascontiguousarray(src, np.uint8)
    dst = np.zeros_like(src)
    lib().oracle_blur_u8(_p(src), src.shape[1], src.shape[0], _p(dst), ksize)
    return dst


def fast_atan2(y, x):
    return lib().oracle_fast_atan2(float(y), float(x))


def fast_detect(img, threshold):
    img = np.ascontiguousarray(img, np.uint8)
    cap = img.size
    out = np.zeros(cap, KP_DTYPE)
    n = lib().oracle_fast_detect(_p(img), img.shape[1], img.shape[0], threshold, _p(out), cap)
    return out[:n].copy()


def fast_score_map(img):
    img = np.ascontiguousarray(img, np.uint8)
    out = np.zeros(img.shape, np.int32)
    lib().oracle_fast_score_map(_p(img), img.shape[1], img.shape[0], _p(out))
    return out


def distribute(kps, minX, maxX, minY, maxY, N):
    kps = np.ascontiguousarray(kps)
    out = np.zeros(max(len(kps), 1), KP_DTYPE)
    n = lib().oracle_distribute(_p(kps), len(kps), minX, maxX, minY, maxY, N, _p(out))
    return out[:n].copy()


# ---------------------------------------------------------------------------------------------- matching
KL_DTYPE = np.dtype([("startX", "<f4"), ("startY", "<f4"), ("endX", "<f4"), ("endY", "<f4"),
                     ("lineLength", "<f4"), ("angle", "<f4"), ("octave", "<i4")])


@_rec.entry("descriptor_distance", ref_match_available)
def descriptor_distance(a, b, impl="oracle"):
    a = np.ascontiguousarray(a, np.uint8); b = np.ascontiguousarray(b, np.uint8)
    f = _fn("descriptor_distance", impl); f.argtypes = [C.c_void_p, C.c_void_p]
    return f(_p(a), _p(b))


def assign_grid(keys, bounds):
    keys = np.ascontiguousarray(keys); b = np.asarray(bounds, np.float32)
    start = np.zeros(64 * 48 + 1, np.int32); items = np.zeros(max(len(keys), 1), np.int32)
    n = lib().oracle_assign_grid(_p(keys), len(keys), _p(b), _p(start), _p(items))
    return start, items[:n]


@_rec.entry("search_for_initialization", ref_match_available)
def search_for_initialization(k1, d1, k2, d2, bounds, prev_matched, window=100, nnratio=0.9, check_ori=True, impl="oracle"):
    k1 = np.ascontiguousarray(k1); k2 = np.ascontiguousarray(k2)
    d1 = np.ascontiguousarray(d1, np.uint8); d2 = np.ascontiguousarray(d2, np.uint8)
    pm = np.ascontiguousarray(prev_matched, np.float32).copy()
    m = np.zeros(max(len(k1), 1), np.int32)
    b = np.asarray(bounds, np.float32)
    f = _fn("search_for_initialization", impl)
    f.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_float, C.c_int]
    nm = f(_p(k1), _p(d1), len(k1), _p(k2), _p(d2), len(k2), _p(b), _p(pm), _p(m), window, nnratio, int(check_ori))
    return nm, m[:len(k1)], pm


@_rec.entry("search_by_projection_last", ref_match_available)
def search_by_projection_last(kc, dc, bounds, Tcw, K, scale_factors, last_valid, last_pos, last_desc, last_octave,
                              last_angle, th, check_ori=True, preassigned=None, impl="oracle"):
    kc = np.ascontiguousarray(kc); dc = np.ascontiguousarray(dc, np.uint8)
    m = np.zeros(max(len(kc), 1), np.int32)
    f = _fn("search_by_projection_last", impl)
    f.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_int, C.c_void_p, C.c_void_p]
    arrs = [np.asarray(bounds, np.float32), np.ascontiguousarray(Tcw, np.float32), np.asarray(K, np.float32),
            np.ascontiguousarray(scale_factors, np.float32)]
    lv = np.ascontiguousarray(last_valid, np.uint8); lp = np.ascontiguousarray(last_pos, np.float32)
    ld = np.ascontiguousarray(last_desc, np.uint8); lo = np.ascontiguousarray(last_octave, np.int32)
    la = np.ascontiguousarray(last_angle, np.float32)
    pre = None if preassigned is None else np.ascontiguousarray(preassigned, np.uint8)
    nm = f(_p(kc), _p(dc), len(kc), _p(arrs[0]), _p(arrs[1]), _p(arrs[2]), _p(arrs[3]), len(lv), _p(lv), _p(lp), _p(ld),
           _p(lo), _p(la), th, int(check_ori), _p(pre), _p(m))
    return nm, m[:len(kc)]


@_rec.entry("search_by_projection_points", ref_match_available)
def search_by_projection_points(k, d, bounds, scale_factors, in_view, proj, level, view_cos, mp_desc, th, nnratio=0.8,
                                preassigned=None, impl="oracle"):
    k = np.ascontiguousarray(k); d = np.ascontiguousarray(d, np.uint8)
    m = np.zeros(max(len(k), 1), np.int32)
    f = _fn("search_by_projection_points", impl)
    f.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                  C.c_void_p, C.c_void_p, C.c_float, C.c_float, C.c_void_p, C.c_void_p]
    b = np.asarray(bounds, np.float32); sf = np.ascontiguousarray(scale_factors, np.float32)
    iv = np.ascontiguousarray(in_view, np.uint8); pr = np.ascontiguousarray(proj, np.float32)
    lv = np.ascontiguousarray(level, np.int32); vc = np.ascontiguousarray(view_cos, np.float32)
    md = np.ascontiguousarray(mp_desc, np.uint8)
    pre = None if preassigned is None else np.ascontiguousarray(preassigned, np.uint8)
    nm = f(_p(k), _p(d), len(k), _p(b), _p(sf), len(iv), _p(iv), _p(pr), _p(lv), _p(vc), _p(md), th, nnratio, _p(pre), _p(m))
    return nm, m[:len(k)]


def bf_knn2(d1, d2):
    d1 = np.ascontiguousarray(d1, np.uint8); d2 = np.ascontiguousarray(d2, np.uint8)
    idx = np.zeros((max(len(d1), 1), 2), np.int32); dist = np.zeros((max(len(d1), 1), 2), np.int32)
    lib().oracle_bf_knn2(_p(d1), len(d1), _p(d2), len(d2), _p(idx), _p(dist))
    return idx[:len(d1)], dist[:len(d1)]


@_rec.entry("frame_bf_match", ref_match_available)
def frame_bf_match(d1, d2, th=50.0, nnratio=0.7, impl="oracle"):
    d1 = np.ascontiguousarray(d1, np.uint8); d2 = np.ascontiguousarray(d2, np.uint8)
    m = np.zeros(max(len(d1), 1), np.int32)
    f = _fn("frame_bf_match", impl)
    f.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_float, C.c_float, C.c_void_p]
    f(_p(d1), len(d1), _p(d2), len(d2), th, nnratio, _p(m))
    return m[:len(d1)]


@_rec.entry("search_double", ref_match_available)
def search_double(d1, d2, nnratio=0.7, impl="oracle"):
    d1 = np.ascontiguousarray(d1, np.uint8); d2 = np.ascontiguousarray(d2, np.uint8)
    m = np.zeros(max(len(d1), 1), np.int32)
    f = _fn("search_double", impl)
    f.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_float, C.c_void_p]
    nm = f(_p(d1), len(d1), _p(d2), len(d2), nnratio, _p(m))
    return nm, m[:len(d1)]


# ---------------------------------------------------------------------------------------------- pose-only LM
def pose_optimization(mode, Tcw, K, pt_obs, pt_inv_sigma2, pt_Xw, line_func, line_Xw):
    Tcw = np.ascontiguousarray(Tcw, np.float32); K = np.ascontiguousarray(K, np.float32)
    po = np.ascontiguousarray(pt_obs, np.float32).reshape(-1, 2); pw = np.ascontiguousarray(pt_inv_sigma2, np.float32)
    px = np.ascontiguousarray(pt_Xw, np.float32).reshape(-1, 3)
    lf = np.ascontiguousarray(line_func, np.float64).reshape(-1, 3); lx = np.ascontiguousarray(line_Xw, np.float64).reshape(-1, 6)
    Tout = np.zeros((4, 4), np.float32)
    pout = np.zeros(max(len(po), 1), np.uint8); lout = np.zeros(max(len(lf), 1), np.uint8)
    its = C.c_int(0)
    f = lib().oracle_pose_optimization
    f.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    n = f(mode, _p(Tcw), _p(K), len(po), _p(po), _p(pw), _p(px), len(lf), _p(lf), _p(lx), _p(Tout), _p(pout), _p(lout),
          C.byref(its))
    return n, Tout, pout[:len(po)].astype(bool), lout[:len(lf)].astype(bool), its.value


# ---------------------------------------------------------------------------------------------- lines (LSD + LBD)
KEYLINE_DTYPE = np.dtype([("angle", "<f4"), ("class_id", "<i4"), ("octave", "<i4"), ("ptx", "<f4"), ("pty", "<f4"),
                          ("response", "<f4"), ("size", "<f4"), ("startPointX", "<f4"), ("startPointY", "<f4"),
                          ("endPointX", "<f4"), ("endPointY", "<f4"), ("sPointInOctaveX", "<f4"),
                          ("sPointInOctaveY", "<f4"), ("ePointInOctaveX", "<f4"), ("ePointInOctaveY", "<f4"),
                          ("lineLength", "<f4"), ("numOfPixels", "<i4")])
assert KEYLINE_DTYPE.itemsize == 68


def lsd_detect(img, order_mode=1):
    """cv::createLineSegmentDetector()->detect(img) -> (n,4) float32 [x1,y1,x2,y2]."""
    img = np.ascontiguousarray(img, np.uint8)
    cap = 20000
    out = np.zeros((cap, 4), np.float32)
    n = lib().oracle_lsd_detect(_p(img), img.shape[1], img.shape[0], order_mode, _p(out), cap)
    return out[:n].copy()


def lsd_stages(img):
    img = np.ascontiguousarray(img, np.uint8)
    sw, sh = C.c_int(), C.c_int()
    w8, h8 = int(round(img.shape[1] * 0.8)) + 2, int(round(img.shape[0] * 0.8)) + 2
    sc = np.zeros(w8 * h8, np.uint8); mg = np.zeros(w8 * h8, np.float64); an = np.zeros(w8 * h8, np.float64)
    lib().oracle_lsd_stages(_p(img), img.shape[1], img.shape[0], _p(sc), _p(mg), _p(an), C.byref(sw), C.byref(sh))
    n = sw.value * sh.value
    return (sc[:n].reshape(sh.value, sw.value), mg[:n].reshape(sh.value, sw.value), an[:n].reshape(sh.value, sw.value))


def lbd_sobel(img):
    img = np.ascontiguousarray(img, np.uint8)
    dx = np.zeros(img.shape, np.int16); dy = np.zeros(img.shape, np.int16)
    lib().oracle_lbd_sobel(_p(img), img.shape[1], img.shape[0], _p(dx), _p(dy))
    return dx, dy


def lbd_compute(img, keylines, want_float=False):
    img = np.ascontiguousarray(img, np.uint8); kl = np.ascontiguousarray(keylines)
    desc = np.zeros((max(len(kl), 1), 32), np.uint8)
    dv = np.zeros((max(len(kl), 1), 72), np.float32) if want_float else None
    lib().oracle_lbd_compute(_p(img), img.shape[1], img.shape[0], _p(kl), len(kl), _p(desc), _p(dv))
    return (desc[:len(kl)], dv[:len(kl)]) if want_float else desc[:len(kl)]


def line_extract(img, mask=None, nfeatures=200, min_line_length=0.0, order_mode=1):
    """LINEextractor::operator() -> (keylines[68 B records], descriptors n x 32, line functions n x 3)."""
    img = np.ascontiguousarray(img, np.uint8)
    cap = nfeatures + 2
    kl = np.zeros(cap, KEYLINE_DTYPE); desc = np.zeros((cap, 32), np.uint8); lf = np.zeros((cap, 3), np.float64)
    m = None if mask is None else np.ascontiguousarray(mask, np.uint8)
    f = lib().oracle_line_extract
    f.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_double, C.c_int, C.c_void_p, C.c_void_p,
                  C.c_void_p, C.c_int]
    n = f(_p(img), img.shape[1], img.shape[0], _p(m), nfeatures, float(min_line_length), order_mode, _p(kl), _p(desc),
          _p(lf), cap)
    assert n >= 0
    return kl[:n].copy(), desc[:n].copy(), lf[:n].copy()


# ---------------------------------------------------------------------------------------------- local BA
def local_ba(p, stop_flag=None):
    """p: dict from synth.synth_ba_problem.  Returns dict(kf_Tcw, pt_Xw, ln_Xw, pe_erase, le_erase, le_erase_kf, its)."""
    n_kf, n_pt, n_ln, n_pe, n_le = len(p["kf_fixed"]), len(p["pt_Xw"]), len(p["ln_Xw"]), len(p["pe_kf"]), len(p["le_kf"])
    out = dict(kf_Tcw=np.zeros((n_kf, 16), np.float32), pt_Xw=np.zeros((max(n_pt, 1), 3), np.float32),
               ln_Xw=np.zeros((max(n_ln, 1), 6), np.float64), pe_erase=np.zeros(max(n_pe, 1), np.uint8),
               le_erase=np.zeros(max(n_le, 1), np.uint8), le_erase_kf=np.zeros(max(n_le, 1), np.int32))
    its = C.c_int(0)
    sf = None if stop_flag is None else np.ascontiguousarray(stop_flag, np.int32)
    f = lib().oracle_local_ba
    f.argtypes = [C.c_int] + [C.c_void_p] * 4 + [C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int] + [C.c_void_p] * 4 + \
                 [C.c_int] + [C.c_void_p] * 3 + [C.c_void_p] * 8
    a = {k: np.ascontiguousarray(v) for k, v in p.items() if isinstance(v, np.ndarray)}
    f(n_kf, _p(a["kf_Tcw"]), _p(a["kf_fixed"]), _p(a["kf_K"]), _p(a["K_end"]), n_pt, _p(a["pt_Xw"]), n_ln, _p(a["ln_Xw"]), n_pe,
      _p(a["pe_kf"]), _p(a["pe_pt"]), _p(a["pe_obs"]), _p(a["pe_inv_sigma2"]), n_le, _p(a["le_kf"]), _p(a["le_ln"]), _p(a["le_func"]),
      _p(sf), _p(out["kf_Tcw"]), _p(out["pt_Xw"]), _p(out["ln_Xw"]), _p(out["pe_erase"]), _p(out["le_erase"]),
      _p(out["le_erase_kf"]), C.byref(its))
    out["its"] = its.value
    for k, n in (("pt_Xw", n_pt), ("ln_Xw", n_ln), ("pe_erase", n_pe), ("le_erase", n_le), ("le_erase_kf", n_le)):
        out[k] = out[k][:n]
    return out


def global_ba(p, n_iterations=5, robust=True, stop_flag=None):
    """Optimizer::BundleAdjustment with lines (Optimizer.cc:275-638).  Returns dict(kf_Tcw, pt_Xw, ln_Xw, its)."""
    n_kf, n_pt, n_ln, n_pe, n_le = len(p["kf_fixed"]), len(p["pt_Xw"]), len(p["ln_Xw"]), len(p["pe_kf"]), len(p["le_kf"])
    out = dict(kf_Tcw=np.zeros((n_kf, 16), np.float32), pt_Xw=np.zeros((max(n_pt, 1), 3), np.float32),
               ln_Xw=np.zeros((max(n_ln, 1), 6), np.float64))
    its = C.c_int(0)
    sf = None if stop_flag is None else np.ascontiguousarray(stop_flag, np.int32)
    f = lib().oracle_global_ba
    f.argtypes = [C.c_int] + [C.c_void_p] * 3 + [C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int] + [C.c_void_p] * 4 + \
                 [C.c_int] + [C.c_void_p] * 3 + [C.c_int, C.c_int] + [C.c_void_p] * 5
    a = {k: np.ascontiguousarray(v) for k, v in p.items() if isinstance(v, np.ndarray)}
    f(n_kf, _p(a["kf_Tcw"]), _p(a["kf_fixed"]), _p(a["kf_K"]), n_pt, _p(a["pt_Xw"]), n_ln, _p(a["ln_Xw"]), n_pe,
      _p(a["pe_kf"]), _p(a["pe_pt"]), _p(a["pe_obs"]), _p(a["pe_inv_sigma2"]), n_le, _p(a["le_kf"]), _p(a["le_ln"]), _p(a["le_func"]),
      int(n_iterations), int(bool(robust)), _p(sf), _p(out["kf_Tcw"]), _p(out["pt_Xw"]), _p(out["ln_Xw"]), C.byref(its))
    out["its"] = its.value
    out["pt_Xw"] = out["pt_Xw"][:n_pt]; out["ln_Xw"] = out["ln_Xw"][:n_ln]
    return out


# ---------------------------------------------------------------------------------------------- line matching by projection
def _compact_kl(kl68):
    """68-byte KeyLine records -> the 7-field flat records oracle_match.cpp reads."""
    out = np.zeros(len(kl68), KL_DTYPE)
    for f in ("lineLength", "angle", "octave"):
        out[f] = kl68[f]
    out["startX"], out["startY"], out["endX"], out["endY"] = kl68["startPointX"], kl68["startPointY"], kl68["endPointX"], kl68["endPointY"]
    return out


def assign_grid_lines(kl68, bounds):
    k = _compact_kl(kl68); b = np.asarray(bounds, np.float32)
    cap = max(len(k), 1) * 120
    start = np.zeros(64 * 48 + 1, np.int32); items = np.zeros(cap, np.int32)
    f = lib().oracle_assign_grid_lines
    f.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
    n = f(_p(k), len(k), _p(b), _p(start), _p(items), cap)
    return start, items[:n]


@_rec.entry("line_search_by_projection_last", ref_match_available)
def line_search_by_projection_last(kl68, lfunc, desc, bounds, last_valid, proj, last_desc, last_length, th, preassigned=None, impl="oracle"):
    k = _compact_kl(kl68); m = np.zeros(max(len(k), 1), np.int32)
    f = _fn("line_search_by_projection_last", impl)
    f.argtypes = [C.c_void_p] * 3 + [C.c_int, C.c_void_p, C.c_int] + [C.c_void_p] * 4 + [C.c_float, C.c_void_p, C.c_void_p]
    a = [np.ascontiguousarray(lfunc, np.float64), np.ascontiguousarray(desc, np.uint8), np.asarray(bounds, np.float32),
         np.ascontiguousarray(last_valid, np.uint8), np.ascontiguousarray(proj, np.float32), np.ascontiguousarray(last_desc, np.uint8),
         np.ascontiguousarray(last_length, np.float32)]
    pre = None if preassigned is None else np.ascontiguousarray(preassigned, np.uint8)
    nm = f(_p(k), _p(a[0]), _p(a[1]), len(k), _p(a[2]), len(a[3]), _p(a[3]), _p(a[4]), _p(a[5]), _p(a[6]), th, _p(pre), _p(m))
    return nm, m[:len(k)]


@_rec.entry("line_search_by_projection_lines", ref_match_available)
def line_search_by_projection_lines(kl68, lfunc, desc, bounds, in_view, proj, view_cos, ml_desc, th, nnratio=0.7, preassigned=None, impl="oracle"):
    k = _compact_kl(kl68); m = np.zeros(max(len(k), 1), np.int32)
    f = _fn("line_search_by_projection_lines", impl)
    f.argtypes = [C.c_void_p] * 3 + [C.c_int, C.c_void_p, C.c_int] + [C.c_void_p] * 4 + [C.c_float, C.c_float, C.c_void_p, C.c_void_p]
    a = [np.ascontiguousarray(lfunc, np.float64), np.ascontiguousarray(desc, np.uint8), np.asarray(bounds, np.float32),
         np.ascontiguousarray(in_view, np.uint8), np.ascontiguousarray(proj, np.float32), np.ascontiguousarray(view_cos, np.float32),
         np.ascontiguousarray(ml_desc, np.uint8)]
    pre = None if preassigned is None else np.ascontiguousarray(preassigned, np.uint8)
    nm = f(_p(k), _p(a[0]), _p(a[1]), len(k), _p(a[2]), len(a[3]), _p(a[3]), _p(a[4]), _p(a[5]), _p(a[6]), th, nnratio, _p(pre), _p(m))
    return nm, m[:len(k)]


# ----------------------------------------------------------------- Frame glue (oracle_frame.cpp; reference src/Frame.cc)
def _f32(a):
    return np.ascontiguousarray(a, np.float32)


def undistort_map(K, D, w, h):
    """cv::initUndistortRectifyMap(K, D, I, K, (w,h), CV_32F) (Frame.cc:220)."""
    mx = np.empty((h, w), np.float32); my = np.empty((h, w), np.float32)
    K = _f32(K); D = _f32(D)
    lib().oracle_undistort_map(_p(K), _p(D), C.c_int(w), C.c_int(h), _p(mx), _p(my))
    return mx, my


def remap_linear(src, mx, my):
    """cv::remap(src, dst, mx, my, INTER_LINEAR) with BORDER_CONSTANT 0 (Frame.cc:221)."""
    src = np.ascontiguousarray(src, np.uint8); h, w = src.shape
    dst = np.empty_like(src)
    mx = _f32(mx); my = _f32(my)
    lib().oracle_remap(_p(src), C.c_int(w), C.c_int(h), _p(mx), _p(my), _p(dst))
    return dst


def undistort_remap(src, K, D):
    src = np.ascontiguousarray(src, np.uint8); h, w = src.shape
    dst = np.empty_like(src)
    K = _f32(K); D = _f32(D)
    lib().oracle_undistort_remap(_p(src), C.c_int(w), C.c_int(h), _p(K), _p(D), _p(dst))
    return dst


def undistort_keypoints(kps, K, D):
    """Frame::UndistortKeyPoints (Frame.cc:915-945)."""
    kps = np.ascontiguousarray(kps, KP_DTYPE)
    out = np.empty_like(kps)
    K = _f32(K); D = _f32(D)
    lib().oracle_undistort_keypoints(_p(kps), C.c_int(len(kps)), _p(K), _p(D), _p(out))
    return out


def image_bounds(K, D, w, h):
    """Frame::ComputeImageBounds (Frame.cc:947-985) -> [minX, minY, maxX, maxY]."""
    b = np.empty(4, np.float32)
    K = _f32(K); D = _f32(D)
    lib().oracle_image_bounds(_p(K), _p(D), C.c_int(w), C.c_int(h), _p(b))
    return b


def is_in_frustum_points(Tcw, Ow, K, bounds, log_scale_factor, n_levels, cos_limit, pos, normal, min_dist, max_dist):
    """Frame::isInFrustum(MapPoint*) (Frame.cc:560-620)."""
    n = len(pos)
    Tcw = _f32(Tcw); Ow = _f32(Ow); K = _f32(K); bounds = _f32(bounds)
    pos = _f32(pos); normal = _f32(normal); min_dist = _f32(min_dist); max_dist = _f32(max_dist)
    inview = np.zeros(n, np.uint8); proj = np.zeros((n, 2), np.float32); level = np.zeros(n, np.int32); vc = np.zeros(n, np.float32)
    lib().oracle_is_in_frustum_points(_p(Tcw), _p(Ow), _p(K), _p(bounds), C.c_float(log_scale_factor), C.c_int(n_levels),
                                      C.c_float(cos_limit), C.c_int(n), _p(pos), _p(normal), _p(min_dist), _p(max_dist),
                                      _p(inview), _p(proj), _p(level), _p(vc))
    return inview, proj, level, vc


def is_in_frustum_lines(Tcw, Ow, K, bounds, log_scale_factor, cos_limit, pos, normal, min_dist, max_dist):
    """Frame::isInFrustum(MapLine*) (Frame.cc:622-702)."""
    n = len(pos)
    Tcw = _f32(Tcw); Ow = _f32(Ow); K = _f32(K); bounds = _f32(bounds)
    pos = np.ascontiguousarray(pos, np.float64); normal = np.ascontiguousarray(normal, np.float64)
    min_dist = _f32(min_dist); max_dist = _f32(max_dist)
    inview = np.zeros(n, np.uint8); proj = np.zeros((n, 4), np.float32); level = np.zeros(n, np.int32); vc = np.zeros(n, np.float32)
    lib().oracle_is_in_frustum_lines(_p(Tcw), _p(Ow), _p(K), _p(bounds), C.c_float(log_scale_factor), C.c_float(cos_limit),
                                     C.c_int(n), _p(pos), _p(normal), _p(min_dist), _p(max_dist), _p(inview), _p(proj),
                                     _p(level), _p(vc))
    return inview, proj, level, vc


# ----------------------------------------------------------------- LocalMapping matchers (ORBmatcher.cc:720-1065)
def _csr(fv):
    """fv: dict node -> list of feature indices (DBoW2::FeatureVector) -> (nodes asc, start, items)."""
    nodes = np.array(sorted(fv), np.uint32)
    start = np.zeros(len(nodes) + 1, np.int32); items = []
    for i, nd in enumerate(nodes):
        items += list(fv[int(nd)]); start[i + 1] = len(items)
    return nodes, start, np.array(items, np.int32).reshape(-1)


@_rec.entry("search_for_triangulation", ref_match_available)
def search_for_triangulation(k1, d1, has_mp1, k2, d2, has_mp2, fv1, fv2, F12, Cw1, R2w, t2w, K2, scale_factors2, level_sigma2_2,
                             check_orientation=True, impl="oracle"):
    k1 = np.ascontiguousarray(k1, KP_DTYPE); k2 = np.ascontiguousarray(k2, KP_DTYPE)
    d1 = np.ascontiguousarray(d1, np.uint8); d2 = np.ascontiguousarray(d2, np.uint8)
    m1 = np.ascontiguousarray(has_mp1, np.uint8); m2 = np.ascontiguousarray(has_mp2, np.uint8)
    n1a, s1, i1 = _csr(fv1); n2a, s2, i2 = _csr(fv2)
    F = _f32(F12); Cw = _f32(Cw1); R = _f32(R2w); t = _f32(t2w); K = _f32(K2); sf = _f32(scale_factors2); sg = _f32(level_sigma2_2)
    out = np.full(len(k1), -1, np.int32)
    f = _fn("search_for_triangulation", impl); f.restype = C.c_int
    nm = f(_p(k1), _p(d1), _p(m1), C.c_int(len(k1)), _p(k2), _p(d2), _p(m2), C.c_int(len(k2)),
                                           _p(n1a), _p(s1), _p(i1), C.c_int(len(n1a)), _p(n2a), _p(s2), _p(i2), C.c_int(len(n2a)),
                                           _p(F), _p(Cw), _p(R), _p(t), _p(K), _p(sf), _p(sg), C.c_int(int(check_orientation)), _p(out))
    return nm, out


@_rec.entry("fuse_search", ref_match_available)
def fuse_search(keys, desc, bounds, Tcw, Ow, K, scale_factors, inv_level_sigma2, log_scale_factor, skip, pos, normal, min_dist,
                max_dist, mp_desc, th=3.0, impl="oracle"):
    keys = np.ascontiguousarray(keys, KP_DTYPE); desc = np.ascontiguousarray(desc, np.uint8)
    b = _f32(bounds); T = _f32(Tcw); O = _f32(Ow); Kc = _f32(K); sf = _f32(scale_factors); iv = _f32(inv_level_sigma2)
    n_mp = len(pos)
    sk = None if skip is None else np.ascontiguousarray(skip, np.uint8)
    pos = _f32(pos); normal = _f32(normal); mn = _f32(min_dist); mx = _f32(max_dist); md = np.ascontiguousarray(mp_desc, np.uint8)
    bi = np.zeros(n_mp, np.int32); bd = np.zeros(n_mp, np.int32)
    args = [_p(keys), _p(desc), C.c_int(len(keys)), _p(b), _p(T), _p(O), _p(Kc), _p(sf), _p(iv), C.c_float(log_scale_factor), C.c_int(len(sf)),
            C.c_int(n_mp), _p(sk), _p(pos), _p(normal), _p(mn), _p(mx), _p(md), C.c_float(th), _p(bi)]
    if impl == "oracle":
        _fn("fuse_search", impl)(*args, _p(bd))
        return bi, bd
    f = _fn("fuse_search", impl); f.restype = C.c_int     # ORBmatcher::Fuse itself: (chosen keypoint per map point, nFused)
    return bi, f(*args)


@_rec.entry("lsd_search_for_triangulation", ref_match_available)
def lsd_search_for_triangulation(d1, has_ml1, d2, has_ml2, nnratio=0.8, is_double=True, th=80.0, impl="oracle"):
    """LSDmatcher::SearchForTriangulation(pKF1, pKF2, vMatchedPairs, isDouble) (LSDmatcher.cpp:727-776)."""
    d1 = np.ascontiguousarray(d1, np.uint8).reshape(-1, 32); d2 = np.ascontiguousarray(d2, np.uint8).reshape(-1, 32)
    m1 = np.ascontiguousarray(has_ml1, np.uint8); m2 = np.ascontiguousarray(has_ml2, np.uint8)
    out = np.full(len(d1), -1, np.int32)
    f = _fn("lsd_search_for_triangulation", impl); f.restype = C.c_int
    nm = f(_p(d1), _p(m1), C.c_int(len(d1)), _p(d2), _p(m2), C.c_int(len(d2)), C.c_float(th), C.c_float(nnratio), C.c_int(int(is_double)), _p(out))
    return nm, out


@_rec.entry("search_by_bow", ref_match_available)
def search_by_bow(kK, dK, has_mp_kf, kF, dF, fvK, fvF, nnratio=0.7, check_orientation=True, impl="oracle"):
    """ORBmatcher::SearchByBoW(pKF, F, vpMapPointMatches) (ORBmatcher.cc:187-327) -> (nmatches, matchesF[nF])."""
    kK = np.ascontiguousarray(kK, KP_DTYPE); kF = np.ascontiguousarray(kF, KP_DTYPE)
    dK = np.ascontiguousarray(dK, np.uint8); dF = np.ascontiguousarray(dF, np.uint8); mp = np.ascontiguousarray(has_mp_kf, np.uint8)
    n1a, s1, i1 = _csr(fvK); n2a, s2, i2 = _csr(fvF)
    out = np.full(len(kF), -1, np.int32)
    f = _fn("search_by_bow", impl); f.restype = C.c_int
    nm = f(_p(kK), _p(dK), _p(mp), C.c_int(len(kK)), _p(kF), _p(dF), C.c_int(len(kF)), _p(n1a), _p(s1), _p(i1),
                                C.c_int(len(n1a)), _p(n2a), _p(s2), _p(i2), C.c_int(len(n2a)), C.c_float(nnratio),
                                C.c_int(int(check_orientation)), _p(out))
    return nm, out


@_rec.entry("search_by_projection_keyframe", ref_match_available)
def search_by_projection_keyframe(kc, dc, bounds, Tcw, Ow, K, scale_factors, log_scale_factor, kf_valid, pos, mp_desc, min_dist,
                                  max_dist, kf_angle, th, orb_dist, check_orientation=True, preassigned=None, impl="oracle"):
    """ORBmatcher::SearchByProjection(CurrentFrame, pKF, sAlreadyFound, th, ORBdist) (ORBmatcher.cc:1587-1716).
    impl="ref": the reference itself; it derives the camera centre from Tcw and returns it as a third value."""
    kc = np.ascontiguousarray(kc, KP_DTYPE); dc = np.ascontiguousarray(dc, np.uint8)
    b = _f32(bounds); T = _f32(Tcw); O = _f32(Ow); Kc = _f32(K); sf = _f32(scale_factors)
    v = np.ascontiguousarray(kf_valid, np.uint8); pos = _f32(pos); md = np.ascontiguousarray(mp_desc, np.uint8)
    mn = _f32(min_dist); mx = _f32(max_dist); ang = _f32(kf_angle)
    pre = None if preassigned is None else np.ascontiguousarray(preassigned, np.uint8)
    out = np.full(len(kc), -1, np.int32)
    if impl == "ref":
        ow = np.zeros(3, np.float32)
        f = _fn("search_by_projection_keyframe", "ref"); f.restype = C.c_int
        nm = f(_p(kc), _p(dc), C.c_int(len(kc)), _p(b), _p(T), _p(Kc), _p(sf), C.c_int(len(sf)), C.c_float(log_scale_factor), C.c_int(len(v)), _p(v),
               _p(pos), _p(md), _p(mn), _p(mx), _p(ang), C.c_float(th), C.c_int(orb_dist), C.c_int(int(check_orientation)), _p(pre), _p(out), _p(ow))
        return nm, out, ow
    L = lib(); L.oracle_search_by_projection_keyframe.restype = C.c_int
    nm = L.oracle_search_by_projection_keyframe(_p(kc), _p(dc), C.c_int(len(kc)), _p(b), _p(T), _p(O), _p(Kc), _p(sf), C.c_int(len(sf)),
                                                C.c_float(log_scale_factor), C.c_int(len(v)), _p(v), _p(pos), _p(md), _p(mn), _p(mx),
                                                _p(ang), C.c_float(th), C.c_int(orb_dist), C.c_int(int(check_orientation)), _p(pre),
                                                _p(out))
    return nm, out


@_rec.entry("search_by_bow_keyframes", ref_match_available)
def search_by_bow_keyframes(k1, d1, mp1, k2, d2, mp2, fv1, fv2, nnratio=0.75, check_orientation=True, impl="oracle"):
    """ORBmatcher::SearchByBoW(pKF1, pKF2, vpMatches12) (ORBmatcher.cc:574-709) -> (nmatches, matches12[n1])."""
    k1 = np.ascontiguousarray(k1, KP_DTYPE); k2 = np.ascontiguousarray(k2, KP_DTYPE)
    d1 = np.ascontiguousarray(d1, np.uint8); d2 = np.ascontiguousarray(d2, np.uint8)
    m1 = np.ascontiguousarray(mp1, np.uint8); m2 = np.ascontiguousarray(mp2, np.uint8)
    n1a, s1, i1 = _csr(fv1); n2a, s2, i2 = _csr(fv2)
    out = np.full(len(k1), -1, np.int32)
    f = _fn("search_by_bow_keyframes", impl); f.restype = C.c_int
    nm = f(_p(k1), _p(d1), _p(m1), C.c_int(len(k1)), _p(k2), _p(d2), _p(m2), C.c_int(len(k2)), _p(n1a),
                                          _p(s1), _p(i1), C.c_int(len(n1a)), _p(n2a), _p(s2), _p(i2), C.c_int(len(n2a)),
                                          C.c_float(nnratio), C.c_int(int(check_orientation)), _p(out))
    return nm, out


def distinctive_descriptors(desc, offsets):
    """MapPoint::ComputeDistinctiveDescriptors (MapPoint.cc:249-314) for a CSR list of map points -> best index per point."""
    desc = np.ascontiguousarray(desc, np.uint8).reshape(-1, 32); off = np.ascontiguousarray(offsets, np.int32)
    best = np.zeros(len(off) - 1, np.int32)
    lib().oracle_distinctive_descriptors(_p(desc), _p(off), C.c_int(len(off) - 1), _p(best))
    return best


@_rec.entry("ref_distinctive_descriptors", ref_match_available, ref_only=True)
def ref_distinctive_descriptors(desc, offsets):
    """MapPoint::ComputeDistinctiveDescriptors of the reference itself -> the 32 bytes each point ends up with."""
    desc = np.ascontiguousarray(desc, np.uint8).reshape(-1, 32); off = np.ascontiguousarray(offsets, np.int32)
    out = np.zeros((len(off) - 1, 32), np.uint8)
    f = _fn("distinctive_descriptors", "ref"); f.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    f(_p(desc), _p(off), len(off) - 1, _p(out))
    return out


@_rec.entry("predict_scale", ref_match_available)
def predict_scale(dist, max_dist, log_scale_factor, n_levels, impl="oracle"):
    """MapPoint::PredictScale(currentDist, pKF): the oracle's restatement, or (impl="ref") the reference itself."""
    d = _f32(dist); mx = _f32(max_dist); out = np.zeros(len(d), np.int32)
    f = _fn("predict_scale", impl); f.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_float, C.c_int, C.c_void_p]
    f(_p(d), _p(mx), len(d), log_scale_factor, n_levels, _p(out))
    return out


def ref_predict_scale(dist, max_dist, log_scale_factor, n_levels):
    return predict_scale(dist, max_dist, log_scale_factor, n_levels, impl="ref")


@_rec.entry("lsd_fuse_search", ref_match_available)
def lsd_fuse_search(keylines, kf_point_desc, bounds, Tcw, Ow, K, scale_line, log_scale_factor_line, skip, pos, normal, min_dist, max_dist,
                    ml_desc, th=3.0, impl="oracle"):
    """Search half of LSDmatcher::Fuse (LSDmatcher.cpp:860-1011) -> (best_idx, best_dist, stop_at);
    impl="ref": LSDmatcher::Fuse itself -> (chosen keyline per map line, Fuse's return value)."""
    kl = np.ascontiguousarray(keylines); pd = np.ascontiguousarray(kf_point_desc, np.uint8).reshape(-1, 32)
    b = _f32(bounds); T = _f32(Tcw); O = _f32(Ow); Kc = _f32(K)
    n = len(pos)
    sk = np.ascontiguousarray(skip, np.uint8); P = np.ascontiguousarray(pos, np.float64); Nn = np.ascontiguousarray(normal, np.float64)
    mn = _f32(min_dist); mx = _f32(max_dist); md = np.ascontiguousarray(ml_desc, np.uint8).reshape(-1, 32)
    bi = np.zeros(n, np.int32); bd = np.zeros(n, np.int32); stop = C.c_int(n)
    if impl == "ref":
        ret = C.c_int(0)
        _fn("lsd_fuse_search", "ref")(_p(kl), C.c_int(len(kl)), _p(pd), C.c_int(len(pd)), _p(b), _p(T), _p(O), _p(Kc), C.c_float(scale_line), C.c_int(1),
                                      C.c_float(log_scale_factor_line), C.c_int(n), _p(sk), _p(P), _p(Nn), _p(mn), _p(mx), _p(md), C.c_float(th),
                                      _p(bi), C.byref(ret))
        return bi, ret.value
    lib().oracle_lsd_fuse_search(_p(kl), C.c_int(len(kl)), _p(pd), C.c_int(len(pd)), _p(b), _p(T), _p(O), _p(Kc), C.c_float(scale_line), C.c_int(1),
                                 C.c_float(log_scale_factor_line), C.c_int(n), _p(sk), _p(P), _p(Nn), _p(mn), _p(mx), _p(md), C.c_float(th),
                                 _p(bi), _p(bd), C.byref(stop))
    return bi, bd, stop.value
