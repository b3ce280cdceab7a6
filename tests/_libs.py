"""ctypes loaders shared by the tests: the oracle restatement, the real reference build
(oracle/_ref, when present) and synthetic-input generators.  TEST INFRASTRUCTURE only."""
import ctypes as C
import hashlib
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")


class Image(C.Structure):
    _fields_ = [("w", C.c_uint), ("h", C.c_uint), ("data", C.c_void_p)]


class Keypoint(C.Structure):
    _fields_ = [("x", C.c_uint), ("y", C.c_uint), ("response", C.c_uint), ("angle", C.c_float),
                ("descriptor", C.c_uint32 * 8)]


class Point(C.Structure):
    _fields_ = [("x", C.c_uint), ("y", C.c_uint)]


class Rect(C.Structure):
    _fields_ = [("x", C.c_uint), ("y", C.c_uint), ("w", C.c_uint), ("h", C.c_uint)]


class Cascade(C.Structure):
    _fields_ = [
        ("window_w", C.c_uint16), ("window_h", C.c_uint16),
        ("nfeatures", C.c_uint16), ("nweaks", C.c_uint16), ("nstages", C.c_uint16),
        ("features", C.c_void_p), ("weak_feature_idx", C.c_void_p),
        ("weak_left_val", C.c_void_p), ("weak_right_val", C.c_void_p),
        ("weak_subset_offset", C.c_void_p), ("weak_num_subsets", C.c_void_p),
        ("subsets", C.c_void_p), ("stage_weak_start", C.c_void_p), ("stage_nweaks", C.c_void_p),
        ("stage_threshold", C.c_void_p),
    ]


MATCH_DTYPE = np.dtype([("idx1", "<u4"), ("idx2", "<u4"), ("distance", "<u4")])
KP_DTYPE = np.dtype([("x", "<u4"), ("y", "<u4"), ("response", "<u4"), ("angle", "<f4"),
                     ("descriptor", "<u4", (8,))])
RECT_DTYPE = np.dtype([("x", "<u4"), ("y", "<u4"), ("w", "<u4"), ("h", "<u4")])
# struct gs_blob (reference grayskull.h:29-34): u16 label + 2 padding bytes, area, box, centroid = 32 bytes
BLOB_DTYPE = np.dtype({"names": ["label", "area", "bx", "by", "bw", "bh", "cx", "cy"],
                       "formats": ["<u2", "<u4", "<u4", "<u4", "<u4", "<u4", "<u4", "<u4"],
                       "offsets": [0, 4, 8, 12, 16, 20, 24, 28], "itemsize": 32})
assert KP_DTYPE.itemsize == 48 and RECT_DTYPE.itemsize == 16 and C.sizeof(Cascade) == 96


def ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def img(a):
    """numpy (h, w) uint8 array -> struct gs_image by value"""
    assert a.dtype == np.uint8 and a.flags.c_contiguous
    return Image(a.shape[1], a.shape[0], a.ctypes.data)


def build_oracle():
    subprocess.run(["make", "-s", "-C", ORACLE_DIR, "all"], check=True)


_cache = {}


def oracle():
    """our C restatement (oracle/libgs_oracle.so)"""
    if "o" not in _cache:
        path = os.path.join(ORACLE_DIR, "libgs_oracle.so")
        if not os.path.exists(path) or os.path.getmtime(path) < os.path.getmtime(
                os.path.join(ORACLE_DIR, "gs_oracle.c")):
            build_oracle()
        lib = C.CDLL(path)
        lib.gso_fast.restype = C.c_uint
        lib.gso_orb_extract.restype = C.c_uint
        lib.gso_lbp_window.restype = C.c_uint
        lib.gso_lbp_detect.restype = C.c_uint
        lib.gso_compute_orientation.restype = C.c_float
        lib.gso_sinf.restype = C.c_float
        lib.gso_sinf.argtypes = [C.c_float]
        lib.gso_atan2f.restype = C.c_float
        lib.gso_atan2f.argtypes = [C.c_float, C.c_float]
        lib.gso_match_orb.restype = C.c_uint
        lib.gso_lbp_depth_map.restype = None
        lib.gso_lbp_depth_map.argtypes = [C.c_void_p, C.c_void_p, C.c_uint, C.c_uint, C.c_float, C.c_int, C.c_void_p]
        lib.gso_filter.restype = None
        lib.gso_filter.argtypes = [C.c_void_p, C.c_void_p, C.c_uint, C.c_uint, C.c_void_p, C.c_uint, C.c_uint, C.c_uint]
        lib.gso_match_template.restype = None
        lib.gso_match_template.argtypes = [C.c_void_p, C.c_uint, C.c_uint, C.c_void_p, C.c_uint, C.c_uint, C.c_void_p]
        lib.gso_find_best_match.restype = C.c_uint
        lib.gso_find_best_match.argtypes = [C.c_void_p, C.c_uint, C.c_uint]
        lib.gso_histogram.restype = None
        lib.gso_histogram.argtypes = [C.c_void_p, C.c_uint, C.c_uint, C.c_void_p]
        lib.gso_otsu_from_hist.restype = C.c_uint
        lib.gso_otsu_from_hist.argtypes = [C.c_void_p, C.c_uint]
        lib.gso_otsu_threshold.restype = C.c_uint
        lib.gso_otsu_threshold.argtypes = [C.c_void_p, C.c_uint, C.c_uint]
        lib.gso_threshold.restype = None
        lib.gso_threshold.argtypes = [C.c_void_p, C.c_uint, C.c_uint, C.c_uint]
        lib.gso_match_orb.argtypes = [C.c_void_p, C.c_uint, C.c_void_p, C.c_uint, C.c_void_p, C.c_uint, C.c_float]
        lib.gso_blobs.restype = C.c_uint
        lib.gso_blobs.argtypes = [C.c_void_p, C.c_uint, C.c_uint, C.c_void_p, C.c_void_p, C.c_uint]
        lib.gso_blob_corners.restype = None
        lib.gso_blob_corners.argtypes = [C.c_void_p, C.c_uint, C.c_uint, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.gso_perspective_correct.restype = None
        lib.gso_perspective_correct.argtypes = [C.c_void_p, C.c_uint, C.c_uint, C.c_void_p, C.c_uint, C.c_uint, C.c_void_p]
        lib.gso_compute_orientation.argtypes = [C.c_void_p, C.c_uint, C.c_uint, C.c_uint, C.c_uint, C.c_uint]
        lib.gso_lbp_window.argtypes = [C.c_void_p, C.c_void_p, C.c_uint, C.c_uint, C.c_int, C.c_int,
                                       C.c_float]
        lib.gso_lbp_detect.argtypes = [C.c_void_p, C.c_void_p, C.c_uint, C.c_uint, C.c_void_p,
                                       C.c_uint, C.c_float, C.c_float, C.c_float, C.c_int]
        _cache["o"] = lib
    return _cache["o"]


def have_ref():
    return os.path.exists(os.path.join(ORACLE_DIR, "_ref", "libgs_ref.so"))


def ref():
    """the UNMODIFIED reference header compiled as a shared object (oracle/_ref)"""
    if "r" not in _cache:
        lib = C.CDLL(os.path.join(ORACLE_DIR, "_ref", "libgs_ref.so"))
        for name in ("gs_blur", "gs_sobel", "gs_erode", "gs_dilate", "gs_resize", "gs_downsample"):
            getattr(lib, name).restype = None
        lib.gs_blur.argtypes = [Image, Image, C.c_uint]
        lib.gs_sobel.argtypes = [Image, Image]
        lib.gs_erode.argtypes = [Image, Image]
        lib.gs_dilate.argtypes = [Image, Image]
        lib.gs_resize.argtypes = [Image, Image]
        lib.gs_downsample.argtypes = [Image, Image]
        lib.gs_adaptive_threshold.argtypes = [Image, Image, C.c_uint, C.c_int]
        lib.gs_adaptive_threshold.restype = None
        lib.gs_integral.argtypes = [Image, C.c_void_p]
        lib.gs_integral.restype = None
        lib.gs_fast.argtypes = [Image, Image, C.c_void_p, C.c_uint, C.c_uint]
        lib.gs_fast.restype = C.c_uint
        lib.gs_compute_orientation.argtypes = [Image, C.c_uint, C.c_uint, C.c_uint]
        lib.gs_compute_orientation.restype = C.c_float
        lib.gs_brief_descriptor.argtypes = [Image, C.c_void_p]
        lib.gs_brief_descriptor.restype = None
        lib.gs_orb_extract.argtypes = [Image, C.c_void_p, C.c_uint, C.c_uint, C.c_void_p]
        lib.gs_orb_extract.restype = C.c_uint
        lib.gs_lbp_window.argtypes = [C.c_void_p, C.c_void_p, C.c_uint, C.c_uint, C.c_int, C.c_int,
                                      C.c_float]
        lib.gs_lbp_window.restype = C.c_uint
        lib.gs_lbp_detect.argtypes = [C.c_void_p, C.c_void_p, C.c_uint, C.c_uint, C.c_void_p,
                                      C.c_uint, C.c_float, C.c_float, C.c_float, C.c_int]
        lib.gs_lbp_detect.restype = C.c_uint
        lib.gs_match_orb.argtypes = [C.c_void_p, C.c_uint, C.c_void_p, C.c_uint, C.c_void_p, C.c_uint, C.c_float]
        lib.gs_match_orb.restype = C.c_uint
        lib.gs_filter.argtypes = [Image, Image, Image, C.c_uint]
        lib.gs_filter.restype = None
        lib.gs_match_template.argtypes = [Image, Image, Image]
        lib.gs_match_template.restype = None
        lib.gs_find_best_match.argtypes = [Image]
        lib.gs_find_best_match.restype = Point
        lib.gs_histogram.argtypes = [Image, C.c_void_p]
        lib.gs_histogram.restype = None
        lib.gs_otsu_threshold.argtypes = [Image]
        lib.gs_otsu_threshold.restype = C.c_uint8
        lib.gs_threshold.argtypes = [Image, C.c_uint8]
        lib.gs_threshold.restype = None
        lib.gs_blobs.argtypes = [Image, C.c_void_p, C.c_void_p, C.c_uint]
        lib.gs_blobs.restype = C.c_uint
        lib.gs_blob_corners.argtypes = [Image, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.gs_blob_corners.restype = None
        lib.gs_perspective_correct.argtypes = [Image, Image, C.c_void_p]
        lib.gs_perspective_correct.restype = None
        lib.ref_frontalface.restype = C.c_void_p
        lib.ref_sort_keypoints.argtypes = [C.c_void_p, C.c_uint]
        lib.ref_sort_keypoints.restype = None
        _cache["r"] = lib
    return _cache["r"]


def digest(x):
    """16-byte digest of an output or an input tuple: arrays by dtype, shape and bytes, Python ints as int64, floats
    as float64 (exact for the c_float results), tuples / lists element by element, RefDigest as itself"""
    if isinstance(x, RefDigest):
        return x
    h = hashlib.blake2b(digest_size=16)

    def feed(v):
        if isinstance(v, (tuple, list)):
            h.update(b"(%d" % len(v))
            for e in v:
                feed(e)
        elif isinstance(v, np.ndarray):
            h.update(v.dtype.str.encode() + repr(v.shape).encode()); h.update(np.ascontiguousarray(v).tobytes())
        elif isinstance(v, (bool, int, np.integer)):
            h.update(b"i"); h.update(np.int64(v).tobytes())
        elif isinstance(v, (float, np.floating)):
            h.update(b"f"); h.update(np.float64(v).tobytes())
        elif isinstance(v, str):
            h.update(b"s" + v.encode())
        else:
            raise TypeError(type(v))
    feed(x)
    return RefDigest(h.digest())


class RefDigest(bytes):
    """a reference output known by its digest only (replayed from tests/golden/ref_digests.npz)"""


def same(want, got):
    """exact equality of a reference output (array, scalar or RefDigest) and an oracle output"""
    return digest(want) == digest(got)


REF_DIGESTS = os.path.join(ROOT, "tests", "golden", "ref_digests.npz")


class RefRecord:
    """The compiled reference (oracle/_ref/libgs_ref.so) as the differential tests see it: `R.blur(a, 5)` is what
    the reference's gs_blur returns for that input.  By default every call is replayed from
    tests/golden/ref_digests.npz: the stored entry must have been made from the same operation and inputs, and
    its output digest is returned (compare with `same`).  With GS_REF_RECORD=1 and oracle/_ref built, the
    reference itself is called, the test compares against its real outputs, and the stream is (re)written.

    Two costs of storing digests instead of arrays: a replayed mismatch says which call differs, not where in the
    output (re-run with GS_REF_RECORD=1 to compare real arrays); and the input digests pin the inputs the tests draw
    from numpy's Generator streams, so a numpy release that changes those streams fails every call with "is not the
    recorded one" until the file is re-recorded with the reference build."""

    def __init__(self, name):
        self.name, self.pos, self.rows = name, 0, []
        self.record = os.environ.get("GS_REF_RECORD") == "1"
        if self.record:
            assert have_ref(), "GS_REF_RECORD=1 needs oracle/_ref/libgs_ref.so (make -C oracle REF=<reference tree>)"
        else:
            z = np.load(REF_DIGESTS)
            self.stored = z[name]             # (calls, 2, 16) uint8: input digest, output digest

    def __getattr__(self, op):
        if op not in _REF_OPS:
            raise AttributeError(op)
        return lambda *args: self._call(op, args)

    def _call(self, op, args):
        key = digest((op,) + tuple(args))
        if self.record:
            out = _REF_OPS[op](ref(), *args)
            self.rows.append((key, digest(out)))
            return out
        assert self.pos < len(self.stored), "%s: more reference calls than recorded (%s)" % (self.name, op)
        k, out = bytes(self.stored[self.pos, 0]), bytes(self.stored[self.pos, 1])
        assert k == key, "%s: call %d (%s%r) is not the recorded one" % (self.name, self.pos, op, tuple(
            a if np.isscalar(a) else getattr(a, "shape", "...") for a in args))
        self.pos += 1
        return RefDigest(out)

    def finish(self):
        if not self.record:
            assert self.pos == len(self.stored), "%s: %d of %d recorded calls made" % (self.name, self.pos, len(self.stored))
            return
        rows = np.frombuffer(b"".join(k + o for k, o in self.rows), np.uint8).reshape(-1, 2, 16)
        old = dict(np.load(REF_DIGESTS)) if os.path.exists(REF_DIGESTS) else {}
        old[self.name] = rows
        np.savez_compressed(REF_DIGESTS, **old)


def _into(fn, shape_of=lambda a: a.shape, fill=0):
    """a reference call fn(dst, src, *args) that writes a uint8 image of shape shape_of(src)"""
    def run(R, a, *args):
        d = np.full(shape_of(a), fill, np.uint8)
        getattr(R, fn)(img(d), img(a), *args)
        return d
    return run


def _ref_resize(R, a, dw, dh):
    d = np.empty((dh, dw), np.uint8)
    R.gs_resize(img(d), img(a))
    return d


def _ref_integral(R, a):
    ii = np.empty(a.shape, np.uint32)
    R.gs_integral(img(a), ptr(ii))
    return ii


def _ref_fast(R, a, sm0, cap, t):
    sm, k = sm0.copy(), np.zeros(cap, KP_DTYPE)
    n = R.gs_fast(img(a), img(sm), ptr(k), cap, t)
    return sm, k[:n]


def _ref_orb(R, a, nk, t):
    k, sm = np.zeros(nk, KP_DTYPE), np.zeros_like(a)
    return k[:R.gs_orb_extract(img(a), ptr(k), nk, t, ptr(sm))]


def _ref_sort(R, k):
    k = k.copy()
    R.ref_sort_keypoints(ptr(k), len(k))
    return k


def _ref_libm(fn, *cols):
    f = getattr(C.CDLL("libm.so.6"), fn)
    f.restype, f.argtypes = C.c_float, [C.c_float] * len(cols)
    return np.array([f(*(float(c[i]) for c in cols)) for i in range(len(cols[0]))], np.float32)


def _ref_lbp_detect(R, ii, mr, sf, mn, mx, st):
    rr = np.zeros(mr, RECT_DTYPE)
    return rr[:R.gs_lbp_detect(R.ref_frontalface(), ptr(ii), ii.shape[1], ii.shape[0], ptr(rr), mr, sf, mn, mx, st)]


def _ref_match_orb(R, k1, k2, mm, md):
    m = np.zeros(max(mm, 1), MATCH_DTYPE)
    return m[:R.gs_match_orb(ptr(k1), len(k1), ptr(k2), len(k2), ptr(m), mm, md)]


def _ref_histogram(R, a):
    h = np.zeros(256, np.uint32)
    R.gs_histogram(img(a), ptr(h))
    return h


def _ref_threshold(R, a, t):
    x = a.copy()
    R.gs_threshold(img(x), t)
    return x


def _ref_filter(R, a, k, norm):
    d = np.zeros_like(a)
    R.gs_filter(img(d), img(a), img(k), norm)
    return d


def _ref_match_template(R, a, tmpl):
    rw, rh = a.shape[1] - tmpl.shape[1] + 1, a.shape[0] - tmpl.shape[0] + 1
    rr = np.zeros((rh, rw), np.uint8)
    R.gs_match_template(img(a), img(tmpl), img(rr))
    p = R.gs_find_best_match(img(rr))
    return rr, p.y * rw + p.x


def _ref_find_best_match(R, r):
    p = R.gs_find_best_match(img(r))
    return p.x, p.y


def _ref_blobs(R, a, nb):
    labels, blobs = np.full(a.shape, 0x5555, np.uint16), np.zeros(nb, BLOB_DTYPE)
    m = R.gs_blobs(img(a), ptr(labels), ptr(blobs), nb)
    return labels, blobs[:m]


def blobs_result(labels, blobs):
    """(labels, defined gs_blob fields as an (n, 8) int64 array): what the blob tests compare"""
    return labels, np.array(blob_fields(blobs), np.int64).reshape(-1, 8)


def _ref_blob_corners(R, a, nb, j):
    labels, blobs = _ref_blobs(R, a, nb)
    c = np.zeros((4, 2), np.uint32)
    R.gs_blob_corners(img(a), ptr(labels), ptr(blobs[j:j + 1]), ptr(c))
    return c


def _ref_perspective(R, src, dw, dh, c):
    d = np.empty((dh, dw), np.uint8)
    R.gs_perspective_correct(img(d), img(src), ptr(c))
    return d


_REF_OPS = {
    "blur": _into("gs_blur"),
    "adaptive": _into("gs_adaptive_threshold"),
    "erode": _into("gs_erode"),
    "dilate": _into("gs_dilate"),
    "sobel77": _into("gs_sobel", fill=77),
    "downsample": _into("gs_downsample", lambda a: (a.shape[0] // 2, a.shape[1] // 2)),
    "resize": _ref_resize,
    "integral": _ref_integral,
    "fast": _ref_fast,
    "orb_extract": _ref_orb,
    "sort_keypoints": _ref_sort,
    "libm_sinf": lambda R, xs: _ref_libm("sinf", xs),
    "libm_atan2f": lambda R, ys, xs: _ref_libm("atan2f", ys, xs),
    "lbp_detect": _ref_lbp_detect,
    "lbp_window": lambda R, ii, x, y, s: R.gs_lbp_window(R.ref_frontalface(), ptr(ii), ii.shape[1], ii.shape[0], x, y, s),
    "match_orb": _ref_match_orb,
    "histogram": _ref_histogram,
    "otsu": lambda R, a: int(R.gs_otsu_threshold(img(a))),
    "threshold": _ref_threshold,
    "filter": _ref_filter,
    "match_template": _ref_match_template,
    "find_best_match": _ref_find_best_match,
    "blobs": lambda R, a, nb: blobs_result(*_ref_blobs(R, a, nb)),
    "blob_corners": _ref_blob_corners,
    "perspective": _ref_perspective,
    "orientation": lambda R, a, x, y, r: R.gs_compute_orientation(img(a), x, y, r),
}


class HostCascade:
    """frontalface tables from the committed fixture, as a struct gs_lbp_cascade on the host"""

    def __init__(self, path=None):
        path = path or os.path.join(ROOT, "grayskull_b200", "data", "frontalface.npz")
        z = np.load(path)
        self.arrays = {k: np.ascontiguousarray(z[k]) for k in z.files}
        a = self.arrays
        self.struct = Cascade(int(a["window"][0]), int(a["window"][1]), len(a["features"]) // 4,
                              len(a["weak_feature_idx"]), len(a["stage_threshold"]),
                              a["features"].ctypes.data, a["weak_feature_idx"].ctypes.data,
                              a["weak_left_val"].ctypes.data, a["weak_right_val"].ctypes.data,
                              a["weak_subset_offset"].ctypes.data, a["weak_num_subsets"].ctypes.data,
                              a["subsets"].ctypes.data, a["stage_weak_start"].ctypes.data,
                              a["stage_nweaks"].ctypes.data, a["stage_threshold"].ctypes.data)

    @property
    def ptr(self):
        return C.addressof(self.struct)


def xorshift_frame(w, h, f=0):
    """SURVEY.md 8(d) synthetic input: 64-bit xorshift, seed 0x9E3779B97F4A7C15 + f, top byte"""
    n = w * h
    out = np.empty(n, np.uint8)
    s = np.uint64((0x9E3779B97F4A7C15 + f) & 0xFFFFFFFFFFFFFFFF)
    # vectorised in blocks: xorshift is sequential, so run it in a small python loop over a
    # jump-free chunk using numpy scalars only for small frames; large frames use the C-speed
    # generator below.
    if n > 1 << 16:
        return _xorshift_big(w, h, f)
    s = int(s)
    M = (1 << 64) - 1
    for i in range(n):
        s ^= (s << 13) & M
        s ^= s >> 7
        s ^= (s << 17) & M
        out[i] = s >> 56
    return out.reshape(h, w)


def _xorshift_big(w, h, f):
    # numpy's PCG is fine for big parity inputs; the exact xorshift stream only matters for the
    # documented small fixtures.  Seeded per frame for reproducibility.
    rng = np.random.default_rng(0x9E3779B9 + f)
    return rng.integers(0, 256, size=(h, w), dtype=np.uint8)


def natural_like(w, h, seed=0):
    """smooth-ish random image (sum of blobs + noise) so FAST/LBP see structure"""
    rng = np.random.default_rng(seed)
    small = rng.integers(0, 256, size=((h + 7) // 8 + 1, (w + 7) // 8 + 1)).astype(np.float32)
    up = np.kron(small, np.ones((8, 8), np.float32))[:h, :w]
    noise = rng.normal(0, 12, size=(h, w)).astype(np.float32)
    return np.clip(up * 0.7 + noise + 30, 0, 255).astype(np.uint8)


def blob_fields(b):
    """the defined fields of a gs_blob array (the 2 padding bytes after `label` are not part of the contract)"""
    return [tuple(int(b[k][i]) for k in BLOB_DTYPE.names) for i in range(len(b))]


def binary_like(w, h, seed, density=0.5, smooth=3):
    """0 / 255 image with blobs of assorted sizes (thresholded smooth noise) plus salt noise: many small
    components, a few large ones, touching the borders"""
    rng = np.random.default_rng(seed)
    a = rng.random((h + 2 * smooth, w + 2 * smooth)).astype(np.float32)
    k = 2 * smooth + 1
    c = np.cumsum(np.cumsum(np.pad(a, ((1, 0), (1, 0))), 0), 1)
    box = (c[k:, k:] - c[:-k, k:] - c[k:, :-k] + c[:-k, :-k]) / (k * k)
    img = (box[:h, :w] > np.quantile(box, 1 - density)).astype(np.uint8) * 255
    salt = rng.random((h, w))
    img[salt < 0.02] = 255
    img[salt > 0.98] = 0
    img[rng.random((h, w)) < 0.01] = 130          # values just above / below the >= 128 foreground test
    img[rng.random((h, w)) < 0.01] = 127
    return np.ascontiguousarray(img)


def desc_sets(rng, n1, n2, dup=0.3):
    """descriptor sets with near-duplicates and exact duplicates so ties and the ratio test trigger"""
    k1 = np.zeros(n1, KP_DTYPE); k2 = np.zeros(n2, KP_DTYPE)
    k2["descriptor"] = rng.integers(0, 2**32, (n2, 8), dtype=np.uint64).astype(np.uint32)
    k1["descriptor"] = rng.integers(0, 2**32, (n1, 8), dtype=np.uint64).astype(np.uint32)
    for i in range(n1):
        if n2 and rng.random() < dup:
            j = int(rng.integers(0, n2))
            d = k2["descriptor"][j].copy()
            for _ in range(int(rng.integers(0, 40))):
                d[int(rng.integers(0, 8))] ^= np.uint32(1 << int(rng.integers(0, 32)))
            k1["descriptor"][i] = d
    if n2 > 4:                                   # exact duplicates inside set 2: best == second
        k2["descriptor"][1] = k2["descriptor"][0]
    return k1, k2


FILTER_KERNELS = {   # (weights as int8 rows, norm): the reference's presets (grayskull.h:249-253) and stress cases
    "sharpen": ([[0, -1, 0], [-1, 5, -1], [0, -1, 0]], 1),
    "emboss": ([[-2, -1, 0], [-1, 1, 1], [0, 1, 2]], 1),
    "box": ([[1, 1, 1], [1, 1, 1], [1, 1, 1]], 9),
    "gaussian": ([[1, 2, 1], [2, 4, 2], [1, 2, 1]], 16),
    "emboss_norm3": ([[-2, -1, 0], [-1, 1, 1], [0, 1, 2]], 3),       # negative sums with norm > 1 -> 255
    "extreme": ([[127, -128, 127], [-128, 127, -128], [127, -128, 127]], 7),
    "huge_norm": ([[1, 1, 1], [1, 1, 1], [1, 1, 1]], 3000000000),     # norm above 2^31
    "big_norm_neg": ([[-1, 0, 0], [0, 0, 0], [0, 0, 0]], 20000000),   # (2^32 - s) / norm below 255
    "k5": ([[1, 4, 6, 4, 1], [4, 16, 24, 16, 4], [6, 24, 36, 24, 6], [4, 16, 24, 16, 4], [1, 4, 6, 4, 1]], 256),
    "k2x4": ([[1, -2, 3, -4], [5, 6, -7, 8]], 5),                     # even sizes: taps at -kw/2 .. kw-1-kw/2
    "k1x1": ([[3]], 2),
    "k7x3": ([[1, 0, -1, 2, -1, 0, 1], [2, 0, -2, 4, -2, 0, 2], [1, 0, -1, 2, -1, 0, 1]], 4),
}


def filter_kernel(name):
    rows, norm = FILTER_KERNELS[name]
    return np.ascontiguousarray(np.array(rows, np.int8).view(np.uint8)), norm


def check_next_golden(impl):
    """tests/golden/next_golden.npz (made by the REAL reference, tools/make_golden.py) against `impl`, an object
    with gs_histogram(a), gs_otsu_threshold(a), gs_threshold(a, t), gs_filter(dst, src, kernel_u8, norm),
    gs_match_template(img, tmpl), gs_find_best_match(res) -> (x, y), gs_orb(a, nkps, t), gs_match_orb(k1, k2, mm, md).
    Shared by the oracle test (CPU) and the CUDA test (GPU) so the checking logic itself is exercised on both."""
    z = np.load(os.path.join(ROOT, "tests", "golden", "next_golden.npz"))
    for tag in [str(t) for t in z["tags"]]:
        a = np.ascontiguousarray(z[tag + "img"])
        assert np.array_equal(impl.gs_histogram(a), z[tag + "hist"]), tag
        t = int(z[tag + "otsu"])
        assert impl.gs_otsu_threshold(a) == t, tag
        assert np.array_equal(impl.gs_threshold(a.copy(), t), z[tag + "threshold_otsu"]), tag
        for name in ("sharpen", "emboss", "box", "gaussian", "emboss_norm3", "k5", "k2x4"):
            k, norm = filter_kernel(name)
            assert np.array_equal(impl.gs_filter(np.zeros_like(a), a, k, norm), z[tag + "filter_" + name]), (tag, name)
        res = impl.gs_match_template(a, np.ascontiguousarray(z[tag + "tmpl"]))
        assert np.array_equal(res, z[tag + "tmatch"]), tag
        assert tuple(impl.gs_find_best_match(res)) == tuple(int(v) for v in z[tag + "tmatch_best"]), tag
        ka, kb = impl.gs_orb(a, 300, 20), impl.gs_orb(np.ascontiguousarray(z[tag + "shifted"]), 300, 20)
        assert ka.tobytes() == z[tag + "kps_a"].tobytes() and kb.tobytes() == z[tag + "kps_b"].tobytes(), tag
        m = impl.gs_match_orb(ka, kb, 300, 60.0)
        assert m.tobytes() == z[tag + "matches"].tobytes() and len(m) > 20, tag


def oracle_chain(cascade_ptr, frame, **params):
    """the C5 chain of grayskull_b200/pipeline.py (blur r=5 -> sobel -> orb_extract / integral + lbp_detect on
    the sobel map) on one frame through the oracle restatement"""
    import sys
    O, L = oracle(), sys.modules[__name__]
    p = dict(radius=5, nkps=1250, threshold=20, max_rects=4096, scale_factor=1.1, min_scale=1.0, max_scale=4.0, step=2)
    p.update(params)
    h, w = frame.shape
    b = np.empty_like(frame)
    O.gso_blur(L.ptr(b), L.ptr(frame), w, h, p["radius"])
    s = np.zeros_like(frame)
    O.gso_sobel(L.ptr(s), L.ptr(b), w, h)
    k = np.zeros(p["nkps"], L.KP_DTYPE)
    sm = np.zeros_like(frame)
    nk = O.gso_orb_extract(L.ptr(s), w, h, L.ptr(k), p["nkps"], p["threshold"], L.ptr(sm))
    t = np.empty(frame.shape, np.uint32)
    O.gso_integral(L.ptr(s), w, h, L.ptr(t))
    r = np.zeros(p["max_rects"], L.RECT_DTYPE)
    nr = O.gso_lbp_detect(cascade_ptr, L.ptr(t), w, h, L.ptr(r), p["max_rects"], p["scale_factor"], p["min_scale"],
                          p["max_scale"], p["step"])
    return {"sobel": s, "kps": k[:nk], "rects": r[:nr]}
