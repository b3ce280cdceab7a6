"""Pins the oracle (oracle/gs_oracle.c): (a) the literal vectors of the reference's own test.c,
(b) differential runs against the real reference build on random inputs (its outputs recorded as digests in
tests/golden/ref_digests.npz, see _libs.RefRecord), (c) the reference-generated fixtures in tests/golden/.  CPU only."""
import hashlib
import os

import numpy as np

import _libs as L

O = L.oracle()
GOLD = os.path.join(L.ROOT, "tests", "golden")


def o_blur(a, r):
    d = np.empty_like(a); O.gso_blur(L.ptr(d), L.ptr(a), a.shape[1], a.shape[0], r); return d
def o_adaptive(a, r, c):
    d = np.empty_like(a); O.gso_adaptive_threshold(L.ptr(d), L.ptr(a), a.shape[1], a.shape[0], r, c); return d
def o_morph(a, dil):
    d = np.empty_like(a); O.gso_morph(L.ptr(d), L.ptr(a), a.shape[1], a.shape[0], dil); return d
def o_sobel(a, fill=0):
    d = np.full_like(a, fill); O.gso_sobel(L.ptr(d), L.ptr(a), a.shape[1], a.shape[0]); return d
def o_resize(a, dw, dh):
    d = np.empty((dh, dw), np.uint8); O.gso_resize(L.ptr(d), dw, dh, L.ptr(a), a.shape[1], a.shape[0]); return d
def o_down(a):
    d = np.empty((a.shape[0] // 2, a.shape[1] // 2), np.uint8); O.gso_downsample(L.ptr(d), L.ptr(a), a.shape[1], a.shape[0]); return d
def o_integral(a):
    ii = np.empty(a.shape, np.uint32); O.gso_integral(L.ptr(a), a.shape[1], a.shape[0], L.ptr(ii)); return ii
def o_fast(a, sm, nkps, t):
    k = np.zeros(nkps, L.KP_DTYPE)
    n = O.gso_fast(L.ptr(a), a.shape[1], a.shape[0], L.ptr(sm), sm.shape[1], sm.shape[0], L.ptr(k), nkps, t)
    return k[:n]
def o_orb(a, sm, nkps, t):
    k = np.zeros(nkps, L.KP_DTYPE)
    n = O.gso_orb_extract(L.ptr(a), a.shape[1], a.shape[0], L.ptr(k), nkps, t, L.ptr(sm))
    return k[:n]
def o_detect(cas, ii, max_rects, sf, mn, mx, step):
    r = np.zeros(max_rects, L.RECT_DTYPE)
    n = O.gso_lbp_detect(cas.ptr, L.ptr(ii), ii.shape[1], ii.shape[0], L.ptr(r), max_rects, sf, mn, mx, step)
    return r[:n]


# ---------------------------------------------------------------- (a) reference test.c vectors
def test_kat_resize():  # reference test.c:24-68
    a = np.array([[0, 50, 100, 150], [25, 75, 125, 175], [50, 100, 150, 200], [75, 125, 175, 225]], np.uint8)
    d = o_resize(a, 2, 2)
    assert d.tolist() == [[37, 137], [87, 187]]
    up = o_resize(d, 4, 4)
    assert up.tolist() == [[37, 62, 112, 137], [49, 74, 124, 149], [74, 99, 149, 174], [87, 112, 162, 187]]
    s = np.array([[10, 20], [30, 40]], np.uint8)
    assert o_resize(s, 2, 2).tolist() == s.tolist()


def test_kat_blur():  # reference test.c:72-86
    a = np.zeros((3, 3), np.uint8); a[1, 1] = 255
    d = o_blur(a, 1)
    assert d[1, 1] == 28 and d[0, 0] == 63


def test_kat_morph():  # reference test.c:88-119, same inputs and assertions
    a = np.zeros((5, 5), np.uint8); a[1:4, 1:4] = 255
    e = o_morph(a, 0)
    assert e[2, 2] == 255 and e[1, 1] == 0
    b = np.zeros((5, 5), np.uint8); b[2, 2] = 255
    d = o_morph(b, 1)
    assert d[2, 2] == 255 and d[1, 2] == 255 and d[3, 2] == 255 and d[2, 1] == 255 and d[2, 3] == 255
    assert d[0, 0] == 0


def test_kat_sobel():  # reference test.c:121-149, same inputs and assertions
    a = np.zeros((5, 5), np.uint8); a[:, 2:] = 255
    d = o_sobel(a)
    assert d[2, 2] > 100 and d[3, 2] > 100 and d[2, 0] == 0
    b = np.zeros((5, 5), np.uint8); b[2:, :] = 255
    d = o_sobel(b)
    assert d[2, 2] > 100 and d[2, 3] > 100 and d[0, 2] == 0


def test_kat_adaptive():  # reference test.c:198-229, both full 5x5 tables
    W = 255
    a = np.array([[50, 50, 200, 50, 50]] * 3 + [[200, 200, 100, 200, 200]] * 2, np.uint8)
    t0 = [[0, 0, W, 0, 0], [0, 0, W, 0, 0], [0, 0, W, 0, 0], [W, W, 0, W, W], [0, W, 0, W, 0]]
    t5 = [[W, 0, W, 0, W], [W, 0, W, 0, W], [0, 0, W, 0, 0], [W, W, 0, W, W], [W, W, 0, W, W]]
    assert o_adaptive(a, 1, 0).tolist() == t0
    assert o_adaptive(a, 1, 5).tolist() == t5


def test_kat_integral():  # reference test.c:289-307
    a = np.arange(1, 10, dtype=np.uint8).reshape(3, 3)
    ii = o_integral(a)
    assert ii.tolist() == [[1, 3, 6], [5, 12, 21], [12, 27, 45]]
    # gs_integral_sum(ii, 3, 1, 1, 2, 2) == 28
    assert int(ii[2, 2]) + int(ii[0, 0]) - int(ii[0, 2]) - int(ii[2, 0]) == 28


def test_quirk_probes():  # SURVEY Appendix B quirk probes
    a = np.full((7, 7), 5, np.uint8); a[3, 3] = 3
    sm = np.zeros((7, 7), np.uint8)
    k = o_fast(a, sm, 10, 20)
    assert len(k) == 1 and sm[3, 3] == 2 and k[0]["response"] == 2
    a = np.full((7, 7), 105, np.uint8); a[3, 3] = 103
    assert len(o_fast(a, np.zeros((7, 7), np.uint8), 10, 20)) == 0
    a = np.full((7, 7), 5, np.uint8); a[3, 3] = 3
    sm = np.zeros((7, 7), np.uint8); sm[2, 2] = 200
    assert len(o_fast(a, sm, 10, 20)) == 0 and sm[2, 2] == 200
    assert o_sobel(np.zeros((5, 5), np.uint8), fill=77)[0, 0] == 77


# ---------------------------------------------------------------- (b) differential vs real reference
def _rand_images(rng, count, lo=1, hi=40):
    for i in range(count):
        w, h = int(rng.integers(lo, hi)), int(rng.integers(lo, hi))
        mode = i % 3
        if mode == 0: a = rng.integers(0, 256, (h, w))
        elif mode == 1: a = rng.integers(0, 40, (h, w))
        else: a = (rng.integers(0, 2, (h, w)) * 255)
        yield np.ascontiguousarray(a.astype(np.uint8))


def test_diff_stencils():
    R = L.RefRecord("test_diff_stencils"); rng = np.random.default_rng(1)
    for a in _rand_images(rng, 120):
        h, w = a.shape
        for r in (0, 1, 2, 5, 9):
            assert L.same(R.blur(a, r), o_blur(a, r)), ("blur", w, h, r)
            c = int(rng.integers(-30, 30))
            assert L.same(R.adaptive(a, r, c), o_adaptive(a, r, c)), ("adaptive", w, h, r, c)
        assert L.same(R.erode(a), o_morph(a, 0))
        assert L.same(R.dilate(a), o_morph(a, 1))
        if w >= 3 and h >= 3:  # the reference's unsigned loop bounds need w,h >= 1; <3 is a no-op only for >= 1... keep to the contract
            assert L.same(R.sobel77(a), o_sobel(a, 77))
        if w >= 2 and h >= 2:
            assert L.same(R.downsample(a), o_down(a))
        dw, dh = int(rng.integers(1, 50)), int(rng.integers(1, 50))
        assert L.same(R.resize(a, dw, dh), o_resize(a, dw, dh)), ("resize", w, h, dw, dh)
        assert L.same(R.integral(a), o_integral(a))
    R.finish()


def test_diff_box_medium_radii():
    """the radii the GPU suite runs k_box_mid's four instantiations at (r mod 4 = 0..3), oracle against the compiled
    reference on small ragged images: the GPU parity test for those radii compares with the oracle, so the oracle is
    pinned there too (the round-2 goldens hold 8 / 9 / 11 / 15 / 31)"""
    R = L.RefRecord("test_diff_box_medium_radii"); rng = np.random.default_rng(17)
    for i, a in enumerate(_rand_images(rng, 24)):
        h, w = a.shape
        for r in (10, 12, 13, 16, 17, 22):
            assert L.same(R.blur(a, r), o_blur(a, r)), ("blur", w, h, r)
            c = int(rng.integers(-60, 60))
            assert L.same(R.adaptive(a, r, c), o_adaptive(a, r, c)), ("adaptive", w, h, r, c)
    R.finish()


def test_diff_fast_orb():
    R = L.RefRecord("test_diff_fast_orb"); rng = np.random.default_rng(2)
    for i, a in enumerate(_rand_images(rng, 150, lo=7, hi=70)):
        h, w = a.shape
        t = [0, 255, 300, int(rng.integers(0, 64)), 20][i % 5]
        cap = int(rng.integers(1, 400))
        sm0 = (rng.integers(0, 256, a.shape) * (rng.random(a.shape) < 0.05)).astype(np.uint8) if i % 2 else np.zeros_like(a)
        sm_o = sm0.copy()
        ko = o_fast(a, sm_o, cap, t)
        assert L.same(R.fast(a, sm0, cap, t), (sm_o, ko)), ("fast", w, h, t, cap)
    for i in range(12):
        a = L.natural_like(160 + 8 * i, 120 + 4 * i, seed=i)
        nk = [50, 500, 1250][i % 3]
        ko = o_orb(a, np.zeros_like(a), nk, 20)
        assert len(ko) > 0
        assert L.same(R.orb_extract(a, nk, 20), ko), ("orb", i)
    R.finish()


def test_diff_sort_is_stable_descending():
    R = L.RefRecord("test_diff_sort_is_stable_descending"); rng = np.random.default_rng(3)
    for n in (2, 3, 17, 400, 1500):
        k = np.zeros(n, L.KP_DTYPE)
        k["response"] = rng.integers(1, 12, n); k["x"] = np.arange(n)
        b = k.copy()
        O.gso_sort_keypoints(L.ptr(b), n)
        assert L.same(R.sort_keypoints(k), b)
    R.finish()


def test_diff_trig_sample():
    """the oracle's restated sinf / atan2f against the C library's, which the reference calls"""
    import math
    R = L.RefRecord("test_diff_trig_sample"); rng = np.random.default_rng(4)
    xs = np.concatenate([rng.uniform(-4.8, 4.8, 20000), [0.0, -0.0, math.pi, -math.pi, 1e-5, 0.7853981]]).astype(np.float32)
    assert L.same(R.libm_sinf(xs), np.array([O.gso_sinf(float(x)) for x in xs], np.float32))
    m = rng.integers(-1200000, 1200001, (20000, 2))
    m[::50, 0] = 0; m[::77, 1] = 0
    assert L.same(R.libm_atan2f(m[:, 0], m[:, 1]), np.array([O.gso_atan2f(float(y), float(x)) for y, x in m], np.float32))
    R.finish()


def test_diff_lbp():
    R = L.RefRecord("test_diff_lbp"); cas = L.HostCascade(); rng = np.random.default_rng(5)
    for i in range(6):
        w, h = 96 + 16 * i, 80 + 12 * i
        a = L.natural_like(w, h, seed=10 + i) if i % 2 else rng.integers(0, 256, (h, w)).astype(np.uint8)
        ii = o_integral(a)
        for (mr, sf, mn, mx, st) in ((1000, 1.1, 1.0, 4.0, 2), (7, 1.2, 1.0, 3.0, 1), (1000, 1.25, 1.5, 2.0, 3)):
            ro = o_detect(cas, ii, mr, sf, mn, mx, st)
            assert L.same(R.lbp_detect(ii, mr, sf, mn, mx, st), ro), ("lbp", i, mr, sf)
        # the fixture cascade (committed .npz) and the reference's struct agree window by window
        for _ in range(200):
            x, y = int(rng.integers(0, w - 24)), int(rng.integers(0, h - 24))
            s = float(np.float32(rng.uniform(1.0, 2.5)))
            assert L.same(R.lbp_window(ii, x, y, s), O.gso_lbp_window(cas.ptr, L.ptr(ii), w, h, x, y, s))
    R.finish()


def test_lbp_depth_map_agrees_with_window():
    """gso_lbp_depth_map (analysis helper for tools/lbp_model.py): depth == nstages exactly where the window fires"""
    cas = L.HostCascade()
    nst = len(cas.arrays["stage_threshold"])
    a = L.natural_like(160, 120, 21)
    ii = o_integral(a)
    for s in (1.0, 1.5):
        s = float(np.float32(s)); win = int(np.float32(24) * np.float32(s))
        nx, ny = (160 - win) // 2 + 1, (120 - win) // 2 + 1
        depth = np.zeros((ny, nx), np.uint8)
        O.gso_lbp_depth_map(cas.ptr, L.ptr(ii), 160, 120, s, 2, L.ptr(depth))
        assert depth.max() <= nst and (depth == 0).any()
        for yi in range(0, ny, 3):
            for xi in range(0, nx, 3):
                assert (depth[yi, xi] == nst) == bool(O.gso_lbp_window(cas.ptr, L.ptr(ii), 160, 120, 2 * xi, 2 * yi, s))


def test_diff_match_orb():
    R = L.RefRecord("test_diff_match_orb"); rng = np.random.default_rng(6)
    for (n1, n2, mm, md) in ((50, 60, 300, 60.0), (300, 257, 40, 60.0), (7, 0, 10, 60.0), (0, 9, 10, 60.0), (120, 1, 500, 300.0),
                             (90, 33, 500, 10.0), (64, 64, 500, 0.0), (200, 500, 500, 255.5)):
        k1, k2 = L.desc_sets(rng, n1, n2)
        mo = np.zeros(max(mm, 1), L.MATCH_DTYPE)
        b = O.gso_match_orb(L.ptr(k1), n1, L.ptr(k2), n2, L.ptr(mo), mm, md)
        assert L.same(R.match_orb(k1, k2, mm, md), mo[:b]), (n1, n2, mm, md, b)
    R.finish()


def otsu_images(rng):
    """bimodal, flat, two-level, dark-heavy, noise and near-tie images: exercises wb == 0 skips, the wf == 0
    break and fp32 ties in varBetween"""
    out = []
    for (w, h) in ((3, 3), (64, 48), (257, 31), (640, 480), (1, 1), (5, 1)):
        out.append(rng.integers(0, 256, (h, w), dtype=np.uint8))
        a = np.where(rng.random((h, w)) < 0.3, rng.normal(60, 12, (h, w)), rng.normal(190, 20, (h, w)))
        out.append(np.clip(a, 0, 255).astype(np.uint8))
        out.append(np.full((h, w), int(rng.integers(0, 256)), np.uint8))
        b = np.full((h, w), 10, np.uint8); b.flat[:: max(1, (w * h) // 7)] = 250
        out.append(b)
        out.append((rng.integers(0, 2, (h, w)) * 255).astype(np.uint8))
        out.append(rng.integers(100, 104, (h, w), dtype=np.uint8))
    out.append(L.natural_like(1920, 1080, 3))
    return out


def test_testc_histogram_threshold_otsu():
    """the literal vectors of the reference's test.c:150-196"""
    a = np.array([[0, 50, 100], [50, 100, 150], [100, 150, 200]], np.uint8)
    hist = np.zeros(256, np.uint32); O.gso_histogram(L.ptr(a), 3, 3, L.ptr(hist))
    assert hist[0] == 1 and hist[50] == 2 and hist[100] == 3 and hist[150] == 2 and hist[200] == 1 and hist.sum() == 9
    t = np.array([[50, 150], [75, 200]], np.uint8); O.gso_threshold(L.ptr(t), 2, 2, 100)
    assert t.tolist() == [[0, 255], [0, 255]]
    assert O.gso_otsu_threshold(L.ptr(np.array([[40, 50, 60], [45, 55, 50], [190, 200, 210]], np.uint8)), 3, 3) == 60
    assert O.gso_otsu_threshold(L.ptr(np.array([[0, 85], [170, 255]], np.uint8)), 2, 2) == 85
    assert O.gso_otsu_threshold(L.ptr(np.full((2, 2), 128, np.uint8)), 2, 2) == 0


def test_diff_histogram_otsu_threshold():
    R = L.RefRecord("test_diff_histogram_otsu_threshold"); rng = np.random.default_rng(8)
    for a in otsu_images(rng):
        h, w = a.shape
        ho = np.zeros(256, np.uint32)
        O.gso_histogram(L.ptr(a), w, h, L.ptr(ho))
        assert L.same(R.histogram(a), ho) and np.array_equal(ho, np.bincount(a.ravel(), minlength=256))
        to = O.gso_otsu_threshold(L.ptr(a), w, h)
        assert L.same(R.otsu(a), to), (a.shape, to)
        for t in (0, 100, 255, int(to)):
            y = a.copy()
            O.gso_threshold(L.ptr(y), w, h, t)
            assert L.same(R.threshold(a, t), y)
    # synthetic histograms: fp32 rounding in the sums matters once counts are large
    for _ in range(200):
        hist = (rng.integers(0, 1 << int(rng.integers(1, 24)), 256) * (rng.random(256) < rng.random())).astype(np.uint32)
        if hist.sum() == 0:
            continue
        img = np.repeat(np.arange(256, dtype=np.uint8), hist)[None, :]
        if img.size > 1 << 26:
            continue
        assert L.same(R.otsu(np.ascontiguousarray(img)), O.gso_otsu_from_hist(L.ptr(hist), int(hist.sum())))
    R.finish()


def test_testc_template_matching():
    """the literal vectors of the reference's test.c:309-349"""
    img = np.array([[0, 0, 0, 0, 0], [0, 100, 150, 200, 0], [0, 125, 175, 225, 0], [0, 110, 160, 210, 0], [0, 0, 0, 0, 0]], np.uint8)
    t = np.ascontiguousarray(img[1:4, 1:4])
    res = np.zeros((3, 3), np.uint8)
    O.gso_match_template(L.ptr(img), 5, 5, L.ptr(t), 3, 3, L.ptr(res))
    assert O.gso_find_best_match(L.ptr(res), 3, 3) == 1 * 3 + 1 and res[1, 1] == 255
    s = np.full((4, 4), 50, np.uint8); s[1:3, 1:3] = 255
    res = np.zeros((3, 3), np.uint8)
    O.gso_match_template(L.ptr(s), 4, 4, L.ptr(np.full((2, 2), 255, np.uint8)), 2, 2, L.ptr(res))
    assert O.gso_find_best_match(L.ptr(res), 3, 3) == 4


def test_diff_filter():
    R = L.RefRecord("test_diff_filter"); rng = np.random.default_rng(9)
    for (w, h) in ((1, 1), (2, 3), (5, 4), (33, 17), (64, 48), (257, 63)):
        a = rng.integers(0, 256, (h, w), dtype=np.uint8)
        for name in L.FILTER_KERNELS:
            k, norm = L.filter_kernel(name)
            do = np.zeros_like(a)
            O.gso_filter(L.ptr(do), L.ptr(a), w, h, L.ptr(k), k.shape[1], k.shape[0], norm)
            assert L.same(R.filter(a, k, norm), do), (w, h, name)
    R.finish()


def test_diff_match_template():
    R = L.RefRecord("test_diff_match_template"); rng = np.random.default_rng(10)
    for (w, h, tw, th) in ((5, 5, 3, 3), (4, 4, 2, 2), (64, 48, 8, 8), (37, 29, 37, 29), (50, 40, 1, 1), (90, 31, 17, 5), (33, 70, 4, 33)):
        a = L.natural_like(w, h, w + h)
        y0, x0 = int(rng.integers(0, h - th + 1)), int(rng.integers(0, w - tw + 1))
        t = np.ascontiguousarray(a[y0:y0 + th, x0:x0 + tw]).copy()
        t = np.clip(t.astype(np.int16) + rng.integers(-3, 4, t.shape), 0, 255).astype(np.uint8)
        for tmpl in (t, rng.integers(0, 256, (th, tw), dtype=np.uint8), np.zeros((th, tw), np.uint8)):
            rw, rh = w - tw + 1, h - th + 1
            ro = np.zeros((rh, rw), np.uint8)
            O.gso_match_template(L.ptr(a), w, h, L.ptr(tmpl), tw, th, L.ptr(ro))
            assert L.same(R.match_template(a, tmpl), (ro, O.gso_find_best_match(L.ptr(ro), rw, rh))), (w, h, tw, th)
    z = np.zeros((3, 4), np.uint8)
    assert L.same(R.find_best_match(z), (0, 0)) and O.gso_find_best_match(L.ptr(z), 4, 3) == 0
    R.finish()


# ---------------------------------------------------------------- (c) committed golden fixtures
def _read_pgm(path):
    with open(path, "rb") as f:
        assert f.readline().strip() == b"P5"
        w, h = map(int, f.readline().split()); assert int(f.readline()) == 255
        return np.frombuffer(f.read(w * h), np.uint8).reshape(h, w).copy()


class _OracleImpl:
    """the oracle behind the interface _libs.check_next_golden expects"""

    @staticmethod
    def gs_histogram(a):
        h = np.zeros(256, np.uint32); O.gso_histogram(L.ptr(a), a.shape[1], a.shape[0], L.ptr(h)); return h

    @staticmethod
    def gs_otsu_threshold(a):
        return O.gso_otsu_threshold(L.ptr(a), a.shape[1], a.shape[0])

    @staticmethod
    def gs_threshold(a, t):
        O.gso_threshold(L.ptr(a), a.shape[1], a.shape[0], t); return a

    @staticmethod
    def gs_filter(dst, src, k, norm):
        O.gso_filter(L.ptr(dst), L.ptr(src), src.shape[1], src.shape[0], L.ptr(k), k.shape[1], k.shape[0], norm); return dst

    @staticmethod
    def gs_match_template(img, tmpl):
        res = np.zeros((img.shape[0] - tmpl.shape[0] + 1, img.shape[1] - tmpl.shape[1] + 1), np.uint8)
        O.gso_match_template(L.ptr(img), img.shape[1], img.shape[0], L.ptr(tmpl), tmpl.shape[1], tmpl.shape[0], L.ptr(res))
        return res

    @staticmethod
    def gs_find_best_match(res):
        b = O.gso_find_best_match(L.ptr(res), res.shape[1], res.shape[0]); return (b % res.shape[1], b // res.shape[1])

    @staticmethod
    def gs_orb(a, nkps, t):
        return o_orb(a, np.zeros_like(a), nkps, t)

    @staticmethod
    def gs_match_orb(k1, k2, mm, md):
        m = np.zeros(max(mm, 1), L.MATCH_DTYPE)
        n = O.gso_match_orb(L.ptr(k1), len(k1), L.ptr(k2 if len(k2) else np.zeros(1, L.KP_DTYPE)), len(k2), L.ptr(m), mm, md)
        return m[:n]


def test_golden_next_rows():
    """tests/golden/next_golden.npz: the 8(f) rows as computed by the real reference on lena and two synthetic images"""
    L.check_next_golden(_OracleImpl)


def test_survey_appendix_b_values(tmp_path):
    """SURVEY.md Appendix B: values the reference produced on testdata/lena.pgm when the survey was written, checked
    against the committed fixture (which the GPU golden tests compare the CUDA path with) and against the oracle"""
    z = np.load(os.path.join(GOLD, "lena_golden.npz"))
    a = z["lena"]

    def pgm_md5(img):
        return hashlib.md5(b"P5\n%d %d\n255\n" % (img.shape[1], img.shape[0]) + img.tobytes()).hexdigest()

    assert pgm_md5(a) == "66bd37186e4510052eefa3a52eef8188"
    assert pgm_md5(z["sobel"]) == "27cd5834468e2c0351475aacb7b5fc29" == pgm_md5(o_sobel(a))
    assert pgm_md5(z["blur1"]) == "53bfdf15397839728afd776749848584" == pgm_md5(o_blur(a, 1))
    assert pgm_md5(o_blur(a, 5)) == "24dd5d5b6898d8e6328410fa28c5e1f6" == pgm_md5(z["blur5"])
    assert pgm_md5(z["blur9"]) == "8c9c1e0db5ee451f7044b9bb96dcdb35"
    assert pgm_md5(z["adaptive_15_5"]) == "b4de7a7037676f5808c892b353362d4d" == pgm_md5(o_adaptive(a, 15, 5))
    assert pgm_md5(z["resize_128x64"]) == "96b030c4a2a50011a27efdfd5212a790" == pgm_md5(o_resize(a, 128, 64))
    k = z["fast_kps"]
    assert len(k) == 325 and (k[0]["x"], k[0]["y"], k[0]["response"]) == (56, 11, 2)
    assert (k[-1]["x"], k[-1]["y"], k[-1]["response"]) == (24, 124, 14)
    k = o_orb(a, np.zeros_like(a), 500, 20)
    assert k.tobytes() == z["orb_kps"].tobytes() and len(k) == 280
    assert (k[0]["x"], k[0]["y"], k[0]["response"]) == (49, 65, 63) and k[0]["descriptor"][0] == 0x6ebed143
    assert abs(float(k[0]["angle"]) - 0.3026622) < 1e-6
    r = z["lbp_rects"]
    assert len(r) == 10 and [tuple(int(v) for v in r[i]) for i in range(5)] == [
        (54, 52, 46, 46), (52, 46, 51, 51), (48, 48, 51, 51), (54, 48, 51, 51), (52, 50, 51, 51)]
    ii = o_integral(a)
    assert len(o_detect(L.HostCascade(), ii, 1000, 1.2, 1.0, 4.0, 1)) == 20
    # the reference CLI built as upstream builds it (oracle/_ref/nanomagick_cpu); the GPU suite checks that the
    # overlay build reproduces this binary's outputs byte for byte
    exe = os.path.join(L.ORACLE_DIR, "_ref", "nanomagick_cpu")
    if os.path.exists(exe):
        import subprocess
        src = tmp_path / "lena.pgm"
        src.write_bytes(b"P5\n128 128\n255\n" + a.tobytes())
        for args, md5 in ((["keypoints", "100", "20"], "c3745a335c3f6d53da8fe13cadf3c9a9"), (["faces", "2"], "0fdde3c4c3121ebe696b2e9100615e6e"),
                          (["sobel"], "27cd5834468e2c0351475aacb7b5fc29")):
            out = tmp_path / "o.pgm"
            assert subprocess.run([exe] + args + [str(src), str(out)], capture_output=True).returncode == 0
            assert hashlib.md5(out.read_bytes()).hexdigest() == md5, args
        r = subprocess.run([exe, "orb", str(src), str(src), str(tmp_path / "orb.pgm")], capture_output=True, text=True)
        assert "Template: 340 keypoints, Scene: 340 keypoints, Matches: 300" in r.stdout


def test_golden_lena():
    """tests/golden/lena_golden.npz was produced by the real reference (tools/make_golden.py)"""
    z = np.load(os.path.join(GOLD, "lena_golden.npz"))
    a = z["lena"]
    assert hashlib.md5(a.tobytes()).hexdigest() == str(z["lena_md5"])
    assert np.array_equal(o_sobel(a), z["sobel"])
    for r in (1, 5, 9):
        assert np.array_equal(o_blur(a, r), z["blur%d" % r])
    assert np.array_equal(o_adaptive(a, 15, 5), z["adaptive_15_5"])
    assert np.array_equal(o_morph(a, 0), z["erode"]) and np.array_equal(o_morph(a, 1), z["dilate"])
    assert np.array_equal(o_resize(a, 128, 64), z["resize_128x64"])
    assert np.array_equal(o_down(a), z["downsample"])
    assert np.array_equal(o_integral(a), z["integral"])
    sm = np.zeros_like(a)
    k = o_fast(a, sm, 5000, 20)
    assert k.tobytes() == z["fast_kps"].tobytes() and np.array_equal(sm, z["fast_scoremap"])
    assert len(k) == 325 and (k[0]["x"], k[0]["y"], k[0]["response"]) == (56, 11, 2)  # SURVEY App. B
    k = o_orb(a, np.zeros_like(a), 500, 20)
    assert k.tobytes() == z["orb_kps"].tobytes() and len(k) == 280
    cas = L.HostCascade()
    r = o_detect(cas, o_integral(a), 1000, 1.1, 1.0, 4.0, 2)
    assert r.tobytes() == z["lbp_rects"].tobytes() and len(r) == 10


# ---- round 2: SURVEY.md 8(f) N4 rows and the r > 15 orientation -------------------------------------------
def _o_blobs(a, nb):
    labels = np.full(a.shape, 0x5555, np.uint16)
    blobs = np.zeros(nb, L.BLOB_DTYPE)
    m = O.gso_blobs(L.ptr(a), a.shape[1], a.shape[0], L.ptr(labels), L.ptr(blobs), nb)
    return labels, blobs[:m]


def test_testc_blobs():  # reference test.c:232-257, same image and expectations
    Wv = 255
    a = np.array([[Wv, Wv, 0, 0, Wv, 0], [Wv, 0, 0, Wv, Wv, 0], [0, 0, Wv, Wv, 0, 0], [Wv, Wv, Wv, 0, 0, Wv],
                  [0, Wv, 0, 0, 0, Wv]], np.uint8)
    labels, blobs = _o_blobs(a, 10)
    assert L.blob_fields(blobs) == [(1, 3, 0, 0, 2, 2, 0, 0), (2, 9, 0, 0, 5, 5, 2, 2), (6, 2, 5, 3, 1, 2, 5, 3)]


def test_diff_blobs_corners():
    R = L.RefRecord("test_diff_blobs_corners"); rng = np.random.default_rng(77)
    cases = 0
    for i in range(60):
        w, h = int(rng.integers(1, 90)), int(rng.integers(1, 70))
        a = L.binary_like(w, h, 1000 + i, density=float(rng.uniform(0.2, 0.8)), smooth=int(rng.integers(0, 4)))
        if i % 7 == 0:
            a = rng.integers(0, 256, (h, w)).astype(np.uint8)             # grey noise: values around the 128 test
        for nb in (2000, int(rng.integers(1, 30)), 1):
            lo, bo = _o_blobs(a, nb)
            assert L.same(R.blobs(a, nb), L.blobs_result(lo, bo)), (i, w, h, nb)
            for j in range(min(len(bo), 5)):
                co = np.zeros((4, 2), np.uint32)
                O.gso_blob_corners(L.ptr(a), w, h, L.ptr(lo), L.ptr(bo[j:j + 1]), L.ptr(co))
                assert L.same(R.blob_corners(a, nb, j), co), (i, nb, j)
                cases += 1
    assert cases > 200
    R.finish()


def test_diff_perspective_and_large_orientation():
    R = L.RefRecord("test_diff_perspective_and_large_orientation")
    rng = np.random.default_rng(78)
    for i in range(40):
        sw, sh = int(rng.integers(1, 120)), int(rng.integers(1, 90))
        src = rng.integers(0, 256, (sh, sw)).astype(np.uint8)
        dw, dh = int(rng.integers(1, 70)), int(rng.integers(1, 60))
        c = rng.integers(0, max(sw, sh) + 30, (4, 2)).astype(np.uint32)
        do = np.empty((dh, dw), np.uint8)
        O.gso_perspective_correct(L.ptr(do), dw, dh, L.ptr(src), sw, sh, L.ptr(c))
        assert L.same(R.perspective(src, dw, dh, c), do), (i, sw, sh, dw, dh)
    a = np.clip(L.natural_like(300, 260, 5).astype(np.int32) + 100, 0, 255).astype(np.uint8)
    for r in (2, 15, 16, 30, 64, 100):
        for _ in range(6):
            x, y = int(rng.integers(r, 300 - r)), int(rng.integers(r, 260 - r))
            go = O.gso_compute_orientation(L.ptr(a), 300, 260, x, y, r)
            assert L.same(R.orientation(a, x, y, r), go), (x, y, r)
    R.finish()


def test_golden_round2_oracle_rows():
    """the oracle against the reference-generated round-2 fixtures (runs without /root/reference)"""
    z = np.load(os.path.join(L.ROOT, "tests", "golden", "round2_golden.npz"))
    for tag in z["blob_tags"]:
        a = np.ascontiguousarray(z["blob_img_" + str(tag)])
        for nb in (1000, 7, 1):
            lo, bo = _o_blobs(a, nb)
            assert np.array_equal(lo, z["blob_%s_n%d_labels" % (tag, nb)]), (tag, nb)
            assert np.array_equal(np.array(L.blob_fields(bo), np.int64).reshape(-1, 8), z["blob_%s_n%d_blobs" % (tag, nb)]), (tag, nb)
        key = "blob_%s_corners" % tag
        if key in z.files:
            lo, bo = _o_blobs(a, 1000)
            for j, want in enumerate(z[key]):
                c = np.zeros((4, 2), np.uint32)
                O.gso_blob_corners(L.ptr(a), a.shape[1], a.shape[0], L.ptr(lo), L.ptr(bo[j:j + 1]), L.ptr(c))
                assert np.array_equal(c, want), (tag, j)
    src = np.ascontiguousarray(z["persp_src"])
    for qi, q in enumerate(z["persp_quads"]):
        for (dw, dh) in ((160, 100), (33, 47), (1, 1), (2, 5)):
            d = np.empty((dh, dw), np.uint8)
            O.gso_perspective_correct(L.ptr(d), dw, dh, L.ptr(src), src.shape[1], src.shape[0], L.ptr(np.ascontiguousarray(q)))
            assert np.array_equal(d, z["persp_q%d_%dx%d" % (qi, dw, dh)]), (qi, dw, dh)
    a = np.ascontiguousarray(z["orient_img"])
    for (x, y, r), want in zip(z["orient_xyr"], z["orient_angle"]):
        got = O.gso_compute_orientation(L.ptr(a), a.shape[1], a.shape[0], int(x), int(y), int(r))
        assert np.float32(got).tobytes() == np.float32(want).tobytes(), (x, y, r)
    for tag in z["radius_tags"]:
        a = np.ascontiguousarray(z["radius_img_" + str(tag)])
        for r in z["radii"]:
            d = np.empty_like(a); O.gso_blur(L.ptr(d), L.ptr(a), a.shape[1], a.shape[0], int(r))
            assert np.array_equal(d, z["blur%d_%s" % (int(r), tag)])
            d = np.empty_like(a); O.gso_adaptive_threshold(L.ptr(d), L.ptr(a), a.shape[1], a.shape[0], int(r), 5 - int(r))
            assert np.array_equal(d, z["adaptive%d_%s" % (int(r), tag)])
