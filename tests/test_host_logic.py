"""CPU-only tests: the C-ABI library loads and exports every symbol include/*.h declares, the
drop-in header compiles the reference's own callers unmodified, the exact-division constants of
the box filter are valid for every clipped count, and the frame sharding works across ranks
(world_size 2, gloo).  No compute call is made on the library here (there is no GPU)."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import _libs as L

ROOT = L.ROOT


def _declared(header):
    txt = open(os.path.join(ROOT, "include", header)).read()
    txt = txt[txt.rindex('extern "C" {'):]
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(gs_[a-z0-9_]+)\s*\(", txt)))


def test_library_exports_every_declared_symbol():
    sys.path.insert(0, ROOT)
    from grayskull_b200 import build, _lib
    build.build()
    handle = C.CDLL(_lib.LIB_PATH)          # loads without a GPU or a driver
    declared = _declared("grayskull.h") + _declared("grayskull_b200.h")
    assert len(declared) > 40
    for name in declared:
        assert hasattr(handle, name), name
        assert name in _lib.SIGNATURES, "binding table is missing %s" % name
    assert sorted(_lib.SIGNATURES) == sorted(set(declared))
    lib = _lib.lib()
    assert b"sm_100a" in lib.gs_b200_version()
    assert lib.gs_b200_device_count() >= 0


def test_sass_is_sm100a_with_tma():
    """the shipped cubin targets sm_100a and the tiled kernels really use TMA (UTMALDG)"""
    from grayskull_b200 import _lib
    out = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out
    assert "UTMALDG" in out and "SYNCS" in out
    assert "VIMNMX3.U16x2" in out and "HMNMX2" in out      # packed-lane arithmetic, not scalar bytes


def test_struct_layouts_match_reference():
    assert C.sizeof(L.Image) == 16 and C.sizeof(L.Rect) == 16 and C.sizeof(L.Keypoint) == 48
    assert C.sizeof(L.Cascade) == 96
    if L.have_ref():
        R = L.ref()
        R.ref_sizeof.restype = C.c_uint
        assert [R.ref_sizeof(i) for i in range(4)] == [16, 16, 48, 96]


def test_reference_callers_compile_unmodified_against_dropin_header():
    """overlay mode: oracle/Makefile compiles the reference's test.c and nanomagick.c, unmodified, with their own
    strict flags (-std=c99 -Wall -Wextra -Werror -pedantic; a warning fails build()) against include/ and links
    them with libgrayskull_b200.so into oracle/_ref/.  Both executables must take the hot path from the library:
    every one of these symbols is an import, none is inlined CPU code."""
    exes = {name: os.path.join(L.ORACLE_DIR, "_ref", name) for name in ("test_overlay", "nanomagick_overlay")}
    if not all(os.path.exists(e) for e in exes.values()):
        pytest.skip("overlay builds not present (build() makes them where the reference tree is readable)")
    for name, exe in exes.items():
        needed = subprocess.run(["readelf", "-d", exe], capture_output=True, text=True).stdout
        assert "[libgrayskull_b200.so]" in needed, name
        syms = subprocess.run(["nm", "-D", "--undefined-only", exe], capture_output=True, text=True).stdout
        wanted = (("gs_blur", "gs_sobel", "gs_erode", "gs_dilate", "gs_adaptive_threshold", "gs_resize", "gs_integral",
                   "gs_histogram", "gs_otsu_threshold", "gs_threshold", "gs_match_template", "gs_find_best_match")
                  if name == "test_overlay" else ("gs_blur", "gs_sobel", "gs_fast", "gs_orb_extract", "gs_match_orb", "gs_lbp_detect", "gs_integral"))
        for sym in wanted:
            assert re.search(r"\bU %s\b" % sym, syms), (name, sym)


def test_standalone_header_compiles_as_c99(tmp_path):
    src = tmp_path / "t.c"
    src.write_text('#include "grayskull_b200.h"\n'
                   "int main(void) { struct gs_image a = gs_alloc(4, 4); gs_set(a, 1, 1, 9);\n"
                   "  unsigned ii[16] = {0}; int ok = gs_get(a, 1, 1) == 9 && gs_integral_sum(ii, 4, 1, 1, 2, 2) == 0;\n"
                   "  gs_free(a); return ok ? 0 : 1; }\n")
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", "-fsyntax-only",
                        "-I", os.path.join(ROOT, "include"), str(src)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_standalone_header_pgm_io(tmp_path):
    """P5 reader / writer of the stand-alone header (reference grayskull.h:111-136 semantics): round trip, header
    with comments and mixed white space, wrong maxval / truncated data rejected"""
    src = tmp_path / "pgm.c"
    src.write_text('#include <string.h>\n#include "grayskull.h"\n'
                   "int main(int argc, char **argv) {\n"
                   "  struct gs_image a = gs_alloc(5, 3); unsigned i; (void)argc;\n"
                   "  for (i = 0; i < 15; i++) a.data[i] = (uint8_t)(i * 17 + 10);\n"
                   "  if (gs_write_pgm(a, argv[1]) != 0) return 2;\n"
                   "  { struct gs_image b = gs_read_pgm(argv[1]);\n"
                   "    if (!gs_valid(b) || b.w != 5 || b.h != 3 || memcmp(a.data, b.data, 15)) return 3;\n    gs_free(b); }\n"
                   "  { struct gs_image c = gs_read_pgm(argv[2]);\n"
                   "    if (!gs_valid(c) || c.w != 2 || c.h != 2 || c.data[0] != 10 || c.data[3] != 'A') return 4;\n    gs_free(c); }\n"
                   "  if (gs_valid(gs_read_pgm(argv[3])) || gs_valid(gs_read_pgm(argv[4])) || gs_valid(gs_read_pgm(argv[5]))) return 5;\n"
                   "  gs_free(a); return 0; }\n")
    exe = str(tmp_path / "pgm")
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"),
                        "-o", exe, str(src)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    (tmp_path / "c.pgm").write_bytes(b"P5\n# made by hand\n2\t2\n# another\n255\n" + bytes([10, 0, 1, 65]))
    (tmp_path / "bad16.pgm").write_bytes(b"P5\n2 2\n65535\n" + bytes(8))
    (tmp_path / "short.pgm").write_bytes(b"P5\n4 4\n255\n" + bytes(7))
    r = subprocess.run([exe, str(tmp_path / "rt.pgm"), str(tmp_path / "c.pgm"), str(tmp_path / "bad16.pgm"),
                        str(tmp_path / "short.pgm"), str(tmp_path / "missing.pgm")])
    assert r.returncode == 0
    assert (tmp_path / "rt.pgm").read_bytes()[:11] == b"P5\n5 3\n255\n"


def test_cli_is_built_and_has_no_cpu_path(tmp_path):
    """gsb_magick (grayskull_b200/cli) builds with the library and refuses to do anything without inputs / a GPU"""
    from grayskull_b200 import build, _lib
    build.build()
    exe = os.path.join(os.path.dirname(_lib.LIB_PATH), "gsb_magick")
    assert os.path.exists(exe)
    r = subprocess.run([exe, "blur:2", str(tmp_path / "o"), str(tmp_path / "missing.pgm")], capture_output=True, text=True)
    assert r.returncode == 1 and "gsb_magick:" in r.stderr
    assert subprocess.run([exe], capture_output=True).returncode == 1


def test_bench_reference_arm_contract():
    """`bench.py --impl reference`: one JSON line with the contract's keys, timed on the host cores; under torchrun
    only rank 0 works and prints"""
    import json
    import sys
    env = dict(os.environ)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stderr[-500:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "Mpixels/s" and d["value"] > 0 and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    env.update(RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1"],
                       capture_output=True, text=True, env=env, timeout=120)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_box_division_constants_are_exact():
    """box.cu: fma_rd(2^23 + S, m*2^-24, 2^23 - m/2) == 2^23 + floor(S*m / 2^24), and
    floor(S*m/2^24) == S // count for every count <= 225 and every S <= 255*count."""
    for count in range(1, 226):
        m = (16777216 + count - 1) // count
        assert m <= 16777216                                  # m is an exact float
        assert (2 * 8388608 - m) % 1 == 0 and (8388608 - m / 2) * 2 == int((8388608 - m / 2) * 2)
        S = np.arange(0, 255 * count + 1, dtype=np.int64)
        assert np.array_equal((S * m) >> 24, S // count), count
        assert ((S * m) >> 24).max() <= 255
        # exactness of the fused multiply-add before its single rounding: the exact value is
        # 2^23 + S*m/2^24 < 2^24, so round-down lands on the integer part
        assert (S.max() * m) / 2 ** 24 < 2 ** 23


def test_wide_box_division_is_exact():
    """box.cu k_box_wide: interior quotients come from fma_rd(float(S), m * 2^-k, 2^23) with k = 23 + floor(log2 count),
    m = ceil(2^k / count): m must be an exact float (< 2^24) and floor(S*m / 2^k) == S // count for every window sum
    S <= 255 * count, count = (2r+1)^2, r = 8..63 (the radii box_wide_magic accepts); clipped counts use
    floor(fdiv_rn(S, count)), exact because S/count is at least 1/count > half an ulp away from the next integer."""
    for r in range(8, 64):
        count = (2 * r + 1) ** 2
        k = 23 + int(np.floor(np.log2(count)))
        m = ((1 << k) + count - 1) // count
        assert m < 1 << 24, r
        e = m * count - (1 << k)
        assert 255 * count * e < 1 << k, r                       # the host-side acceptance test of box_wide_magic
        step = 1 if r <= 20 else 7                               # every S for the common radii, a stride beyond
        S = np.arange(0, 255 * count + 1, step, dtype=np.int64)
        S = np.concatenate([S, np.arange(count - 1, 255 * count + 1, count), np.arange(0, 255 * count + 1, count)])
        assert np.array_equal([int(v) for v in (S.astype(object) * m) >> k] if r > 50 else (S * m) >> k, S // count), r
        assert float(S.max()) * m / 2.0 ** k < 2 ** 23
    # the fdiv path: worst cases q*d + (d - 1) for d up to 241^2 (r = 120), in float32 arithmetic
    for d in (289, 961, 16129, 16641, 58081, 65025, 241 * 241):
        q = np.arange(0, 256, dtype=np.int64)
        for f in (d - 1, d - 2, 0, 1):
            S = q * d + f
            S = S[S < 1 << 24]
            got = np.floor(S.astype(np.float32) / np.float32(d)).astype(np.int64)
            assert np.array_equal(got, S // d), (d, f)


def _box_mid_row_model(C, r, R8, w_img, xs, look_ahead=True):
    """One H-phase row of box.cu k_box_mid, restated on a byte buffer: the row of 256 u16 column sums is laid out as the
    V-phase stores it (4 u16 of zero pad, then groups of four columns as two pair words (c0,c2) (c1,c3)); the walk reads
    64-bit groups, forms W + D_k through the (word, half) selection of dp2a_elem, and writes the 8 output sums of step t
    over bytes [8 + 8t, 16 + 8t) of the SAME buffer -- with the next step's groups read BEFORE that store, as the kernel
    orders them.  Returns the window sums of the steps that reach into the image."""
    buf = np.zeros(130 * 4, np.uint8)
    u16 = buf.view(np.uint16)
    for l in range(32):                                          # V-phase store of lane l: words 2 + 4l .. 5 + 4l
        c = C[8 * l: 8 * l + 8]
        u16[4 + 8 * l: 12 + 8 * l] = [c[0], c[2], c[1], c[3], c[4], c[6], c[5], c[7]]
    RM, LM = r & 3, (3 - (r & 3)) & 3
    ge0, gl0 = (R8 + r + 4) >> 2, (R8 - r + 3) >> 2
    outw = 256 - 2 * R8
    iters = outw >> 3

    def grp(g):                                                  # a 64-bit group: four u16 in storage order
        assert 0 <= g <= 64, ("group outside the lane's row", g)
        return buf[8 * g: 8 * g + 8].view(np.uint16).copy()

    def elem(a, b, idx):                                         # dp2a_elem: word idx & 1, half (idx >> 1) & 1 of group a / b
        g = a if idx < 4 else b
        return int(g[2 * (idx & 1) + ((idx >> 1) & 1)])
    L0, E0 = grp(gl0), grp(ge0)
    W = sum(elem(L0, L0, k) for k in range(LM, 4)) + sum(int(grp(g).sum()) for g in range(gl0 + 1, ge0)) + \
        sum(elem(E0, E0, k) for k in range(RM))
    xo = xs + R8
    t_img = min(iters, (w_img - xo + 7) >> 3)
    u_in = (60 - ge0) >> 1
    out = []
    EA, LA = [grp(ge0 + 1), grp(ge0 + 2)], [grp(gl0 + 1), grp(gl0 + 2)]
    Ep, Lp = E0, L0
    zero = np.zeros(4, np.uint16)
    for t in range(t_img):
        # look-ahead of step t+1, guarded exactly like the kernel's tail steps (the unguarded loop runs while t + 1 <= u_in)
        Ln = [grp(gl0 + 2 * t + 3), grp(gl0 + 2 * t + 4)]
        if t <= u_in:
            En = [grp(ge0 + 2 * t + 3), grp(ge0 + 2 * t + 4)]
        else:
            En = [grp(ge0 + 2 * t + 3) if ge0 + 2 * t + 3 <= 64 else zero, zero]
        sums = []
        for s_ in range(2):
            Ea, La = (Ep, Lp) if s_ == 0 else (EA[0], LA[0])
            D = 0
            for k in range(4):
                D += elem(Ea, EA[s_], RM + k) - elem(La, LA[s_], LM + k)
                sums.append(W + D)
            W += D
        out.append(sums)
        buf[8 + 8 * t: 16 + 8 * t] = 0xAB                        # the packed quotients overwrite the consumed head of the row
        Ep, Lp, EA, LA = EA[1], LA[1], En, Ln
    return np.array(out, np.int64).reshape(-1)


def test_box_mid_row_walk_matches_direct_window_sums():
    """box.cu k_box_mid, H-phase index arithmetic (r mod 4 element positions, permuted pair layout, first / last groups,
    in-place output store, look-ahead guards) against direct window sums, for every radius the kernel takes and strips at
    the left edge, in the interior and hanging over the right edge of the image"""
    rng = np.random.default_rng(5)
    for r in list(range(8, 41)) + [47, 48, 63, 64, 77, 100, 119, 120]:
        R8 = (r + 7) // 8 * 8
        outw = 256 - 2 * R8
        assert outw >= 16
        for w_img in (outw * 3 + 40, 4096, 8 * ((r + 9) // 8)):
            strips = (w_img + outw - 1) // outw
            for strip in sorted({0, strips // 2, strips - 1}):
                xs = strip * outw - R8
                cols = np.arange(xs, xs + 256)
                C = np.where((cols >= 0) & (cols < w_img), rng.integers(0, (2 * r + 1) * 255 + 1, 256), 0).astype(np.int64)
                got = _box_mid_row_model(C, r, R8, w_img, xs)
                Cp = np.concatenate([np.zeros(r + 1, np.int64), C, np.zeros(r + 1, np.int64)])
                want = np.array([Cp[c + 1: c + 2 * r + 2].sum() for c in range(R8, R8 + len(got))])
                assert np.array_equal(got, want), (r, w_img, strip)
                assert len(got) >= min(outw, w_img - (xs + R8)), (r, w_img, strip)   # every in-image output is produced


def test_filter_magic_division_is_exact():
    """filter.cu fast path: for norm >= 2, min(255, umulhi((u32)sum, floor(2^32/norm)+1)) equals the reference's
    `sum = sum / norm` (int converted to unsigned, quotient back to int, clamp 0..255) for every sum the host check
    admits: pos_max * norm < 2^32 and (2^32 - neg_max) / norm >= 256"""
    rng = np.random.default_rng(41)

    def ref(sv, norm):
        q = (sv.astype(np.int64) & 0xFFFFFFFF) // norm            # (unsigned)sum / norm
        v = np.where(q >= 1 << 31, q - (1 << 32), q)              # back into an int
        return np.clip(v, 0, 255)

    def fast(sv, norm):
        m = (1 << 32) // norm + 1
        hi = ((sv.astype(np.int64) & 0xFFFFFFFF).astype(object) * m) >> 32
        return np.minimum(np.array(hi, dtype=np.int64), 255)

    cases = [(9, 255 * 9, 0), (16, 255 * 16, 0), (3, 255 * 4, 255 * 4), (7, 255 * 127 * 5, 255 * 128 * 4), (2, 32385 * 9, 32640 * 9),
             (255, 65025, 3000), (4096, 255 * 127 * 9, 255 * 128 * 9)]
    for _ in range(40):
        norm = int(rng.integers(2, 1 << int(rng.integers(2, 24))))
        pos = int(rng.integers(0, min((1 << 32) // norm, 255 * 127 * 9) + 1))
        neg = int(rng.integers(0, 255 * 128 * 9 + 1))
        cases.append((norm, pos, neg))
    checked = 0
    for norm, pos, neg in cases:
        if not (pos * norm < (1 << 32) and ((1 << 32) - neg) // norm >= 256):
            continue                                               # the host sends these to the generic kernel
        if pos + neg <= 400000:
            sv = np.arange(-neg, pos + 1, dtype=np.int64)
        else:
            sv = np.unique(np.concatenate([rng.integers(-neg, pos + 1, 200000), np.arange(-min(neg, 2000), min(pos, 2000) + 1),
                                           np.arange(max(pos - 2000, 0), pos + 1), np.arange(-neg, min(-neg + 2000, 0) + 1),
                                           (np.arange(0, pos // norm + 1)[:5000] * norm), (np.arange(1, pos // norm + 1)[:5000] * norm - 1)]))
        assert np.array_equal(fast(sv, norm), ref(sv, norm)), (norm, pos, neg)
        checked += 1
    assert checked >= 20


def test_otsu_parallel_form_matches_sequential_scan():
    """histogram.cu k_otsu: serial prefix sums + per-threshold variance + FIRST-maximum reduction over the valid
    thresholds must pick the same threshold as the reference's sequential loop (checked through the oracle)"""
    import _libs as L
    O = L.oracle()
    rng = np.random.default_rng(42)
    f32 = np.float32
    for it in range(300):
        hist = (rng.integers(0, 1 << int(rng.integers(1, 22)), 256) * (rng.random(256) < rng.random())).astype(np.uint32)
        if it % 7 == 0:
            hist[:] = 0; hist[int(rng.integers(0, 256))] = 1000           # one level only
        if it % 11 == 0:
            hist[int(rng.integers(0, 128))] = hist[int(rng.integers(128, 256))] = 77777   # exact ties are likely
        npix = int(hist.sum())
        if npix == 0:
            continue
        total = f32(0)
        for i in range(256):
            total = f32(total + f32(f32(i) * f32(hist[i])))
        wb = np.cumsum(hist.astype(np.int64))
        sum_b = np.zeros(256, f32); acc = f32(0)
        for t in range(256):
            acc = f32(acc + f32(f32(t) * f32(hist[t]))); sum_b[t] = acc
        wf = npix - wb
        valid = (wb > 0) & (wf > 0)
        with np.errstate(divide="ignore", invalid="ignore"):
            m_b = (sum_b / wb.astype(f32)).astype(f32)
            m_f = ((f32(total) - sum_b).astype(f32) / wf.astype(f32)).astype(f32)
            diff = (m_b - m_f).astype(f32)
            var = (((wb.astype(f32) * wf.astype(f32)).astype(f32) * diff).astype(f32) * diff).astype(f32)
        best = 0
        if valid.any():
            v = np.where(valid, var, f32(-1))
            best = int(np.argmax(v))                                      # first maximum
        assert best == O.gso_otsu_from_hist(L.ptr(hist), npix), it


def test_match_key_trick_matches_sequential_scan():
    """match.cu: the two smallest (distance << 22 | index) keys with M represented by ceil(M) << 22 reproduce the
    reference's float scan (best / second / first best index, acceptance test) for any max_distance"""
    rng = np.random.default_rng(43)
    f32 = np.float32
    for it in range(3000):
        n2 = int(rng.integers(0, 40))
        d = rng.integers(0, 257, n2) if it % 3 else rng.integers(0, 8, n2)
        md = f32(rng.choice([0.0, 0.5, 3.0, 7.0, 60.0, 64.5, 255.0, 255.5, 256.0, 300.0, -1.0, -0.5, 0.99, 1e9]))
        M = f32(md + f32(1))
        best, second, bidx = M, M, 0
        for j, dj in enumerate(d):
            fd = f32(dj)
            if fd < best:
                second, best, bidx = best, fd, j
            elif fd < second:
                second = fd
        accept_ref = bool(best <= md and best < f32(f32(0.8) * second))
        thr = int(min(max(np.ceil(float(M)), 0.0), 257.0))
        sentinel = thr << 22
        keys = sorted([sentinel, sentinel] + [(int(dj) << 22) + j for j, dj in enumerate(d)])
        b, s2 = keys[0], keys[1]
        fb = M if b >= sentinel else f32(b >> 22)
        fs = M if s2 >= sentinel else f32(s2 >> 22)
        accept = bool(fb <= md and fb < f32(f32(0.8) * fs))
        assert accept == accept_ref and fb == best and fs == second, (it, md, list(d))
        if accept:
            assert (b & ((1 << 22) - 1)) == bidx


def test_lbp_window_count_matches_enumeration():
    cas = L.HostCascade()
    # (the reference's loops, enumerated in python with fp32 arithmetic)
    def count(iw, ih, sf, mn, mx, step):
        n, scale = 0, np.float32(mn)
        while scale <= np.float32(mx):
            ww, wh = int(np.float32(24) * scale), int(np.float32(24) * scale)
            if ww > iw or wh > ih:
                break
            n += len(range(0, ih - wh + 1, step)) * len(range(0, iw - ww + 1, step))
            scale = np.float32(scale * np.float32(sf))
        return n
    assert count(3840, 2160, 1.1, 1.0, 4.0, 2) == 30016520          # SURVEY.md 8(d)
    from grayskull_b200 import _lib
    lib = _lib.lib()
    for args in ((3840, 2160, 1.1, 1.0, 4.0, 2), (128, 128, 1.2, 1.0, 4.0, 1), (100, 37, 1.1, 1.0, 4.0, 2), (20, 20, 1.1, 1.0, 4.0, 1)):
        assert lib.gs_b200_lbp_window_count(cas.ptr, *args) == count(*args), args


def test_shard_ranges_cover_every_frame_once():
    from grayskull_b200.shard import shard_range
    for n in (0, 1, 7, 256, 8192, 1000):
        for world in (1, 2, 3, 4, 8):
            spans = [shard_range(n, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(spans[i][1] == spans[i + 1][0] for i in range(world - 1))
            assert max(b - a for a, b in spans) - min(b - a for a, b in spans) <= 1


_WORKER = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from grayskull_b200.shard import scatter_frames, gather_frames, gather_many, shard_range
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%s" % sys.argv[2], rank=int(sys.argv[3]), world_size=2)
rank = dist.get_rank()
n, h, w = 7, 5, 16
full = (torch.arange(n * h * w, dtype=torch.int64) % 251).to(torch.uint8).reshape(n, h, w) if rank == 0 else None
mine = scatter_frames(full, n, (h, w), torch.uint8, "cpu")
lo, hi = shard_range(n, rank, 2)
want = (torch.arange(n * h * w, dtype=torch.int64) % 251).to(torch.uint8).reshape(n, h, w)[lo:hi]
assert torch.equal(mine, want), rank
out = gather_frames(255 - mine, n)          # a per-frame "op", then the gather
if rank == 0:
    assert torch.equal(out, 255 - (torch.arange(n * h * w, dtype=torch.int64) % 251).to(torch.uint8).reshape(n, h, w))
else:
    assert out is None
# several result tensors (maps, records, per-frame counts) in one group, into preallocated root buffers
recs = torch.arange(lo, hi, dtype=torch.int32).reshape(-1, 1, 1).repeat(1, 3, 4) * 7
cnts = torch.arange(lo, hi, dtype=torch.int32) + 100
pre = [torch.zeros((n, h, w), dtype=torch.uint8), torch.zeros((n, 3, 4), dtype=torch.int32), torch.zeros((n,), dtype=torch.int32)] if rank == 0 else None
res = gather_many([mine, recs, cnts], n, out=pre)
if rank == 0:
    assert res is pre and torch.equal(res[0], want_all := (torch.arange(n * h * w, dtype=torch.int64) % 251).to(torch.uint8).reshape(n, h, w))
    assert torch.equal(res[1], torch.arange(n, dtype=torch.int32).reshape(-1, 1, 1).repeat(1, 3, 4) * 7)
    assert torch.equal(res[2], torch.arange(n, dtype=torch.int32) + 100)
else:
    assert res is None
dist.barrier(); dist.destroy_process_group(); print("ok", rank)
'''


_WORKER_RUN = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from grayskull_b200.shard import ShardedRun, shard_range
world = int(sys.argv[4])
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%s" % sys.argv[2], rank=int(sys.argv[3]), world_size=world)
rank = dist.get_rank()

class FakePipe:      # a per-frame "op" with two result tensors: the schedule and the index arithmetic are what is tested
    def __init__(self, n, h, w):
        self.out = torch.zeros((n, h, w), dtype=torch.uint8); self.tag = torch.zeros((n,), dtype=torch.int32)
    def run(self, frames, lo):
        m = frames.shape[0]
        if m == 0:
            return
        self.out[lo:lo + m] = 255 - frames
        self.tag[lo:lo + m] = frames.reshape(m, -1)[:, 0].to(torch.int32) + 1000
    def results(self, m):
        return {"out": self.out[:m], "tag": self.tag[:m]}

h, w = 3, 8
for n in (7, 2, 13):                 # ragged shards, a rank with an empty shard (n=2, world=3), several pieces
    full = ((torch.arange(n * h * w, dtype=torch.int64) * 7) % 251).to(torch.uint8).reshape(n, h, w)
    lo, hi = shard_range(n, rank, world)
    for mode in ("serial", 1, 2, 5):
        pipe = FakePipe(hi - lo, h, w)
        run = ShardedRun(pipe, n, h, w, torch.device("cpu"), keys=("out", "tag"))
        if mode == "serial":
            run.run_serial(full if rank == 0 else None)
        else:
            run.run_overlapped(full if rank == 0 else None, mode)
        dist.barrier()
        if rank == 0:
            assert torch.equal(run.gathered[0], 255 - full), (n, mode)
            assert torch.equal(run.gathered[1], full.reshape(n, -1)[:, 0].to(torch.int32) + 1000), (n, mode)
dist.barrier(); dist.destroy_process_group(); print("ok", rank)
'''


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_run_schedule_gloo(tmp_path, world):
    """ShardedRun (scatter -> per-rank pipeline -> gather; whole shard and in overlapped pieces) on a CPU group:
    ragged shards, an empty shard, more pieces than frames"""
    script = tmp_path / "worker_run.py"
    script.write_text(_WORKER_RUN)
    port = str(30500 + (os.getpid() + world) % 1000)
    procs = [subprocess.Popen([sys.executable, str(script), ROOT, port, str(r), str(world)], stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(world)]
    outs = [p.communicate(timeout=300)[0] for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o


def test_scatter_gather_world_size_2_gloo(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    port = str(29500 + os.getpid() % 1000)
    procs = [subprocess.Popen([sys.executable, str(script), ROOT, port, str(r)], stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=240)[0] for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o
