"""Pins the CPU restatement (oracle/*.c) before anything trusts it:
  1. known-answer checksums measured on the reference build (SURVEY.md section 6 / BASELINE.md section 2),
  2. the unmodified reference objects (oracle/_ref/libugref.so) on ragged sizes, as recorded in tests/golden/reference_*.json,
  3. committed golden vectors generated from the reference (tests/golden/make_golden.py),
  4. the colour-coefficient limits test of the reference (test/misc_test.c:46-87).
"""
import ctypes
import os

import numpy as np
import pytest

import util

UYVY, YUYV, RGBA, RGB, BGR, RG48, V210, Y216, Y416, VUYA, R10K, R12L, DVS10 = 2, 3, 1, 12, 20, 27, 7, 30, 31, 4, 5, 6, 8

PAIRS = [(V210, UYVY), (YUYV, UYVY), (UYVY, YUYV), (UYVY, RGB), (YUYV, RGB), (UYVY, RGBA), (RGB, UYVY), (BGR, UYVY), (RGBA, UYVY),
         (RG48, UYVY), (RGB, RGBA), (RGBA, RGB), (RGBA, RGBA), (RGB, RGB), (BGR, RGB), (UYVY, UYVY),
         (UYVY, V210), (Y216, V210), (V210, Y216), (V210, Y416), (V210, RGB),
         (RG48, RGB), (RG48, RGBA), (RG48, R10K), (RGBA, RG48), (RGB, RG48), (UYVY, Y216), (UYVY, Y416), (Y216, UYVY), (Y416, UYVY),
         (VUYA, Y416), (VUYA, UYVY), (VUYA, RGB), (RGBA, VUYA), (R10K, RGBA), (R10K, RGB), (R10K, RG48), (RGBA, R10K),
         (Y416, RG48), (Y416, RGB), (Y416, RGBA), (Y416, R10K), (Y416, V210), (RG48, Y416), (RG48, Y216), (RG48, V210), (UYVY, RG48),
         (R10K, Y416), (R10K, UYVY),
         (R12L, RGB), (R12L, RGBA), (R12L, RG48), (R12L, R10K), (R12L, Y416), (R12L, UYVY), (RGB, R12L), (RGBA, R12L), (RG48, R12L),
         (Y416, R12L), (DVS10, UYVY), (DVS10, V210), (V210, RG48)]


def test_known_answer_checksums(orc):
    """chk = sum of output bytes over an LCG(seed 12345) frame; values from the reference build."""
    w, h = 1920, 1080
    out = util.convert_cpu(orc, "orc_convert", UYVY, RGB, util.lcg_bytes(w * h * 2), w, h)
    assert int(out.astype(np.uint64).sum()) == 798567039


@pytest.mark.parametrize("inc,outc,chk", [(UYVY, RGB, 12776800531), (RGB, UYVY, 8377299523), (V210, UYVY, 8460379454)])
def test_known_answer_checksums_8k(orc, inc, outc, chk):
    w, h = 7680, 4320
    src = util.lcg_bytes(orc.orc_vc_get_linesize(w, inc) * h)
    out = util.convert_cpu(orc, "orc_convert", inc, outc, src, w, h)
    assert int(out.astype(np.uint64).sum()) == chk


@pytest.mark.parametrize("depth", [0, 8, 10, 12, 16])
def test_color_coeffs_vs_reference(orc, depth):
    a = (ctypes.c_int * 14)()
    for cs in (0, 1, 2):
        orc.orc_get_color_coeffs(cs, depth, a)
        assert list(a) == util.ref_color_coeffs(cs, depth), (cs, depth)


def test_color_coeff_range(orc):
    """misc_test_color_coeff_range, test/misc_test.c:46-87: black/white/primaries land within 1<<(d-8) of the limits"""
    c = (ctypes.c_int * 14)()
    for d in (8, 10, 12, 16):
        orc.orc_get_color_coeffs(0, d, c)
        y_r, y_g, y_b, cb_r, cb_g, cb_b, cr_r, cr_g, cr_b = list(c)[:9]
        mx, tol = (1 << d) - 1, 1 << (d - 8)
        lo, hi_y, hi_c, mid = 1 << (d - 4), 235 << (d - 8), 240 << (d - 8), 1 << (d - 1)
        white = ((mx * (y_r + y_g + y_b)) >> 14) + lo
        assert abs(white - hi_y) <= tol
        assert abs(((mx * cb_b) >> 14) + mid - hi_c) <= tol      # blue -> max Cb
        assert abs(((mx * cr_r) >> 14) + mid - hi_c) <= tol      # red  -> max Cr
        assert abs(((mx * (cb_r + cb_g)) >> 14) + mid - lo) <= tol


@pytest.mark.parametrize("inc,outc", PAIRS)
def test_line_converters_vs_reference(orc, inc, outc):
    sizes = [(1, 2), (2, 1), (6, 3), (16, 1), (17, 5), (47, 3), (48, 2), (50, 4), (127, 9), (130, 2), (256, 3)]
    cases = []  # per size: the source and the keyword arguments of every conversion of it
    for i, (w, h) in enumerate(sizes):
        src = util.rng_bytes(orc.orc_vc_get_linesize(w, inc) * h, 1000 + i)
        kws = [{"shifts": shifts} for shifts in ((0, 8, 16), (16, 8, 0), (8, 16, 24))]
        # a dst_len that is not a whole number of pixel groups (vc_get_size instead of linesize, ragged tails)
        kws += [{"dst_len": dl} for dl in sorted({orc.orc_vc_get_size(w, outc), max(orc.orc_vc_get_size(w, outc) - 4, 0) // 4 * 4})]
        cases.append((w, h, src, kws))

    def run(lib, fn, w, h, src, kws):
        return util.digest(*[util.convert_cpu(lib, fn, inc, outc, src, w, h, **kw) for kw in kws])

    def theirs():
        ref = util.ref_cpu()
        return {"has_decoder": ref.ref_has_decoder(inc, outc), "linesize": [ref.ref_vc_get_linesize(w, inc) for w, _ in sizes],
                "out": [run(ref, "ref_convert", *c) for c in cases]}
    want = util.reference("oracle_pinning", f"line/{inc}/{outc}", theirs)
    assert orc.orc_has_decoder(inc, outc) and want["has_decoder"]
    assert [orc.orc_vc_get_linesize(w, inc) for w, _ in sizes] == want["linesize"]
    for c, d in zip(cases, want["out"], strict=True):
        assert run(orc, "orc_convert", *c) == d, (c[0], c[1], c[3])


def test_v210_to_p010_vs_reference(orc):
    for i, (w, h) in enumerate([(6, 2), (48, 4), (50, 6), (96, 5), (100, 7), (1920, 4), (7, 8), (13, 9)]):
        src = util.v210_noise(w, h, 50 + i)
        ls = ((w + 5) // 6 * 6) * 2 + 32

        def run(lib, fn):
            y = np.full(ls * h, 0xAB, dtype=np.uint8)
            c = np.full(ls * ((h + 1) // 2), 0xCD, dtype=np.uint8)
            getattr(lib, fn)(w, h, y.ctypes.data, ls, c.ctypes.data, ls, src.ctypes.data)
            return [util.digest(y), util.digest(c)]
        assert run(orc, "orc_v210_to_p010le") == util.reference("oracle_pinning", f"v210_to_p010le/{w}x{h}",
                                                                 lambda: run(util.ref_cpu(), "ref_v210_to_p010le")), (w, h)


def test_v210_p010_identity(orc):
    """the idea of ff_codec_conversions_test_pX10_from_to_v210 (test/ff_codec_conversions_test.cpp:346-401) without
    FFmpeg: every 10-bit luma sample survives v210 -> P010 exactly (<<6), chroma of equal rows too."""
    w, h = 1920, 4
    src = util.v210_noise(w, 1, 7)
    src = np.tile(src, h)  # identical rows => chroma average is the identity
    y = np.zeros(w * 2 * h, dtype=np.uint8)
    c = np.zeros(w * 2 * (h // 2), dtype=np.uint8)
    orc.orc_v210_to_p010le(w, h, y.ctypes.data, w * 2, c.ctypes.data, w * 2, src.ctypes.data)
    words = src.view(np.uint32).reshape(h, -1)[:, :w // 6 * 4].reshape(h, -1, 4)
    luma = np.stack([(words[:, :, 0] >> 10) & 0x3ff, words[:, :, 1] & 0x3ff, (words[:, :, 1] >> 20) & 0x3ff,
                     (words[:, :, 2] >> 10) & 0x3ff, words[:, :, 3] & 0x3ff, (words[:, :, 3] >> 20) & 0x3ff], axis=2)
    assert np.array_equal(y.view(np.uint16).reshape(h, w), (luma.reshape(h, w) << 6).astype(np.uint16))
    chroma = np.stack([words[:, :, 0] & 0x3ff, (words[:, :, 0] >> 20) & 0x3ff, (words[:, :, 1] >> 10) & 0x3ff,
                       words[:, :, 2] & 0x3ff, (words[:, :, 2] >> 20) & 0x3ff, (words[:, :, 3] >> 10) & 0x3ff], axis=2)
    assert np.array_equal(c.view(np.uint16).reshape(h // 2, w), (chroma[::2].reshape(h // 2, w) << 6).astype(np.uint16))


def test_golden_vectors(orc):
    """fixtures generated from the reference by tests/golden/make_golden.py (travel to the GPU box, no reference needed)"""
    path = os.path.join(util.ROOT, "tests", "golden", "pixfmt_golden.npz")
    g = np.load(path)
    cases = [k[:-4] for k in g.files if k.endswith("_src") and k.startswith("c")]
    assert len(cases) >= 16
    for k in cases:
        inc, outc, w, h = [int(v) for v in g[k + "_meta"]]
        out = util.convert_cpu(orc, "orc_convert", inc, outc, g[k + "_src"], w, h)
        assert np.array_equal(out, g[k + "_dst"]), k
    y = np.zeros_like(g["p010_y"])
    c = np.zeros_like(g["p010_c"])
    w, h, ls = [int(v) for v in g["p010_meta"]]
    src = g["p010_src"]  # keep the array alive while ctypes holds its pointer
    orc.orc_v210_to_p010le(w, h, y.ctypes.data, ls, c.ctypes.data, ls, src.ctypes.data)
    assert np.array_equal(y, g["p010_y"]) and np.array_equal(c, g["p010_c"])
