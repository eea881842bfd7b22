"""The line converters pixfmt_conv.h exports outside the decoders[] table (SURVEY.md section 8 row A9): vc_copylineABGRtoRGB, BGRAtoRGB,
ToRGBA_inplace, UYVYtoGrayscale.  CPU: restatement == unmodified reference objects; GPU: ugb200_vc_copyline == restatement."""
import ctypes

import numpy as np
import pytest

import util

FUNCS = {"ABGRtoRGB": (1, 4, 3), "BGRAtoRGB": (2, 4, 3), "ToRGBA_inplace": (3, 4, 4), "UYVYtoGrayscale": (4, 2, 1)}  # id, bytes/px in, out
SIZES = [(1, 2), (3, 1), (7, 3), (8, 2), (9, 2), (16, 1), (17, 5), (50, 4), (130, 2), (256, 3)]
SHIFTS = [(0, 8, 16), (16, 8, 0), (8, 16, 24), (24, 16, 8)]


def run_cpu(lib, fn, fid, src, w, h, bi, bo, shifts, dst_len=None):
    sp, dp = w * bi, w * bo
    dst = np.full(dp * h + 64, 0xCD, np.uint8)
    srcp = np.concatenate([src, np.zeros(4096, np.uint8)])
    f = getattr(lib, fn)
    f.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_long, ctypes.c_void_p, ctypes.c_long, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int]
    assert f(fid, dst.ctypes.data, dp, srcp.ctypes.data, sp, dp if dst_len is None else dst_len, h, *shifts) == 0
    return dst[:dp * h]


@pytest.mark.parametrize("name", list(FUNCS))
def test_restatement_equals_reference(orc, name):
    fid, bi, bo = FUNCS[name]
    srcs = [util.rng_bytes(w * bi * h, 300 + i) for i, (w, h) in enumerate(SIZES)]

    def run(lib, fn, src, w, h):  # every shift and dst_len of one size
        return util.digest(*[run_cpu(lib, fn, fid, src, w, h, bi, bo, shifts, dl)
                             for shifts in SHIFTS for dl in (None, max(w * bo - 2, 0), max(w * bo - bo, 0))])
    want = util.reference("named_line_converters", name, lambda: [run(util.ref_cpu(), "ref_copyline_named", s, w, h) for s, (w, h) in zip(srcs, SIZES)])
    for src, (w, h), d in zip(srcs, SIZES, want, strict=True):
        assert run(orc, "orc_copyline_named", src, w, h) == d, (name, w, h)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(FUNCS))
def test_gpu_equals_restatement(orc, name):
    import torch
    from ultragrid_b200 import api
    fid, bi, bo = FUNCS[name]
    for i, (w, h) in enumerate(SIZES + [(1920, 1080)]):
        src = util.rng_bytes(w * bi * h, 400 + i)
        for shifts in SHIFTS[:2] + SHIFTS[3:]:
            want = run_cpu(orc, "orc_copyline_named", fid, src, w, h, bi, bo, shifts)
            d_src = torch.from_numpy(np.concatenate([src, np.zeros(64, np.uint8)])).cuda()
            d_dst = torch.full((w * bo * h,), 0xCD, dtype=torch.uint8, device="cuda")
            api.vc_copyline(name, d_src, d_dst, w * bo, h, w * bi, w * bo, shifts)
            assert np.array_equal(d_dst.cpu().numpy(), want), (name, w, h, shifts)
    if name == "ToRGBA_inplace":  # dst == src
        w, h = 333, 7
        src = util.rng_bytes(w * 4 * h, 9)
        want = run_cpu(orc, "orc_copyline_named", fid, src, w, h, 4, 4, (16, 8, 0))
        buf = torch.from_numpy(src.copy()).cuda()
        api.vc_copyline(name, buf, buf, w * 4, h, w * 4, w * 4, (16, 8, 0))
        assert np.array_equal(buf.cpu().numpy(), want)
