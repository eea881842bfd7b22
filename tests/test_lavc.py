"""libavcodec bridge conversions (SURVEY.md section 8f rank 3; include/ugb200_lavc.h).  The reference file cannot be compiled here (FFmpeg headers
absent) - PARITY UNPINNED against it; CPU part: the restatement oracle/lavc_oracle.c against what the tree does pin (colour coefficients of the
unmodified color_space.c, identities through the unmodified to_planar.c / from_planar.c); GPU part: kernels == restatement, byte for byte."""
import ctypes

import numpy as np
import pytest

import util

RGBA, UYVY, R10k, R12L, V210, RGB, RG48 = 1, 2, 5, 6, 7, 12, 27
_vp, _i = ctypes.c_void_p, ctypes.c_int


class Coeffs(ctypes.Structure):
    _fields_ = [(n, _i) for n in ("y_r", "y_g", "y_b", "cb_r", "cb_g", "cb_b", "cr_r", "cr_g", "cr_b")]


def coeffs(depth):
    """get_color_coeffs(CS_DFL, depth) of the UNMODIFIED src/color_space.c"""
    return Coeffs(*util.ref_color_coeffs(0, depth)[:9])


def planes_for(shapes, fill=0xA5):
    bufs = [np.full(ls * rows, fill, np.uint8) for ls, rows in shapes]
    p = (_vp * 3)(*[b.ctypes.data for b in bufs] + [None] * (3 - len(bufs)))
    ls = (_i * 3)(*[s[0] for s in shapes] + [0] * (3 - len(shapes)))
    return bufs, p, ls


def lavc_cpu(orc, in_codec, fmt, src, w, h, pad=0):
    from ultragrid_b200 import api
    shapes = api.av_plane_shapes(fmt, w, h, pad)
    bufs, p, ls = planes_for(shapes)
    if in_codec == V210:
        orc.orc_lavc_v210({"YUV420P10LE": 0, "YUV422P10LE": 1, "YUV444P10LE": 2, "YUV444P16LE": 3}[fmt], src.ctypes.data, w, h, p, ls)
    elif in_codec == UYVY:
        orc.orc_lavc_uyvy(1 if fmt == "YUV444P" else 0, src.ctypes.data, w, h, p, ls)
    elif fmt == "GBRP":
        orc.orc_lavc_gbrp(3 if in_codec == RGB else 4, src.ctypes.data, w, h, p, ls)
    else:
        depth = 8 if fmt == "YUV444P" else int(fmt[7:9])
        kind = {R10k: 0, RG48: 1, R12L: 2, RGB: 3}[in_codec]
        orc.orc_lavc_rgb(kind, depth, 1 if "422" in fmt else 0, ctypes.byref(coeffs(depth)), src.ctypes.data, w, h, p, ls)
    return bufs, shapes


PAIRS = [(V210, "YUV420P10LE"), (V210, "YUV422P10LE"), (V210, "YUV444P10LE"), (V210, "YUV444P16LE"), (UYVY, "YUV422P"), (UYVY, "YUV444P"),
         (R10k, "YUV444P10LE"), (R10k, "YUV444P12LE"), (R10k, "YUV444P16LE"), (RG48, "YUV444P10LE"), (RG48, "YUV444P12LE"), (RG48, "YUV444P16LE"),
         (R12L, "YUV444P10LE"), (R12L, "YUV444P12LE"), (R12L, "YUV444P16LE"), (R12L, "YUV422P10LE"), (R12L, "YUV422P12LE"), (R12L, "YUV422P16LE"),
         (RGB, "YUV444P"), (RGB, "GBRP"), (RGBA, "GBRP")]


def source(orc, in_codec, w, h, seed):
    if in_codec == V210:
        return util.v210_noise(w, h, seed)
    return util.rng_bytes(orc.orc_vc_get_linesize(w, in_codec) * h, seed)


def test_support_table_and_hook_refusals():
    from ultragrid_b200 import _lib, api
    L = _lib.load()
    for inc, fmt in PAIRS + [(V210, "P010LE"), (UYVY, "NV12"), (UYVY, "YUV420P")]:
        assert L.ugb200_to_lavc_supported(inc, api.AV_PIXFMT[fmt]), (inc, fmt)
    assert not L.ugb200_to_lavc_supported(UYVY, api.AV_PIXFMT["YUV444P16LE"]) and not L.ugb200_to_lavc_supported(V210, api.AV_PIXFMT["GBRP"])
    assert not L.ugb200_to_lavc_vid_conv_init(UYVY, 0, 16, api.AV_PIXFMT["YUV422P"])    # bad size
    assert not L.ugb200_to_lavc_vid_conv_init(UYVY, 64, 16, api.AV_PIXFMT["GBRP"])      # unsupported pair
    assert not L.ugb200_get_av_to_uv_conversion(api.AV_PIXFMT["NV12"], UYVY)


def test_restatement_v210_identities_through_reference_functions(orc):
    """v210 -> yuv422p10le -> (UNMODIFIED yuv422p10le_to_v210, from_planar.c:295-333) == the v210 frame (30 valid bits per word), and
    v210 -> yuv420p10le == UNMODIFIED v210_to_p010le >> 6 (to_planar.c:64-155): the idea of test/ff_codec_conversions_test.cpp:346-401"""
    w, h = 96, 6
    src = util.v210_noise(w, h, 4)
    bufs, shapes = lavc_cpu(orc, V210, "YUV422P10LE", src, w, h)

    def back():  # the planes and what the reference packs them back into
        ref = util.ref_cpu()
        out = np.zeros_like(src)
        ref.ref_yuv422p10le_to_v210.argtypes = [_i, _i, _vp, ctypes.c_uint, _vp, _vp, _vp, ctypes.c_uint, ctypes.c_uint]
        ref.ref_yuv422p10le_to_v210(w, h, out.ctypes.data, len(src) // h, bufs[0].ctypes.data, bufs[1].ctypes.data, bufs[2].ctypes.data, shapes[0][0], shapes[1][0])
        return {"planes": util.digest(*bufs), "v210": util.digest(out)}
    want = util.reference("lavc", "yuv422p10le_to_v210", back)
    assert util.digest(*bufs) == want["planes"] and want["v210"] == util.digest(src)
    # 4:2:0: luma and averaged chroma against the reference's P010 converter (samples there sit in the 10 MSBs, chroma interleaved)
    bufs, shapes = lavc_cpu(orc, V210, "YUV420P10LE", src, w, h)

    def p010():
        y, c = np.zeros(w * 2 * h, np.uint8), np.zeros(w * h, np.uint8)
        util.ref_cpu().ref_v210_to_p010le(w, h, y.ctypes.data, w * 2, c.ctypes.data, w * 2, src.ctypes.data)
        cc = (c.view(np.uint16) >> 6).reshape(h // 2, w)
        return [util.digest(y.view(np.uint16) >> 6), util.digest(cc[:, 0::2]), util.digest(cc[:, 1::2])]
    want = util.reference("lavc", "v210_to_p010le", p010)
    assert [util.digest(b.view(np.uint16)) for b in bufs] == want


def test_restatement_rgb_matrix_against_reference_line_converters(orc):
    """RG48 -> yuv444p16le uses the same Q14 matrix at depth 16 as the reference's vc_copylineRG48toY416 -style converters use: spot values by hand
    (coefficients from the unmodified color_space.c), limited-range offsets, and a white / black / primary sanity sweep"""
    c = coeffs(16)
    src = np.array([[65535, 65535, 65535], [0, 0, 0], [65535, 0, 0], [0, 65535, 0], [0, 0, 65535], [12345, 23456, 34567]], np.uint16)
    w, h = len(src), 1
    bufs, _ = lavc_cpu(orc, RG48, "YUV444P16LE", src.view(np.uint8).reshape(-1), w, h)
    Y, CB, CR = (b.view(np.uint16)[:w].astype(np.int64) for b in bufs)
    for i, (r, g, b) in enumerate(src.astype(np.int64)):
        assert Y[i] == ((r * c.y_r + g * c.y_g + b * c.y_b) >> 14) + 4096
        assert CB[i] == (((r * c.cb_r + g * c.cb_g + b * c.cb_b) >> 14) + 32768) % 65536
        assert CR[i] == (((r * c.cr_r + g * c.cr_g + b * c.cr_b) >> 14) + 32768) % 65536
    assert abs(int(Y[0]) - 60160) <= 8 and Y[1] == 4096 and abs(int(CB[0]) - 32768) <= 2  # white = 235 << 8, black = 16 << 8, grey chroma


@pytest.mark.gpu
@pytest.mark.parametrize("inc,fmt", PAIRS)
def test_gpu_to_lavc_equals_restatement(orc, inc, fmt):
    import torch
    from ultragrid_b200 import api
    for k, (w, h, pad) in enumerate([(48, 4, 0), (96, 6, 32), (100, 5, 0), (8, 2, 0), (1920, 16, 64), (1922, 3, 10)]):
        if inc == V210 and fmt == "YUV420P10LE" and h % 2:
            h += 1
        src = source(orc, inc, w, h, 300 + k)
        want, shapes = lavc_cpu(orc, inc, fmt, src, w, h, pad)
        planes = [torch.full((ls * rows,), 0xA5, dtype=torch.uint8, device="cuda") for ls, rows in shapes]
        got = api.to_lavc(inc, fmt, torch.from_numpy(src).cuda(), w, h, planes=planes, pad=pad)
        for i, (g, wnt) in enumerate(zip(got, want)):
            assert np.array_equal(g.cpu().numpy(), wnt), (w, h, pad, i)


@pytest.mark.gpu
def test_gpu_delegated_conversions_equal_to_planar(orc):
    """v210 -> P010LE, UYVY -> NV12 / YUV420P go through the to_planar kernels (as the reference delegates, to_lavc_vid_conv.c:132-135,186-189)"""
    import torch
    from ultragrid_b200 import api
    w, h = 96, 8
    src = util.v210_noise(w, h, 9)
    y, c = api.to_lavc(V210, "P010LE", torch.from_numpy(src).cuda(), w, h)
    wy, wc = np.zeros(w * 2 * h, np.uint8), np.zeros(w * h, np.uint8)
    orc.orc_v210_to_p010le(w, h, wy.ctypes.data, w * 2, wc.ctypes.data, w * 2, src.ctypes.data)
    assert np.array_equal(y.cpu().numpy(), wy) and np.array_equal(c.cpu().numpy(), wc)


@pytest.mark.gpu
def test_gpu_hook_shape_host_frame_in_device_planes_out(orc):
    """to_lavc_vid_conv_cuda_init / to_lavc_vid_conv_cuda / _destroy (to_lavc_vid_conv_cuda.h:60-65): host frame in like the reference's hook"""
    import torch
    from ultragrid_b200 import _lib, api
    L = _lib.load()
    w, h = 1920, 1080
    src = util.rng_bytes(w * 2 * h, 77)
    st = L.ugb200_to_lavc_vid_conv_init(UYVY, w, h, api.AV_PIXFMT["YUV444P"])  # the format the reference's hook names
    assert st
    p = ctypes.cast(L.ugb200_to_lavc_vid_conv(st, src.ctypes.data, 0), ctypes.POINTER(api.AvPlanes)).contents
    want, shapes = lavc_cpu(orc, UYVY, "YUV444P", src, w, h)
    for i in range(3):
        ls = p.linesize[i]
        host = np.zeros(ls * h, np.uint8)
        assert L.cuda_wrapper_memcpy(host.ctypes.data, p.data[i], host.size, 1) == 0
        assert np.array_equal(host.reshape(h, ls)[:, :w], want[i].reshape(h, -1)[:, :w])
    h_st = ctypes.c_void_p(st)
    L.ugb200_to_lavc_vid_conv_destroy(ctypes.byref(h_st))
    assert not h_st.value


@pytest.mark.gpu
@pytest.mark.parametrize("out_codec", [UYVY, RGB, RGBA, V210])
def test_gpu_from_lavc_yuv422p_to_any_codec(orc, out_codec):
    """av_to_uv_convert_cuda shape: YUV422P planes (the format from_lavc_vid_conv_cuda.h:55-57 declares) -> UYVY, and on through the line converters"""
    import torch
    from ultragrid_b200 import api
    w, h = 192, 10
    uyvy = util.rng_bytes(w * 2 * h, 5)
    u = uyvy.reshape(h, w // 2, 4)
    Y = np.ascontiguousarray(np.stack([u[:, :, 1], u[:, :, 3]], axis=2).reshape(h, w))
    Cb, Cr = np.ascontiguousarray(u[:, :, 0]), np.ascontiguousarray(u[:, :, 2])
    planes = [torch.from_numpy(a.reshape(-1)).cuda() for a in (Y, Cb, Cr)]
    pitch = orc.orc_vc_get_linesize(w, out_codec)
    dst = torch.zeros(pitch * h, dtype=torch.uint8, device="cuda")
    api.from_lavc("YUV422P", out_codec, planes, [w, w // 2, w // 2], w, h, dst, pitch)
    want = uyvy if out_codec == UYVY else util.convert_cpu(orc, "orc_convert", UYVY, out_codec, uyvy, w, h)
    assert np.array_equal(dst.cpu().numpy(), want)
