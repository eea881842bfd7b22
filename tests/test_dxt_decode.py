"""DXT1 / DXT5-YCoCg decode (SURVEY.md section 8f rank 1).  Contract for DXT5-YCoCg: the reference's CPU tool cuda_dxt/dxt62tga.c:24-108
(double arithmetic), compiled unmodified into oracle/_ref; DXT1 follows the same rule for its colour block (no CPU decoder in the tree)."""
import ctypes

import numpy as np
import pytest

import util


def orc_decode(orc, blocks, w, h, dxt_type, bgr=0, pitch=None):
    pitch = pitch or w * 3
    out = np.full(pitch * h, 0xCD, np.uint8)
    fn = orc.orc_dxt1_to_rgb if dxt_type == 1 else orc.orc_dxt5ycocg_to_rgb
    fn.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_long, ctypes.c_int]
    fn.restype = None
    fn(blocks.ctypes.data, out.ctypes.data, w, h, pitch, bgr)
    return out


def hard_blocks(n_bytes, seed):
    """any bit pattern is a valid block: noise, plus blocks with equal / swapped endpoints and extreme alpha"""
    b = util.rng_bytes(n_bytes, seed).copy()
    b[:64] = 0
    b[64:128] = 255
    return b


def test_dxt5ycocg_decoder_restatement_equals_reference_tool(orc):
    for seed, (w, h) in enumerate([(4, 4), (64, 16), (256, 64), (1920, 1080)]):
        blk = hard_blocks(w * h, seed)

        def theirs():
            ref = util.ref_cpu()
            ref.ref_dxt5ycocg_to_bgr.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int]
            want = np.zeros(w * h * 3, np.uint8)
            ref.ref_dxt5ycocg_to_bgr(blk.ctypes.data, want.ctypes.data, w, h)
            return util.digest(want)
        assert util.digest(orc_decode(orc, blk, w, h, 6, bgr=1)) == util.reference("dxt_decode", f"dxt5ycocg_to_bgr/{w}x{h}", theirs), (w, h)


def test_dxt_roundtrip_psnr_cpu(orc):
    """encode with the restated encoders, decode: the blocks describe the image"""
    from test_jpeg import natural_rgb, psnr
    w, h = 256, 128
    rgb = natural_rgb(w, h, 4).reshape(-1).copy()
    for t, fn, nbytes, floor in ((1, orc.orc_rgb_to_dxt1, w * h // 2, 30.0), (6, orc.orc_rgb_to_dxt6, w * h, 33.0)):
        out = np.zeros(nbytes, np.uint8)
        fn.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int]
        assert fn(rgb.ctypes.data, out.ctypes.data, w, h) == 0
        assert psnr(orc_decode(orc, out, w, h, t), rgb) > floor


@pytest.mark.gpu
@pytest.mark.parametrize("dxt_type", [1, 6])
@pytest.mark.parametrize("w,h", [(4, 4), (64, 16), (260, 36), (1920, 1080), (7680, 4320)])
def test_gpu_decode_equals_oracle(orc, dxt_type, w, h):
    import torch
    from ultragrid_b200 import api
    blk = hard_blocks(w * h // (2 if dxt_type == 1 else 1), w + dxt_type)
    d = torch.from_numpy(blk).cuda()
    for bgr in (0, 1):
        assert np.array_equal(api.dxt_to_rgb(d, w, h, dxt_type, bgr=bool(bgr)).cpu().numpy(), orc_decode(orc, blk, w, h, dxt_type, bgr))
    if w <= 260:  # padded rows: bytes outside the image stay untouched
        pitch = w * 3 + 20
        out = torch.full((pitch * h,), 0xCD, dtype=torch.uint8, device="cuda")
        api.dxt_to_rgb(d, w, h, dxt_type, out=out, out_pitch=pitch)
        assert np.array_equal(out.cpu().numpy(), orc_decode(orc, blk, w, h, dxt_type, pitch=pitch))


@pytest.mark.gpu
def test_gpu_encode_decode_roundtrip_8k(orc):
    import torch
    from ultragrid_b200 import api
    from test_jpeg import natural_rgb, psnr
    w, h = 7680, 4320
    rgb = natural_rgb(w, h, 6).reshape(-1)
    uyvy = torch.from_numpy(util.convert_cpu(orc, "orc_convert", 12, 2, rgb, w, h)).cuda()
    for t, floor in ((1, 30.0), (6, 33.0)):
        back = api.dxt_to_rgb(api.uyvy_to_dxt(uyvy, w, h, dxt_type=t), w, h, t).cpu().numpy()
        assert psnr(back, rgb) > floor

