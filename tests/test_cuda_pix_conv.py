"""src/utils/cuda_pix_conv.cu of the reference (SURVEY.md section 8f rank 4): cuda_RGB_to_RGBA, cuda_RGBA_to_RGB, cuda_UYVY_to_RGBA,
cuda_RGBA_to_UYVY with the reference's C++ names.  GPU: libugb200 == the UNMODIFIED reference file built for sm_100a (oracle/_ref; its outputs
recorded in tests/golden/reference_cuda_pix_conv.json) == the CPU restatement, byte for byte."""
import ctypes
import os

import numpy as np
import pytest

import util

NAMES = {"RGB_to_RGBA": ("_Z16cuda_RGB_to_RGBAPhmS_mmmP11CUstream_st", 0, 3, 4), "RGBA_to_RGB": ("_Z16cuda_RGBA_to_RGBPhmS_mmmP11CUstream_st", 1, 4, 3),
         "UYVY_to_RGBA": ("_Z17cuda_UYVY_to_RGBAPhmS_mmmP11CUstream_st", 2, 2, 4), "RGBA_to_UYVY": ("_Z17cuda_RGBA_to_UYVYPhmS_mmmP11CUstream_st", 3, 4, 2)}
ARGS = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_size_t, ctypes.c_size_t, ctypes.c_void_p]


def test_library_exports_the_reference_cxx_symbols():
    from ultragrid_b200 import _lib
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for sym, *_ in NAMES.values():
        assert hasattr(lib, sym), sym


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(NAMES))
def test_gpu_equals_reference_kernels_and_restatement(orc, name):
    import torch
    from ultragrid_b200 import _lib
    lib = ctypes.CDLL(_lib.LIB_PATH)
    sym, kind, bi, bo = NAMES[name]
    orc.orc_cuda_pix_conv.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_int]
    orc.orc_cuda_pix_conv.restype = None
    for i, (w, h, pad) in enumerate([(2, 1, 0), (5, 3, 0), (16, 2, 0), (17, 5, 4), (64, 4, 16), (130, 3, 8), (1920, 1080, 0), (7680, 16, 0)]):  # pitches stay 4-byte aligned: the reference stores uchar4
        wi = (w + 1) // 2 * 2 if bi == 2 else w  # UYVY rows hold whole pairs
        sp, dp = wi * bi + pad, ((w + 1) // 2 * 2 if bo == 2 else w) * bo + pad
        src = util.rng_bytes(sp * h, 900 + i)
        want = np.full(dp * h, 0xCD, np.uint8)
        orc.orc_cuda_pix_conv(kind, want.ctypes.data, dp, src.ctypes.data, sp, w, h)
        d_src = torch.from_numpy(src).cuda()

        def run(L):
            fn = getattr(L, sym)
            fn.argtypes, fn.restype = ARGS, None
            d_dst = torch.full((dp * h,), 0xCD, dtype=torch.uint8, device="cuda")
            fn(d_dst.data_ptr(), dp, d_src.data_ptr(), sp, w, h, None)
            torch.cuda.synchronize()
            return d_dst.cpu().numpy()
        o = run(lib)
        assert np.array_equal(o, want), (name, w, h, pad, np.flatnonzero(o != want)[:8])
        theirs = util.reference("cuda_pix_conv", f"{name}/{w}x{h}+{pad}",
                                lambda: util.digest(run(ctypes.CDLL(os.path.join(util.ORACLE_DIR, "_ref", "libcuda_pix_conv_ref.so")))))
        assert util.digest(want) == theirs, (name, w, h, pad)
