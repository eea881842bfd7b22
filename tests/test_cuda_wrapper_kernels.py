"""src/cuda_wrapper/kernels.cu of the reference (SURVEY.md section 8f rank 4): postprocess_rg48_to_r12l / preprocess_r12l_to_rg48, the CUDA callbacks the
Comprimato J2K modules hand to the codec, under their own C++ names (include/cuda_wrapper_kernels.hpp).  GPU: libugb200 == the UNMODIFIED reference file built
for sm_100a (oracle/_ref/libcuda_wrapper_kernels_ref.so) == the pinned CPU line converters, byte for byte where the reference's result is defined."""
import ctypes
import os

import numpy as np
import pytest

import util

RG48, R12L = 27, 6
POST = "_Z24postprocess_rg48_to_r12lPvS_miiP25cmpto_j2k_dec_comp_formatiS_mS_mS_mS_"
PRE = "_Z23preprocess_r12l_to_rg48PvS_miiP25cmpto_j2k_enc_comp_formatiS_mS_mS_"
VP, SZ, I = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int
POST_ARGS = [VP, VP, SZ, I, I, VP, I, VP, SZ, VP, SZ, VP, SZ, VP]
PRE_ARGS = [VP, VP, SZ, I, I, VP, I, VP, SZ, VP, SZ, VP]


def test_codec_ids():
    from ultragrid_b200 import Codec
    assert (int(Codec.RG48), int(Codec.R12L)) == (RG48, R12L)


def test_library_exports_the_reference_cxx_symbols():
    from ultragrid_b200 import _lib
    lib = ctypes.CDLL(_lib.LIB_PATH)
    assert hasattr(lib, POST) and hasattr(lib, PRE)


def entry_points(path):
    """(postprocess_rg48_to_r12l, preprocess_r12l_to_rg48) of libugb200, or of the reference build when path is given"""
    from ultragrid_b200 import _lib
    L = ctypes.CDLL(path or _lib.LIB_PATH)
    post, pre = getattr(L, POST), getattr(L, PRE)
    post.argtypes, post.restype, pre.argtypes, pre.restype = POST_ARGS, I, PRE_ARGS, I
    return post, pre


REF = os.path.join(util.ORACLE_DIR, "_ref", "libcuda_wrapper_kernels_ref.so")  # its outputs are recorded in tests/golden/reference_cuda_wrapper_kernels.json


SIZES = [(8, 1), (16, 3), (64, 2), (256, 5), (1920, 8), (7680, 4), (4, 2), (9, 3), (30, 2), (1000, 3), (1921, 2), (255, 4)]


@pytest.mark.gpu
@pytest.mark.parametrize("w,h", SIZES)
def test_rg48_to_r12l_equals_reference_kernel(orc, w, h):
    import torch
    nb = (w + 7) // 8
    src = util.rng_bytes(w * 6 * h, 700 + w)
    d_src = torch.from_numpy(src).cuda()

    def run(path):
        post, _ = entry_points(path)
        d_dst = torch.full((nb * 36 * h,), 0xCD, dtype=torch.uint8, device="cuda")
        assert post(None, None, 0, w, h, None, 3, d_src.data_ptr(), src.size, None, 0, d_dst.data_ptr(), d_dst.numel(), None) == 0
        torch.cuda.synchronize()
        return d_dst.cpu().numpy().reshape(h, nb * 36)
    outs = [run(None)]
    # the whole groups are vc_copylineRG48toR12L of the pinned oracle
    want = util.convert_cpu(orc, "orc_convert", RG48, R12L, src, w, h, src_pitch=w * 6, dst_pitch=nb * 36, dst_len=nb * 36).reshape(h, nb * 36)
    full = w // 8 * 36
    defined = full + (w % 8) * 36 // 8  # bytes of the last group that depend only on samples inside the row (4.5 bytes per pixel, rounded down)
    assert np.array_equal(outs[0][:, :full], want[:, :full])
    # the reference kernel: its defined bytes equal ours (and so the oracle's whole groups)
    assert util.digest(outs[0][:, :defined]) == util.reference("cuda_wrapper_kernels", f"rg48_to_r12l/{w}x{h}", lambda: util.digest(run(REF)[:, :defined]))
    if w % 8:  # the partial group is written (the CPU line converter stops before it): its defined bytes are the packed samples
        s16 = src.view(np.uint16).reshape(h, w * 3)[:, w // 8 * 24:] >> 4
        bits = np.zeros((h, 36), np.uint8)
        for k in range(s16.shape[1]):
            v = s16[:, k].astype(np.uint32) << (12 * k % 8)
            bits[:, 12 * k // 8] |= (v & 0xFF).astype(np.uint8)
            bits[:, 12 * k // 8 + 1] |= (v >> 8).astype(np.uint8)
        n = defined - full
        assert np.array_equal(outs[0][:, full:defined], bits[:, :n])


@pytest.mark.gpu
@pytest.mark.parametrize("w,h", SIZES)
def test_r12l_to_rg48_equals_reference_kernel(orc, w, h):
    import torch
    nb = (w + 7) // 8
    src = util.rng_bytes(nb * 36 * h, 800 + w)
    d_src = torch.from_numpy(src).cuda()

    def run(path):
        _, pre = entry_points(path)
        d_dst = torch.full((w * 6 * h + 64,), 0xCD, dtype=torch.uint8, device="cuda")
        assert pre(None, None, 0, w, h, None, 3, d_src.data_ptr(), src.size, d_dst.data_ptr(), w * 6 * h, None) == 0
        torch.cuda.synchronize()
        return d_dst.cpu().numpy()
    o = run(None)
    want = util.convert_cpu(orc, "orc_convert", R12L, RG48, src, w, h, src_pitch=nb * 36, dst_pitch=w * 6, dst_len=w * 6)
    assert np.array_equal(o[:w * 6 * h], want)
    assert np.all(o[w * 6 * h:] == 0xCD)  # exactly size_x * 6 bytes per row, nothing behind the frame
    # the reference kernel wrote the same bytes, and nothing else
    assert util.digest(o) == util.reference("cuda_wrapper_kernels", f"r12l_to_rg48/{w}x{h}", lambda: util.digest(run(REF)))
