"""GPU parity of the DXT entry points, through the C ABI.

Bit-exact oracle = the UNMODIFIED reference kernel (cuda_dxt/cuda_dxt.cu) built for sm_100a with the same nvcc
(oracle/_ref/libcuda_dxt_ref.so); its outputs for these inputs are recorded in tests/golden/reference_dxt_gpu.json.  The CPU restatement
(oracle/dxt_oracle.c) is compared too and must agree except where MUFU.RCP rounding flips a DXT1 index.
"""
import ctypes

import numpy as np
import pytest

import util

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def api():
    from ultragrid_b200 import api as a
    return a


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def ref_dxt(name, src_dev, w, h, dxt_type=1):
    """the reference kernel's output (recorded: see util.reference)"""
    out = torch.empty(w * abs(h) // 2 * (1 if dxt_type == 1 else 2), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    rc = getattr(util.ref_gpu(), name)(ctypes.c_void_p(src_dev.data_ptr()), ctypes.c_void_p(out.data_ptr()), w, h, None)
    assert rc == 0
    return out


def special_blocks_rgb(w, h, seed):
    """frames made of hard cases: flat, two-colour, negative covariance, near-equal endpoints, gradients, extremes"""
    rng = np.random.default_rng(seed)
    img = np.zeros((h, w, 3), dtype=np.uint8)
    for by in range(h // 4):
        for bx in range(w // 4):
            kind = (bx + 7 * by) % 8
            blk = img[by * 4:by * 4 + 4, bx * 4:bx * 4 + 4]
            if kind == 0:
                blk[:] = rng.integers(0, 256, 3)
            elif kind == 1:
                a, b = rng.integers(0, 256, (2, 3))
                blk[:] = np.where(rng.integers(0, 2, (4, 4, 1)) == 1, a, b)
            elif kind == 2:  # red up, blue down: negative r/b covariance
                t = rng.integers(0, 256, (4, 4))
                blk[:, :, 0], blk[:, :, 1], blk[:, :, 2] = t, rng.integers(0, 256), 255 - t
            elif kind == 3:  # endpoints one 565 step apart
                base = rng.integers(0, 248, 3)
                blk[:] = base + rng.integers(0, 9, (4, 4, 3))
            elif kind == 4:
                g = np.linspace(0, 255, 16).reshape(4, 4).astype(np.uint8)
                blk[:, :, 0], blk[:, :, 1], blk[:, :, 2] = g, g.T, 255 - g
            elif kind == 5:
                blk[:] = rng.choice([0, 255], (4, 4, 3))
            elif kind == 6:
                blk[:] = rng.integers(120, 136, (4, 4, 3))
            else:
                blk[:] = rng.integers(0, 256, (4, 4, 3))
    return img.reshape(-1)


FRAMES = ["noise", "testcard", "special"]


def make_packed3(kind, w, h, seed=1):
    if kind == "noise":
        return util.rng_bytes(w * h * 3, seed)
    if kind == "testcard":
        return util.testcard_rgb(w, h)
    return special_blocks_rgb(w, h, seed)


@pytest.mark.parametrize("name", ["cuda_rgb_to_dxt1", "cuda_yuv_to_dxt1", "cuda_rgb_to_dxt6", "cuda_yuv_to_dxt6"])
@pytest.mark.parametrize("kind", FRAMES)
@pytest.mark.parametrize("w,h", [(4, 4), (64, 36), (1920, 1080), (3840, 2160), (1924, -1080), (200, -52)])
def test_packed3_bit_exact_vs_reference_kernel(api, name, kind, w, h):
    src = dev(make_packed3(kind, w, abs(h), seed=w + abs(h)))
    mine = api.compat_to_dxt(name, src, w, h)
    theirs = util.reference("dxt_gpu", f"packed3/{name}/{kind}/{w}x{h}", lambda: util.digest(ref_dxt(name, src, w, h, dxt_type=1 if name.endswith("1") else 6)))
    assert util.digest(mine) == theirs


@pytest.mark.parametrize("kind", FRAMES)
@pytest.mark.parametrize("w,h", [(8, 4), (36, 20), (1920, 1080), (7680, 4320), (3844, -2160)])
def test_fused_uyvy_dxt6_equals_reference_pipeline(api, orc, kind, w, h):
    """config 5: UYVY -> DXT5-YCoCg; reference path = cuda_yuv422_to_yuv444 + cuda_yuv_to_dxt6"""
    ah = abs(h)
    if kind == "testcard":
        uyvy = util.testcard_uyvy(w, ah, orc)
    elif kind == "noise":
        uyvy = util.rng_bytes(w * ah * 2, 199 + w)
    else:
        uyvy = util.convert_cpu(orc, "orc_convert", 12, 2, special_blocks_rgb(w, ah, 6), w, ah)
    e = np.zeros(w * ah * 3, dtype=np.uint8)
    orc.orc_yuv422_to_yuv444(uyvy.ctypes.data, e.ctypes.data, w * ah)
    theirs = util.reference("dxt_gpu", f"fused_dxt6/{kind}/{w}x{h}", lambda: util.digest(ref_dxt("cuda_yuv_to_dxt6", dev(e), w, h, dxt_type=6)))
    mine = api.uyvy_to_dxt(dev(uyvy), w, h, dxt_type=6)
    assert util.digest(mine) == theirs


def test_cpu_oracle_dxt6_is_bit_exact(orc):
    """DXT5-YCoCg has no approximate instruction on its path: oracle/dxt_oracle.c must equal the reference kernel exactly"""
    w, h = 512, 256
    for name, fn, kind in (("cuda_rgb_to_dxt6", "orc_rgb_to_dxt6", "noise"), ("cuda_yuv_to_dxt6", "orc_yuv_to_dxt6", "noise"),
                           ("cuda_rgb_to_dxt6", "orc_rgb_to_dxt6", "special"), ("cuda_rgb_to_dxt6", "orc_rgb_to_dxt6", "testcard")):
        src = make_packed3(kind, w, h, seed=21)
        theirs = util.reference("dxt_gpu", f"cpu_dxt6/{name}/{kind}", lambda: util.digest(ref_dxt(name, dev(src), w, h, dxt_type=6)))
        mine = np.zeros(w * h // 16 * 4, dtype=np.uint32)
        assert getattr(orc, fn)(src.ctypes.data, mine.ctypes.data, w, h) == 0
        assert util.digest(mine) == theirs, (name, kind)


@pytest.mark.parametrize("kind", FRAMES)
@pytest.mark.parametrize("w,h", [(8, 4), (4, 8), (36, 20), (1920, 1080), (3840, 2160), (7680, 4320), (3844, -2160)])
def test_fused_uyvy_dxt1_equals_reference_pipeline(api, orc, kind, w, h):
    """config 2/metric: UYVY -> DXT1.  Reference path (src/video_compress/cuda_dxt.cpp:223-257):
    cuda_yuv422_to_yuv444 then cuda_yuv_to_dxt1.  pix_count must be a multiple of 256 for the reference kernel."""
    ah = abs(h)
    if kind == "testcard":
        uyvy = util.testcard_uyvy(w, ah, orc)
    elif kind == "noise":
        uyvy = util.rng_bytes(w * ah * 2, 99 + w)
    else:
        rgb = special_blocks_rgb(w, ah, 5)
        uyvy = util.convert_cpu(orc, "orc_convert", 12, 2, rgb, w, ah)
    src = dev(uyvy)
    mine = api.uyvy_to_dxt(src, w, h, dxt_type=1)
    torch.cuda.synchronize()

    def pipeline():
        if (w * ah) % 256 == 0:
            yuv444 = torch.empty(w * ah * 3, dtype=torch.uint8, device="cuda")
            assert util.ref_gpu().cuda_yuv422_to_yuv444(ctypes.c_void_p(src.data_ptr()), ctypes.c_void_p(yuv444.data_ptr()), w * ah, None) == 0
        else:  # reference expander would run out of bounds: expand on the CPU oracle instead
            e = np.zeros(w * ah * 3, dtype=np.uint8)
            orc.orc_yuv422_to_yuv444(uyvy.ctypes.data, e.ctypes.data, w * ah)
            yuv444 = dev(e)
        return {"yuv444": util.digest(yuv444), "dxt1": util.digest(ref_dxt("cuda_yuv_to_dxt1", yuv444, w, h))}
    theirs = util.reference("dxt_gpu", f"fused_dxt1/{kind}/{w}x{h}", pipeline)
    assert util.digest(mine) == theirs["dxt1"]
    # and the ABI-compat two-step path of the product gives the same bytes
    mine444 = api.yuv422_to_yuv444(src, w * ah)
    assert util.digest(mine444) == theirs["yuv444"]
    assert util.digest(api.compat_to_dxt("cuda_yuv_to_dxt1", mine444, w, h)) == theirs["dxt1"]


def test_fused_uyvy_pitch_and_unaligned_fallbacks(api, orc):
    w, h = 36, 16  # wb = 9 (odd) -> one-block-per-thread kernel
    uyvy = util.rng_bytes(w * h * 2, 3)
    e = np.zeros(w * h * 3, dtype=np.uint8)
    orc.orc_yuv422_to_yuv444(uyvy.ctypes.data, e.ctypes.data, w * h)
    theirs = util.reference("dxt_gpu", f"fallbacks/{w}x{h}", lambda: util.digest(ref_dxt("cuda_yuv_to_dxt1", dev(e), w, h)))
    assert util.digest(api.uyvy_to_dxt(dev(uyvy), w, h)) == theirs
    # padded rows
    pitch = w * 2 + 24
    padded = np.zeros(pitch * h, dtype=np.uint8)
    padded.reshape(h, pitch)[:, :w * 2] = uyvy.reshape(h, w * 2)
    assert util.digest(api.uyvy_to_dxt(dev(padded), w, h, pitch=pitch)) == theirs


def test_argument_checks_match_reference(api):
    """cuda_dxt.cu:745-747: -1 for sizes not divisible by 4 or misaligned pointers"""
    from ultragrid_b200 import _lib
    L = _lib.load()
    buf = torch.zeros(4096, dtype=torch.uint8, device="cuda")
    out = torch.zeros(4096, dtype=torch.uint8, device="cuda")
    p, o = buf.data_ptr(), out.data_ptr()
    assert L.cuda_rgb_to_dxt1(p, o, 6, 4, None) == -1
    assert L.cuda_rgb_to_dxt1(p, o, 8, 6, None) == -1
    assert L.cuda_rgb_to_dxt1(p + 4, o, 8, 8, None) == -1
    assert L.cuda_rgb_to_dxt1(p, o + 4, 8, 8, None) == -1
    assert L.cuda_rgb_to_dxt1(p, o, 8, 8, None) == 0
    assert L.ugb200_uyvy_to_dxt1_async(p, o, 8, 8, 8, None) == -1  # pitch < 2*w


def test_cpu_oracle_vs_reference_kernel(orc):
    """pins oracle/dxt_oracle.c: palettes identical, index words differ only where MUFU.RCP != 1/x"""
    w, h = 1024, 512
    for name, fn in (("cuda_rgb_to_dxt1", "orc_rgb_to_dxt1"), ("cuda_yuv_to_dxt1", "orc_yuv_to_dxt1")):
        src = util.rng_bytes(w * h * 3, 77)
        mine = np.zeros(w * h // 16 * 2, dtype=np.uint32)
        assert getattr(orc, fn)(src.ctypes.data, mine.ctypes.data, w, h) == 0
        mine = mine.reshape(-1, 2)

        def kernel():  # the reference's palettes and index words, the latter as the blocks where they differ from this oracle's
            theirs = ref_dxt(name, dev(src), w, h).cpu().numpy().view(np.uint32).reshape(-1, 2)
            diff = np.flatnonzero(mine[:, 1] != theirs[:, 1])
            return {"palettes": util.digest(theirs[:, 0]), "indices": util.digest(theirs[:, 1]), "index_diff": [[int(i), int(theirs[i, 1])] for i in diff]}
        ref = util.reference("dxt_gpu", f"cpu_dxt1/{name}", kernel)
        assert util.digest(mine[:, 0]) == ref["palettes"]
        theirs = mine[:, 1].copy()
        for i, v in ref["index_diff"]:
            theirs[i] = v
        assert util.digest(theirs) == ref["indices"], "index words of the oracle changed outside the recorded differences"
        bad = np.count_nonzero(mine[:, 1] != theirs)
        assert bad <= len(mine) * 1e-3, bad


def test_dxt1_blocks_decode_close_to_source(api, orc):
    """sanity (not parity): decoded DXT1 of a smooth image is close to the image"""
    w, h = 256, 256
    yy, xx = np.mgrid[0:h, 0:w]
    img = np.stack([xx, yy, (xx + yy) // 2], axis=2).astype(np.uint8).reshape(-1)
    enc = api.compat_to_dxt("cuda_rgb_to_dxt1", dev(img), w, h).cpu().numpy()
    dec = np.zeros(w * h * 3, dtype=np.uint8)
    orc.orc_dxt1_decode(enc.ctypes.data, dec.ctypes.data, w, h)
    mse = np.mean((dec.astype(np.float64) - img) ** 2)
    assert 10 * np.log10(255 ** 2 / mse) > 35
