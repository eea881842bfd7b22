"""video_compress module layer: converter selection against the reference (CPU), module behaviour on the GPU."""
import ctypes

import numpy as np
import pytest

import util
from test_jpeg import natural_rgb, orc_encode

RGBA, UYVY, YUYV, V210, RGB, BGR, RG48 = 1, 2, 3, 7, 12, 20, 27


def test_registry_and_option_parsing_fail_cleanly():
    from ultragrid_b200 import compress
    with pytest.raises(RuntimeError):
        compress.Compress("no_such_module")
    with pytest.raises(RuntimeError):
        compress.Compress("cuda_dxt:DXT3")  # usage error like cuda_dxt.cpp:113-117
    with pytest.raises(RuntimeError):
        compress.Compress("GPUJPEG:bogus=1")
    with pytest.raises(RuntimeError):
        compress.Compress("GPUJPEG:lanes=0")
    for bad in ("GPUJPEG:0", "GPUJPEG:101", "GPUJPEG:quality=0", "GPUJPEG:subsampling=411", "GPUJPEG:restart=-1"):
        with pytest.raises(RuntimeError):
            compress.Compress(bad)


@pytest.mark.parametrize("cfg", ["GPUJPEG:90", "GPUJPEG:90:8", "GPUJPEG:quality=80:restart=4", "GPUJPEG:q=75:interleaved", "GPUJPEG:Y709", "GPUJPEG:RGB:subsampling=444",
                                 "GPUJPEG:Y601full:alpha:lanes=2"])
def test_gpujpeg_option_grammar_of_the_reference(cfg):
    """state_video_compress_gpujpeg::parse_fmt (gpujpeg.cpp:371-424): positional quality / restart interval and every keyword parse; whether a colour
    space or subsampling can be honoured is decided against the first frame's format"""
    from ultragrid_b200 import compress
    c = compress.Compress(cfg)
    c.push(None, 0, 0, 0)
    assert c.pop(16) is None
    c.close()


@pytest.mark.parametrize("cfg", ["GPUJPEG", "GPUJPEG:q=90:lanes=1", "GPUJPEG:lanes=4", "cuda_dxt:DXT5", "cuda_dxt_sync"])
def test_module_lifecycle_without_frames(cfg):
    """init / done with no frame in between, and the poison pill through every lane (src/video_compress.h:143-147): host logic only, no GPU work"""
    from ultragrid_b200 import compress
    c = compress.Compress(cfg)
    c.close()
    c = compress.Compress(cfg)
    c.push(None, 0, 0, 0)
    assert c.pop(16) is None
    c.close()


@pytest.mark.parametrize("cands", [(RGB, UYVY), (UYVY, RGB), (UYVY, RGB, RGBA), (RGBA, RGB), (UYVY,), (YUYV, UYVY)])
def test_get_best_decoder_from_matches_reference(cands):
    """where both sides have the converters, the selection (pixfmt_desc ranking 'dsc') must agree with the reference"""
    from ultragrid_b200 import compress
    incs = (RGBA, UYVY, YUYV, V210, RGB, BGR, RG48)

    def selections():  # per input codec: the reference's choice and the candidates it has a converter to
        ref = util.ref_cpu()
        ref.ref_get_best_decoder_from.argtypes = [ctypes.c_int, ctypes.POINTER(ctypes.c_int), ctypes.c_int]
        arr = (ctypes.c_int * len(cands))(*cands)
        return [[ref.ref_get_best_decoder_from(inc, arr, len(cands)), [c for c in cands if ref.ref_has_decoder(inc, c)]] for inc in incs]
    checked = 0
    for inc, (theirs, usable) in zip(incs, util.reference("vcompress", "best_decoder/" + ",".join(map(str, cands)), selections), strict=True):
        if not all(compress.get_best_decoder_from(inc, [c]) == c for c in usable):
            continue  # the reference knows a converter that is not on the device yet: selection may legitimately differ
        assert compress.get_best_decoder_from(inc, cands) == theirs, (inc, cands)
        checked += 1
    assert checked >= 3


# ---- GPU ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("cfg,inc", [("cuda_dxt", UYVY), ("cuda_dxt:DXT1", RGB), ("cuda_dxt:DXT5", UYVY), ("cuda_dxt:DXT5", RGB),
                                     ("cuda_dxt:DXT1", V210), ("cuda_dxt:DXT1", RGBA), ("cuda_dxt:DXT5", YUYV)])
def test_cuda_dxt_module_equals_kernel_path(orc, cfg, inc):
    """host frame in -> pooled host frame out equals the device kernels run by hand (and hence the reference kernels)"""
    import torch
    from ultragrid_b200 import api, compress
    w, h = 1920, 1080
    src = util.rng_bytes(orc.orc_vc_get_linesize(w, inc) * h, 12 + inc) if inc != V210 else util.v210_noise(w, h, 3)
    dxt_type = 6 if cfg.endswith("DXT5") else 1
    d = torch.from_numpy(src).cuda()
    if inc in (UYVY, RGB):
        mid, mid_codec = d, inc
    else:
        mid_codec = compress.get_best_decoder_from(inc, [RGB, UYVY])
        mid = api.pixfmt_convert(inc, mid_codec, d, w, h)
    if mid_codec == UYVY:
        want = api.uyvy_to_dxt(mid, w, h, dxt_type=dxt_type)
    else:
        want = api.compat_to_dxt("cuda_rgb_to_dxt1" if dxt_type == 1 else "cuda_rgb_to_dxt6", mid, w, h)
    want = want.cpu().numpy()
    c = compress.Compress(cfg)
    for rep in range(3):  # three frames through the same state: pool reuse, no reconfiguration
        c.push(src, w, h, inc)
        got, codec, seq = c.pop(w * h)
        assert codec == (11 if dxt_type == 6 else 9) and seq == rep
        assert np.array_equal(got, want)
    c.push(d, w, h, inc)  # device-resident input (mem_location == CUDA_MEM)
    got, _, _ = c.pop(w * h)
    assert np.array_equal(got, want)
    # pipelined use of the asynchronous shape: five frames pushed back to back (3 in flight), popped in order, zero-copy
    frames = [src.copy() for _ in range(5)]
    frames[2][:] = 0
    for f in frames:
        c.push(f, w, h, inc)
    c.push(None, 0, 0, 0)
    for i in range(5):
        view, codec, seq = c.pop_ref()
        assert seq == 4 + i
        assert np.array_equal(view, want) == (i != 2)
    assert c.pop_ref() is None
    c.close()
    # the same module behind the reference's synchronous tile API
    c = compress.Compress(cfg.replace("cuda_dxt", "cuda_dxt_sync"))
    c.push(src, w, h, inc)
    got, _, _ = c.pop(w * h)
    assert np.array_equal(got, want)
    c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("devices,cfg", [([0], "GPUJPEG:q=90:lanes=1"), ([0], "GPUJPEG:q=90"), ([0, 0, 0], "GPUJPEG:q=90:lanes=1"),
                                         ([0, 0], "GPUJPEG:q=90:lanes=2")])
def test_gpujpeg_module_keeps_order_and_matches_oracle(orc, devices, cfg):
    """async frame API with 1 encoder (inline, the reference's single-device shape), with the default 3 lanes on one device, with one
    worker per cuda_devices[] entry (all on GPU 0) and with both: results pop in submission order and carry the oracle's bytes"""
    from ultragrid_b200 import compress
    compress.set_cuda_devices(devices)
    try:
        w, h, n = 640, 360, 7
        frames = [util.convert_cpu(orc, "orc_convert", RGB, UYVY, natural_rgb(w, h, 100 + i).reshape(-1), w, h) for i in range(n)]
        want = [orc_encode(orc, f, w, h, UYVY, 90) for f in frames]
        c = compress.Compress(cfg)
        for f in frames:
            c.push(f, w, h, UYVY)
        c.push(None, 0, 0, 0)
        for i in range(n):
            got, codec, seq = c.pop(w * h * 3)
            assert codec == 13 and seq == i
            assert got.tobytes() == want[i], i
        assert c.pop(w * h * 3) is None
        c.close()
    finally:
        compress.set_cuda_devices([0])


@pytest.mark.gpu
def test_gpujpeg_module_options_against_the_input_format(orc):
    """interleaved RGB through the module == the oracle's single-scan stream; an internal colour space / subsampling that would need a transform
    inside the codec drops the frame with a message (no silently different stream); the native ones pass"""
    from test_jpeg import orc_encode_interleaved_rgb
    from ultragrid_b200 import compress
    w, h = 320, 184
    rgb = natural_rgb(w, h, 4).reshape(-1)
    uyvy = util.convert_cpu(orc, "orc_convert", RGB, UYVY, rgb, w, h)
    c = compress.Compress("GPUJPEG:75:interleaved:RGB:subsampling=444")
    c.push(rgb, w, h, RGB)
    got, _, _ = c.pop(w * h * 3 + 4096)
    assert got.tobytes() == orc_encode_interleaved_rgb(orc, rgb, w, h, 75)
    c.close()
    c = compress.Compress("GPUJPEG:75:Y709:subsampling=422:lanes=1")
    c.push(uyvy, w, h, UYVY)
    got, _, _ = c.pop(w * h * 3 + 4096)
    assert got.tobytes() == orc_encode(orc, uyvy, w, h, UYVY, 75)
    c.close()
    for cfg, frame, codec in (("GPUJPEG:Y601:lanes=1", uyvy, UYVY), ("GPUJPEG:Y709:lanes=1", rgb, RGB), ("GPUJPEG:subsampling=420:lanes=1", uyvy, UYVY)):
        c = compress.Compress(cfg)
        c.push(frame, w, h, codec)
        c.push(None, 0, 0, 0)
        assert c.pop(w * h * 3 + 4096) is None  # the failed frame is skipped (gpujpeg.cpp:194-198), then end of stream
        c.close()


@pytest.mark.gpu
def test_gpujpeg_module_rgb_and_conversion_input(orc):
    from ultragrid_b200 import compress
    w, h = 320, 184
    rgb = natural_rgb(w, h, 4).reshape(-1)
    c = compress.Compress("GPUJPEG:q=75:restart=16")
    c.push(rgb, w, h, RGB)
    got, _, _ = c.pop(w * h * 3)
    assert got.tobytes() == orc_encode(orc, rgb, w, h, RGB, 75, ri=16)
    yuyv = util.rng_bytes(w * h * 2, 8)
    c.push(yuyv, w, h, YUYV)  # converted on the device to UYVY first
    got, _, _ = c.pop(w * h * 3)
    uyvy = util.convert_cpu(orc, "orc_convert", YUYV, UYVY, yuyv, w, h)
    assert got.tobytes() == orc_encode(orc, uyvy, w, h, UYVY, 75, ri=16)
    c.close()


@pytest.mark.parametrize("cfg", ["cuda_dxt", "cuda_dxt_sync"])
def test_cuda_dxt_bad_format_does_not_hang_and_recovers_sequence(cfg):
    """a frame whose size is not divisible by 4 fails configure_with() before any CUDA call (cuda_dxt.cpp:148-151).  The reference returns
    NULL; here push + pop must stay in step: an empty result comes back (pop reports failure) instead of pop blocking for ever.  Host logic only."""
    import threading
    from ultragrid_b200 import compress
    c = compress.Compress(cfg)
    bad = np.zeros(6 * 6 * 2, dtype=np.uint8)
    result = []

    def work():
        for _ in range(2):  # twice: the failed configuration must not be remembered as the current one
            c.push(bad, 6, 6, UYVY)
            try:
                result.append(c.pop(64))
            except RuntimeError as e:
                result.append(str(e))
    t = threading.Thread(target=work, daemon=True)
    t.start()
    t.join(timeout=20)
    assert not t.is_alive(), "pop() blocked after a failed reconfiguration"
    assert len(result) == 2 and all(isinstance(r, str) and "compress_pop failed" in r for r in result), result
    c.push(None, 0, 0, 0)
    assert c.pop(16) is None
    c.close()
