"""JPEG wire contract (SURVEY.md section 8f rank 2): the encoder's stream as an UNMODIFIED UltraGrid receiver/sender sees it.
The reference's own parser src/utils/jpeg_reader.c (compiled into oracle/_ref) must accept the UYVY stream and classify it as RFC 2435
compatible (type 0 = 4:2:2, +64 = restart markers, dynamic quantisation tables), with the Annex K Huffman tables it requires."""
import ctypes

import numpy as np
import pytest

import util
from test_jpeg import RGB, UYVY, natural_rgb, orc_encode


def read_stream(s):
    """what the reference's src/utils/jpeg_reader.c reads from the stream: jpeg_reader_read_image_info's return, its 16 info ints and the
    quantisation tables, and jpeg_get_rtp_hdr_data's return and its 6 ints"""
    ref = util.ref_cpu()
    out, qt, hf = (ctypes.c_int * 16)(), np.zeros(128, np.uint8), np.zeros(1088, np.uint8)
    rc = ref.ref_jpeg_read_info(s.ctypes.data, len(s), out, qt.ctypes.data, hf.ctypes.data)
    rtp = (ctypes.c_int * 6)()
    rtp_rc = ref.ref_jpeg_get_rtp_hdr_data(s.ctypes.data, len(s), rtp)
    return {"rc": rc, "info": list(out), "qt": qt.tolist(), "rtp_rc": rtp_rc, "rtp": list(rtp)}


def rebuild(rtp, qt, scan):
    """what the reference's src/utils/jpeg_writer.c writes around an RFC 2435 payload (create_jpeg_frame, src/rtp/rtpdec_jpeg.c:150-200): headers made
    from the payload's type, size, restart interval and tables, the scan, EOI.  Recorded as those headers and that trailer for these inputs."""
    def theirs():
        ref = util.ref_cpu()
        out = np.zeros(len(scan) + 2048, np.uint8)
        q = np.array(qt, np.uint8)
        ref.ref_jpeg_writer_rebuild.restype = ctypes.c_long
        ref.ref_jpeg_writer_rebuild.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_long, ctypes.c_void_p]
        n = ref.ref_jpeg_writer_rebuild(rtp[2], rtp[0], rtp[1], rtp[4], q.ctypes.data, scan.ctypes.data, len(scan), out.ctypes.data)
        assert 0 < n <= len(out)
        head = n - len(scan) - 2
        assert np.array_equal(out[head:head + len(scan)], scan)
        return {"rtp": list(rtp), "qt": list(qt), "head": out[:head].tobytes().hex(), "tail": out[n - 2:n].tobytes().hex()}
    want = util.reference("jpeg_wire", f"rebuild/{rtp[0]}x{rtp[1]}/{rtp[2]}/{rtp[4]}", theirs)
    assert (list(rtp), list(qt)) == (want["rtp"], want["qt"]), "the writer was recorded for another payload"
    return np.concatenate([np.frombuffer(bytes.fromhex(want["head"]), np.uint8), scan, np.frombuffer(bytes.fromhex(want["tail"]), np.uint8)])


@pytest.mark.parametrize("w,h,q,ri", [(200, 120, 90, 0), (1920, 1080, 75, 8), (98, 50, 50, 1)])
def test_reference_reader_accepts_uyvy_stream(orc, w, h, q, ri):
    src = util.convert_cpu(orc, "orc_convert", RGB, UYVY, natural_rgb(w, h, 5).reshape(-1), w, h)
    s = np.frombuffer(orc_encode(orc, src, w, h, UYVY, q, ri), np.uint8).copy()
    r = util.reference("jpeg_wire", f"read/{w}x{h}/q{q}/ri{ri}/stream", lambda: {"stream": util.digest(s), **read_stream(s)})
    assert r["stream"] == util.digest(s), "the reader was recorded for another stream"
    out, qt = r["info"], r["qt"]
    assert r["rc"] == 0
    width, height, ncomp, color_spec, interleaved, dri = out[:6]
    assert (width, height, ncomp, interleaved, dri) == (w, h, 3, 1, ri or 4)
    assert color_spec == 1  # JPEG_COLOR_SPEC_YCBCR_JPEG: JFIF, no transform marker (jpeg_reader.h:52-60)
    assert out[6:15] == [2, 1, 1, 1, 1, 1, 0, 1, 1]  # sampling h, v; quantisation-table map
    assert s[out[15] - 14:out[15] - 12].tolist() == [0xFF, 0xDA]  # entropy-coded data starts right behind the 14-byte SOS
    # the quantisation tables the reader extracted are Annex K scaled by the IJG rule (zig-zag order in the stream)
    lum = (ctypes.c_uint8 * 64)()
    orc.orc_jpeg_scaled_qtable.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
    orc.orc_jpeg_scaled_qtable(0, q, lum)
    zz = [0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22,
          15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63]
    assert qt[:64] == [lum[n] for n in zz]
    # RFC 2435: accepted, type 0 (4:2:2) + 64 (restart markers), Q = 255 (tables in-band)
    assert r["rtp_rc"] == 1
    assert r["rtp"][:5] == [w, h, 64, 255, ri or 4]


def test_reference_reader_and_adobe_rgb(orc):
    """The RGB stream carries a standard Adobe APP14 (length 14, 'Adobe', version 100, flags, transform 0) that libjpeg honours
    (tests/test_jpeg.py).  The reference's reader compares SIX bytes with "Adobe" (src/utils/jpeg_reader.c:822-832), so it reads the
    transform one byte late and rejects every standard APP14; RGB is not RFC 2435 material anyway (:1078-1090)."""
    w, h = 64, 32
    s = np.frombuffer(orc_encode(orc, natural_rgb(w, h, 5).reshape(-1).copy(), w, h, RGB, 90), np.uint8).copy()
    r = util.reference("jpeg_wire", "read/adobe_rgb", lambda: {"stream": util.digest(s), **read_stream(s)})
    assert r["stream"] == util.digest(s), "the reader was recorded for another stream"
    assert r["rc"] == -1


@pytest.mark.parametrize("w,h,q,ri", [(200, 120, 90, 0), (1920, 1080, 75, 8), (96, 48, 50, 2)])
def test_rtp_round_trip_through_reference_reader_and_writer(orc, w, h, q, ri):
    """Sender side (jpeg_get_rtp_hdr_data, src/utils/jpeg_reader.c:1092-1160) strips our stream to the RFC 2435 payload - type, Q = 255 with both
    quantisation tables in-band, restart interval, scan data; receiver side (create_jpeg_frame, src/rtp/rtpdec_jpeg.c:150-200) rebuilds a JPEG around
    that payload with the reference's own src/utils/jpeg_writer.c:215-382.  The rebuilt stream must decode to exactly the pixels of the original:
    the encoder's tables and scan layout are what an unmodified UltraGrid receiver assumes (Annex K Huffman tables, component 0 -> table 0, 2x1 luma)."""
    from test_jpeg import decode_ycc
    src = util.convert_cpu(orc, "orc_convert", RGB, UYVY, natural_rgb(w, h, 15).reshape(-1), w, h)
    s = np.frombuffer(orc_encode(orc, src, w, h, UYVY, q, ri), np.uint8).copy()
    r = util.reference("jpeg_wire", f"read/{w}x{h}/q{q}/ri{ri}/round_trip", lambda: {"stream": util.digest(s), **read_stream(s)})
    assert r["stream"] == util.digest(s), "the reader was recorded for another stream"
    assert r["rtp_rc"] == 1 and r["rc"] == 0
    rw, rh, rtype, rq, rri, off = r["rtp"]
    assert rw % 8 == 0 and rh % 8 == 0 and rw // 8 < 256 and rh // 8 < 256  # what the 8-bit size fields of the RTP header can carry
    scan = s[off:len(s) - 2]  # the payload: entropy-coded data without the EOI
    assert s[-2:].tolist() == [0xFF, 0xD9]
    rebuilt = rebuild(r["rtp"], r["qt"], scan)
    a, b = decode_ycc(s.tobytes(), w, h), decode_ycc(rebuilt.tobytes(), w, h)
    assert np.array_equal(a, b)


@pytest.mark.gpu
def test_gpu_decoder_reads_the_stream_rebuilt_by_the_reference_writer(orc):
    """the same round trip with the CUDA encoder at the sender and the CUDA decoder at the receiver"""
    from ultragrid_b200 import api
    w, h = 1920, 1080
    src = util.convert_cpu(orc, "orc_convert", RGB, UYVY, natural_rgb(w, h, 16).reshape(-1), w, h)
    enc = api.JpegEncoder()
    s = np.frombuffer(enc.encode(src, w, h, UYVY, quality=85), np.uint8).copy()
    enc.close()
    r = util.reference("jpeg_wire", f"read/{w}x{h}/q85/gpu", lambda: {"stream": util.digest(s), **read_stream(s)})
    assert r["stream"] == util.digest(s), "the reader was recorded for another stream"
    assert r["rtp_rc"] == 1 and r["rc"] == 0
    rebuilt = rebuild(r["rtp"], r["qt"], s[r["rtp"][5]:len(s) - 2])
    dec = api.JpegDecoder()
    a = dec.decode(s.tobytes(), UYVY)
    b = dec.decode(rebuilt.tobytes(), UYVY)
    dec.close()
    assert np.array_equal(a, b)
