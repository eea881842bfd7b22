"""Test helpers: deterministic frame generators and ctypes access to the checkers under oracle/.

oracle/ is test infrastructure: it is loaded here (tests), by __graft_entry__.smoke() and by bench.py's
cpu_baseline / --impl reference legs only.
"""
import atexit
import ctypes
import hashlib
import json
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")

_vp, _i, _l, _u = ctypes.c_void_p, ctypes.c_int, ctypes.c_long, ctypes.c_uint


# ---- deterministic inputs -------------------------------------------------------------------------
def lcg_bytes(n, seed=12345):
    """LCG of SURVEY.md section 6: s = s*1664525 + 1013904223 (mod 2^32), byte = s >> 24."""
    a, c = 1664525, 1013904223
    blk = 1 << 16
    ak = np.empty(blk, dtype=np.uint64)
    ck = np.empty(blk, dtype=np.uint64)
    A, C = 1, 0
    for i in range(blk):
        A = (A * a) & 0xFFFFFFFF
        C = (C * a + c) & 0xFFFFFFFF
        ak[i], ck[i] = A, C
    out = np.empty(n, dtype=np.uint8)
    s, pos = seed, 0
    while pos < n:
        m = min(blk, n - pos)
        v = (ak[:m] * np.uint64(s) + ck[:m]) & np.uint64(0xFFFFFFFF)
        out[pos:pos + m] = (v >> np.uint64(24)).astype(np.uint8)
        s, pos = int(v[m - 1]), pos + m
    return out


def rng_bytes(n, seed):
    return np.random.default_rng(seed).integers(0, 256, size=n, dtype=np.uint8)


def v210_noise(width, height, seed):
    """random v210 frame, 30 valid bits per word (as test/ff_codec_conversions_test.cpp:355)"""
    ls = (width + 47) // 48 * 128
    w = np.random.default_rng(seed).integers(0, 1 << 30, size=ls // 4 * height, dtype=np.uint32)
    return w.view(np.uint8).copy()


RECT_COLORS = [0xff0000ff, 0xff00ff00, 0xffff0000, 0xff00ffff, 0xffffff00, 0xffff00ff]  # testcard_common.c:51-58


def testcard_rgba(width, height):
    """`-t testcard:pattern=bars` RGBA image (src/utils/video_pattern_generator.cpp:235-281)."""
    img = np.zeros((height, width), dtype=np.uint32)

    def fill(x, y, w, h, color):  # testcard_fillRect, testcard_common.c:60-71
        img[max(y, 0):min(y + h, height), max(x, 0):min(x + w, width)] = color

    col_num, ncol = 0, 6
    rs = (width + ncol - 1) // ncol
    for j in range(0, height, rs):
        grey = 0xFF010101
        if j == rs * 2:
            fill(0, j, width, rs // 4, 0xFFFFFFFF)
            fill(0, j + rs * 3 // 4, width, rs - rs * 3 // 4, 0xFF000000)
        for i in range(0, width, rs):
            if j != rs * 2:
                fill(i, j, rs, min(rs, height - j), RECT_COLORS[col_num])
                col_num = (col_num + 1) % ncol
            else:
                fill(i, j + rs // 4, rs, rs // 2, grey)
                grey = (grey + 0x00010101 * (255 // ncol)) & 0xFFFFFFFF
    return img.view(np.uint8).reshape(height, width, 4).copy()


def testcard_rgb(width, height):
    """RG48 expansion keeps the 8-bit value in the high byte (video_pattern_generator.cpp:180-196) and
    vc_copylineRG48toRGB takes the high byte back, so the RGB testcard is the RGBA one minus alpha."""
    return np.ascontiguousarray(testcard_rgba(width, height)[:, :, :3]).reshape(-1)


def testcard_uyvy(width, height, orc):
    """UYVY testcard as testcard_convert_buffer makes it: vc_copylineRG48toUYVY on the high bytes ==
    vc_copylineRGBtoUYVY on the 8-bit RGB (same vc_copylineToUYVY body, pixfmt_conv.c:1008-1053)."""
    rgb = testcard_rgb(width, height)
    out = np.zeros(width * 2 * height, dtype=np.uint8)
    rc = orc.orc_convert(12, 2, out.ctypes.data, width * 2, rgb.ctypes.data, width * 3, width * 2, height, 0, 8, 16)
    assert rc == 0
    return out


# ---- checkers ---------------------------------------------------------------------------------------
def _build_oracle():
    subprocess.run(["make", "-s", "-C", ORACLE_DIR, "libugoracle.so"], check=True, capture_output=True)


_ORC = None


def oracle():
    """my CPU restatement, oracle/libugoracle.so (built on demand; needs only gcc)."""
    global _ORC
    if _ORC is not None:
        return _ORC
    path = os.path.join(ORACLE_DIR, "libugoracle.so")
    srcs = [os.path.join(ORACLE_DIR, f) for f in os.listdir(ORACLE_DIR) if f.endswith(".c") and f != "ref_shim.c"]
    if not os.path.exists(path) or any(os.path.getmtime(s) > os.path.getmtime(path) for s in srcs):
        _build_oracle()
    L = ctypes.CDLL(path)
    L.orc_convert.argtypes = [_i, _i, _vp, _l, _vp, _l, _i, _i, _i, _i, _i]
    L.orc_has_decoder.argtypes = [_i, _i]
    L.orc_vc_get_linesize.argtypes = [_u, _i]
    L.orc_vc_get_size.argtypes = [_u, _i]
    L.orc_get_color_coeffs.argtypes = [_i, _i, _vp]
    L.orc_v210_to_p010le.argtypes = [_i, _i, _vp, _u, _vp, _u, _vp]
    L.orc_v210_to_p010le.restype = None
    for n in ("orc_rgb_to_dxt1", "orc_yuv_to_dxt1", "orc_rgb_to_dxt6", "orc_yuv_to_dxt6"):
        getattr(L, n).argtypes = [_vp, _vp, _i, _i]
    L.orc_uyvy_to_dxt1.argtypes = [_vp, _vp, _i, _i, _l]
    L.orc_uyvy_to_dxt6.argtypes = [_vp, _vp, _i, _i, _l]
    L.orc_yuv422_to_yuv444.argtypes = [_vp, _vp, _i]
    L.orc_yuv422_to_yuv444.restype = None
    L.orc_dxt1_decode.argtypes = [_vp, _vp, _i, _i]
    L.orc_dxt1_decode.restype = None
    _ORC = L
    return L


def ref_cpu():
    """unmodified reference CPU objects, oracle/_ref/libugref.so, or None when not built."""
    path = os.path.join(ORACLE_DIR, "_ref", "libugref.so")
    if not os.path.exists(path):
        return None
    L = ctypes.CDLL(path)
    L.ref_convert.argtypes = [_i, _i, _vp, _l, _vp, _l, _i, _i, _i, _i, _i]
    L.ref_convert_parallel.argtypes = [_i, _i, _vp, _i, _vp, _i, _i, _i]
    L.ref_has_decoder.argtypes = [_i, _i]
    L.ref_vc_get_linesize.argtypes = [_u, _i]
    L.ref_vc_get_size.argtypes = [_u, _i]
    L.ref_get_color_coeffs.argtypes = [_i, _i, _vp]
    L.ref_get_color_coeffs.restype = None
    L.ref_v210_to_p010le.argtypes = [_i, _i, _vp, _u, _vp, _u, _vp]
    L.ref_v210_to_p010le.restype = None
    L.ref_v210_to_p010le_parallel.argtypes = [_i, _i, _vp, _u, _vp, _u, _vp, _i]
    L.ref_v210_to_p010le_parallel.restype = None
    return L


def ref_gpu():
    """unmodified reference cuda_dxt.cu built for sm_100a (oracle/_ref/libcuda_dxt_ref.so), or None."""
    path = os.path.join(ORACLE_DIR, "_ref", "libcuda_dxt_ref.so")
    if not os.path.exists(path):
        return None
    L = ctypes.CDLL(path)  # RTLD_LOCAL: its cuda_*_to_dxt* do not clash with the product's
    for n in ("cuda_rgb_to_dxt1", "cuda_yuv_to_dxt1", "cuda_rgb_to_dxt6", "cuda_yuv_to_dxt6"):
        getattr(L, n).argtypes = [_vp, _vp, _i, _i, _vp]
    L.cuda_yuv422_to_yuv444.argtypes = [_vp, _vp, _i, _vp]
    return L


# ---- recorded results of the reference ----------------------------------------------------------------
# The reference builds under oracle/_ref/ need the reference source tree, which a checkout of this project does not have.  What they
# returned for the tests' inputs is stored in tests/golden/reference_<group>.json, so the comparisons run everywhere.  To record them again,
# build oracle/_ref/ and run the tests with UGB200_RECORD_REFERENCE=<dir>: compute() then calls the reference and the results are written
# to <dir>/reference_<group>.json.
RECORD_DIR = os.environ.get("UGB200_RECORD_REFERENCE")
_golden, _recorded = {}, {}


def digest(*arrays):
    """128-bit BLAKE2b of the bytes of the arrays (numpy or torch), in order: compares large outputs exactly without storing them"""
    h = hashlib.blake2b(digest_size=16)
    for a in arrays:
        if hasattr(a, "cpu"):
            a = a.cpu().numpy()
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def reference(group, key, compute):
    """what the reference returned for one test input: compute() (JSON-able: ints, lists, dicts, digests) when recording, else the stored value"""
    if RECORD_DIR:
        value = json.loads(json.dumps(compute()))
        _recorded.setdefault(group, {})[key] = value
        return value
    if group not in _golden:
        with open(os.path.join(GOLDEN_DIR, f"reference_{group}.json")) as f:
            _golden[group] = json.load(f)
    assert key in _golden[group], f"no recorded reference result {group}:{key} (record it with UGB200_RECORD_REFERENCE)"
    return _golden[group][key]


def ref_color_coeffs(cs, depth):
    """get_color_coeffs(cs, depth) of the unmodified src/color_space.c: the 14 ints it fills"""
    def theirs():
        out = (_i * 14)()
        lib = ref_cpu()
        lib.ref_get_color_coeffs(cs, depth, out)
        return list(out)
    return reference("color_space", f"{cs}/{depth}", theirs)


@atexit.register
def _write_recorded():
    for group, table in _recorded.items():
        path = os.path.join(RECORD_DIR, f"reference_{group}.json")
        if os.path.exists(path):
            with open(path) as f:
                table = {**json.load(f), **table}
        with open(path, "w") as f:  # one entry per line keeps diffs of the fixtures readable
            f.write("{\n" + ",\n".join(f"{json.dumps(k)}: {json.dumps(table[k])}" for k in sorted(table)) + "\n}\n")


def convert_cpu(lib, fn, in_c, out_c, src, width, height, dst_len=None, src_pitch=None, dst_pitch=None, shifts=(0, 8, 16),
                linesize=None):
    """run a whole-buffer conversion through the oracle (fn='orc_convert') or the reference (fn='ref_convert')"""
    ls = linesize or oracle().orc_vc_get_linesize
    src_pitch = ls(width, in_c) if src_pitch is None else src_pitch
    dst_pitch = ls(width, out_c) if dst_pitch is None else dst_pitch
    dst_len = ls(width, out_c) if dst_len is None else dst_len
    srcp = np.concatenate([src, np.zeros(4096, dtype=np.uint8)])  # zero slack (>= MAX_PADDING, video_codec.h:61): over-reads see zeros, like the GPU path
    dst = np.zeros(dst_pitch * height + 64, dtype=np.uint8)
    rc = getattr(lib, fn)(in_c, out_c, dst.ctypes.data, dst_pitch, srcp.ctypes.data, src_pitch, dst_len, height, *shifts)
    assert rc == 0, rc
    return dst[:dst_pitch * height]
