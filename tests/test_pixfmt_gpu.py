"""GPU parity of the whole-buffer line converters and the planar converter against the pinned CPU oracle
(byte-exact), golden fixtures from the reference, and full-size known answers."""
import os

import numpy as np
import pytest

import util
from test_oracle_pinning import PAIRS, RGB, UYVY, V210

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def api():
    from ultragrid_b200 import api as a
    return a


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.mark.parametrize("inc,outc", PAIRS)
def test_line_converters_vs_oracle(api, orc, inc, outc):
    assert api.pixfmt_supported(inc, outc)
    for i, (w, h) in enumerate([(1, 2), (2, 1), (6, 3), (16, 1), (17, 5), (47, 3), (48, 2), (50, 4), (127, 9), (130, 2), (256, 3),
                                (1920, 16), (1922, 3)]):
        src = util.rng_bytes(orc.orc_vc_get_linesize(w, inc) * h, 2000 + i)
        for shifts in ((0, 8, 16), (16, 8, 0), (8, 16, 24)):
            want = util.convert_cpu(orc, "orc_convert", inc, outc, src, w, h, shifts=shifts)
            got = api.pixfmt_convert(inc, outc, dev(src), w, h, shifts=shifts).cpu().numpy()
            assert np.array_equal(got, want), (w, h, shifts)
        for dl in {orc.orc_vc_get_size(w, outc), max(orc.orc_vc_get_size(w, outc) - 4, 0) // 4 * 4}:
            want = util.convert_cpu(orc, "orc_convert", inc, outc, src, w, h, dst_len=dl)
            got = api.pixfmt_convert(inc, outc, dev(src), w, h, dst_len=dl).cpu().numpy()
            assert np.array_equal(got, want), (w, h, dl)


@pytest.mark.parametrize("inc,outc", PAIRS)
def test_staged_and_direct_launch_forms_agree(api, orc, inc, outc):
    """every converter through all four launch forms (line_conv_kernel / line_conv_staged_kernel<in, out>) on 16-byte aligned pitches: identical and == oracle"""
    try:
        for i, (w, h) in enumerate([(64, 2), (192, 3), (1920, 5), (2048 + 64, 2), (7680, 2)]):
            si, so = orc.orc_vc_get_linesize(w, inc), orc.orc_vc_get_linesize(w, outc)
            sp, dp = (si + 15) // 16 * 16 + 32, (so + 15) // 16 * 16 + 16
            src = util.rng_bytes(sp * h, 2100 + i)
            want = util.convert_cpu(orc, "orc_convert", inc, outc, src, w, h, src_pitch=sp, dst_pitch=dp)
            got = []
            for mode in (0, 1, 2, 3):  # direct, input + output staged, output only, input only
                api.pixfmt_staged_mode(mode)
                got.append(api.pixfmt_convert(inc, outc, dev(src), w, h, src_pitch=sp, dst_pitch=dp).cpu().numpy())
            assert all(np.array_equal(g, want) for g in got), (w, h, [np.array_equal(g, want) for g in got])
            for dl in (so, max(so - 20, 0) // 4 * 4):  # a dst_len that ends inside a 16-byte unit
                want = util.convert_cpu(orc, "orc_convert", inc, outc, src, w, h, src_pitch=sp, dst_pitch=dp, dst_len=dl)
                for mode in (1, 2, 3):
                    api.pixfmt_staged_mode(mode)
                    g1 = api.pixfmt_convert(inc, outc, dev(src), w, h, src_pitch=sp, dst_pitch=dp, dst_len=dl).cpu().numpy()
                    assert np.array_equal(g1, want), (w, h, dl, mode)
    finally:
        api.pixfmt_staged_mode(-1)


def test_unaligned_pitches_take_the_guarded_path(api, orc):
    w, h = 100, 5
    for inc, outc in ((UYVY, RGB), (RGB, UYVY), (V210, UYVY)):
        sp, dp = orc.orc_vc_get_linesize(w, inc) + 4, orc.orc_vc_get_linesize(w, outc) + 12
        src = util.rng_bytes(sp * h, 31)
        want = util.convert_cpu(orc, "orc_convert", inc, outc, src, w, h, src_pitch=sp, dst_pitch=dp)
        got = api.pixfmt_convert(inc, outc, dev(src), w, h, src_pitch=sp, dst_pitch=dp).cpu().numpy()
        assert np.array_equal(got, want)


def test_golden_vectors_on_gpu(api):
    g = np.load(os.path.join(util.ROOT, "tests", "golden", "pixfmt_golden.npz"))
    for k in [k[:-4] for k in g.files if k.endswith("_src") and k.startswith("c")]:
        inc, outc, w, h = [int(v) for v in g[k + "_meta"]]
        got = api.pixfmt_convert(inc, outc, dev(g[k + "_src"]), w, h).cpu().numpy()
        assert np.array_equal(got, g[k + "_dst"]), k
    w, h, ls = [int(v) for v in g["p010_meta"]]
    y, c = api.v210_to_p010le(dev(g["p010_src"]), w, h, ls_y=ls, ls_c=ls)
    assert np.array_equal(y.cpu().numpy(), g["p010_y"]) and np.array_equal(c.cpu().numpy(), g["p010_c"])


@pytest.mark.parametrize("inc,outc,w,h,chk", [(UYVY, RGB, 1920, 1080, 798567039), (UYVY, RGB, 7680, 4320, 12776800531),
                                             (RGB, UYVY, 7680, 4320, 8377299523), (V210, UYVY, 7680, 4320, 8460379454)])
def test_known_answers_full_size(api, orc, inc, outc, w, h, chk):
    """config 1 (1080p UYVY->RGB) and the 8K checksums measured on the reference build (SURVEY.md section 6)"""
    src = util.lcg_bytes(orc.orc_vc_get_linesize(w, inc) * h)
    got = api.pixfmt_convert(inc, outc, dev(src), w, h)
    assert int(got.to(torch.int64).sum().item()) == chk


def test_v210_to_p010_vs_oracle(api, orc):
    for i, (w, h) in enumerate([(6, 2), (48, 4), (50, 6), (96, 5), (100, 7), (1920, 4), (7, 8), (13, 9), (7680, 16)]):
        src = util.v210_noise(w, h, 50 + i)
        ls = ((w + 5) // 6 * 6) * 2 + 32
        y0 = np.full(ls * h, 0xAB, dtype=np.uint8)
        c0 = np.full(ls * ((h + 1) // 2), 0xCD, dtype=np.uint8)
        y, c = y0.copy(), c0.copy()
        orc.orc_v210_to_p010le(w, h, y.ctypes.data, ls, c.ctypes.data, ls, src.ctypes.data)
        gy, gc = api.v210_to_p010le(dev(src), w, h, out_y=dev(y0), out_c=dev(c0), ls_y=ls, ls_c=ls)
        assert np.array_equal(gy.cpu().numpy(), y), (w, h)
        assert np.array_equal(gc.cpu().numpy(), c), (w, h)


def test_v210_to_p010_8k_properties(api):
    """config 4 at full size through size-independent properties: luma is an exact <<6 repack and the chroma of a
    frame whose rows are all equal is the identity."""
    w, h = 7680, 4320
    row = util.v210_noise(w, 1, 11)
    src = np.tile(row, h)
    y, c = api.v210_to_p010le(dev(src), w, h)
    words = torch.from_numpy(row.view(np.int32).astype(np.int64)).cuda().reshape(-1, 4)
    luma = torch.stack([(words[:, 0] >> 10) & 0x3ff, words[:, 1] & 0x3ff, (words[:, 1] >> 20) & 0x3ff,
                        (words[:, 2] >> 10) & 0x3ff, words[:, 3] & 0x3ff, (words[:, 3] >> 20) & 0x3ff], dim=1).reshape(-1) << 6
    chroma = torch.stack([words[:, 0] & 0x3ff, (words[:, 0] >> 20) & 0x3ff, (words[:, 1] >> 10) & 0x3ff,
                          words[:, 2] & 0x3ff, (words[:, 2] >> 20) & 0x3ff, (words[:, 3] >> 10) & 0x3ff], dim=1).reshape(-1) << 6
    yv = y.view(torch.int16).to(torch.int64).bitwise_and(0xffff).reshape(h, w)
    cv = c.view(torch.int16).to(torch.int64).bitwise_and(0xffff).reshape(h // 2, w)
    assert torch.equal(yv, luma.expand(h, w))
    assert torch.equal(cv, chroma.expand(h // 2, w))


def test_v210_to_p010_8k_full_frame_vs_reference(api, orc):
    """BASELINE config 4 at its full size with real arithmetic in every chroma sample: a 7680x4320 frame of 30-bit noise (rows all different, so
    the (row0 + row1) / 2 average of to_planar.c:133-138 is exercised everywhere) memcmp-equal to the UNMODIFIED reference function
    (oracle/_ref: ref_v210_to_p010le) and to the restatement"""
    w, h = 7680, 4320
    src = util.v210_noise(w, h, 77)
    gy, gc = api.v210_to_p010le(dev(src), w, h)
    gy, gc = gy.cpu().numpy(), gc.cpu().numpy()

    def run(lib, fn):
        y, c = np.zeros(w * 2 * h, np.uint8), np.zeros(w * h, np.uint8)
        getattr(lib, fn)(w, h, y.ctypes.data, w * 2, c.ctypes.data, w * 2, src.ctypes.data)
        return y, c
    y, c = run(orc, "orc_v210_to_p010le")
    assert np.array_equal(gy, y) and np.array_equal(gc, c)
    theirs = util.reference("pixfmt_gpu", f"v210_to_p010le/{w}x{h}", lambda: [util.digest(a) for a in run(util.ref_cpu(), "ref_v210_to_p010le")])
    assert [util.digest(gy), util.digest(gc)] == theirs
    # the average is not the identity on this frame: more than a third of the chroma words differ from plain row 0
    words = src.view(np.uint32).reshape(h, -1, 4)[0::2]
    cb0 = ((words[:, :, 0] & 0x3ff) << 6).astype(np.uint16)
    assert np.count_nonzero(gc.view(np.uint16).reshape(h // 2, w)[:, 0::6] != cb0[:, : w // 6]) > cb0[:, : w // 6].size // 3
