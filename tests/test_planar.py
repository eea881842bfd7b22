"""Packed<->planar whole-buffer converters (SURVEY.md section 8 rows A10/A11): src/to_planar.c and src/from_planar.c of the reference.
  * CPU: the restatement (oracle/planar_oracle.c) against the unmodified reference objects (oracle/_ref/libugref.so; their outputs recorded in tests/golden);
  * GPU: ugb200_<name> through the C ABI against the restatement, byte for byte, including the bytes that must stay untouched."""
import numpy as np
import pytest

import planar_cases as pc
import util

SIZES = [(16, 2), (17, 3), (24, 1), (48, 4), (50, 5), (130, 3), (256, 6)]


def _sizes_for(name, vs_ref):
    out = []
    for w, h in SIZES:
        if name == "yuv420_to_i420" and (w % 2 or h % 2):
            continue  # asserted by the reference (from_planar.c:371-372)
        if vs_ref and name.endswith("_to_r12l") and w % 8:
            continue  # partial last group = uninitialised stack in the reference (from_planar.c:78-86)
        out.append((w, h))
    return out


@pytest.fixture(scope="module")
def orc():
    return util.oracle()


@pytest.mark.parametrize("name,depth", pc.all_cases())
def test_oracle_vs_reference(orc, name, depth):
    sizes = _sizes_for(name, True)
    cases = [[pc.Case(name, w, h, seed=10 * i + mode, mode=mode, depth=depth, valid_bits=valid, shifts=((0, 8, 16), (16, 8, 0), (8, 16, 24))[mode])
              for mode in (0, 1, 2) for valid in (True, False)] for i, (w, h) in enumerate(sizes)]

    def run(lib, prefix, size_cases):  # every output plane of every case of one size
        return util.digest(*[o for c in size_cases for o in c.run_cpu(lib, prefix)])
    want = util.reference("planar", f"{name}/{depth}", lambda: [run(util.ref_cpu(), "", cs) for cs in cases])
    for (w, h), cs, d in zip(sizes, cases, want, strict=True):
        assert run(orc, "orc_", cs) == d, (name, depth, w, h)


@pytest.mark.gpu
@pytest.mark.parametrize("name,depth", pc.all_cases())
def test_gpu_vs_oracle(orc, name, depth):
    import torch
    from ultragrid_b200 import _lib
    lib = _lib.load()
    for i, (w, h) in enumerate(_sizes_for(name, False) + [(1920, 1080), (1918, 1079)]):
        if name == "yuv420_to_i420" and (w % 2 or h % 2):
            continue
        for mode, offset in ((0, 0), (1, 0), (2, 0), (0, 2)):
            if w > 1000 and mode == 1:
                continue
            c = pc.Case(name, w, h, seed=100 + 10 * i + mode, mode=mode, depth=depth, valid_bits=(mode != 1), shifts=((0, 8, 16), (16, 8, 0), (8, 16, 24))[mode])
            a, b = c.run_cpu(orc, "orc_"), c.run_gpu(lib, torch, offset)
            for k, (x, y) in enumerate(zip(a, b)):
                assert np.array_equal(x, y), (name, depth, w, h, mode, offset, k, np.flatnonzero(x != y)[:8])
