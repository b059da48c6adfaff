"""The cooperative copies of yk_k_emit on the CPU-emulated kernels (tests/emu), built with groups of 32 nibble words / range
tiles, super-groups of 4 groups and a corner list of 32 entries.  A gradient group then copies its colours in several
rounds as soon as it emits more than 32 corners, and a range group whose tiles all code 4 quadrants copies 3 x 128 chunks,
four rounds of its 32 threads.  The emulated yk_k_emit asserts that each group's own scan total equals the total
yk_k_owner counted."""
import os
import subprocess

import numpy as np
import pytest

import cases
from parity import check_image
from strips_check import check_against_oracle
from yaik_b200 import capi, strips

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tests", "emu", "_build", "emit_expand")
LIB = os.path.join(OUT, "libyaik_b200_emu.so")
THREADS, LIST = 32, 32


@pytest.fixture(scope="module")
def emu_lib():
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "tests", "emu"), "OUT=" + OUT,
                    "CXX=" + os.environ.get("CXX", "g++") + f" -DYK_EMIT_THREADS={THREADS} -DYK_SUPER=4 -DYK_EMIT_LIST={LIST}"],
                   check=True)
    return capi.load_library(LIB)


def _run(lib, planes, stages):
    c, h, w = planes.shape
    ctx = capi.Context(w, h, planes=4, slots=1, lib=lib)
    try:
        check_image(ctx, planes, stages, fused=True)
        return ctx.fetch_all(0)
    finally:
        ctx.close()


@pytest.mark.parametrize("planes", [np.full((3, 256, 256), 77, np.int32), cases._smooth_noisy(256, 256, 41, 1)],
                         ids=["flat256", "ramp256"])
def test_corner_rounds(emu_lib, planes):
    # 256 x 256: the 16x16 pass has 32 nibble words, one group, whose corners need more than one round of the list
    res = _run(emu_lib, planes, ("grad", "r2"))
    assert res["passes"][0]["rgb"].size > 3 * LIST


def test_full_chunk_groups(emu_lib):
    planes = cases._noise(256, 256, 3, 42)
    res = _run(emu_lib, planes, ("grad", "r2"))
    tiles = (256 // 8) ** 2
    for q in res["r2"]:
        assert q["type"].size == 3 * tiles and q["idx"].size == 64 * tiles       # every tile codes all four quadrants


def test_mixed_image(emu_lib):
    planes, stages = cases.SMALL_CASES["synth256_rgba"]()
    ctx = capi.Context(256, 256, planes=4, slots=1, lib=emu_lib)
    try:
        check_image(ctx, planes, stages, fused=True)
    finally:
        ctx.close()


def test_strips(emu_lib):
    planes = cases._smooth_noisy(128, 192, 43, 1)
    ctxs = [capi.Context(128, 192, planes=3, slots=1, lib=emu_lib) for _ in range(3)]
    try:
        check_against_oracle(strips.LocalTransport(ctxs).run(planes, n_strips=3), planes)
    finally:
        for c in ctxs:
            c.close()
