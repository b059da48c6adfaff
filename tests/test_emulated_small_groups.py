"""Emission offsets from group totals on the CPU-emulated kernels (tests/emu), built with groups of 32 nibble words / range
tiles and super-groups of 4 groups.  At the product's sizes (512 and 32) every image up to 256 x 256 lies in one
super-group; here a 256 x 256 image has 32 range groups in 8 super-groups, so the two-level base sum, rows of range tiles
that straddle two groups, and lattice rows whose owners span groups are all exercised.  The emulated yk_k_emit asserts that
each group's own scan total equals the total yk_k_owner counted."""
import os
import subprocess

import pytest

import cases
from parity import check_image
from strips_check import check_against_oracle
from yaik_b200 import capi, strips

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tests", "emu", "_build", "small_groups")
LIB = os.path.join(OUT, "libyaik_b200_emu.so")


@pytest.fixture(scope="module")
def emu_lib():
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "tests", "emu"), "OUT=" + OUT,
                    "CXX=" + os.environ.get("CXX", "g++") + " -DYK_EMIT_THREADS=32 -DYK_SUPER=4"], check=True)
    return capi.load_library(LIB)


CASES = ["synth256_rgb_3bit", "alpha_island256", "patchy_72x40", "patchy128", "mip32_rgba", "noise_hi", "flat64", "r1_signed96"]


@pytest.mark.parametrize("name", CASES)
def test_small_groups_match_oracle(emu_lib, name):
    planes, stages = cases.SMALL_CASES[name]()
    ctx = capi.Context(256, 256, planes=4, slots=1, lib=emu_lib)
    try:
        check_image(ctx, planes, stages, fused=True)
    finally:
        ctx.close()


def test_small_groups_stage_by_stage_calls(emu_lib):
    planes, stages = cases.SMALL_CASES["patchy_72x40"]()
    ctx = capi.Context(128, 64, planes=4, slots=1, lib=emu_lib)
    try:
        check_image(ctx, planes, ("grad", "r2"), fused=False)
    finally:
        ctx.close()


def test_small_groups_strips(emu_lib):
    planes = cases._patchy(128, 192, 41, 4, 3)
    ctxs = [capi.Context(128, 192, planes=3, slots=1, lib=emu_lib) for _ in range(3)]
    try:
        check_against_oracle(strips.LocalTransport(ctxs).run(planes, n_strips=3), planes)
    finally:
        for c in ctxs:
            c.close()
