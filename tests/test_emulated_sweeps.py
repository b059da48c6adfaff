"""Oracle sweeps through the CPU-emulated kernels (sizes up to 256): DynamicTileEncode (R1) on random shapes, modes,
uploads and call paths; the alpha stage on random islands; rejectFactor 0..64; multi-slot batches with fused R1; seeded
sequences of loads and programs on the slots of one context.  Bit for bit against the C oracle; seeds are fixed."""
import os
import subprocess

import numpy as np
import pytest

import sweeps
from parity import check_image, check_results, fused_stages
from yaik_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU = os.path.join(ROOT, "tests", "emu", "_build", "libyaik_b200_emu.so")


@pytest.fixture(scope="module")
def emu_lib():
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "tests", "emu")], check=True)
    return capi.load_library(EMU)


def _host_bytes(a):
    """Device memory of the emulated build is host memory."""
    return a.ctypes.data, a


def _run(lib, planes, stages, fused, packed, **kw):
    c, h, w = planes.shape
    ctx = capi.Context(w, h, planes=4, slots=1, lib=lib)
    try:
        ctx.set_upload_format(packed)
        check_image(ctx, planes, stages, fused=fused, **kw)
    finally:
        ctx.close()


@pytest.mark.parametrize("i", range(30))
def test_r1_sweep(emu_lib, i):
    planes, stages, fused, packed = sweeps.r1_case(i, 256)
    _run(emu_lib, planes, stages, fused, packed)


@pytest.mark.parametrize("i", range(12))
def test_alpha_sweep(emu_lib, i):
    planes, stages, fused, packed = sweeps.alpha_case(i, 256)
    _run(emu_lib, planes, stages, fused, packed)


@pytest.mark.parametrize("fused", [True, False], ids=["fused", "stage_by_stage"])
@pytest.mark.parametrize("reject", sweeps.REJECT_FACTORS)
def test_reject_factor_sweep(emu_lib, reject, fused):
    w, h = ((64, 64), (96, 80), (136, 72))[reject % 3]
    planes = sweeps.reject_content(w, h, reject, 8000 + reject)
    _run(emu_lib, planes, ("grad", "r2", "r1"), fused, reject % 2 == 0, reject=reject)


def test_reject_factor_abi_contract(emu_lib):
    planes = sweeps.reject_content(64, 64, 5, 8100)
    ctx = capi.Context(64, 64, planes=4, slots=1, lib=emu_lib)
    try:
        ctx.set_image(planes)
        for bad in (-1, 65):
            for call in (lambda r: ctx.analyze(capi.STAGE_GRADIENT, reject=r), lambda r: ctx.prepare_quad_smooth(reject=r),
                         lambda r: ctx.gradient_pass(4, 4, reject=r), lambda r: ctx.strip_run(reject=r),
                         lambda r: ctx.strip_phase(0, reject=r)):
                with pytest.raises(capi.YaikError) as e:
                    call(bad)
                assert e.value.code == sweeps.YK_ERR_ARG, bad
        ctx.analyze(capi.STAGE_GRADIENT, reject=5)
        with pytest.raises(capi.YaikError) as e:           # the cascade was prepared with another factor
            ctx.gradient_pass(4, 4, reject=3)
        assert e.value.code == sweeps.YK_ERR_STATE
        check_results(ctx, planes, ("grad",), reject=5)    # the refused call consumed nothing
    finally:
        ctx.close()


@pytest.mark.parametrize("n_slots,r1", [(2, "r1"), (3, "r1_3bit"), (3, "r1")])
def test_batch_with_fused_r1(emu_lib, n_slots, r1):
    """One yk_analyze over n_slots slots with ALPHA | GRADIENT | RANGE1D | RANGEDYN(3): RGB and RGBA images side by side,
    every slot against the oracle."""
    d = sweeps._Draw(8200, n_slots * 2 + (r1 == "r1"))
    side = 64 << d.int(2)
    stages = ("alpha", "grad", "r2", r1)
    imgs = [sweeps.rgba_island_image(d, side, 8300 + 10 * n_slots + k) if k != 1 else sweeps.rgb_content(d, side, side, 8400 + k)
            for k in range(n_slots)]
    ctx = capi.Context(side, side, planes=4, slots=n_slots, lib=emu_lib)
    try:
        for k, im in enumerate(imgs):
            ctx.set_image(im, k)
        ctx.analyze(fused_stages(imgs[0], stages), slot0=0, n_slots=n_slots)
        for k, im in enumerate(imgs):
            check_results(ctx, im, stages, slot=k, r1_fused=True)
    finally:
        ctx.close()


@pytest.mark.parametrize("seq,n_slots", [(0, 2), (1, 3)])
def test_slot_reuse_sequence(emu_lib, seq, n_slots):
    ctx = capi.Context(128, 128, planes=4, slots=n_slots, lib=emu_lib)
    try:
        sweeps.run_sequence(ctx, sweeps.reuse_sequence(seq, n_slots, 10, 128), _host_bytes)
    finally:
        ctx.close()


def test_reuse_sequences_cover_the_transitions():
    """The opening of every sequence holds the transitions the slot flags exist for."""
    for seq, n_slots in ((0, 2), (1, 3)):
        steps = sweeps.reuse_sequence(seq, n_slots, 10, 128)
        seen = set()
        for k, a in enumerate(steps):
            for later in steps[k + 1:]:               # the next step on the same slot
                if later[0] != a[0]:
                    continue
                pa, pb = a[2], later[2]
                if pb.shape[1] * pb.shape[2] < pa.shape[1] * pa.shape[2]:
                    seen.add("small after large")
                if pa.shape[0] == 3 and pb.shape[0] == 4:
                    seen.add("rgba after rgb")
                if pa.shape[0] == 4 and pb.shape[0] == 3 and later[3] == "fused_r1":
                    seen.add("fused r1 on rgb after rgba")
                if a[3] == "fused_r1" and later[3] == "r1_only" and a[4] == later[4]:
                    seen.add("r1 only after fused r1")
                if pa.min() < 0 and later[1] == "packed" and pb.min() >= 0:
                    seen.add("packed after int32 fallback")
                break
        assert seen >= {"small after large", "rgba after rgb", "fused r1 on rgb after rgba", "r1 only after fused r1",
                        "packed after int32 fallback"}, (seq, seen)
