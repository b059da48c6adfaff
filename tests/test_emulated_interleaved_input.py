"""Interleaved 8-bit input (yk_set_image_interleaved / _device and yk_k_unpack8) through the CPU-emulated kernels: every
stage after such a load matches the oracle, and the slot behaves like one loaded by a packed yk_set_image (chroma,
batches with packed slots, strips).  Host memory stands for device memory in the emulated build, so the device variant
reads the caller's buffer itself: row padding, a misaligned base and widths that end inside a 16-pixel group take the
kernel's byte path there, aligned rows its 16-byte path."""
import os
import subprocess
import sys

import numpy as np
import pytest

import cases
from interleaved import Interleaved, loader
from parity import check_image, results_digest
from yaik_b200 import capi
from yaik_b200.synth import make_image, SEED_BASE, _rand

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU = os.path.join(ROOT, "tests", "emu", "_build", "libyaik_b200_emu.so")
ASAN_CXX = os.environ.get("ASAN_CXX", "/usr/bin/g++")
YK_ERR_ARG, YK_ERR_CAPACITY = -2, -3


@pytest.fixture(scope="module")
def emu_lib():
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "tests", "emu")], check=True)
    return capi.load_library(EMU)


def _ctx(lib, w, h, planes=4, slots=1):
    return capi.Context(w, h, planes=planes, slots=slots, lib=lib)


SMALL = ["patchy_72x40", "synth256_rgba", "alpha_island128", "synth256_rgb_3bit", "mip8_rgb", "ramp64_a2"]
# variant: entry point, bytes per pixel (None: one per plane), row padding, base offset from a 16-byte boundary
VARIANTS = {
    "host": ("host", None, 0, 0),
    "device": ("device", None, 0, 0),
    "host_rgba_for_rgb": ("host", 4, 0, 0),
    "device_rgba_for_rgb": ("device", 4, 0, 0),
    "device_padded": ("device", None, 24, 0),
    "host_padded_offset": ("host", None, 5, 9),
    "device_offset": ("device", None, 0, 1),
    "device_padded_offset": ("device", None, 3, 15),
}


@pytest.mark.parametrize("variant", sorted(VARIANTS))
@pytest.mark.parametrize("name", SMALL)
def test_small_cases_match_oracle(emu_lib, name, variant):
    planes, stages = cases.SMALL_CASES[name]()
    how, ch, pad, off = VARIANTS[variant]
    if ch == 4:              # four bytes per pixel, three planes: the alpha bytes are ignored
        planes, stages = planes[:3], tuple(s for s in stages if s != "alpha")
    c, h, w = planes.shape
    ctx = _ctx(emu_lib, w, h)
    try:
        check_image(ctx, planes, stages, fused=True, load=loader(how, ch, pad, off))
        if "r1" in stages or "r1_3bit" in stages or "grad" in stages:
            check_image(ctx, planes, stages, fused=False, load=loader(how, ch, pad, off))
    finally:
        ctx.close()


@pytest.mark.parametrize("ch", [3, 4])
@pytest.mark.parametrize("w", [36, 40, 44, 48])
def test_widths_ending_inside_a_16_pixel_group(emu_lib, w, ch):
    """w = 4, 8, 12 and 0 mod 16, aligned rows (16-byte path for whole groups, byte path for the last one) and misaligned.
    RGBA: the state download and R1 are left out, their alpha box on a non-square image lies outside the alpha stage's domain."""
    h = 24
    planes = make_image(w, h, ch, SEED_BASE + 40 + w) if ch == 4 else cases._patchy(w, h, 60 + w, 4, 3)
    stages = ("alpha", "grad") if ch == 4 else ("grad",)
    if w % 8 == 0:                                   # R2 / R1: multiples of 8
        stages += ("r2",) if ch == 4 else ("r2", "r1")
    ctx = _ctx(emu_lib, w, h)
    try:
        for how, pad, off in (("host", 0, 0), ("device", (16 - w * ch % 16) % 16, 0), ("device", 4, 6)):
            check_image(ctx, planes, stages, state=(ch == 3), load=loader(how, None, pad, off))
    finally:
        ctx.close()


def _random_case(i):
    r = _rand(991, i, np.arange(8, dtype=np.uint64))
    w = 4 * (1 + int(r[0] % np.uint64(48)))          # 4 .. 192
    h = 4 * (1 + int(r[1] % np.uint64(40)))          # 4 .. 160
    kind = int(r[2] % np.uint64(3))
    if kind == 0:
        planes = cases._patchy(w, h, 1100 + i, 4, 1 + int(r[3] % np.uint64(4)))
    elif kind == 1:
        planes = make_image(w, h, 3, SEED_BASE + 900 + i)
    else:
        planes = cases._noise(w, h, 3, 3100 + i, 90, 90 + int(r[3] % np.uint64(12)))
    stages = ("grad", "r2") if w % 8 == 0 and h % 8 == 0 else ("grad",)
    how = "host" if r[4] % np.uint64(2) else "device"
    ch = 3 + int(r[5] % np.uint64(2))
    pad = int(r[6] % np.uint64(3)) * 7
    off = int(r[7] % np.uint64(16))
    return planes, stages, (how, ch, pad, off)


@pytest.mark.parametrize("i", range(12))
def test_random_shapes_match_oracle(emu_lib, i):
    planes, stages, (how, ch, pad, off) = _random_case(i)
    c, h, w = planes.shape
    ctx = _ctx(emu_lib, w, h)
    try:
        check_image(ctx, planes, stages, fused=(i % 3 != 0), load=loader(how, ch, pad, off))
    finally:
        ctx.close()


@pytest.mark.parametrize("k", [0, 1, 2])
def test_chroma_after_interleaved_load_equals_int32_load(emu_lib, k):
    name, pre, cfg, modes = cases.CHROMA_CASES[k]
    planes, _ = cases.SMALL_CASES[name]()
    c, h, w = planes.shape
    st = (capi.STAGE_ALPHA if ("alpha" in pre and c == 4) else 0) | (capi.STAGE_GRADIENT if "grad" in pre else 0)
    out = []
    for how in ("int32", "host", "device"):
        ctx = _ctx(emu_lib, w, h)
        try:
            if how == "int32":
                ctx.set_upload_format(False)
                ctx.set_image(planes)
            else:
                loader(how, None, 4, 3)(ctx, planes, 0)
            if st:
                ctx.analyze(st)
            out.append(ctx.chroma(cfg, modes))
        finally:
            ctx.close()
    for got in out[1:]:
        for key in ("Y", "workCo", "workCg"):
            assert np.array_equal(got[key], out[0][key]), key
        for a, b in zip(got["coded"], out[0]["coded"]):
            assert a["constraint"] == b["constraint"] and a["n_nibbles"] == b["n_nibbles"]
            for key in ("nibbles", "defs", "dst"):
                assert np.array_equal(a[key], b[key]), key


@pytest.mark.parametrize("order", ["interleaved_first", "packed_first"])
def test_batch_of_interleaved_and_packed_slots_equals_single_runs(emu_lib, order):
    imgs = [make_image(128, 128, 4, SEED_BASE + 30), make_image(128, 128, 4, SEED_BASE + 31)]
    st = capi.STAGE_ALPHA | capi.STAGE_GRADIENT | capi.STAGE_RANGE1D
    single = []
    for im in imgs:
        ctx = _ctx(emu_lib, 128, 128)
        try:
            ctx.set_image(im); ctx.analyze(st)
            single.append(results_digest(ctx.fetch_all(0)))
        finally:
            ctx.close()
    ctx = _ctx(emu_lib, 128, 128, slots=2)
    try:
        k = 0 if order == "interleaved_first" else 1
        loader("device" if k else "host", None, 8, 0)(ctx, imgs[k], k)
        ctx.set_image(imgs[1 - k], 1 - k)
        ctx.analyze(st, slot0=0, n_slots=2)
        assert [results_digest(ctx.fetch_all(s)) for s in (0, 1)] == single
    finally:
        ctx.close()


def test_binding_takes_a_strided_array(emu_lib):
    """Context.set_image_interleaved: an H x W x C uint8 array whose row stride exceeds W * C."""
    planes, stages = cases.SMALL_CASES["synth256_rgba"]()
    img = Interleaved(planes, pad=32)
    arr = img.array()
    assert arr.strides[0] == 256 * 4 + 32
    ctx = _ctx(emu_lib, 256, 256)
    try:
        check_image(ctx, planes, ("alpha", "grad", "r2"), load=lambda c, p, s: c.set_image_interleaved(arr, slot=s))
        check_image(ctx, planes[:3], ("grad", "r2"), load=lambda c, p, s: c.set_image_interleaved(arr, n_planes=3, slot=s))
    finally:
        ctx.close()


@pytest.mark.parametrize("ch", [3, 4])
def test_strips_load_rows_of_one_interleaved_image(emu_lib, ch):
    """LocalTransport.run with a loader: every strip's rows are a pointer y0 * rowBytes into one interleaved image."""
    from strips_check import check_against_oracle
    from yaik_b200 import strips
    w, h, n = 96, 200, 3
    planes = make_image(w, h, ch, SEED_BASE + 50) if ch == 4 else cases._patchy(w, h, 51, 4, 3)
    img = Interleaved(planes, pad=16)
    ctxs = [_ctx(emu_lib, w, h, planes=ch) for _ in range(n)]
    try:
        def load(ctx, y0, sh):
            ctx.set_image_interleaved_device(img.ptr + y0 * img.row_bytes, img.row_bytes, ch, ch, w, sh)
        merged = strips.LocalTransport(ctxs).run(planes, n_strips=n, load=load)
        check_against_oracle(merged, planes)
    finally:
        for c in ctxs:
            c.close()


@pytest.mark.parametrize("fn", ["yk_set_image_interleaved", "yk_set_image_interleaved_device"])
def test_argument_errors(emu_lib, fn):
    ctx = _ctx(emu_lib, 64, 64, planes=3)
    f = getattr(emu_lib, fn)
    buf = np.zeros(64 * 64 * 4 + 64, np.uint8)
    p = buf.ctypes.data
    try:
        assert f(ctx.ctx, 0, None, 256, 4, 3, 64, 64) == YK_ERR_ARG              # NULL pixels
        assert f(None, 0, p, 256, 4, 3, 64, 64) == YK_ERR_ARG                    # NULL context
        assert f(ctx.ctx, 1, p, 256, 4, 3, 64, 64) == YK_ERR_ARG                 # no such slot
        for ch in (1, 2, 5):
            assert f(ctx.ctx, 0, p, 320, ch, 3, 64, 64) == YK_ERR_ARG            # channels
        assert f(ctx.ctx, 0, p, 192, 3, 4, 64, 64) == YK_ERR_ARG                 # nPlanes 4 from 3 channels
        assert f(ctx.ctx, 0, p, 256, 4, 2, 64, 64) == YK_ERR_ARG                 # nPlanes 2
        assert f(ctx.ctx, 0, p, 255, 4, 3, 64, 64) == YK_ERR_ARG                 # rowBytes < w * channels
        assert f(ctx.ctx, 0, p, 191, 3, 3, 64, 64) == YK_ERR_ARG
        assert f(ctx.ctx, 0, p, 256, 4, 3, 62, 64) == YK_ERR_ARG                 # w not a multiple of 4
        assert f(ctx.ctx, 0, p, 256, 4, 3, 64, 2) == YK_ERR_ARG                  # h < 4
        assert f(ctx.ctx, 0, p, 256, 4, 3, -4, 64) == YK_ERR_ARG
        assert f(ctx.ctx, 0, p, 512, 4, 3, 68, 64) == YK_ERR_CAPACITY            # wider than the context
        assert f(ctx.ctx, 0, p, 256, 4, 3, 64, 68) == YK_ERR_CAPACITY            # taller
        assert f(ctx.ctx, 0, p, 256, 4, 4, 64, 64) == YK_ERR_CAPACITY            # nPlanes > maxPlanes
        assert f(ctx.ctx, 0, p, 256, 4, 3, 64, 64) == 0
        assert f(ctx.ctx, 0, p, 192, 3, 3, 64, 64) == 0
    finally:
        ctx.close()


def _libasan():
    try:
        p = subprocess.run([ASAN_CXX, "-print-file-name=libasan.so"], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:
        return None
    return p if os.path.isabs(p) and os.path.exists(p) else None


def test_interleaved_input_runs_clean_under_asan():
    """The source buffers end exactly at the last pixel's last byte: a read past it by the host copy or the unpack kernel
    (as emulated) aborts the AddressSanitizer build."""
    libasan = _libasan()
    if not libasan:
        pytest.skip("no g++ with libasan here")
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "tests", "emu"), "asan", "ASAN_CXX=" + ASAN_CXX], check=True)
    lib = os.path.join(ROOT, "tests", "emu", "_build", "libyaik_b200_emu_asan.so")
    env = dict(os.environ, LD_PRELOAD=libasan, ASAN_OPTIONS="detect_leaks=0:abort_on_error=1", PYTHONPATH=os.pathsep.join([ROOT, os.path.join(ROOT, "tests")]))
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "asan_interleaved_cases.py"), lib], capture_output=True, text=True, timeout=900,
                       env=env, cwd=os.path.join(ROOT, "tests"))
    assert r.returncode == 0 and "asan interleaved cases ok" in r.stdout, (r.stdout[-1000:], r.stderr[-3000:])
