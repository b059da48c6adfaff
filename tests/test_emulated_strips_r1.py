"""DynamicTileEncode (R1) of a strip set on the CPU, through the emulated build of the kernels (tests/emu): every strip codes
the blocks of the image's walk whose top row it holds, and the merged streams equal the oracle's on the whole image (or,
outside the oracle's alpha domain, one context coding the whole image)."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import cases
from strips_check import check_against_oracle
from strips_r1_check import check_r1, oracle_r1, r1_stage, whole_image_r1
from yaik_b200 import capi, strips
from yaik_b200.synth import make_image, SEED_BASE, _rand

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU = os.path.join(ROOT, "tests", "emu", "_build", "libyaik_b200_emu.so")
YK_ERR_ARG, YK_ERR_STATE, YK_ERR_UNSUPPORTED = -2, -5, -6


@pytest.fixture(scope="module")
def emu_lib():
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "tests", "emu")], check=True)
    return capi.load_library(EMU)


def _run(lib, planes, n, mode3, packed=True):
    c, h, w = planes.shape
    ctxs = [capi.Context(w, h, planes=c, slots=1, lib=lib) for _ in range(n)]
    try:
        for ctx in ctxs:
            ctx.set_upload_format(packed)
        return strips.LocalTransport(ctxs).run(planes, n_strips=n, r1=r1_stage(mode3))
    finally:
        for ctx in ctxs:
            ctx.close()


def _hand_made_box(w=256):
    """Rows 0-31, rows w-32..w-1 and columns 0-15 transparent: the box starts below row 0 and ends above the last row, so
    the walk's last block rows (y + 8 > ch) and its extra block lie in the last of 4 strips, which codes nothing."""
    a = np.full((w, w), 255, np.int32)
    a[:32] = 0
    a[w - 32:] = 0
    a[:, :16] = 0
    return cases._with_alpha(cases._patchy(w, w, 61, 4, 3), a)


@pytest.mark.parametrize("mode3", [False, True])
@pytest.mark.parametrize("name,w,h,n", [("patchy", 128, 192, 2), ("patchy", 128, 192, 3), ("ramp", 64, 136, 2), ("synth", 128, 256, 4)])
def test_strips_r1_rgb_matches_oracle(emu_lib, name, w, h, n, mode3):
    planes = (cases._patchy(w, h, 41, 4, 3) if name == "patchy" else cases._smooth_noisy(w, h, 42, 2) if name == "ramp"
              else make_image(w, h, 3, SEED_BASE + 3))
    merged = _run(emu_lib, planes, n, mode3)
    check_r1(merged, oracle_r1(planes, mode3))
    check_against_oracle(merged, planes)


@pytest.mark.parametrize("i", range(6))
def test_strips_r1_random_shapes(emu_lib, i):
    """Random widths and heights inside R1's domain (multiples of 8, >= 32), strip counts, modes and both upload formats."""
    r = _rand(4343, i, np.arange(6, dtype=np.uint64))
    w = 8 * (4 + int(r[0] % np.uint64(20)))              # 32 .. 184
    h = 8 * (9 + int(r[1] % np.uint64(24)))              # 72 .. 256
    n = 2 + int(r[2] % np.uint64(3))
    planes = cases._patchy(w, h, 600 + i, 4, 1 + int(r[3] % np.uint64(4)))
    mode3 = bool(r[4] % np.uint64(2))
    merged = _run(emu_lib, planes, n, mode3, packed=i % 2 == 0)
    check_r1(merged, oracle_r1(planes, mode3))
    check_against_oracle(merged, planes)


@pytest.mark.parametrize("mode3", [False, True])
@pytest.mark.parametrize("case", ["make128x2", "make256x4", "hand_made_box", "opaque"])
def test_strips_r1_rgba_matches_oracle(emu_lib, case, mode3):
    if case == "make128x2":
        planes, n = make_image(128, 128, 4, SEED_BASE + 16), 2
    elif case == "make256x4":
        planes, n = make_image(256, 256, 4, SEED_BASE + 12), 4
    elif case == "hand_made_box":
        planes, n = _hand_made_box(), 4
    else:                                                 # box == image: the alpha rejection is discarded (EC.cpp:1400-1403)
        planes, n = cases._with_alpha(cases._patchy(128, 128, 62, 4, 3), np.full((128, 128), 255, np.int32)), 2
    merged = _run(emu_lib, planes, n, mode3)
    check_r1(merged, oracle_r1(planes, mode3))
    check_against_oracle(merged, planes)
    if case == "hand_made_box":
        assert merged["r1"][0]["constraint"] == [16, 32, 240, 192]


def test_strips_r1_last_strip_codes_nothing(emu_lib):
    planes = _hand_made_box()
    ctxs = [capi.Context(256, 256, planes=4, slots=1, lib=emu_lib) for _ in range(4)]
    try:
        strips.LocalTransport(ctxs).run(planes, n_strips=4, r1=capi.STAGE_RANGEDYN)
        last = ctxs[3].range_dyn(0)
        assert last["n_nibbles"] == 0 and last["defs"].size == 0 and last["constraint"] == [16, 32, 240, 192]
    finally:
        for ctx in ctxs:
            ctx.close()


@pytest.mark.parametrize("mode3", [False, True])
def test_strips_r1_rgba_rectangle_matches_whole_image_context(emu_lib, mode3):
    """128x256 RGBA in 3 strips: outside the oracle's alpha domain, so against one emulated context on the whole image."""
    planes = make_image(128, 256, 4, SEED_BASE + 19)
    merged = _run(emu_lib, planes, 3, mode3)
    whole = capi.Context(128, 256, planes=4, slots=1, lib=emu_lib)
    try:
        check_r1(merged, whole_image_r1(whole, planes, mode3))
    finally:
        whole.close()


def test_strips_r1_two_gloo_ranks_host_transport(emu_lib):
    """world_size 2, one strip per rank over gloo, the alpha box gathered on the control plane (RGBA), both modes."""
    script = os.path.join(ROOT, "tests", "strips_r1_rank.py")
    for k, extra in enumerate((["--planes", "3"], ["--planes", "4", "--mode3"])):
        env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT=str(30100 + os.getpid() % 500 + k), YK_STRIPS_LIB=EMU)
        procs = [subprocess.Popen([sys.executable, script, "--rank", str(r), "--world", "2", "--backend", "gloo", "--mode", "host",
                                   "--w", "128", "--h", "128", *extra], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
                 for r in range(2)]
        outs = [p.communicate(timeout=600)[0] for p in procs]
        assert all(p.returncode == 0 for p in procs), "\n".join(outs)
        assert "strips r1 ok" in outs[0]


def _strip_pair(lib, c, w, h):
    """Two strips of a w x h image with c planes, configured, phase 0 not run yet."""
    planes = cases._patchy(w, h, 43, 4, 3)
    if c == 4:
        planes = cases._with_alpha(planes, np.full((h, w), 255, np.int32))
    rows = strips.strip_rows(h, 2)
    ctxs = []
    for y0, sh in rows:
        ctx = capi.Context(w, h, planes=c, slots=1, lib=lib)
        ctx.set_image(planes[:, y0:y0 + sh], 0)
        ctx.strip_config(h, y0)
        ctxs.append(ctx)
    return ctxs


def test_strips_r1_errors(emu_lib):
    L = emu_lib
    box = lambda *v: (C.c_int * 4)(*v)
    rgb = _strip_pair(emu_lib, 3, 64, 128)
    rgba = _strip_pair(emu_lib, 4, 64, 128)
    try:
        a = rgb[0]
        assert L.yk_strip_range_dyn(a.ctx, 0, 0, None) == YK_ERR_STATE                    # phase 0 has not run
        assert L.yk_strip_range_dyn(a.ctx, 0, 0, box(0, 0, 64, 128)) == YK_ERR_ARG        # a box for an RGB strip
        for ctx in rgb + rgba:
            ctx.strip_phase(0)
        assert L.yk_range_dyn(a.ctx, 0, 0, 0, None, 0, None, None, 0, None, None, None) == YK_ERR_STATE     # not coded yet
        b = rgba[1]
        assert L.yk_strip_range_dyn(b.ctx, 0, 0, None) == YK_ERR_ARG                      # none for an RGBA strip
        for bad in ((0, 0, 65, 128), (0, 0, 64, 129), (-8, 0, 64, 128), (0, -1, 64, 128), (8, 0, 8, 128), (0, 40, 64, 40)):
            assert L.yk_strip_range_dyn(b.ctx, 0, 0, box(*bad)) == YK_ERR_ARG, bad           # outside [0, w) x [0, imgH), or empty
        assert L.yk_strip_range_dyn(b.ctx, 0, 0, box(0, 0, 64, 128)) == 0
        assert L.yk_strip_range_dyn(a.ctx, 0, 1, None) == 0
        nib = np.zeros(4096, np.uint8); defs = np.zeros(256, np.uint16)
        nn, nd = C.c_int(), C.c_int()
        args = lambda ctx, mode3, dst: (ctx.ctx, 0, 0, mode3, nib.ctypes.data_as(C.c_void_p), nib.size, C.byref(nn),
                                        defs.ctypes.data_as(C.c_void_p), defs.size, C.byref(nd), None, dst)
        assert L.yk_range_dyn(*args(a, 0, None)) == YK_ERR_STATE                            # coded in the other mode
        assert L.yk_range_dyn(*args(a, 1, None)) == 0
        dst = np.zeros((64, 64), np.int32)
        assert L.yk_range_dyn(*args(a, 1, dst.ctypes.data_as(C.c_void_p))) == YK_ERR_UNSUPPORTED   # no write-back on strips
        # the host-free protocol: stage bits, and R1 of an RGBA strip set
        for sets in (rgb, rgba):
            arr = (C.c_void_p * 2)(*[ctx.ctx for ctx in sets])
            assert L.yk_strips_link(arr, 2, 0) == 0
        arr3 = (C.c_void_p * 2)(*[ctx.ctx for ctx in rgb])
        arr4 = (C.c_void_p * 2)(*[ctx.ctx for ctx in rgba])
        assert L.yk_strip_run_stages(a.ctx, 0, 3, capi.STAGE_GRADIENT) == YK_ERR_ARG
        assert L.yk_strip_run_stages(a.ctx, 0, 3, capi.STAGE_RANGEDYN | capi.STAGE_RANGEDYN3) == YK_ERR_ARG
        assert L.yk_strips_run_stages(arr3, 2, 0, 3, capi.STAGE_RANGEDYN | capi.STAGE_ALPHA) == YK_ERR_ARG
        assert L.yk_strip_run_stages(b.ctx, 0, 3, capi.STAGE_RANGEDYN) == YK_ERR_UNSUPPORTED
        assert L.yk_strips_run_stages(arr4, 2, 0, 3, capi.STAGE_RANGEDYN3) == YK_ERR_UNSUPPORTED
        assert L.yk_strip_run_stages(b.ctx, 0, 3, 0) == YK_ERR_UNSUPPORTED                 # the emulation cannot wait for flags
    finally:
        for ctx in rgb + rgba:
            ctx.close()
    # not a strip; w / imgH outside R1's domain
    whole = capi.Context(64, 64, planes=3, slots=1, lib=emu_lib)
    try:
        whole.set_image(cases._patchy(64, 64, 44, 4, 3), 0)
        assert L.yk_strip_range_dyn(whole.ctx, 0, 0, None) == YK_ERR_STATE
    finally:
        whole.close()
    for w, h in ((36, 128), (24, 128), (64, 28)):
        narrow = capi.Context(w, h, planes=3, slots=1, lib=emu_lib)
        try:
            narrow.set_image(cases._patchy(w, h, 45, 4, 3), 0)
            narrow.strip_config(h, 0)
            narrow.strip_phase(0)
            assert L.yk_strip_range_dyn(narrow.ctx, 0, 0, None) == YK_ERR_ARG, (w, h)
        finally:
            narrow.close()


def _libasan():
    try:
        p = subprocess.run([os.environ.get("ASAN_CXX", "/usr/bin/g++"), "-print-file-name=libasan.so"], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:
        return None
    return p if os.path.isabs(p) and os.path.exists(p) else None


def test_strips_r1_runs_clean_under_asan():
    """Contexts exactly as large as their strips: a row read at the image's y instead of the strip's aborts the
    AddressSanitizer build."""
    libasan = _libasan()
    if not libasan:
        pytest.skip("no g++ with libasan here")
    asan_cxx = os.environ.get("ASAN_CXX", "/usr/bin/g++")
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "tests", "emu"), "asan", "ASAN_CXX=" + asan_cxx], check=True)
    lib = os.path.join(ROOT, "tests", "emu", "_build", "libyaik_b200_emu_asan.so")
    env = dict(os.environ, LD_PRELOAD=libasan, ASAN_OPTIONS="detect_leaks=0:abort_on_error=1", PYTHONPATH=os.pathsep.join([ROOT, os.path.join(ROOT, "tests")]))
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "asan_strips_r1_cases.py"), lib], capture_output=True, text=True, timeout=900,
                       env=env, cwd=os.path.join(ROOT, "tests"))
    assert r.returncode == 0 and "asan strips r1 cases ok" in r.stdout, (r.stdout[-1000:], r.stderr[-3000:])
