"""DynamicTileEncode (R1) of tile-row strips on the GPU (-m gpu): the host-barrier protocol (yk_strip_range_dyn after phase
0) and the host-free one (yk_strips_run_stages), against the oracle on the whole image or against one context coding the
whole image."""
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
from yaik_b200.synth import make_image, SEED_BASE

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    return capi.load_library()        # raises if libyaik_b200.so is missing: no fallback


def _planes(w, h, c=3):
    return make_image(w, h, c, SEED_BASE + 3) if w >= 512 else cases._patchy(w, h, 43, 4, 3)


def _contexts(lib, planes, n):
    c, h, w = planes.shape
    return [capi.Context(w, h, planes=c, slots=1, lib=lib) for _ in range(n)]


def _close(ctxs):
    for c in ctxs:
        c.close()


@pytest.mark.parametrize("mode3", [False, True])
@pytest.mark.parametrize("w,h,n", [(256, 512, 2), (256, 512, 4), (192, 328, 3), (2048, 1024, 4)])
def test_strips_r1_host_barrier_matches_oracle(lib, w, h, n, mode3):
    planes = _planes(w, h)
    ctxs = _contexts(lib, planes, n)
    try:
        merged = strips.LocalTransport(ctxs).run(planes, n_strips=n, r1=r1_stage(mode3))
        check_r1(merged, oracle_r1(planes, mode3))
        check_against_oracle(merged, planes)
    finally:
        _close(ctxs)


@pytest.mark.parametrize("mode3", [False, True])
@pytest.mark.parametrize("w,h,n", [(256, 512, 2), (2048, 1024, 4), (192, 328, 3)])
def test_strips_r1_host_free_matches_oracle(lib, w, h, n, mode3):
    """Three images back to back on every strip's stream, R1 between exchange 2 and phase 1; the last one's streams."""
    planes = _planes(w, h)
    ctxs = _contexts(lib, planes, n)
    try:
        merged = strips.LocalTransport(ctxs).run_device_flags(planes, n_strips=n, images=3, r1=r1_stage(mode3))
        check_r1(merged, oracle_r1(planes, mode3))
        check_against_oracle(merged, planes)
    finally:
        _close(ctxs)


def test_strips_r1_host_free_alternating_with_and_without_r1(lib):
    """One strip set, images with and without R1 in turn: a run without R1 leaves no R1 streams behind."""
    w, h, n = 256, 512, 2
    planes = _planes(w, h)
    ctxs = _contexts(lib, planes, n)
    try:
        rows = strips.strip_rows(h, n)
        for ctx, (y0, sh) in zip(ctxs, rows):
            ctx.set_image(planes[:, y0:y0 + sh], 0)
            ctx.strip_config(h, y0)
        arr = (C.c_void_p * n)(*[ctx.ctx for ctx in ctxs])
        assert ctxs[0].L.yk_strips_link(arr, n, 0) == 0
        wants = {m: oracle_r1(planes, m) for m in (False, True)}
        for stages in (capi.STAGE_RANGEDYN, 0, capi.STAGE_RANGEDYN3, 0, capi.STAGE_RANGEDYN, capi.STAGE_RANGEDYN3):
            for ctx in ctxs:
                ctx.strip_run(stages=stages)
            for ctx in ctxs:
                ctx.sync()
            if stages == 0:
                for ctx in ctxs:
                    with pytest.raises(capi.YaikError) as e:
                        ctx.range_dyn(0)
                    assert e.value.code == -5
            else:
                mode3 = stages == capi.STAGE_RANGEDYN3
                merged = strips.merge_results([strips.collect_results(ctx, r1=stages) for ctx in ctxs])
                check_r1(merged, wants[mode3])
                check_against_oracle(merged, planes)
    finally:
        _close(ctxs)


def test_strips_r1_4096x16384_host_free_matches_whole_image(lib):
    """67 Mpixel RGB (the 2048² texture tiled), 4 strips of 4096 rows host-free with R1: equal arrays to one context coding
    the whole image with yk_analyze(GRADIENT | RANGE1D | RANGEDYN)."""
    base = make_image(2048, 2048, 3, SEED_BASE + 3)
    planes = np.ascontiguousarray(np.tile(base, (1, 8, 2)))
    assert planes.shape == (3, 16384, 4096)
    ctxs = [capi.Context(4096, 4096, planes=3, slots=1, lib=lib) for _ in range(4)]
    try:
        merged = strips.LocalTransport(ctxs).run_device_flags(planes, n_strips=4, r1=capi.STAGE_RANGEDYN)
    finally:
        _close(ctxs)
    whole = capi.Context(4096, 16384, planes=3, slots=1, lib=lib)
    try:
        check_r1(merged, whole_image_r1(whole, planes, False), "4096x16384 in 4 strips")
    finally:
        whole.close()


def _hand_made_box(w=256):
    a = np.full((w, w), 255, np.int32)
    a[:32] = 0
    a[w - 32:] = 0
    a[:, :16] = 0
    return cases._with_alpha(cases._patchy(w, w, 61, 4, 3), a)


@pytest.mark.parametrize("mode3", [False, True])
@pytest.mark.parametrize("case", ["holes512", "hand_made_box"])
def test_strips_r1_rgba_host_barrier_matches_oracle(lib, case, mode3):
    planes, n = (make_image(512, 512, 4, SEED_BASE + 12), 4) if case == "holes512" else (_hand_made_box(), 4)
    ctxs = _contexts(lib, planes, n)
    try:
        merged = strips.LocalTransport(ctxs).run(planes, n_strips=n, r1=r1_stage(mode3))
        check_r1(merged, oracle_r1(planes, mode3))
        check_against_oracle(merged, planes)
    finally:
        _close(ctxs)


def test_strips_r1_host_free_rgba_is_unsupported(lib):
    planes = make_image(256, 256, 4, SEED_BASE + 12)
    ctxs = _contexts(lib, planes, 2)
    try:
        with pytest.raises(capi.YaikError) as e:
            strips.LocalTransport(ctxs).run_device_flags(planes, n_strips=2, r1=capi.STAGE_RANGEDYN)
        assert e.value.code == -6
    finally:
        _close(ctxs)


def test_strips_r1_two_ranks_ipc_peer_copies():
    """Two processes (two GPUs when the box has them, else both on GPU 0), halo exchange by CUDA IPC + peer copies, R1."""
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT=str(29900 + os.getpid() % 300))
    procs = [subprocess.Popen([sys.executable, os.path.join(ROOT, "tests", "strips_r1_rank.py"), "--rank", str(r), "--world", "2",
                               "--backend", "gloo", "--mode", "ipc", "--w", "512", "--h", "1024"],
                              env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=600)[0] for p in procs]
    assert all(p.returncode == 0 for p in procs), "\n".join(outs)
    assert "strips r1 ok" in outs[0]
