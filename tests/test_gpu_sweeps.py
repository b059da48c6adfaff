"""The oracle sweeps of tests/test_emulated_sweeps.py on the CUDA library at larger sizes, on both analysis kernels
(int32 uploads for yk_k_analyze, packed uploads for yk_k_analyze_u8), plus what only the GPU schedules: R1's look-back
over 128 units at 2048 x 2048, the pipelined configuration bench.py times with R1 behind the analysis, and slot reuse on a
context bound to a non-default stream."""
import numpy as np
import pytest

import sweeps
from parity import check_image, check_results, fused_stages, results_digest
from yaik_b200 import capi
from yaik_b200.synth import make_image, SEED_BASE

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def lib():
    return capi.load_library()


@pytest.fixture(scope="module")
def ctx(lib):
    c = capi.Context(1024, 1024, planes=4, slots=1, lib=lib)
    yield c
    c.close()


def _device_bytes(a):
    import torch
    t = torch.from_numpy(np.ascontiguousarray(a)).cuda()
    torch.cuda.synchronize()
    return t.data_ptr(), t


def _run(ctx, planes, stages, fused, packed, **kw):
    ctx.set_upload_format(packed)
    try:
        check_image(ctx, planes, stages, fused=fused, **kw)
    finally:
        ctx.set_upload_format(True)


@pytest.mark.parametrize("i", range(24))
def test_r1_sweep(ctx, i):
    planes, stages, fused, packed = sweeps.r1_case(100 + i, 1024)
    _run(ctx, planes, stages, fused, packed)


@pytest.mark.parametrize("i", range(12))
def test_alpha_sweep(ctx, i):
    planes, stages, fused, packed = sweeps.alpha_case(100 + i, 1024)
    _run(ctx, planes, stages, fused, packed, state=planes.shape[1] <= 512)


@pytest.mark.parametrize("packed", [True, False], ids=["u8", "int32"])
@pytest.mark.parametrize("fused", [True, False], ids=["fused", "stage_by_stage"])
@pytest.mark.parametrize("reject", sweeps.REJECT_FACTORS)
def test_reject_factor_sweep(ctx, reject, fused, packed):
    w, h = ((512, 512), (520, 296), (1024, 200))[reject % 3]
    planes = sweeps.reject_content(w, h, reject, 8500 + reject)
    _run(ctx, planes, ("grad", "r2", "r1"), fused, packed, reject=reject)


@pytest.mark.parametrize("packed", [True, False], ids=["u8", "int32"])
@pytest.mark.parametrize("n_slots,r1", [(2, "r1"), (3, "r1_3bit")])
def test_batch_with_fused_r1(lib, n_slots, r1, packed):
    d = sweeps._Draw(8600, n_slots * 2 + packed)
    side = 512
    stages = ("alpha", "grad", "r2", r1)
    imgs = [sweeps.rgba_island_image(d, side, 8700 + 10 * n_slots + k) if k != 1 else sweeps.rgb_content(d, side, side, 8800 + k)
            for k in range(n_slots)]
    c = capi.Context(side, side, planes=4, slots=n_slots, lib=lib)
    try:
        c.set_upload_format(packed)
        for k, im in enumerate(imgs):
            c.set_image(im, k)
        c.analyze(fused_stages(imgs[0], stages), slot0=0, n_slots=n_slots)
        for k, im in enumerate(imgs):
            check_results(c, im, stages, slot=k, r1_fused=True, state=False)
    finally:
        c.close()


@pytest.mark.parametrize("r1", ["r1", "r1_3bit"])
def test_r1_2048_rgba_with_alpha(lib, r1):
    """The bench texture with an island cut into its alpha: R1's offsets kernel over 128 look-back units, its constraint
    box from the alpha stage, fused and per plane, against the oracle."""
    planes = make_image(2048, 2048, 4, SEED_BASE + 1).copy()
    planes[3, :, 1800:] = 0
    planes[3, :72, :] = 0
    c = capi.Context(2048, 2048, planes=4, slots=1, lib=lib)
    try:
        c.set_upload_format(r1 == "r1")
        check_image(c, planes, ("alpha", "grad", r1), state=False)
    finally:
        c.close()


def _load_device_planes(c, planes, slot):
    ch, h, w = planes.shape
    ptrs = []
    for i in range(ch):
        ptrs.append(c.device_plane(slot, i))
        c.copy_from_host(ptrs[-1], np.ascontiguousarray(planes[i], dtype=np.int32))
    c.set_image_device(ptrs, ch, w, h, slot)


def test_bench_configuration_with_r1_matches_oracle(lib):
    """bench.py's with_r1 step: 8 contexts on 8 CUDA streams, analysis launches of a quarter of the SMs, int32 planes
    resident in HBM, ALPHA | GRADIENT | RANGE1D | RANGEDYN on 8 distinct 2048 x 2048 RGBA textures issued round-robin.
    The first two textures' R1 streams against the oracle; after 6 rounds every context's results and R1 streams equal a
    single-context, full-SM run's."""
    import torch
    st = capi.STAGE_ALPHA | capi.STAGE_GRADIENT | capi.STAGE_RANGE1D | capi.STAGE_RANGEDYN
    imgs = [make_image(2048, 2048, 4, SEED_BASE + 1 + i) for i in range(8)]
    c0 = capi.Context(2048, 2048, planes=4, slots=1, lib=lib)
    want = []
    try:
        c0.set_upload_format(False)
        for k, im in enumerate(imgs):
            if k < 2:
                check_image(c0, im, ("alpha", "grad", "r2", "r1"), state=False)      # oracle-verified
                c0.reset_state(0)
            else:
                c0.set_image(im)
            c0.analyze(st)
            want.append((results_digest(c0.fetch_all(0)), sweeps.r1_digest(c0, 0)))
    finally:
        c0.close()
    ctxs = [capi.Context(2048, 2048, planes=4, slots=1, lib=lib) for _ in range(8)]
    streams = [torch.cuda.Stream() for _ in range(8)]
    try:
        for c, s, im in zip(ctxs, streams, imgs):
            c.set_stream(s.cuda_stream); c.set_upload_format(False); c.set_analysis_ctas(c.sm_count() // 4)
            _load_device_planes(c, im, 0)
        for rep in range(6):
            for c in ctxs:
                c.reset_state(0); c.analyze(st)
        got = [(results_digest(c.fetch_all(0)), sweeps.r1_digest(c, 0)) for c in ctxs]
        assert got == want
    finally:
        for c in ctxs:
            c.close()


@pytest.mark.parametrize("seq,n_slots", [(10, 2), (11, 3)])
def test_slot_reuse_sequence_on_a_side_stream(lib, seq, n_slots):
    import torch
    s = torch.cuda.Stream()
    c = capi.Context(512, 512, planes=4, slots=n_slots, lib=lib)
    try:
        c.set_stream(s.cuda_stream)
        sweeps.run_sequence(c, sweeps.reuse_sequence(seq, n_slots, 14, 512), _device_bytes)
    finally:
        c.close()
