"""Interleaved 8-bit input on the B200: yk_set_image_interleaved from pinned and pageable host memory and
yk_set_image_interleaved_device from a CUDA tensor give the results of the int32 yk_set_image of the same samples, and
of the oracle; strips load their rows from one interleaved image; the device buffer can be reused once a load's
unpack kernel has run."""
import ctypes as C

import numpy as np
import pytest

import cases
from interleaved import Interleaved
from parity import check_image, results_digest
from yaik_b200 import capi
from yaik_b200.synth import make_image, SEED_BASE

pytestmark = pytest.mark.gpu

ST = capi.STAGE_ALPHA | capi.STAGE_GRADIENT | capi.STAGE_RANGE1D


@pytest.fixture(scope="module")
def lib():
    return capi.load_library()


class Pinned:
    """The bytes of an Interleaved image in pinned host memory (yk_host_alloc), same row stride."""

    def __init__(self, lib, img: Interleaved):
        self.lib, self.n = lib, img.row_bytes * (img.h - 1) + img.w * img.channels
        self.ptr = lib.yk_host_alloc(self.n)
        assert self.ptr
        C.memmove(self.ptr, img.ptr, self.n)

    def free(self):
        self.lib.yk_host_free(self.ptr)


def _device_bytes(img: Interleaved, offset=0):
    """The bytes of an Interleaved image in a CUDA tensor, starting `offset` bytes into it; returns (tensor, pointer)."""
    import torch
    n = img.row_bytes * (img.h - 1) + img.w * img.channels
    src = np.ctypeslib.as_array(C.cast(img.ptr, C.POINTER(C.c_uint8)), shape=(n,))
    t = torch.empty(offset + n, dtype=torch.uint8, device="cuda")
    t[offset:].copy_(torch.from_numpy(src.copy()))
    torch.cuda.synchronize()
    return t, t.data_ptr() + offset


def gpu_loader(lib, how, channels=None, pad=0, offset=0):
    """parity.check_image `load` hook: "pinned", "pageable" (host entry point) or "device" (from a CUDA tensor)."""
    def load(ctx, planes, slot):
        c = planes.shape[0]
        img = Interleaved(planes, channels, pad, 0)
        if how == "pinned":
            p = Pinned(lib, img)
            ctx.set_image_interleaved_ptr(p.ptr, img.row_bytes, img.channels, c, img.w, img.h, slot)
            ctx.sync()
            p.free()
        elif how == "pageable":
            ctx.set_image_interleaved(img.array(), n_planes=c, slot=slot)
        else:
            t, ptr = _device_bytes(img, offset)
            ctx.set_image_interleaved_device(ptr, img.row_bytes, img.channels, c, img.w, img.h, slot)
            ctx.sync()
            del t
    return load


def _everything(ctx):
    """Digest of the fused run's streams, then DynamicTileEncode of each plane with write-back, then the state download."""
    ctx.analyze(ST)
    out = {"digest": results_digest(ctx.fetch_all(0))}
    for p in range(3):
        r = ctx.range_dyn(p, want_dst=True)
        out[f"r1_{p}"] = (r["nibbles"].tobytes(), r["defs"].tobytes(), r["dst"].tobytes(), tuple(r["constraint"]))
    s = ctx.download_state()
    out["state"] = [s["smoothMap"].tobytes(), s["mipmapMask"].tobytes()] + [a.tobytes() for k in ("mapSmoothTile", "mappedRGB", "recon") for a in s[k]]
    return out


def test_2048_rgba_bench_texture_three_loads_agree(lib):
    import torch
    planes = make_image(2048, 2048, 4, SEED_BASE + 1)
    img = Interleaved(planes)
    got = {}
    ctx = capi.Context(2048, 2048, planes=4, slots=1, lib=lib)
    try:
        ctx.set_upload_format(False)
        ctx.set_image(planes)
        got["int32"] = _everything(ctx)
        pin = Pinned(lib, img)
        ctx.set_image_interleaved_ptr(pin.ptr, img.row_bytes, 4, 4, 2048, 2048)
        got["pinned"] = _everything(ctx)
        pin.free()
        dev = torch.from_numpy(np.ascontiguousarray(np.transpose(planes, (1, 2, 0)).astype(np.uint8))).cuda()      # H x W x 4 uint8
        stream = torch.cuda.current_stream()
        ctx.set_stream(stream.cuda_stream)        # the tensor's copy and the unpack kernel on one stream
        ctx.set_image_interleaved_device(dev.data_ptr(), dev.stride(0), 4, 4, 2048, 2048)
        got["device"] = _everything(ctx)
    finally:
        ctx.close()
    assert got["pinned"] == got["int32"]
    assert got["device"] == got["int32"]


@pytest.mark.parametrize("how,channels,pad,offset", [("pinned", None, 0, 0), ("pageable", None, 40, 0), ("device", None, 0, 0),
                                                     ("device", None, 12, 5), ("pinned", 4, 8, 0), ("device", 4, 0, 3)])
@pytest.mark.parametrize("name", ["synth256_rgba", "patchy_72x40", "alpha_island128", "mip8_rgb", "synth256_rgb_3bit"])
def test_small_cases_match_oracle(lib, name, how, channels, pad, offset):
    planes, stages = cases.SMALL_CASES[name]()
    if channels == 4:
        planes, stages = planes[:3], tuple(s for s in stages if s != "alpha")
    c, h, w = planes.shape
    ctx = capi.Context(w, h, planes=4, slots=1, lib=lib)
    try:
        check_image(ctx, planes, stages, load=gpu_loader(lib, how, channels, pad, offset))
    finally:
        ctx.close()


@pytest.mark.parametrize("how", ["pinned", "device"])
def test_4096_rgb_matches_oracle(lib, how):
    planes = make_image(4096, 4096, 3, SEED_BASE + 4)
    ctx = capi.Context(4096, 4096, planes=3, slots=1, lib=lib)
    try:
        check_image(ctx, planes, ("grad", "r2"), state=False, load=gpu_loader(lib, how))
    finally:
        ctx.close()


def test_strips_load_rows_of_one_interleaved_image(lib):
    """2048 x 1024 RGB in 4 strips on this GPU, each strip a pointer y0 * rowBytes into one interleaved image in HBM."""
    from strips_check import check_against_oracle
    from yaik_b200 import strips
    w, h, n = 2048, 1024, 4
    planes = make_image(w, h, 3, SEED_BASE + 3)
    img = Interleaved(planes, pad=64)
    t, base = _device_bytes(img)
    ctxs = [capi.Context(w, h, planes=3, slots=1, lib=lib) for _ in range(n)]
    try:
        def load(ctx, y0, sh):
            ctx.set_image_interleaved_device(base + y0 * img.row_bytes, img.row_bytes, 3, 3, w, sh)
        merged = strips.LocalTransport(ctxs).run(planes, n_strips=n, load=load)
        check_against_oracle(merged, planes)
    finally:
        for c in ctxs:
            c.close()
    del t


def test_device_buffer_reused_across_contexts(lib):
    """Four contexts on their own streams load from one device buffer; the buffer is overwritten with the next image as soon
    as a load's unpack kernel has run (stream-ordered, no host sync), while the analyses are still queued."""
    import torch
    imgs = [make_image(1024, 1024, 4, SEED_BASE + 60 + i) for i in range(4)]
    want = []
    c0 = capi.Context(1024, 1024, planes=4, slots=1, lib=lib)
    try:
        for im in imgs:
            c0.set_image(im); c0.analyze(ST)
            want.append(results_digest(c0.fetch_all(0)))
    finally:
        c0.close()
    dev_imgs = [torch.from_numpy(np.ascontiguousarray(np.transpose(im, (1, 2, 0)).astype(np.uint8))).cuda() for im in imgs]
    torch.cuda.synchronize()
    buf = torch.empty_like(dev_imgs[0])
    fill = torch.cuda.Stream()
    streams = [torch.cuda.Stream() for _ in imgs]
    ctxs = [capi.Context(1024, 1024, planes=4, slots=1, lib=lib) for _ in imgs]
    try:
        for c, s in zip(ctxs, streams):
            c.set_stream(s.cuda_stream)
        for c, s, d in zip(ctxs, streams, dev_imgs):
            with torch.cuda.stream(fill):
                buf.copy_(d)
            filled = fill.record_event()
            s.wait_event(filled)
            c.set_image_interleaved_device(buf.data_ptr(), buf.stride(0), 4, 4, 1024, 1024)
            fill.wait_event(s.record_event())        # the next copy into buf waits for this unpack only
            c.analyze(ST)
        got = [results_digest(c.fetch_all(0)) for c in ctxs]
    finally:
        for c in ctxs:
            c.close()
    assert got == want
