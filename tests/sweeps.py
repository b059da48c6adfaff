"""Seeded case generators and helpers shared by the oracle sweeps on the CPU-emulated library
(tests/test_emulated_sweeps.py, sizes up to 256) and on the GPU (tests/test_gpu_sweeps.py, larger sizes):
DynamicTileEncode (R1) on random shapes, the alpha stage on random islands, rejectFactor 0..64, multi-slot batches and
seeded sequences of loads and programs on one context's slots.  The same index gives the same case on every run."""
import hashlib

import numpy as np

import cases
from interleaved import Interleaved
from parity import check_chroma, check_image, check_results, fused_stages, results_digest
from yaik_b200 import capi
from yaik_b200.synth import make_image, SEED_BASE, _rand

YK_ERR_ARG, YK_ERR_STATE = -2, -5
REJECT_FACTORS = (0, 1, 2, 4, 5, 8, 16, 33, 64)


class _Draw:
    """Seeded integers: the i-th draw of stream (seed, index)."""

    def __init__(self, seed, index, n=64):
        self.v = _rand(seed, index, np.arange(n, dtype=np.uint64)) >> np.uint64(11)
        self.k = 0

    def int(self, n):
        x = int(self.v[self.k % self.v.size]) % n
        self.k += 1
        return x

    def pick(self, seq):
        return seq[self.int(len(seq))]


def rgb_content(d: _Draw, w, h, seed):
    """Patchy ramp, illustration-like, or full-range noise."""
    kind = d.int(3)
    if kind == 0:
        return cases._patchy(w, h, seed, d.pick((4, 8)), 1 + d.int(4))
    if kind == 1:
        return make_image(w, h, 3, SEED_BASE + seed)
    return cases._noise(w, h, 3, seed, 0, 255)


def signed_planes(w, h, seed):
    """Signed samples inside the reference's R1 domain (see the r1_signed* cases): they go up as int32 whatever the
    upload format, and only DynamicTileEncode takes them."""
    return cases._noise(w, h, 3, seed, -120, 100)


def island(d: _Draw, side):
    """An alpha plane for a side x side image: one rectangle of kept pixels whose corners lie on or off the 16-pixel grid,
    optional holes; or the box over the whole image (the rejection is discarded); or a single kept tile at a corner."""
    kind = d.int(8)
    if kind == 0:                                   # box == image: holes inside, no chunk is written
        holes = [(16, 16, side - 16, 32)] if side >= 64 else []
        return cases._alpha_island(side, side, 0, 0, side, side, holes)
    if kind == 1:                                   # one 16 x 16 tile at a corner, partly covered
        cx, cy = d.pick((0, side - 16)), d.pick((0, side - 16))
        return cases._alpha_island(side, side, cx + d.int(8), cy + d.int(8), cx + 16 - d.int(8), cy + 16 - d.int(8))

    def coord(n):                                   # on the grid, or anywhere
        return 16 * d.int(n // 16 + 1) if d.int(2) else d.int(n + 1)
    while True:
        x0, x1 = sorted((coord(side), coord(side)))
        y0, y1 = sorted((coord(side), coord(side)))
        if x1 > x0 and y1 > y0:
            break
    holes = []
    for _ in range(d.int(3)):
        hx, hy = d.int(side), d.int(side)
        holes.append((hx, hy, min(side, hx + 1 + d.int(40)), min(side, hy + 1 + d.int(40))))
    a = cases._alpha_island(side, side, x0, y0, x1, y1, holes)
    if not a.any():                                 # fully transparent: outside the reference's domain
        a[y0, x0] = 255
    return a


def rgba_island_image(d: _Draw, side, seed):
    return cases._with_alpha(rgb_content(d, side, side, seed), island(d, side))


def r1_case(i, max_side=256):
    """(planes, stages, fused, packed) for DynamicTileEncode: a random multiple-of-8 shape from 32 to max_side (RGBA: a
    power-of-two square with an island), 4- or 3-bit mode, with or without the gradient stage before it."""
    d = _Draw(4242, i)
    mode = "r1_3bit" if d.int(2) else "r1"
    fused, packed = d.int(2) == 0, d.int(2) == 0
    kind = d.int(6)
    if kind == 0:                                   # signed int32 planes, R1 alone
        w, h = 8 * (4 + d.int(max_side // 8 - 3)), 8 * (4 + d.int(max_side // 8 - 3))
        return signed_planes(w, h, 6000 + i), (mode,), fused, packed
    if kind == 1:
        side = 32 << d.int((max_side // 32).bit_length())
        return rgba_island_image(d, side, 6100 + i), ("alpha", "grad", mode), fused, packed
    w, h = 8 * (4 + d.int(max_side // 8 - 3)), 8 * (4 + d.int(max_side // 8 - 3))
    stages = ("grad", mode) if d.int(4) else (mode,)
    return rgb_content(d, w, h, 6200 + i), stages, fused, packed


def alpha_case(i, max_side=256):
    """(planes, stages, fused, packed): a power-of-two RGBA square (32 .. max_side) with a random island, every stage."""
    d = _Draw(4343, i)
    side = 32 << d.int((max_side // 32).bit_length())
    return rgba_island_image(d, side, 6300 + i), ("alpha", "grad", "r2", "r1"), d.int(3) != 0, d.int(2) == 0


def reject_content(w, h, reject, seed):
    """A ramp with patch-wise noise of amplitude up to about rejectFactor: tiles are accepted or rejected at every tile
    size whatever the factor."""
    return cases._patchy(w, h, seed, 4, max(1, reject + 1))


def r1_digest(ctx, slot, mode3=False):
    """SHA-1 over the three R1 streams yk_range_dyn returns for `slot` without a write-back plane (the fused streams when
    yk_analyze coded them in this mode), or the error code."""
    h = hashlib.sha1()
    for p in range(3):
        try:
            r = ctx.range_dyn(p, mode3=mode3, slot=slot)
        except capi.YaikError as e:
            return f"error {e.code}"
        h.update(r["nibbles"].tobytes()); h.update(r["defs"].tobytes())
        h.update(str((r["n_nibbles"], r["constraint"])).encode())
    return h.hexdigest()


def all_digest(ctx, slot):
    """parity.results_digest of yk_fetch_all, or the error code (no analysis has run on the slot's image)."""
    try:
        return results_digest(ctx.fetch_all(slot))
    except capi.YaikError as e:
        return f"error {e.code}"


# ---- loads ------------------------------------------------------------------------------------------------------
LOADS = ("packed", "int32", "device", "interleaved_host", "interleaved_device")


def load_fn(how, device_bytes):
    """A check_image `load` hook.  device_bytes(uint8 array) -> (device address, keep-alive) puts bytes in device memory
    (host memory in the emulated build)."""
    def load(ctx, planes, slot):
        c, h, w = planes.shape
        if how in ("packed", "int32"):
            ctx.set_upload_format(how == "packed")
            ctx.set_image(planes, slot)
            ctx.set_upload_format(True)
        elif how == "device":                       # int32 planes resident in device memory (the slot's own buffers)
            ptrs = []
            for p in range(c):
                ptrs.append(ctx.device_plane(slot, p))
                ctx.copy_from_host(ptrs[-1], np.ascontiguousarray(planes[p], dtype=np.int32))
            ctx.set_image_device(ptrs, c, w, h, slot)
        else:
            img = Interleaved(planes)
            if how == "interleaved_host":
                ctx.set_image_interleaved_ptr(img.ptr, img.row_bytes, img.channels, c, w, h, slot)
            else:
                ptr, keep = device_bytes(img.raw[img.ptr - img.raw.ctypes.data:])
                ctx.set_image_interleaved_device(ptr, img.row_bytes, img.channels, c, w, h, slot)
            ctx.sync()                              # the buffer may go once the call has returned
    return load


# ---- slot-reuse sequences ---------------------------------------------------------------------------------------
PROGRAMS = ("fused", "fused_r1", "stages", "r1_only", "chroma", "reset_again")


def _image(d: _Draw, kind, max_side, seed, side=None):
    if kind == "rgba":
        side = side or 32 << d.int((max_side // 32).bit_length())
        return rgba_island_image(d, min(side, max_side), seed)
    if kind == "signed":
        return signed_planes(8 * (4 + d.int(max_side // 8 - 3)), 8 * (4 + d.int(max_side // 8 - 3)), seed)
    if kind == "noise_large":
        return cases._noise(max_side, max_side, 3, seed, 0, 255)
    w, h = side or 8 * (4 + d.int(max_side // 8 - 3)), side or 8 * (4 + d.int(max_side // 8 - 3))
    return rgb_content(d, w, h, seed)


def reuse_sequence(seq, n_slots, n_random, max_side):
    """A seeded list of steps (slot, load, planes, program, mode3).  It opens with the transitions that decide what a slot
    clears, re-derives or serves from cache, then continues at random:
    large noisy RGB -> small RGBA in the same slot (small after large, RGBA after RGB, alpha state after none);
    fused R1 -> R1 alone in the same mode (the fused-stream cache must not outlive the image);
    RGBA with alpha -> RGB with fused R1 (the alpha stage's flags must not outlive the image);
    signed planes that fall back to int32 -> a packed image."""
    d = _Draw(5151, seq, 256)
    seed = 7000 + 100 * seq
    m3 = d.int(2) == 1
    other = 1 % n_slots
    steps = [
        (0, "packed", _image(d, "noise_large", max_side, seed + 0), "fused_r1", m3),
        (other, "int32", _image(d, "rgba", max_side, seed + 1), "fused_r1", not m3),
        (0, d.pick(LOADS), _image(d, "rgba", max_side, seed + 2, side=32), "fused_r1", m3),
        (0, d.pick(LOADS), _image(d, "rgb", max_side, seed + 3), "r1_only", m3),
        (other, d.pick(LOADS), _image(d, "rgba", max_side, seed + 4), "stages", m3),
        (other, d.pick(("packed", "int32")), _image(d, "rgb", max_side, seed + 5), "fused_r1", m3),
        (0, "packed", _image(d, "signed", max_side, seed + 6), "r1_only", m3),
        (0, "packed", _image(d, "rgb", max_side, seed + 7), "fused", m3),
    ]
    for k in range(n_random):
        kind = d.pick(("rgb", "rgb", "rgba", "rgba", "signed", "noise_large"))
        planes = _image(d, kind, max_side, seed + 10 + k)
        if kind == "signed":
            prog, how = "r1_only", d.pick(("packed", "int32", "device"))
        else:
            prog, how = d.pick(PROGRAMS), d.pick(LOADS)
        steps.append((d.int(n_slots), how, planes, prog, d.int(2) == 1))
    return steps


def chroma_config(d: _Draw, w, h):
    """(halfCoW, halfCoH, halfCgW, halfCgH), (EDownSample of Co, Cg): an axis is halved only where the reduced plane stays
    a multiple of 8 and at least 32 (R1's domain)."""
    ok = (w % 16 == 0 and w >= 64, h % 16 == 0 and h >= 64)
    cfg = tuple(d.int(2) if ok[k % 2] else 0 for k in range(4))
    modes = []
    for k in range(2):
        both = cfg[2 * k] and cfg[2 * k + 1]
        modes.append(d.int(5) if both else d.pick((0, 2)))     # one halved axis: nearest / average only
    return cfg, tuple(modes)


def run_step(ctx, step, device_bytes, index):
    """Run one step of a reuse sequence and compare its outputs with the oracle.  Returns the R1 mode the slot's streams
    were last coded in."""
    slot, how, planes, prog, m3 = step
    c, h, w = planes.shape
    load = load_fn(how, device_bytes)
    r1 = "r1_3bit" if m3 else "r1"
    full = ("alpha", "grad", "r2") if c == 4 else ("grad", "r2")
    if prog == "fused":
        load(ctx, planes, slot)
        ctx.analyze(fused_stages(planes, full), slot0=slot)
        check_results(ctx, planes, full, slot=slot)
    elif prog == "fused_r1":                         # the fused streams stay in the slot for the steps after this one
        load(ctx, planes, slot)
        ctx.analyze(fused_stages(planes, full + (r1,)), slot0=slot)
        check_results(ctx, planes, full + (r1,), slot=slot, r1_fused=True, r1_dst=False)
    elif prog == "stages":
        check_image(ctx, planes, full + (r1,), fused=False, slot=slot, load=load)
    elif prog == "r1_only":
        load(ctx, planes, slot)
        check_results(ctx, planes, (r1,), slot=slot, r1_without_dst=True)
    elif prog == "chroma":
        d = _Draw(5252, index)
        cfg, modes = chroma_config(d, w, h)
        pre = d.pick(((), ("grad",), ("alpha", "grad") if c == 4 else ("grad",)))
        check_chroma(ctx, planes, pre, cfg, modes, slot=slot, load=load)
    elif prog == "reset_again":
        st = fused_stages(planes, full + (r1,))
        load(ctx, planes, slot)
        ctx.analyze(st, slot0=slot)
        ctx.reset_state(slot)
        ctx.analyze(st, slot0=slot)
        check_results(ctx, planes, full + (r1,), slot=slot, r1_fused=True)
    else:
        raise ValueError(prog)
    return m3


def run_sequence(ctx, steps, device_bytes):
    """Every step against the oracle; after each, every other slot's fetch_all and R1 digests are what they were."""
    digests, modes = {}, {}
    for k, step in enumerate(steps):
        slot = step[0]
        try:
            modes[slot] = run_step(ctx, step, device_bytes, k)
        except AssertionError as e:
            raise AssertionError(f"step {k} {step[:2] + (step[2].shape,) + step[3:]}: {e}") from None
        for s, want in digests.items():
            if s != slot:
                got = (all_digest(ctx, s), r1_digest(ctx, s, modes[s]))
                assert got == want, f"step {k} on slot {slot} changed slot {s}'s results"
        digests[slot] = (all_digest(ctx, slot), r1_digest(ctx, slot, modes[slot]))
