"""Shared parity checker: the C-ABI path (CUDA library on the GPU box, or the CPU-emulated build of the same
sources for kernel-logic tests here) against the C oracle on the same input.  Bit-exact or fail."""
import numpy as np

from oracle_py import Oracle, PASS_ORDER
from yaik_b200 import capi


def _eq(a, b, what):
    a = np.asarray(a); b = np.asarray(b)
    if a.shape != b.shape or not np.array_equal(a, b):
        n = min(a.size, b.size)
        diff = np.nonzero(a.ravel()[:n] != b.ravel()[:n])[0]
        first = int(diff[0]) if diff.size else n
        raise AssertionError(f"{what}: sizes {a.size} vs {b.size}, first difference at {first} "
                             f"(got {a.ravel()[first:first + 8].tolist()} want {b.ravel()[first:first + 8].tolist()}), {diff.size} differ")


def results_digest(r) -> str:
    """SHA-1 over everything Context.fetch_all() returned for one image (bitmaps, rgbStreams, TileDone, boxes, R2 streams,
    alpha results): equal digests == identical streams."""
    import hashlib
    h = hashlib.sha1()
    for p in r["passes"]:
        if p is None:
            h.update(b"-")
            continue
        h.update(p["bitmap"].tobytes()); h.update(p["rgb"].tobytes()); h.update(str((p["tiledone"], list(p["bbox"]))).encode())
    for q in r["r2"]:
        h.update(q["idx"].tobytes()); h.update(q["type"].tobytes())
    a = r.get("alpha")
    if a:
        h.update(a["bitmap"].tobytes()); h.update(str((a["bound"], a["remaining"], a["wrote"], a["chunk_bbox"])).encode())
    return h.hexdigest()


def fused_stages(planes: np.ndarray, stages) -> int:
    """The yk_analyze stage flags that run `stages` (as in tests/cases.py) in one call: R1 only inside its domain
    (multiples of 8, at least 32 x 32), alpha only on four planes."""
    c, h, w = planes.shape
    st = ((capi.STAGE_ALPHA if "alpha" in stages and c == 4 else 0) | (capi.STAGE_GRADIENT if "grad" in stages else 0)
          | (capi.STAGE_RANGE1D if "r2" in stages else 0))
    if ("r1" in stages or "r1_3bit" in stages) and w >= 32 and h >= 32 and w % 8 == 0 and h % 8 == 0:
        st |= capi.STAGE_RANGEDYN3 if "r1_3bit" in stages else capi.STAGE_RANGEDYN
    return st


def check_image(ctx: "capi.Context", planes: np.ndarray, stages, *, fused=True, state=True, slot=0, load=None, reject=3):
    """stages as in tests/cases.py.  fused=True: one yk_analyze then getters; False: stage-by-stage calls.
    load(ctx, planes, slot): how the samples get into the context (default: yk_set_image from host planes).
    reject: the rejectFactor of the gradient stage (0..64), passed to yk_analyze, yk_gradient_pass and the oracle."""
    if load is None:
        ctx.set_image(planes, slot)
    else:
        load(ctx, planes, slot)
    st = fused_stages(planes, stages)
    if fused:
        ctx.analyze(st, slot0=slot, reject=reject)
    check_results(ctx, planes, stages, slot=slot, state=state, reject=reject,
                  r1_fused=fused and bool(st & (capi.STAGE_RANGEDYN | capi.STAGE_RANGEDYN3)))


def check_results(ctx: "capi.Context", planes: np.ndarray, stages, *, slot=0, state=True, reject=3, r1_fused=False, r1_without_dst=False,
                  r1_dst=True):
    """The results of `stages` in `slot` against the oracle, once the image is loaded: whatever yk_analyze left there, and
    the getters run the stages it did not (stage by stage).  r1_fused: yk_analyze coded R1, its streams are fetched as they
    are first; r1_without_dst: R1 is also fetched once without a write-back plane when it was not fused; r1_dst: then
    each plane is coded again with the write-back plane (this replaces the fused streams)."""
    c, h, w = planes.shape
    o = Oracle(planes)
    do_alpha = "alpha" in stages and c == 4
    do_grad = "grad" in stages
    do_r2 = "r2" in stages
    do_r1 = "r1" in stages or "r1_3bit" in stages
    if do_alpha:
        want = o.alpha()
        if want is not None:
            got = ctx.alpha_reject(slot)
            assert got["bound"] == want["bound"], ("alpha bound", got["bound"], want["bound"])
            assert got["remaining"] == want["remaining"]
            assert got["wrote"] == want["wrote"]
            assert got["chunk_bbox"] == want["chunk_bbox"]
            _eq(got["bitmap"], want["bitmap"], "alpha bitmap")
    if do_grad:
        for k, (sx, sy) in enumerate(PASS_ORDER):
            want = o.gradient_pass(sx, sy, reject=reject)
            got = ctx.gradient_pass(sx, sy, slot, reject=reject)
            assert got["tiledone"] == want["tiledone"], (f"pass {k} tileDone", got["tiledone"], want["tiledone"])
            _eq(got["bitmap"], want["bitmap"], f"pass {k} bitmap")
            assert got["bbox"] == want["bbox"], (f"pass {k} bbox", got["bbox"], want["bbox"])
            _eq(got["rgb"], want["rgb"], f"pass {k} rgbStream")
    if do_r2:
        for n in range(3):
            want = o.range1d(n)
            got = ctx.range1d(n, slot)
            _eq(got["type"], want["type"], f"R2 type plane {n}")
            _eq(got["idx"], want["idx"], f"R2 idx plane {n}")
    if state and do_grad:
        s = ctx.download_state(slot)
        _eq(s["smoothMap"].ravel(), o.state(0), "smoothMap")
        _eq(s["mipmapMask"].ravel(), o.state(1), "mipmapMask")
        for n in range(3):
            _eq(s["mapSmoothTile"][n].ravel(), o.state(2 + n), f"mapSmoothTile{n}")
            _eq(s["mappedRGB"][n].ravel(), o.state(5 + n), f"mappedRGB{n}")
            _eq(s["recon"][n].ravel(), o.state(8 + n), f"recon{n}")
    if do_r1:
        wants = [o.range_dyn(n, mode3="r1_3bit" in stages, want_dst=True) for n in range(3)]
        if r1_fused or r1_without_dst:        # the streams yk_analyze left on the device / coded without a write-back plane
            what = "fused R1" if r1_fused else "R1 without dst"
            for n in range(3):
                got = ctx.range_dyn(n, mode3="r1_3bit" in stages, slot=slot, want_dst=False)
                assert got["constraint"] == wants[n]["constraint"]
                _eq(got["defs"], wants[n]["defs"], f"{what} defs plane {n}")
                assert got["n_nibbles"] == wants[n]["n_nibbles"]
                _eq(got["nibbles"], wants[n]["nibbles"], f"{what} nibbles plane {n}")
        for n in range(3 if r1_dst else 0):
            want = wants[n]
            got = ctx.range_dyn(n, mode3="r1_3bit" in stages, slot=slot, want_dst=True)
            assert got["constraint"] == want["constraint"]
            _eq(got["defs"], want["defs"], f"R1 defs plane {n}")
            assert got["n_nibbles"] == want["n_nibbles"]
            _eq(got["nibbles"], want["nibbles"], f"R1 nibbles plane {n}")
            _eq(got["dst"], want["dst"], f"R1 dst plane {n}")
    o.close()


def check_chroma(ctx: "capi.Context", planes: np.ndarray, pre, cfg, modes, slot=0, load=None):
    """The chroma front-end (yk_chroma_prepare + yk_range_dyn_chroma x3) after the stages in `pre`, against the oracle.
    load: as in check_image."""
    c, h, w = planes.shape
    o = Oracle(planes)
    if load is None:
        ctx.set_image(planes, slot)
    else:
        load(ctx, planes, slot)
    st = (capi.STAGE_ALPHA if ("alpha" in pre and c == 4) else 0) | (capi.STAGE_GRADIENT if "grad" in pre else 0)
    if st:
        ctx.analyze(st, slot0=slot)
    if "alpha" in pre and c == 4:
        o.alpha()
    if "grad" in pre:
        o.gradient_cascade()
    want = o.chroma(cfg, modes)
    got = ctx.chroma(cfg, modes, slot=slot)
    for k in ("Y", "workCo", "workCg"):
        _eq(got[k], want[k], "chroma plane " + k)
    for n in range(3):
        g, wnt = got["coded"][n], want["coded"][n]
        assert g["constraint"] == wnt["constraint"], (n, g["constraint"], wnt["constraint"])
        _eq(g["defs"], wnt["defs"], f"chroma R1 defs {n}")
        assert g["n_nibbles"] == wnt["n_nibbles"]
        _eq(g["nibbles"], wnt["nibbles"], f"chroma R1 nibbles {n}")
        _eq(g["dst"], wnt["dst"], f"chroma R1 dst {n}")
    o.close()
