"""Tile-row strips: one large image analysed by several contexts / GPUs (SURVEY.md §8e, BASELINE.json configs[3]).

The reference walks an image on one thread; FittingQuadSmooth's results only couple neighbouring tile rows through
(i) the clamped bottom corner samples of a tile row and (ii) the ownership of the lattice points on the shared row.
So an image is cut into strips of whole 64-row swizzle blocks, each strip is an ordinary image of its own context
(``yk_strip_config``), and two small device-to-device copies per strip boundary are all the communication there is:

    exchange 1   first pixel row of strip k+1  ->  halo of strip k          (before ``yk_strip_phase 0``)
    exchange 2   boundary touch words, both directions                       (between phase 0 and phase 1)

DynamicTileEncode (R1) of R, G, B needs no halo: after phase 0 each strip codes the blocks of the image's walk whose top
row it holds (``yk_strip_range_dyn``, with the strip set's merged alpha box for RGBA), and its streams are its slice of
the image's.

Host logic here: the partition, the order of the steps, and the merge of the per-strip results into the image's streams
(bitmaps are consecutive byte ranges, rgb / range streams concatenate in strip order, TileDone adds, boxes merge).
Transports: ``LocalTransport`` (all strips driven by this process: direct peer copies), ``DistTransport`` (one strip per
``torch.distributed`` rank; "ipc" = CUDA IPC handle + peer copy over NVLink, "host" = staged through host memory with
point-to-point send/recv — the form the gloo CPU tests use).  No collective touches the data path.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import capi

BLOCK = 64          # largest swizzle block (include/YAIK_private.h:212-276): strips start on multiples of it


def strip_rows(img_h: int, n: int):
    """[(y0, h)] of at most n strips covering img_h rows: whole 64-row blocks, as even as possible, the last strip takes
    the remainder.  Fewer than n strips come back when the image has fewer blocks."""
    blocks = (img_h + BLOCK - 1) // BLOCK
    n = max(1, min(n, blocks))
    out, b0 = [], 0
    for i in range(n):
        nb = blocks // n + (1 if i < blocks % n else 0)
        y0, y1 = b0 * BLOCK, min(img_h, (b0 + nb) * BLOCK)
        out.append((y0, y1 - y0))
        b0 += nb
    return out


def collect_results(ctx: "capi.Context", slot=0, r2=True, r1=0):
    """Per-strip results through the ordinary getters (after phase 1).  r1 = STAGE_RANGEDYN / STAGE_RANGEDYN3: also the
    strip's DynamicTileEncode streams of R, G, B in that mode (res["r1"], one Context.range_dyn dict per plane)."""
    res = {"passes": [], "r2": []}
    for sx, sy in capi.PASS_ORDER:
        res["passes"].append(ctx.gradient_pass(sx, sy, slot))
    if r2:
        for p in range(3):
            res["r2"].append(ctx.range1d(p, slot))
    if r1:
        res["r1"] = [ctx.range_dyn(p, mode3=r1 == capi.STAGE_RANGEDYN3, slot=slot) for p in range(3)]
    return res


def merged_box(parts):
    """The image's alpha box from the strips' (bound, kept-tile count) pairs: None when no strip kept a tile."""
    boxes = [b for b, n in parts if n > 0]
    if not boxes:
        return None
    return [min(b[0] for b in boxes), min(b[1] for b in boxes), max(b[2] for b in boxes), max(b[3] for b in boxes)]


def merge_alpha(lib, parts, w, h):
    """MipPrefilter's results for the whole image from the strips' per-tile alpha results (Context.alpha_kept, strip order):
    the arrays stack (a strip is a whole number of 16-row tiles, except the last), the boxes merge, the bitmap / remaining
    pixels / chunk box come from yk_alpha_assemble (EC.cpp:1287-1403)."""
    kept = np.ascontiguousarray(np.concatenate([p["kept"] for p in parts], axis=0))
    bound = merged_box([(p["bound"], p["count"]) for p in parts])
    if bound is None:
        return None                                  # fully transparent: outside the reference's domain
    th, tw = kept.shape
    bm = np.zeros(tw * th // 8 + 8, np.uint8)
    nb, rem, wrote = C.c_int(), C.c_int(), C.c_int()
    cb = (C.c_int * 4)()
    rc = lib.yk_alpha_assemble(kept.ctypes.data_as(C.c_void_p), tw, th, w, h, (C.c_int * 4)(*bound), bm.ctypes.data_as(C.c_void_p), bm.size,
                               C.byref(nb), C.byref(rem), C.byref(wrote), cb)
    if rc:
        raise capi.YaikError(rc, "yk_alpha_assemble")
    return dict(bitmap=bm[:nb.value].copy(), bound=bound, remaining=rem.value, wrote=wrote.value, chunk_bbox=list(cb) if wrote.value else [])


def merge_results(parts):
    """Image-level streams from the strips' (in strip order): what one context would have returned for the whole image."""
    out = {"passes": [], "r2": []}
    for k in range(len(capi.PASS_ORDER)):
        ps = [p["passes"][k] for p in parts]
        out["passes"].append(dict(
            bitmap=np.concatenate([p["bitmap"] for p in ps]),
            rgb=np.concatenate([p["rgb"] for p in ps]),
            tiledone=int(sum(p["tiledone"] for p in ps)),
            bbox=[min(p["bbox"][0] for p in ps), min(p["bbox"][1] for p in ps), max(p["bbox"][2] for p in ps), max(p["bbox"][3] for p in ps)]))
    if parts and parts[0]["r2"]:
        for pl in range(3):
            out["r2"].append(dict(idx=np.concatenate([p["r2"][pl]["idx"] for p in parts]),
                                  type=np.concatenate([p["r2"][pl]["type"] for p in parts])))
    if parts and parts[0].get("r1"):
        out["r1"] = []
        for pl in range(3):
            rs = [p["r1"][pl] for p in parts]
            # a strip codes whole 4x4 cells: its nibbles fill whole bytes, so the strips' bytes concatenate unshifted
            assert all(r["n_nibbles"] % 2 == 0 for r in rs), [r["n_nibbles"] for r in rs]
            assert all(r["constraint"] == rs[0]["constraint"] for r in rs), [r["constraint"] for r in rs]
            out["r1"].append(dict(nibbles=np.concatenate([r["nibbles"] for r in rs]), n_nibbles=int(sum(r["n_nibbles"] for r in rs)),
                                  defs=np.concatenate([r["defs"] for r in rs]), dst=None, constraint=list(rs[0]["constraint"])))
    return out


class LocalTransport:
    """Every strip is driven by this process (one or several GPUs): the halo pointers are used directly."""

    def __init__(self, ctxs):
        self.ctxs = ctxs

    def run_device_flags(self, planes: np.ndarray, n_strips=None, reject=3, r2=True, images=1, r1=0):
        """The form without the host in the loop (yk_strips_link / yk_strips_run_stages): every strip enqueues the whole
        image on its stream, the exchanges are ordered by epoch flags in the halos.  `images` > 1 runs the image that many
        times back to back (the last run's results are collected).  r1 = STAGE_RANGEDYN / STAGE_RANGEDYN3: every image
        also codes R1 (RGB only)."""
        c, h, w = planes.shape
        rows = strip_rows(h, n_strips or len(self.ctxs))
        ctxs = self.ctxs[:len(rows)]
        for ctx, (y0, sh) in zip(ctxs, rows):
            ctx.set_image(planes[:, y0:y0 + sh], 0)
            ctx.strip_config(h, y0)
        L = ctxs[0].L
        arr = (C.c_void_p * len(ctxs))(*[ctx.ctx for ctx in ctxs])
        rc = L.yk_strips_link(arr, len(ctxs), 0)
        if rc:
            raise capi.YaikError(rc, "yk_strips_link")
        for _ in range(images):
            rc = L.yk_strips_run_stages(arr, len(ctxs), 0, reject, r1)
            if rc:
                raise capi.YaikError(rc, "yk_strips_run_stages")
        for ctx in ctxs:
            ctx.sync()
        merged = merge_results([collect_results(ctx, r2=r2, r1=r1) for ctx in ctxs])
        if c == 4:
            merged["alpha"] = merge_alpha(L, [ctx.alpha_kept() for ctx in ctxs], w, h)
        return merged

    def run(self, planes: np.ndarray, n_strips=None, reject=3, r2=True, load=None, r1=0):
        """load(ctx, y0, h): puts rows [y0, y0 + h) of the image into slot 0 of ctx (default: yk_set_image of those rows of
        `planes`); e.g. a pointer y0 * rowBytes into one interleaved image, with no copy on the host.
        r1 = STAGE_RANGEDYN / STAGE_RANGEDYN3: DynamicTileEncode of R, G, B after phase 0 (merged["r1"])."""
        c, h, w = planes.shape
        rows = strip_rows(h, n_strips or len(self.ctxs))
        ctxs = self.ctxs[:len(rows)]
        load = load or (lambda ctx, y0, sh: ctx.set_image(planes[:, y0:y0 + sh], 0))
        halos = []
        for ctx, (y0, sh) in zip(ctxs, rows):
            load(ctx, y0, sh)
            ctx.strip_config(h, y0)
            halos.append(ctx.strip_halo())
        # exchange 1: first pixel row of strip k+1 -> halo of strip k
        for k in range(len(rows) - 1):
            src, dst = halos[k + 1], halos[k]
            for p in range(3):
                ctxs[k + 1].copy_async(dst.haloIn + dst.pixelRowInOffset + p * dst.pixelRowStride, src.pixelRowOut[p], src.planeRowBytes)
        for ctx in ctxs:
            ctx.sync()
        for ctx in ctxs:
            ctx.strip_phase(0, reject=reject)
        for ctx in ctxs:
            ctx.sync()
        alpha = None
        if r1:
            if c == 4:          # the image's alpha box: a reduction over every strip
                alpha = merge_alpha(ctxs[0].L, [ctx.alpha_kept() for ctx in ctxs], w, h)
            for ctx in ctxs:
                ctx.strip_range_dyn(mode3=r1 == capi.STAGE_RANGEDYN3, bound=alpha["bound"] if alpha else None)
        # exchange 2: boundary touch words, both directions
        for k in range(len(rows) - 1):
            up, lo = halos[k], halos[k + 1]
            ctxs[k].copy_async(lo.haloIn + lo.touchInTopOffset, up.touchOutBottom, up.touchBytes)
            ctxs[k + 1].copy_async(up.haloIn + up.touchInBottomOffset, lo.touchOutTop, lo.touchBytes)
        for ctx in ctxs:
            ctx.sync()
        for ctx in ctxs:
            ctx.strip_phase(1, reject=reject)
        merged = merge_results([collect_results(ctx, r2=r2, r1=r1) for ctx in ctxs])
        if c == 4:
            merged["alpha"] = alpha or merge_alpha(ctxs[0].L, [ctx.alpha_kept() for ctx in ctxs], w, h)
        return merged


class DistTransport:
    """One strip per torch.distributed rank (ranks >= number of strips idle).  mode "ipc": the halo buffer of the
    neighbour is mapped through a CUDA IPC handle and written with a peer copy (NVLink); mode "host": the two exchanges
    are staged through host memory and sent point to point (works on any backend, used by the gloo tests)."""

    def __init__(self, ctx: "capi.Context", dist, mode="ipc"):
        self.ctx, self.dist, self.mode = ctx, dist, mode
        self.rank, self.world = dist.get_rank(), dist.get_world_size()

    def _sendrecv_host(self, send_to, data, recv_from, nbytes):
        """Point-to-point: send `data` (uint8 array or None) to rank send_to, receive nbytes from recv_from (or None)."""
        import torch
        reqs, got = [], None
        if send_to is not None:
            reqs.append(self.dist.isend(torch.from_numpy(np.ascontiguousarray(data)), dst=send_to))
        if recv_from is not None:
            buf = torch.empty(nbytes, dtype=torch.uint8)
            reqs.append(self.dist.irecv(buf, src=recv_from))
            got = buf
        for r in reqs:
            r.wait()
        return None if got is None else got.numpy()

    def run(self, my_planes, img_h, rows, reject=3, r2=True, r1=0):
        """rows = strip_rows(img_h, world); my_planes = this rank's rows (or None if the rank has no strip).
        r1 = STAGE_RANGEDYN / STAGE_RANGEDYN3: DynamicTileEncode of R, G, B after phase 0, in the box gathered from every
        strip's alpha results (RGBA).  Returns the merged result on rank 0, None elsewhere."""
        dist, ctx, rank = self.dist, self.ctx, self.rank
        n = len(rows)
        active = rank < n
        halo = None
        if active:
            y0, sh = rows[rank]
            ctx.set_image(my_planes, 0)
            ctx.strip_config(img_h, y0)
            halo = ctx.strip_halo()
        above = rank - 1 if active and rank > 0 else None
        below = rank + 1 if active and rank + 1 < n else None
        peers = {}
        if self.mode == "ipc":
            handles = [None] * self.world
            dist.all_gather_object(handles, ctx.ipc_export(halo.haloIn) if active else None)      # control plane only
            for r in (above, below):
                if r is not None:
                    peers[r] = ctx.ipc_open(handles[r])
        # ---- exchange 1: my first pixel row -> halo of the strip above
        if self.mode == "ipc":
            if above is not None:
                for p in range(3):
                    ctx.copy_async(peers[above] + halo.pixelRowInOffset + p * halo.pixelRowStride, halo.pixelRowOut[p], halo.planeRowBytes)
            if active:
                ctx.sync()
            dist.barrier()
        else:
            mine = None
            if above is not None:
                mine = np.concatenate([ctx.copy_to_host(halo.pixelRowOut[p], halo.planeRowBytes) for p in range(3)])
            got = self._sendrecv_host(above, mine, below, 3 * halo.planeRowBytes if below is not None else 0)
            if got is not None:
                for p in range(3):
                    ctx.copy_from_host(halo.haloIn + halo.pixelRowInOffset + p * halo.pixelRowStride, got[p * halo.planeRowBytes:(p + 1) * halo.planeRowBytes])
        if active:
            ctx.strip_phase(0, reject=reject)
            ctx.sync()
        if r1:
            # the image's alpha box is a reduction over every strip: gathered on the control plane, like the IPC handles
            mine = None
            if active and my_planes.shape[0] == 4:
                a = ctx.alpha_kept()
                mine = (a["bound"], a["count"])
            boxes = [None] * self.world
            dist.all_gather_object(boxes, mine)
            rgba = any(b is not None for b in boxes)
            if active:
                ctx.strip_range_dyn(mode3=r1 == capi.STAGE_RANGEDYN3, bound=merged_box([b for b in boxes if b is not None]) if rgba else None)
        # ---- exchange 2: boundary touch words, both directions
        if self.mode == "ipc":
            if above is not None:
                ctx.copy_async(peers[above] + halo.touchInBottomOffset, halo.touchOutTop, halo.touchBytes)
            if below is not None:
                ctx.copy_async(peers[below] + halo.touchInTopOffset, halo.touchOutBottom, halo.touchBytes)
            if active:
                ctx.sync()
            dist.barrier()
        else:
            top = ctx.copy_to_host(halo.touchOutTop, halo.touchBytes) if above is not None else None
            bot = ctx.copy_to_host(halo.touchOutBottom, halo.touchBytes) if below is not None else None
            got_b = self._sendrecv_host(above, top, below, halo.touchBytes if below is not None else 0)     # upwards
            got_t = self._sendrecv_host(below, bot, above, halo.touchBytes if above is not None else 0)     # downwards
            if got_b is not None:
                ctx.copy_from_host(halo.haloIn + halo.touchInBottomOffset, got_b)
            if got_t is not None:
                ctx.copy_from_host(halo.haloIn + halo.touchInTopOffset, got_t)
        part = None
        if active:
            ctx.strip_phase(1, reject=reject)
            part = collect_results(ctx, r2=r2, r1=r1)
        for r, ptr in peers.items():
            ctx.ipc_close(ptr)
        parts = [None] * self.world
        dist.all_gather_object(parts, part)         # host-side result assembly (what the reference's chunk writers would consume)
        return merge_results([p for p in parts[:n]]) if rank == 0 else None
