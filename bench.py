#!/usr/bin/env python
"""bench.py — encoded megapixels/s of the YAIK encoder-analysis stage (alpha-zero tile rejection + 7 gradient passes
+ 8x8 range stage R2) on B200, with the HBM roofline of the dominant kernel and the reference CPU encoder timed on
the same box.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

One "step" = one pass of the hot path over one 2048x2048 RGBA synthetic texture (BASELINE.json configs[1]) per GPU,
inputs resident in HBM.  Inputs rotate over 8 distinct resident images (512 MiB of planes > the 126 MB L2) so every
step reads cold data.  N > 1: one process per GPU, every rank analyses its own textures (sharded by image, no
collective on the data path; weak scaling); time = max over ranks.

--dump-outputs DIR: after the timed steps, rank 0 writes the result streams of its last timed step (step K - 1, texture
(K - 1) mod 8) as DIR/<name>.npy, see dump_outputs().  The textures are seeded, so two builds run with the same arguments
can be compared output for output.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

W = H = 2048
CH = 4
NSLOTS = 8
METRIC = "encoded megapixels/sec (gradient+range stages)"
UNIT = "MP/s"
WORKLOAD = "single synthetic 2048x2048 RGBA texture with alpha holes (alpha bitmap + full tile cascade + R2 range stage) per step"
DUMP_LIMIT = 64 << 20          # bytes --dump-outputs may write in all


def base_config(args):
    """`config` of both arms' lines (identical dictionaries, so that lines of the two arms can be compared)."""
    return {"workload": WORKLOAD, "images_per_step_per_gpu": 1, "sharding": "by image, no collective",
            "stages": "MipPrefilter + 7x FittingQuadSmooth + 3x DynamicTileCompressor, results left in HBM",
            "l2": "GPU arm: inputs rotate over 8 distinct resident 64 MiB textures (512 MiB > 126 MB L2), so every step reads cold planes",
            "timed_regions": f"GPU arm: one region of {args.steps} steps bracketed by barrier + synchronize, after an untimed run of the same region"}


def dump_outputs(path, r):
    """Writes what yk_fetch_all returned for one image (Context.fetch_all) as .npy files: per gradient pass k its bitmap
    and rgbStream (pass<k>_bitmap, pass<k>_rgb, float32) and [TileDone, bbox] (pass<k>_tiledone_bbox, float64); per colour
    plane n the R2 streams (r2_idx<n>, r2_type<n>, float32); the alpha stage's bitmap (alpha_bitmap, float32) and
    [bound, remaining, wrote, chunk bbox] (alpha_bound_remaining_wrote_chunk_bbox, float64, chunk bbox zero when no chunk
    was written).  stream_lengths (float64) holds the length of every stream in that order; a stream of length zero (an
    alpha stage that rejects no tile, say) has no file of its own.  Every value is a byte or an int32, so the conversion
    is exact.  Should the files exceed DUMP_LIMIT, every stream is cut to the same share of its elements, drawn with a
    fixed seed."""
    streams, out = {}, {}
    for k, p in enumerate(r["passes"]):
        if p is not None:
            streams[f"pass{k}_bitmap"] = p["bitmap"]
            streams[f"pass{k}_rgb"] = p["rgb"]
            out[f"pass{k}_tiledone_bbox"] = np.array([p["tiledone"], *p["bbox"]], np.float64)
    for n, q in enumerate(r["r2"]):
        streams[f"r2_idx{n}"] = q["idx"]
        streams[f"r2_type{n}"] = q["type"]
    a = r["alpha"]
    if a:
        streams["alpha_bitmap"] = a["bitmap"]
        out["alpha_bound_remaining_wrote_chunk_bbox"] = np.array([*a["bound"], a["remaining"], a["wrote"], *(a["chunk_bbox"] or [0] * 4)], np.float64)
    out["stream_lengths"] = np.array([v.size for v in streams.values()], np.float64)
    room = DUMP_LIMIT - sum(v.nbytes for v in out.values())
    keep = min(1.0, room / (4 * sum(v.size for v in streams.values()) or 1))
    rng = np.random.default_rng(0)
    for name, v in streams.items():
        if v.size and keep < 1.0:      # over the limit: the same fixed, seeded share of every stream, in stream order
            v = v[np.sort(rng.choice(v.size, int(v.size * keep), replace=False))]
        if v.size:
            out[name] = v.astype(np.float32)
    os.makedirs(path, exist_ok=True)
    for name, v in out.items():
        np.save(os.path.join(path, name + ".npy"), v)


def results_digest(r) -> str:
    """SHA-1 over everything yk_fetch_all returned for one image (the same fields tests/parity.py digests)."""
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


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def sample(self):
        if not self.nv:
            return
        nv = self.nv
        try:
            self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
                     0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting"}
            for bit, n in names.items():
                if r & bit:
                    self.reasons.add(n)
        except Exception:
            pass

    def run(self):
        while not self.stop_flag:
            self.sample()
            time.sleep(0.004)

    def result(self):
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(s)}


def physical_gpu_index(local):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local])
        except Exception:
            return local
    return local


# ------------------------------------------------------------------------------------------------ reference arm
def cpu_reference_run(planes, stages, reps):
    """Run the compiled, unmodified reference (oracle/_ref) or, if absent, the oracle port; returns (seconds per
    image for alpha+gradient+range, kind)."""
    from refrun import have_ref, run_ref
    if have_ref():
        r = run_ref(planes, stages, reps=reps, timeout=3600)
        t = r["time.seconds"]
        return float(t[0] + t[1] + t[2]), "reference"
    from oracle_py import Oracle
    t0 = time.perf_counter()
    for _ in range(reps):
        o = Oracle(planes)
        if planes.shape[0] == 4 and "alpha" in stages:
            o.alpha()
        o.gradient_cascade()
        for p in range(3):
            o.range1d(p)
        o.close()
    return (time.perf_counter() - t0) / reps, "port"


_REF_IMG = {}


def _ref_worker(args):
    """One encoder process: returns the seconds the reference spent in MipPrefilter + 7x FittingQuadSmooth (with its host
    tail) + 3x DynamicTileCompressor, measured inside the process around the member calls (no image generation, no I/O)."""
    side, seed = args
    if (side, seed) not in _REF_IMG:
        from yaik_b200.synth import make_image
        _REF_IMG.clear()
        _REF_IMG[(side, seed)] = make_image(side, side, CH, seed)
    t, kind = cpu_reference_run(_REF_IMG[(side, seed)], ("alpha", "grad", "r2"), 1)
    return t, kind


def run_reference_arm(args):
    """--impl reference: the reference's own CPU implementation of the path on the host cores, all of them (the
    reference is single-threaded, so one independent encoder process per core, each on its own texture)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    from yaik_b200.synth import SEED_BASE
    cores = max(1, min(os.cpu_count() or 1, 64))
    total_steps = args.steps + args.warmup
    budget = 150.0 / max(1, total_steps)                # seconds per step so that the whole run ends within minutes
    side = 2048
    while side > 64 and (side * side / 2.0e6) * 1.3 > budget:      # ~2 MP/s per core measured for the reference
        side //= 2
    with mp.get_context("spawn").Pool(cores) as pool:
        work = [(side, SEED_BASE + 1 + i) for i in range(cores)]
        for _ in range(max(1, args.warmup)):
            pool.map(_ref_worker, work, chunksize=1)
        dt = 0.0
        kind = "port"
        for _ in range(args.steps):
            res = pool.map(_ref_worker, work, chunksize=1)      # all cores busy at once; a step lasts as long as its slowest encoder
            kind = res[0][1]
            dt += max(r[0] for r in res)
    mp_per_step = cores * side * side / 1e6
    value = mp_per_step * args.steps / dt
    sample = (f"{cores} independent encoder processes per step, each one {side}x{side} RGBA synthetic texture "
              f"({'full configs[1] size' if side == 2048 else 'crop-sized sample of configs[1]'}); step time = slowest encoder's in-process stage time")
    line = {"impl": "reference", "metric": METRIC, "value": round(value, 3), "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(1e3 * dt / args.steps, 3), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "config": base_config(args), "sample_side": side,
            "cpu_baseline": {"value": round(value, 3), "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": round(value, 3), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ strips (configs[3])
def _stream_digests(res):
    """Lengths + SHA-1 of every stream of one strip (7 bitmaps, 7 rgbStreams, 3 + 3 range streams) and its counters."""
    import hashlib
    out = []
    for p in res["passes"]:
        out.append(("bitmap", int(p["bitmap"].size), hashlib.sha1(p["bitmap"].tobytes()).hexdigest()))
        out.append(("rgb", int(p["rgb"].size), hashlib.sha1(p["rgb"].tobytes()).hexdigest()))
    for q in res["r2"]:
        out.append(("idx", int(q["idx"].size), hashlib.sha1(q["idx"].tobytes()).hexdigest()))
        out.append(("type", int(q["type"].size), hashlib.sha1(q["type"].tobytes()).hexdigest()))
    return out, [(p["tiledone"], list(p["bbox"])) for p in res["passes"]]


def run_strips(args, torch, dist, lib, rank, world, local, steps, warmup):
    """One side x side RGB image (a seeded 2048x2048 texture tiled over the plane) in tile-row strips, one strip per rank /
    GPU, int32 planes resident in HBM.  Every rank enqueues whole images on its stream (yk_strip_run): the halo exchanges
    are NVLink peer copies into the neighbour's halo (CUDA IPC mapping) ordered by epoch flags on the device - no host
    barrier inside the timed region, no collective on the data path.  Returns the result dictionary on rank 0."""
    import hashlib
    from yaik_b200 import capi, strips
    from yaik_b200.synth import make_image, SEED_BASE
    side = args.strips_side
    rows = strips.strip_rows(side, world)
    active = rank < len(rows)
    base = make_image(2048, 2048, 3, SEED_BASE + 3)
    reps = (side + 2047) // 2048

    def rows_of(y0, sh):
        return np.ascontiguousarray(np.tile(base, (1, reps, reps))[:, y0:y0 + sh, :side])

    # Two strip sets per rank on the same resident planes (own contexts, streams, halos and flags): consecutive images
    # alternate between them, so the ownership / emission kernels of one image run beside the analysis of the next.
    NSETS = 2
    ctxs, halos, sts = [], [], []
    if active:
        y0, sh = rows[rank]
        for k in range(NSETS):
            c = capi.Context(side, sh, planes=3, slots=1, device=local, lib=lib)
            stream_k = torch.cuda.Stream(device=local)
            c.set_stream(stream_k.cuda_stream)
            c.set_upload_format(False)
            if k == 0:
                c.set_image(rows_of(y0, sh), 0)
                c.sync()
            else:
                c.set_image_device([ctxs[0].device_plane(0, p) for p in range(3)], 3, side, sh, 0)
            c.strip_config(side, y0)
            ctxs.append(c); halos.append(c.strip_halo()); sts.append(stream_k)
    ctx = ctxs[0] if active else None
    halo = halos[0] if active else None
    st = sts[0] if active else torch.cuda.Stream(device=local)
    peers = [dict() for _ in range(NSETS)]
    if dist is not None:
        handles = [None] * world
        dist.all_gather_object(handles, [c.ipc_export(h.haloIn) for c, h in zip(ctxs, halos)] if active else None)      # control plane only
        for k in range(NSETS):
            for r in (rank - 1, rank + 1):
                if active and 0 <= r < len(rows):
                    peers[k][r] = ctxs[k].ipc_open(handles[r][k])
        dist.barrier()                                   # every halo is cleared before a neighbour writes into it
    for k in range(NSETS if active else 0):
        ctxs[k].strip_set_peers(peers[k].get(rank - 1), peers[k].get(rank + 1))

    def barrier():
        torch.cuda.synchronize(local)
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(local)

    def run_images(n, nsets):
        for i in range(n):
            if active:
                ctxs[i % nsets].strip_run()

    run_images(max(4, warmup), NSETS)
    barrier()
    sampler = ClockSampler(physical_gpu_index(local))
    sampler.sample(); sampler.start()

    def timed(n, nsets):
        ev0, ev1, j = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True), torch.cuda.Event()
        ev0.record(st)
        if active and nsets > 1:
            sts[1].wait_event(ev0)
        run_images(n, nsets)
        if active and nsets > 1:
            j.record(sts[1]); st.wait_event(j)
        ev1.record(st)
        barrier()
        t_ms = ev0.elapsed_time(ev1)
        if dist is not None:
            t = torch.tensor([t_ms], device=f"cuda:{local}", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            t_ms = float(t.item())
        return t_ms

    # CTAs of the strips' analysis launches, calibrated before the timed run with all ranks running: a launch that takes
    # every SM leaves none for the other set's ownership / emission kernels (a resident analysis CTA holds an SM's whole
    # shared memory), so the two sets take turns instead of overlapping; a launch a little narrower lasts longer but
    # runs beside them.  Pays when a strip's analysis is short (many GPUs), not when it dominates.
    sms = ctx.sm_count() if active else 0
    cal = {}
    cands = [0] if args.strips_ctas >= 0 else [0, sms * 7 // 8, sms * 3 // 4, sms * 5 // 8]
    if args.strips_ctas > 0:
        cands = [args.strips_ctas]
    best = cands[0]
    if len(cands) > 1:
        for n_ctas in cands:
            for c in ctxs:
                c.set_analysis_ctas(n_ctas)
            run_images(2, NSETS)
            barrier()
            cal[n_ctas] = timed(max(4, steps // 2), NSETS) / max(4, steps // 2)
        best = min(cal, key=cal.get)
    for c in ctxs:
        c.set_analysis_ctas(best)
    run_images(2, NSETS)
    barrier()
    ms = timed(steps, NSETS)                             # throughput: images pipelined over the two sets
    ms_single = timed(max(2, steps // 2), 1)             # one set: every image waits for the one before it
    sampler.stop_flag = True; sampler.sample()
    # ---- parity: the strips' streams against one context analysing the whole image (rank 0's GPU), compared through
    # lengths + SHA-1 per stream per strip (the merged streams are the strips' streams one after the other)
    mine = _stream_digests(strips.collect_results(ctx)) if active else None
    parts = [mine]
    if dist is not None:
        parts = [None] * world
        dist.all_gather_object(parts, mine)
    result = None
    if rank == 0:
        whole = capi.Context(side, side, planes=3, slots=1, device=local, lib=lib)
        whole.set_upload_format(False)
        whole.set_image(rows_of(0, side), 0)
        whole.analyze(capi.STAGE_GRADIENT | capi.STAGE_RANGE1D)
        ref = strips.collect_results(whole)
        whole.close()
        streams = []
        for p in ref["passes"]:
            streams += [p["bitmap"], p["rgb"]]
        for q in ref["r2"]:
            streams += [q["idx"], q["type"]]
        offs = [0] * len(streams)
        ok = True
        for part in parts[:len(rows)]:
            for k, (kind, n, sha) in enumerate(part[0]):
                seg = streams[k][offs[k]:offs[k] + n]
                ok = ok and seg.size == n and hashlib.sha1(seg.tobytes()).hexdigest() == sha
                offs[k] += n
        ok = ok and all(offs[k] == streams[k].size for k in range(len(streams)))
        for k, p in enumerate(ref["passes"]):
            ok = ok and p["tiledone"] == sum(part[1][k][0] for part in parts[:len(rows)])
        if not ok:
            raise SystemExit("bench.py: the strips' streams differ from the whole-image run")
        mp = side * side / 1e6
        result = {"metric": METRIC, "value": round(mp * steps / (ms / 1e3), 1), "unit": UNIT, "n_gpus": world, "steps": steps, "ms_per_image": round(ms / steps, 4),
                  "ms_per_image_unpipelined": round(ms_single / max(2, steps // 2), 4),
                  "analysis_ctas": int(best) if best else "one per SM", "analysis_ctas_calibration_ms_per_image": {str(k): round(v, 4) for k, v in cal.items()},
                  "pipelining": "consecutive images alternate between two strip sets per GPU (same resident planes): ownership / emission of one image runs beside the analysis of the next",
                  "workload": f"one {side}x{side} synthetic RGB image in {len(rows)} tile-row strips, one GPU each (BASELINE.json configs[3])",
                  "scaling": "strong", "halo_bytes_per_boundary": int(3 * halo.planeRowBytes + 2 * halo.touchBytes),
                  "exchange": "NVLink P2P copies into the neighbour's halo (CUDA IPC), ordered by epoch flags on the device; no host barrier in the timed region, no collective",
                  "parity_checked": True, "parity_against": "one context analysing the whole image (itself compared with the oracle at 4096x16384 in tests/)",
                  "clocks": sampler.result()}
    if active:
        for k in range(NSETS):
            for ptr in peers[k].values():
                ctxs[k].ipc_close(ptr)
        for c in reversed(ctxs):
            c.close()
    return result


# ------------------------------------------------------------------------------------------------ GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--e2e-steps", type=int, default=384)
    ap.add_argument("--e2e-threads", type=int, default=8, help="host threads (one context each) the end-to-end steps are pipelined over")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--workload", default="batch", choices=["batch", "strips"],
                    help="batch: configs[1] textures sharded by image (the metric's configuration); strips: one 16384x16384 RGB image in tile-row strips over the ranks (configs[3])")
    ap.add_argument("--strips-side", type=int, default=16384)
    ap.add_argument("--strips-ctas", type=int, default=-1, help="CTAs of a strip's analysis launch (-1: calibrated, 0: one per SM)")
    ap.add_argument("--no-strips", action="store_true", help="N > 1, batch workload: skip the strips sub-measurement echoed in the line")
    ap.add_argument("--no-r1", action="store_true", help="skip the second timed region (the step with DynamicTileEncode behind it)")
    ap.add_argument("--no-other", action="store_true", help="skip the informational timing of the stages outside the metric")
    ap.add_argument("--streams", type=int, default=8, help="contexts/streams the steps are pipelined over (1, 2, 4 or 8)")
    ap.add_argument("--analysis-ctas", type=int, default=-1, help="CTAs of the persistent analysis kernel in the pipelined region (-1: a quarter of the SMs with 8 streams, half with 2-4, else one per SM)")
    ap.add_argument("--roofline-steps", type=int, default=100, help="launches of the separate pass that times the dominant kernel alone")
    ap.add_argument("--no-prewarm", action="store_true", help="skip the clock-settling loop (profiling runs under ncu)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed step as DIR/<name>.npy (batch workload of the GPU arm)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.workload != "batch"):
        ap.error("--dump-outputs: only the GPU arm's batch workload")
    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch
    from yaik_b200 import capi
    from yaik_b200.synth import make_image, SEED_BASE

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)

    lib = capi.load_library()          # fails loudly if the CUDA library is missing: there is no fallback
    if args.workload == "strips":
        res = run_strips(args, torch, dist, lib, rank, world, local, max(1, args.steps), args.warmup)
        if rank == 0:
            line = dict(res, warmup=args.warmup, higher_is_better=True, vs_baseline=None, dtype="int32", data="synthetic",
                        config={"workload": res["workload"]})
            print(json.dumps(line), flush=True)
        if dist is not None:
            dist.destroy_process_group()
        return
    # Textures are independent, so consecutive steps are pipelined over NCTX contexts (one CUDA stream each): while
    # one texture is in its emission / range kernels the next one's analysis kernel already runs.
    NCTX = max(1, args.streams)
    ctxs = [capi.Context(W, H, planes=CH, slots=NSLOTS // NCTX, device=local, lib=lib) for _ in range(NCTX)]
    streams = [torch.cuda.Stream(device=local) for _ in range(NCTX)]
    for c, st in zip(ctxs, streams):
        c.set_stream(st.cuda_stream)
        c.set_upload_format(False)     # `value` is measured on int32 planes resident in HBM (the reference's Plane representation)
    sms = ctxs[0].sm_count()
    actas = args.analysis_ctas if args.analysis_ctas >= 0 else (sms // 4 if NCTX >= 8 else (sms // 2 if NCTX > 1 else 0))
    if args.analysis_ctas < 0 and args.steps < 4:      # a timed region of one to three steps cannot fill four quarter-SM launches
        actas = 0 if args.steps <= 1 else sms // args.steps
    for c in ctxs:
        c.set_analysis_ctas(actas)     # launches of neighbouring steps run side by side on disjoint SMs: ramp and tail of one hide behind the others
    ctx, stream = ctxs[0], streams[0]

    # eight distinct textures per rank, one per slot (distinct contents and distinct HBM addresses)
    from concurrent.futures import ThreadPoolExecutor
    with ThreadPoolExecutor(4) as ex:
        imgs = list(ex.map(lambda i: make_image(W, H, CH, SEED_BASE + 1 + 16 * rank + i), range(NSLOTS)))
    for s in range(NSLOTS):
        ctxs[s % NCTX].set_image(imgs[s], s // NCTX)
    STAGES = capi.STAGE_ALPHA | capi.STAGE_GRADIENT | capi.STAGE_RANGE1D

    def step(i):
        c = ctxs[i % NCTX]
        s = (i // NCTX) % (NSLOTS // NCTX)
        c.reset_state(s)
        c.analyze(STAGES, slot0=s)

    def sync_all():
        for c in ctxs:
            c.sync()

    def barrier():
        torch.cuda.synchronize(local)
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(local)

    # untimed: the W warm-up steps asked for, plus enough work for the clocks to settle
    for i in range(max(args.warmup, 3)):
        step(i)
    sync_all()
    t0 = time.perf_counter()
    i = 0
    while not args.no_prewarm and time.perf_counter() - t0 < 0.3:
        for _ in range(50):
            step(i); i += 1
        sync_all()

    lib.yk_profile.argtypes = [C.c_void_p, C.c_int]
    lib.yk_profile_read.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_longlong)]
    sampler = ClockSampler(physical_gpu_index(local))
    joins = [torch.cuda.Event() for _ in streams]
    sampler.sample()
    sampler.start()

    def region(n):
        """n steps, timed from their first launch to the end of the last one on any stream; ms of the slowest rank."""
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)                      # every stream starts after ev0 ...
        for st in streams[1:]:
            st.wait_event(ev0)
        for i in range(n):
            step(i)
        for st, j in zip(streams[1:], joins[1:]):
            j.record(st)
            stream.wait_event(j)                # ... and ev1 is recorded after all of them have finished
        ev1.record(stream)
        sampler.sample()
        barrier()
        t_ms = ev0.elapsed_time(ev1)
        if dist is not None:                    # a region lasts as long as its slowest rank
            t = torch.tensor([t_ms], device=f"cuda:{local}", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            t_ms = float(t.item())
        return t_ms

    # untimed: the same region once more, so that the timed one is not the first run of the event / stream-wait path
    # (the first of several regions measured slower than the others)
    region(args.steps)
    launches0 = sum(c.launch_count() for c in ctxs)
    ms = region(args.steps)
    launches = sum(c.launch_count() for c in ctxs) - launches0
    sampler.stop_flag = True
    sampler.sample()
    last = args.steps - 1                       # the results of the last timed step, before anything else runs on its slot
    dumped = ctxs[last % NCTX].fetch_all((last // NCTX) % (NSLOTS // NCTX)) if args.dump_outputs and rank == 0 else None
    # informational: the kernels' durations inside a pipelined pass (they overlap each other there).  A pass of its own,
    # after the timed regions: the event pair the library records around every launch is host work and two more stream
    # operations per kernel, and the timed region holds the product's own launches only.
    for c in ctxs:
        lib.yk_profile(c.ctx, 1)
    for i in range(max(args.steps, 2 * NCTX)):
        step(i)
    sync_all()
    kms = (C.c_double * 8)(); kcnt = (C.c_longlong * 8)()
    for c in ctxs:
        a = (C.c_double * 8)(); b = (C.c_longlong * 8)()
        lib.yk_profile_read(c.ctx, a, b)
        lib.yk_profile(c.ctx, 0)
        for k in range(8):
            kms[k] += a[k]; kcnt[k] += b[k]
    mp_per_step = W * H / 1e6

    # ---- parity of what was just timed: every context's streams (as left by the last timed step on it) against an untimed
    # run of the same texture on a fresh context with one CTA per SM (the configuration tests/test_gpu_parity.py compares
    # with the oracle at this size).  A mismatch fails the run.
    sync_all()
    got = [results_digest(ctxs[s % NCTX].fetch_all(s // NCTX)) for s in range(NSLOTS)]
    cref = capi.Context(W, H, planes=CH, slots=1, device=local, lib=lib)
    cref.set_upload_format(False)
    want = []
    for s in range(NSLOTS):
        cref.set_image(imgs[s], 0)
        cref.analyze(STAGES)
        want.append(results_digest(cref.fetch_all(0)))
    cref.close()
    if got != want:
        raise SystemExit(f"bench.py: results of the timed configuration differ from the single-context run: {got} vs {want}")
    parity_checked = True
    value = world * mp_per_step * args.steps / (ms / 1e3)

    # algorithmic bytes per image (SURVEY.md §8d): every input plane read once + every emitted pre-entropy stream
    rb = ctx.result_bytes(0)
    alg_bytes = 4 * CH * W * H + sum(rb)
    peak, peak_src = peaks()
    names = ["analyze", "emit", "owner"]
    kern_ms_pipe = {n: (kms[i] / kcnt[i] if kcnt[i] else None) for i, n in enumerate(names)}
    # the dominant kernel timed ALONE (one stream, one CTA per SM, event pair around every launch, inputs rotating over the
    # resident textures so they come from HBM): in the pipelined region above launches of several steps overlap on the
    # device, so their individual durations say nothing about the kernel
    roof = None
    if args.roofline_steps > 0:
        sync_all()
        for c in ctxs:
            c.set_analysis_ctas(0)
            lib.yk_profile(c.ctx, 1)
        for i in range(args.roofline_steps):
            step(i)
            ctxs[i % NCTX].sync()
        akms = (C.c_double * 8)(); akcnt = (C.c_longlong * 8)()
        for c in ctxs:
            a = (C.c_double * 8)(); b = (C.c_longlong * 8)()
            lib.yk_profile_read(c.ctx, a, b)
            lib.yk_profile(c.ctx, 0)
            for k in range(8):
                akms[k] += a[k]; akcnt[k] += b[k]
        kern_ms = {n: (akms[i] / akcnt[i] if akcnt[i] else None) for i, n in enumerate(names)}
        dom = kern_ms["analyze"]
        if dom:
            ach = alg_bytes / (dom * 1e-3) / 1e9
            roof = {"bound": "hbm", "kernel": "yk_k_analyze", "achieved": round(ach, 1), "peak": peak, "unit": "GB/s", "frac": round(ach / peak, 4),
                    "traffic": None, "traffic_source": None, "peak_source": peak_src + ", burst copy figure (kernel timed alone)", "algorithmic_bytes_per_launch": alg_bytes,
                    "how": f"{int(akcnt[0])} launches timed alone after the pipelined region: one stream at a time, one CTA per SM, CUDA event pair around each launch",
                    "kernel_ms": {k: (round(v, 5) if v else None) for k, v in kern_ms.items()},
                    "kernel_ms_inside_pipelined_region": {k: (round(v, 5) if v else None) for k, v in kern_ms_pipe.items()},
                    "whole_step_frac": round(alg_bytes / (ms / args.steps * 1e-3) / 1e9 / peak, 4)}
            tp = os.path.join(ROOT, "profiles", "traffic.json")
            if os.path.exists(tp):
                try:
                    tj = json.load(open(tp))
                    roof["traffic"] = tj.get("yk_k_analyze_dram_bytes_per_launch")
                    roof["traffic_source"] = "constant from the committed ncu --set full capture, profiles/traffic.json: " + str(tj.get("source", "r01q"))
                except Exception:
                    pass

    # ---- the same step with DynamicTileEncode (the README's 3 / 4 bits-per-pixel range stage, R1) of R, G, B behind it:
    # one more launch per step (yk_k_r1_encode, three planes), everything left in HBM.  Timed like `value` (one region),
    # then the kernel alone (one step at a time), then its streams compared with the per-plane API path.
    with_r1 = None
    if not args.no_r1:
        STAGES_R1 = STAGES | capi.STAGE_RANGEDYN

        def step_r1(i):
            c = ctxs[i % NCTX]
            s = (i // NCTX) % (NSLOTS // NCTX)
            c.reset_state(s)
            c.analyze(STAGES_R1, slot0=s)

        for c in ctxs:
            c.set_analysis_ctas(actas)
        for i in range(2 * NCTX):
            step_r1(i)
        sync_all()
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        for st in streams[1:]:
            st.wait_event(ev0)
        n_r1 = max(args.steps, 2 * NCTX)
        for i in range(n_r1):
            step_r1(i)
        for st, j in zip(streams[1:], joins[1:]):
            j.record(st)
            stream.wait_event(j)
        ev1.record(stream)
        barrier()
        r1_ms = ev0.elapsed_time(ev1)
        if dist is not None:
            t = torch.tensor([r1_ms], device=f"cuda:{local}", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            r1_ms = float(t.item())
        # the kernel alone: one step at a time, one CTA per SM for the analysis before it
        for c in ctxs:
            c.set_analysis_ctas(0)
            lib.yk_profile(c.ctx, 1)
        for i in range(max(8, args.roofline_steps // 4)):
            step_r1(i)
            ctxs[i % NCTX].sync()
        rk = (C.c_double * 8)(); rc_ = (C.c_longlong * 8)()
        for c in ctxs:
            a = (C.c_double * 8)(); b = (C.c_longlong * 8)()
            lib.yk_profile_read(c.ctx, a, b)
            lib.yk_profile(c.ctx, 0)
            for k in range(8):
                rk[k] += a[k]; rc_[k] += b[k]
        r1_alone_ms = rk[3] / rc_[3] if rc_[3] else None
        # parity of the fused launch: its streams against the per-plane path (yk_range_dyn, which tests/ compare with the oracle)
        fused = [ctxs[0].range_dyn(p) for p in range(3)]
        cchk = capi.Context(W, H, planes=CH, slots=1, device=local, lib=lib)
        cchk.set_upload_format(False)
        cchk.set_image(imgs[0], 0)
        cchk.analyze(STAGES)
        r1_bytes = 0
        for p in range(3):
            single = cchk.range_dyn(p)
            if not (np.array_equal(single["nibbles"], fused[p]["nibbles"]) and np.array_equal(single["defs"], fused[p]["defs"])):
                raise SystemExit("bench.py: DynamicTileEncode streams of the fused launch differ from the per-plane path")
            r1_bytes += 4 * single["n_nibbles"] + single["nibbles"].size + 2 * single["defs"].size
        cchk.close()
        with_r1 = {"value": round(world * mp_per_step * n_r1 / (r1_ms / 1e3), 2), "unit": UNIT, "ms_per_step": round(r1_ms / n_r1, 5), "steps": n_r1,
                   "stages": "MipPrefilter + 7x FittingQuadSmooth + 3x DynamicTileCompressor + 3x DynamicTileEncode (six LUT modes)",
                   "parity_checked": True,
                   "r1_kernel": {"name": "yk_k_r1_encode (R, G, B in one launch)", "ms_alone": round(r1_alone_ms, 5) if r1_alone_ms else None,
                                 "algorithmic_bytes_per_launch": int(r1_bytes),
                                 "bytes_note": "int32 samples of the coded pixels + the nibble and tile-definition streams, three planes",
                                 "hbm_frac": round(r1_bytes / (r1_alone_ms * 1e-3) / 1e9 / peak, 4) if r1_alone_ms else None,
                                 "bound": "instruction issue / latency (six LUT modes per pixel, an ordered float32 sum per block), not HBM"}}

    # ---- end to end through the public C ABI with HOST buffers: pinned int32 planes in (yk_set_image packs them to bytes
    # on the host and uploads those), every result stream out (yk_fetch_all: pinned arena).  Textures are independent, so
    # the steps are pipelined over a few host threads with one context each (upload, analysis and download overlap).
    e2e = None
    if args.e2e_steps > 0:
        lib.yk_host_alloc.restype = C.c_void_p
        nbytes = W * H * 4
        nthr = max(1, args.e2e_threads)
        per = max(1, args.e2e_steps // nthr)
        # the ranks of a box share its host cores: every rank keeps to its own set, so that one rank's packing threads do
        # not migrate over another's
        cores = sorted(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else list(range(os.cpu_count() or 8))
        if world > 1 and len(cores) >= world:
            share = len(cores) // world
            mine_cores = cores[local * share:(local + 1) * share]
            try:
                os.sched_setaffinity(0, mine_cores)
                cores = mine_cores
            except OSError:
                pass
        # host threads that pack the Plane samples: this rank's cores over its worker threads
        os.environ.setdefault("YK_PACK_THREADS", str(max(1, min(8, len(cores) // nthr + 1))))
        ectx = [capi.Context(W, H, planes=CH, slots=1, device=local, lib=lib) for _ in range(nthr)]
        hps = []
        for t in range(nthr):
            hp = [lib.yk_host_alloc(nbytes) for _ in range(CH)]
            for c in range(CH):
                C.memmove(hp[c], imgs[t % NSLOTS][c].ctypes.data, nbytes)
            hps.append(hp)
        moved = [0] * nthr

        def e2e_step(t):
            c = ectx[t]
            c.set_image_ptrs(hps[t], CH, W, H, slot=0)
            c.analyze(STAGES, slot0=0)
            r = c.fetch_all(0, copy=False)
            moved[t] = sum(r.bitmapBytes) + sum(r.rgbBytes) + 3 * (r.r2IdxBytes + r.r2TypeBytes) + ((W // 16) * (H // 16) if CH == 4 else 0)

        def worker(t, n):
            for _ in range(n):
                e2e_step(t)

        def run_threads(n_each):
            t0 = time.perf_counter()
            ths = [threading.Thread(target=worker, args=(t, n_each)) for t in range(nthr)]
            for th in ths:
                th.start()
            for th in ths:
                th.join()
            torch.cuda.synchronize(local)
            return time.perf_counter() - t0

        def set_mix(n_int32):
            """n_int32 of the worker threads upload the int32 planes as they are (plain pinned DMA, 16 B/pixel over PCIe, no
            host work); the others pack to bytes on the host first (4 B/pixel over PCIe, host-memory-bound)."""
            for t, c in enumerate(ectx):
                c.set_upload_format(t >= n_int32)

        # The upload format is chosen from measured throughput on this box, with all ranks running (they share the host):
        # packing wins while there are cores to pack with, the plain DMA wins when a box's cores are spread over many GPUs,
        # and a mix uses the cores and the PCIe link at the same time.
        calib = {}
        for n_int32 in sorted({0, max(1, nthr // 4), nthr // 2, nthr}):
            set_mix(n_int32)
            run_threads(1)
            barrier()
            dt_c = run_threads(3)
            if dist is not None:
                tc = torch.tensor([dt_c], device=f"cuda:{local}", dtype=torch.float64)
                dist.all_reduce(tc, op=dist.ReduceOp.MAX)
                dt_c = float(tc.item())
            calib[n_int32] = world * mp_per_step * 3 * nthr / dt_c
            barrier()
        best = max(calib, key=calib.get)
        set_mix(best)
        run_threads(1)
        barrier()
        dt = run_threads(per)
        if dist is not None:
            t = torch.tensor([dt], device=f"cuda:{local}", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        pitch = (W + 15) // 16 * 16
        h2d = (best * CH * W * H * 4 + (nthr - best) * CH * pitch * H) // nthr
        e2e = {"value": round(world * mp_per_step * per * nthr / dt, 2), "unit": UNIT, "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int(moved[0]), "steps": per * nthr, "host_threads": nthr,
               "upload": f"{nthr - best} of {nthr} worker threads pack the int32 planes to bytes on the host (4 B/pixel over PCIe), {best} upload them as they are (16 B/pixel, pinned DMA)",
               "upload_calibration_mp_s": {f"{k}_int32_threads": round(v, 1) for k, v in sorted(calib.items())},
               "host_cores_per_rank": len(cores),
               "bound": ("host memory bandwidth / cores (packing)" if best == 0 else ("PCIe (int32 DMA)" if best == nthr else "host packing and PCIe together")),
               "what": "per step: yk_set_image from pinned host int32 planes (64 MiB) + yk_analyze + yk_fetch_all (all result streams to pinned "
                       "host memory); wall clock, steps pipelined over host threads with one context each. The reference's host tails "
                       "(PaletteCompressor + ZSTD-18 inside FittingQuadSmooth, about 3 % of the CPU arm's time) are not part of this figure"}
        for c in ectx:
            c.close()
        for hp in hps:
            for p in hp:
                lib.yk_host_free(C.c_void_p(p))

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        reps = 3
        sec, kind = cpu_reference_run(imgs[0], ("alpha", "grad", "r2"), reps)
        cpu = {"value": round(mp_per_step / sec, 3), "unit": UNIT, "cores": 1, "kind": kind,
               "sample": f"the same 2048x2048 RGBA texture, alpha + 7 gradient passes (incl. the reference's host tail) + R2, {reps} repetitions, 1 thread"}

    # ---- stages of the path that are not part of the metric (informational): DynamicTileEncode (R1) per colour plane and the
    # chroma front-end in the CLI's configuration, device time of their kernels (event pairs around each launch)
    other = None
    if rank == 0 and world == 1 and not args.no_other:
        c = capi.Context(W, H, planes=CH, slots=1, device=local, lib=lib)
        c.set_image(imgs[0], 0)
        c.analyze(capi.STAGE_ALPHA | capi.STAGE_GRADIENT | capi.STAGE_RANGE1D)
        c.sync()
        for it in range(4):
            if it == 1:
                lib.yk_profile(c.ctx, 1)
            for p in range(3):
                c.range_dyn(p)
        a = (C.c_double * 8)(); b = (C.c_longlong * 8)()
        lib.yk_profile_read(c.ctx, a, b)
        r1_us = a[3] / b[3] * 1e3 if b[3] else None
        for it in range(4):
            if it == 1:
                lib.yk_profile(c.ctx, 1)
            c.chroma((1, 0, 1, 0), (2, 2), planes=False)
        lib.yk_profile_read(c.ctx, a, b)
        lib.yk_profile(c.ctx, 0)
        other = {"r1_encode_us_per_plane": round(r1_us, 2) if r1_us else None,
                 "chroma_convert_us": round(a[4] / b[4] * 1e3, 2) if b[4] else None,
                 "chroma_encode_us_per_plane": round(a[3] / b[3] * 1e3, 2) if b[3] else None,
                 "what": "kernel device time on the bench texture after the analysis: yk_k_r1_encode (DynamicTileEncode, all six LUT modes) per "
                         "colour plane; yk_k_chroma (RGB -> YCoCg + half-width Co / Cg) and yk_k_r1_encode averaged over Y, Co, Cg. Not in `value`."}
        c.close()

    # ---- N > 1: the other way the path shards (configs[3]): one large image in tile-row strips over the same ranks
    strips_res = None
    if world > 1 and not args.no_strips:
        for c in ctxs:
            c.close()
        ctxs = []
        torch.cuda.empty_cache()
        strips_res = run_strips(args, torch, dist, lib, rank, world, local, 10, 3)

    if rank == 0:
        line = {"metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": round(ms / args.steps, 5), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "int32", "data": "synthetic",
                "config": base_config(args),
                "run": {"pipelining": f"steps are independent textures, issued round-robin on {NCTX} CUDA streams (contexts); analysis launches of {actas or sms} CTAs on {sms} SMs",
                        "kernels_per_step": "yk_k_analyze (persistent, TMA-staged, range stage fused) + yk_k_owner + yk_k_emit",
                        "region_ms": round(ms, 4)},
                "parity_checked": parity_checked,
                "clocks": sampler.result(), "e2e": e2e, "gpu_launches": int(launches), "roofline": roof, "cpu_baseline": cpu,
                "with_r1": with_r1, "strips": strips_res, "stages_outside_metric": other}
        if dumped is not None:
            dump_outputs(args.dump_outputs, dumped)
        print(json.dumps(line), flush=True)
    for c in ctxs:
        c.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
