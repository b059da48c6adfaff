"""Interleaved 8-bit input against int32 Plane input, on one GPU, on bench.py's seeded 2048x2048 RGBA textures.

    python tools/e2e_interleaved.py [--runs 3] [--e2e-steps 192] [--steps 400] [--out FILE]

  e2e (host buffers in, every result stream out; 8 host threads with one context each, as bench.py's e2e figure):
    (a) pinned int32 planes through yk_set_image, packed to bytes on the host (16 B/pixel read from host memory, 4 B over PCIe)
    (b) pinned interleaved RGBA8 through yk_set_image_interleaved (4 B/pixel over PCIe, no host work)
    every step = load + yk_analyze(ALPHA | GRADIENT | RANGE1D) + yk_fetch_all; arms alternate, `--runs` runs each.
  resident input, steps pipelined as bench.py's `value` (8 contexts on 8 streams, analysis launches of a quarter of the SMs):
    (c) int32 planes in HBM: every step = yk_reset_state + yk_analyze
    (d) interleaved RGBA8 textures in HBM: every step = yk_set_image_interleaved_device (the unpack) + yk_analyze
  yk_k_unpack8 alone: its time per launch from yk_profile slot 5, over eight resident textures in turn (134 MB of input, more
    than the 126 MB L2), with its bytes w * h * (channels + nPlanes) over the 6551 GB/s burst-copy peak measured on a B200.
Every arm's results must have the digests of arm (a); the script exits non-zero otherwise.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

W = H = 2048
CH = 4
NTEX = 8
ST_BITS = 1 | 2 | 4          # ALPHA | GRADIENT | RANGE1D
COPY_PEAK_GBS = 6551.0


def gpu_info(index):
    q = "name,power.limit,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", str(index)], capture_output=True, text=True)
    return dict(zip(q.split(","), [v.strip() for v in r.stdout.strip().split(",")])) if r.returncode == 0 else {"error": r.stderr.strip()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--threads", type=int, default=8)
    ap.add_argument("--e2e-steps", type=int, default=192, help="steps of one e2e run (split over the threads)")
    ap.add_argument("--steps", type=int, default=400, help="steps of one resident-input run")
    ap.add_argument("--unpack-launches", type=int, default=400)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()

    import numpy as np
    import torch
    from parity import results_digest
    from yaik_b200 import capi
    from yaik_b200.synth import make_image, SEED_BASE

    lines = []

    def emit(d):
        print(json.dumps(d), flush=True)
        lines.append(d)

    dev = torch.cuda.current_device()
    emit({"gpu": gpu_info(dev), "torch_device": torch.cuda.get_device_name(dev)})
    nthr = args.threads
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 8)
    os.environ.setdefault("YK_PACK_THREADS", str(max(1, min(8, cores // nthr + 1))))      # as bench.py's e2e
    lib = capi.load_library()
    imgs = [make_image(W, H, CH, SEED_BASE + 1 + i) for i in range(NTEX)]          # bench.py's textures (rank 0)
    hwc = [np.ascontiguousarray(np.transpose(im, (1, 2, 0)).astype(np.uint8)) for im in imgs]
    mp = W * H / 1e6
    failures = []

    # ---- e2e: (a) vs (b) ------------------------------------------------------------------------------------------------
    ectx = [capi.Context(W, H, planes=CH, slots=1, lib=lib) for _ in range(nthr)]
    planes_pinned, inter_pinned = [], []
    for t in range(nthr):
        im = imgs[t % NTEX]
        ps = [lib.yk_host_alloc(W * H * 4) for _ in range(CH)]
        for c in range(CH):
            C.memmove(ps[c], im[c].ctypes.data, W * H * 4)
        planes_pinned.append(ps)
        p = lib.yk_host_alloc(W * H * CH)
        C.memmove(p, hwc[t % NTEX].ctypes.data, W * H * CH)
        inter_pinned.append(p)
    want = {}
    digest = {}

    def e2e_step(t, arm):
        c = ectx[t]
        if arm == "a":
            c.set_image_ptrs(planes_pinned[t], CH, W, H)
        else:
            c.set_image_interleaved_ptr(inter_pinned[t], W * CH, CH, CH, W, H)
        c.analyze(ST_BITS)
        c.fetch_all(0, copy=False)

    def e2e_run(arm, per):
        def worker(t):
            for _ in range(per):
                e2e_step(t, arm)
        ths = [threading.Thread(target=worker, args=(t,)) for t in range(nthr)]
        t0 = time.perf_counter()
        for th in ths:
            th.start()
        for th in ths:
            th.join()
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    for c in ectx:
        c.set_upload_format(True)
    per = max(1, args.e2e_steps // nthr)
    res = {"a": [], "b": []}
    for arm in ("a", "b"):
        e2e_run(arm, 1)                                     # warm-up
        for t in range(nthr):
            digest.setdefault(arm, {})[t % NTEX] = results_digest(ectx[t].fetch_all(0))
    want = digest["a"]
    if digest["b"] != want:
        failures.append("e2e (b) digests differ from (a)")
    for r in range(args.runs):
        for arm in ("a", "b"):
            dt = e2e_run(arm, per)
            res[arm].append(round(mp * per * nthr / dt, 1))
    for arm, what in (("a", "pinned int32 planes, yk_set_image packed to bytes on the host"),
                      ("b", "pinned interleaved RGBA8, yk_set_image_interleaved")):
        emit({"arm": arm, "what": what, "mp_s_runs": res[arm], "steps_per_run": per * nthr, "host_threads": nthr,
              "pack_threads_per_context": int(os.environ["YK_PACK_THREADS"]),
              "h2d_bytes_per_step": (W + 15) // 16 * 16 * H * CH if arm == "a" else W * H * CH,
              "host_bytes_read_per_step": W * H * CH * (4 if arm == "a" else 1)})
    for c in ectx:
        c.close()
    for t in range(nthr):
        for p in planes_pinned[t]:
            lib.yk_host_free(p)
        lib.yk_host_free(inter_pinned[t])

    # ---- resident input, pipelined: (c) vs (d) ------------------------------------------------------------------------------
    ctxs = [capi.Context(W, H, planes=CH, slots=1, lib=lib) for _ in range(NTEX)]
    streams = [torch.cuda.Stream() for _ in range(NTEX)]
    dev_hwc = [torch.from_numpy(a).cuda() for a in hwc]
    torch.cuda.synchronize()
    sms = ctxs[0].sm_count()
    for c, s in zip(ctxs, streams):
        c.set_stream(s.cuda_stream)
        c.set_analysis_ctas(sms // 4)

    def load_c():
        for c, im in zip(ctxs, imgs):
            c.set_upload_format(False)
            c.set_image(im)

    def step(i, arm):
        c = ctxs[i % NTEX]
        if arm == "c":
            c.reset_state(0)
        else:
            d = dev_hwc[i % NTEX]
            c.set_image_interleaved_device(d.data_ptr(), d.stride(0), CH, CH, W, H)
        c.analyze(ST_BITS)

    def region(n, arm):
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(streams[0])
        for s in streams[1:]:
            s.wait_event(ev0)
        for i in range(n):
            step(i, arm)
        for s in streams[1:]:
            streams[0].wait_event(s.record_event())
        ev1.record(streams[0])
        torch.cuda.synchronize()
        return ev0.elapsed_time(ev1)

    res = {"c": [], "d": []}
    for r in range(args.runs):
        for arm in ("c", "d"):
            if arm == "c":
                load_c()
            for i in range(3 * NTEX):
                step(i, arm)
            ms = region(args.steps, arm)
            res[arm].append(round(mp * args.steps / (ms * 1e-3), 1))
            if r == 0:
                got = {k: results_digest(c.fetch_all(0)) for k, c in enumerate(ctxs)}
                if got != want:
                    failures.append(f"resident ({arm}) digests differ from (a)")
    for arm, what in (("c", "int32 planes resident in HBM (bench.py's value): reset + analyze"),
                      ("d", "interleaved RGBA8 resident in HBM: yk_set_image_interleaved_device (unpack) + analyze")):
        emit({"arm": arm, "what": what, "mp_s_runs": res[arm], "steps_per_run": args.steps, "contexts": NTEX, "analysis_ctas": sms // 4})
    for c in ctxs:
        c.close()

    # ---- yk_k_unpack8 alone ----------------------------------------------------------------------------------------------
    lib.yk_profile.argtypes = [C.c_void_p, C.c_int]
    lib.yk_profile_read.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_longlong)]
    ctx = capi.Context(W, H, planes=CH, slots=1, lib=lib)
    try:
        for ch, npl in ((4, 4), (3, 3), (4, 3)):
            srcs = [torch.from_numpy(np.ascontiguousarray(a[:, :, :ch])).cuda() for a in hwc]
            torch.cuda.synchronize()
            for i in range(2 * NTEX):
                ctx.set_image_interleaved_device(srcs[i % NTEX].data_ptr(), W * ch, ch, npl, W, H)
            ctx.sync()
            ms, cnt = (C.c_double * 8)(), (C.c_longlong * 8)()
            lib.yk_profile_read(ctx.ctx, ms, cnt)
            lib.yk_profile(ctx.ctx, 1)
            for i in range(args.unpack_launches):
                ctx.set_image_interleaved_device(srcs[i % NTEX].data_ptr(), W * ch, ch, npl, W, H)
            lib.yk_profile_read(ctx.ctx, ms, cnt)
            lib.yk_profile(ctx.ctx, 0)
            us = ms[5] / max(1, cnt[5]) * 1e3
            nbytes = W * H * (ch + npl)
            emit({"kernel": "yk_k_unpack8", "channels": ch, "n_planes": npl, "w": W, "h": H, "launches": int(cnt[5]),
                  "us_per_launch": round(us, 3), "bytes": nbytes, "gb_s": round(nbytes / (us * 1e-6) / 1e9, 1),
                  "floor_us_at_copy_peak": round(nbytes / (COPY_PEAK_GBS * 1e9) * 1e6, 3),
                  "copy_peak_frac": round(nbytes / (us * 1e-6) / 1e9 / COPY_PEAK_GBS, 3),
                  "inputs": f"{NTEX} resident textures in turn ({NTEX * W * H * ch / 1e6:.0f} MB): mostly read from HBM, not L2"})
            del srcs
    finally:
        ctx.close()

    emit({"digests_equal": not failures, "failures": failures})
    if args.out:
        with open(args.out, "a") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")
    return 1 if failures else 0


if __name__ == "__main__":
    sys.exit(main())
