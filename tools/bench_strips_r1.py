#!/usr/bin/env python
"""DynamicTileEncode (R1) of tile-row strips: one 16384x16384 RGB image over the ranks of a torchrun launch (one GPU each),
the host-free protocol (yk_strip_set_peers over CUDA IPC + yk_strip_run_stages), int32 planes resident in HBM.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 tools/bench_strips_r1.py [--side 16384] [--steps 10] [--reps 3]

Two arms alternate in the same call, `--reps` times each: `--steps` images enqueued back to back on every strip's stream
with stages 0 (the analysis alone) and with YK_STAGE_RANGEDYN; time = CUDA events around the images on each rank's stream,
after a barrier, max over ranks, per image.  On rank 0's GPU one context analyses the whole image with yk_analyze(GRADIENT |
RANGE1D | RANGEDYN), timed the same way (the 1-GPU figure).  Every strip's streams (7 bitmaps, 7 rgbStreams, R2 and R1 of
three planes: lengths + SHA-1) are compared with that context's, whose streams are the strips' concatenated in strip
order; a mismatch fails the run.  The image is bench_strips.py's seeded 2048x2048 texture tiled over the plane.  Rank 0
prints one JSON line with the card's name and power limit (nvidia-smi, read only)."""
import argparse, hashlib, json, os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np


def digests(res):
    """(kind, length, SHA-1) of every stream of one strip or image, in a fixed order."""
    out = []
    for p in res["passes"]:
        out += [("bitmap", p["bitmap"]), ("rgb", p["rgb"])]
    for q in res["r2"]:
        out += [("idx", q["idx"]), ("type", q["type"])]
    for q in res.get("r1", []):
        out += [("r1_nibbles", q["nibbles"]), ("r1_defs", q["defs"])]
    return [(k, int(a.nbytes), hashlib.sha1(a.tobytes()).hexdigest()) for k, a in out]


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
        return [l.strip() for l in r.stdout.strip().splitlines()]
    except Exception as e:
        return [f"nvidia-smi failed: {e}"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--side", type=int, default=16384)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    import torch
    import torch.distributed as dist
    from yaik_b200 import capi, strips
    from yaik_b200.synth import make_image, SEED_BASE
    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dist.init_process_group("gloo")          # control plane only: IPC handles, barriers, the timing reduction
    side = args.side
    rows = strips.strip_rows(side, world)
    active = rank < len(rows)
    base = make_image(2048, 2048, 3, SEED_BASE + 3)
    reps = (side + 2047) // 2048

    def rows_of(y0, sh):
        return np.ascontiguousarray(np.tile(base, (1, reps, reps))[:, y0:y0 + sh, :side])

    lib = capi.load_library()
    ctx, peers = None, {}
    stream = torch.cuda.Stream(device=local)
    if active:
        y0, sh = rows[rank]
        ctx = capi.Context(side, sh, planes=3, slots=1, device=local, lib=lib)
        ctx.set_stream(stream.cuda_stream)
        ctx.set_upload_format(False)
        ctx.set_image(rows_of(y0, sh), 0)
        ctx.strip_config(side, y0)
    handles = [None] * world
    dist.all_gather_object(handles, ctx.ipc_export(ctx.strip_halo().haloIn) if active else None)
    for r in (rank - 1, rank + 1):
        if active and 0 <= r < len(rows):
            peers[r] = ctx.ipc_open(handles[r])
    dist.barrier()                                   # every halo is cleared before a neighbour writes into it
    if active:
        ctx.strip_set_peers(peers.get(rank - 1), peers.get(rank + 1))

    def barrier():
        torch.cuda.synchronize(local)
        dist.barrier()

    def timed(stages, n):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        for _ in range(n):
            if active:
                ctx.strip_run(stages=stages)
        ev1.record(stream)
        barrier()
        t = torch.tensor([ev0.elapsed_time(ev1) / n], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    arms = {"analysis": 0, "analysis+r1": capi.STAGE_RANGEDYN}
    for stages in arms.values():
        timed(stages, args.warmup)
    ms = {k: [] for k in arms}
    for _ in range(args.reps):
        for k, stages in arms.items():
            ms[k].append(timed(stages, args.steps))
    # the last image ran with R1: its streams, per strip
    mine = digests(strips.collect_results(ctx, r1=capi.STAGE_RANGEDYN)) if active else None
    parts = [None] * world
    dist.all_gather_object(parts, mine)
    line = None
    if rank == 0:
        whole = capi.Context(side, side, planes=3, slots=1, device=local, lib=lib)
        whole.set_stream(stream.cuda_stream)
        whole.set_upload_format(False)
        whole.set_image(rows_of(0, side), 0)
        STAGES = capi.STAGE_GRADIENT | capi.STAGE_RANGE1D | capi.STAGE_RANGEDYN

        def whole_timed(n):
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record(stream)
            for _ in range(n):
                whole.reset_state(0)
                whole.analyze(STAGES)
            ev1.record(stream)
            torch.cuda.synchronize(local)
            return ev0.elapsed_time(ev1) / n

        whole_timed(args.warmup)
        whole_ms = [whole_timed(args.steps) for _ in range(args.reps)]
        ref = strips.collect_results(whole, r1=capi.STAGE_RANGEDYN)
        whole.close()
        streams = []
        for p in ref["passes"]:
            streams += [p["bitmap"], p["rgb"]]
        for q in ref["r2"]:
            streams += [q["idx"], q["type"]]
        for q in ref["r1"]:
            streams += [q["nibbles"], q["defs"]]
        flat = [s.view(np.uint8).ravel() for s in streams]
        offs = [0] * len(flat)
        ok = True
        for part in parts[:len(rows)]:
            for k, (kind, n, sha) in enumerate(part):
                seg = flat[k][offs[k]:offs[k] + n]
                ok = ok and seg.size == n and hashlib.sha1(seg.tobytes()).hexdigest() == sha
                offs[k] += n
        ok = ok and all(offs[k] == flat[k].size for k in range(len(flat)))
        if not ok:
            raise SystemExit("bench_strips_r1.py: the strips' streams differ from the whole-image context")
        best = {k: min(v) for k, v in ms.items()}
        info = gpu_info()
        line = {"metric": "ms per image (max over ranks)", "workload": f"one {side}x{side} RGB image (seeded 2048x2048 texture tiled), int32 planes resident, "
                f"{len(rows)} tile-row strips, one GPU each, host-free protocol (CUDA IPC halos, epoch flags)",
                "n_gpus": world, "steps": args.steps, "reps": args.reps,
                "ms_per_image": {k: [round(x, 4) for x in v] for k, v in ms.items()},
                "r1_ms_per_image_added": round(best["analysis+r1"] - best["analysis"], 4),
                "whole_image_1gpu_ms_per_image_gradient_range1d_rangedyn": [round(x, 4) for x in whole_ms],
                "strip_rows": rows, "parity_checked": True,
                "parity_against": "one context on rank 0's GPU: yk_analyze(GRADIENT | RANGE1D | RANGEDYN) of the whole image, every stream's length + SHA-1",
                "gpu_name_power_limit": info[local] if local < len(info) else info}
        print(json.dumps(line), flush=True)
    for ptr in peers.values():
        ctx.ipc_close(ptr)
    if ctx:
        ctx.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
