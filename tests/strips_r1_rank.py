"""One rank of a strip run with DynamicTileEncode (used by tests/test_emulated_strips_r1.py on gloo with the host-staged
transport and by tests/test_gpu_strips_r1.py over CUDA IPC): rank r analyses strip r of a seeded image and codes its R1
streams in the box gathered from every strip; rank 0 checks the merged result against the oracle on the whole image."""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rank", type=int, default=int(os.environ.get("RANK", "0")))
    ap.add_argument("--world", type=int, default=int(os.environ.get("WORLD_SIZE", "1")))
    ap.add_argument("--backend", default="gloo")
    ap.add_argument("--mode", default="host")
    ap.add_argument("--w", type=int, default=128)
    ap.add_argument("--h", type=int, default=128)
    ap.add_argument("--planes", type=int, default=3, choices=[3, 4])
    ap.add_argument("--mode3", action="store_true")
    args = ap.parse_args()
    import torch.distributed as dist
    import cases
    from yaik_b200 import capi, strips
    from yaik_b200.synth import make_image, SEED_BASE
    from strips_check import check_against_oracle
    from strips_r1_check import check_r1, oracle_r1, r1_stage

    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29534")
    dist.init_process_group(args.backend, rank=args.rank, world_size=args.world)
    lib = capi.load_library(os.environ.get("YK_STRIPS_LIB") or None)
    device = 0
    if args.mode == "ipc":
        import torch
        device = args.rank % max(1, torch.cuda.device_count())
    # RGBA: a power-of-two square with alpha holes (the oracle's alpha domain)
    planes = cases._patchy(args.w, args.h, 41, 4, 3) if args.planes == 3 else make_image(args.w, args.h, 4, SEED_BASE + 16)
    rows = strips.strip_rows(args.h, args.world)
    mine = planes[:, rows[args.rank][0]:rows[args.rank][0] + rows[args.rank][1]] if args.rank < len(rows) else None
    ctx = capi.Context(args.w, args.h, planes=args.planes, slots=1, device=device, lib=lib)
    try:
        merged = strips.DistTransport(ctx, dist, mode=args.mode).run(mine, args.h, rows, r1=r1_stage(args.mode3))
        if args.rank == 0:
            check_r1(merged, oracle_r1(planes, args.mode3))
            check_against_oracle(merged, planes)
            print("strips r1 ok:", len(rows), "strips over", args.world, "ranks, transport", args.mode, "planes", args.planes, flush=True)
    finally:
        ctx.close()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
