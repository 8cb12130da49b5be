"""k-NN entropy on sharded particles: forward, backward and both of KNNEntropyEstimator at d = 6, k = 5 for N_total in
{25,000, 1e5, 1e6}, particles split evenly over the ranks, and the three all-gathers (x, r, idx) timed on their own.

Run under torchrun, one process per GPU (world size 1 runs the single-GPU estimator):

    torchrun --nproc_per_node=R scripts/knn_entropy_sharded_bench.py [--reps 5] [--out results.jsonl]

Every timed call starts after a barrier and ends in a device synchronise; a call's time is the slowest rank's CUDA-event
time, the best of --reps after warm-up.  "gathers" is the all-gather of x, r and idx alone.  The card's name, power limit
and maximum SM clock are read in the same run, and the SM clock right after each case.  Rank 0 prints one JSON line per
case; with --out it appends them to that file.

--rank-share R1,R2,... (world size 1): also time, on the one device, what rank 0 of R ranks computes besides the
gathers -- its row search of N / R queries against the N gathered particles, the log sum of the N gathered r, and the
backward of its rows -- as a stand-in for the per-rank pair work where fewer than R GPUs are available.
"""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from mentflow_b200 import distributed as mfd                  # noqa: E402
from mentflow_b200 import ops                                   # noqa: E402
from mentflow_b200.entropy import KNNEntropyEstimator          # noqa: E402


def card(q="name,power.limit,clocks.max.sm"):
    try:
        row = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()[0]
        return dict(zip(q.split(","), [v.strip() for v in row.split(",")]))
    except (OSError, IndexError, subprocess.SubprocessError):
        return {"name": torch.cuda.get_device_name()}


def timed_ms(fn, reps, world, warm=1):
    """best over reps of the slowest rank's time of one call"""
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    best = float("inf")
    for _ in range(reps):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        t = torch.tensor([a.elapsed_time(b)], device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        best = min(best, float(t))
    return best


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--k", type=int, default=5)
    ap.add_argument("--d", type=int, default=6)
    ap.add_argument("--sizes", default="25000,100000,1000000")
    ap.add_argument("--rank-share", default="", help="world size 1: time rank 0's share of R ranks, e.g. 2,4,8")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("knn_entropy_sharded_bench.py needs a CUDA device")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    info = card()
    rows = []
    for n_total in (int(s) for s in args.sizes.split(",")):
        if n_total % world:
            raise SystemExit(f"N_total = {n_total} does not split evenly over {world} ranks")
        n_local = n_total // world
        g = torch.Generator(device=device).manual_seed(n_total)
        x_all = torch.randn(n_total, args.d, generator=g, device=device)
        x = x_all[mfd.shard_slice(n_total, rank, world)].contiguous()
        est = KNNEntropyEstimator(k=args.k)
        reducer = None
        if world > 1:
            reducer = mfd.ShardReducer(equal_shards=True)
            est.reducer = reducer
        xg = x.clone().requires_grad_(True)
        reps = args.reps if n_total < 1_000_000 else max(2, args.reps // 2)

        def fwd():
            with torch.no_grad():
                est(x)

        h = est(xg)

        def bwd():
            xg.grad = None
            h.backward(retain_graph=True)

        def both():
            xg.grad = None
            est(xg).backward()

        r_loc = torch.rand(n_local, device=device)
        i_loc = torch.zeros(n_local, dtype=torch.int32, device=device)

        def gathers():
            reducer.all_gather(x)
            reducer.all_gather(r_loc)
            reducer.all_gather(i_loc)

        t_f, t_b, t_fb = timed_ms(fwd, reps, world), timed_ms(bwd, reps, world), timed_ms(both, reps, world)
        t_g = timed_ms(gathers, max(reps, 5), world) if world > 1 else 0.0
        clock = card("clocks.sm").get("clocks.sm")
        pairs = float(n_total) * n_local          # this rank's rows against the union
        row = {"world": world, "n_total": n_total, "n_per_rank": n_local, "d": args.d, "k": args.k,
               "forward_ms": round(t_f, 4), "backward_ms": round(t_b, 4), "forward_backward_ms": round(t_fb, 4),
               "gathers_ms": round(t_g, 4), "pairs_per_rank": pairs,
               "pairs_per_s_per_rank": float(f"{pairs / (t_f * 1e-3):.4g}"),
               "neg_entropy": float(h.detach()), "gpu": info.get("name"), "power_limit": info.get("power.limit"),
               "sm_clock_max": info.get("clocks.max.sm"), "sm_clock_after": clock}
        if rank == 0:
            print(json.dumps(row), flush=True)
        rows.append(row)
        for share in (int(s) for s in args.rank_share.split(",") if s) if world == 1 else ():
            sl = mfd.shard_slice(n_total, 0, share)
            r_all, idx_all, _ = ops.knn_kth(x_all, args.k)
            g1 = torch.ones((), dtype=torch.float64, device=device)
            t_rows = timed_ms(lambda: ops.knn_kth(x_all, args.k, rows=sl), reps, 1)
            t_log = timed_ms(lambda: ops.knn_logsum(r_all), max(reps, 5), 1)
            t_bwd = timed_ms(lambda: ops.knn_kth_bwd(x_all, r_all, idx_all, g1, rows=sl), max(reps, 5), 1)
            clock = card("clocks.sm").get("clocks.sm")
            row = {"emulated_world": share, "rank": 0, "n_total": n_total, "n_per_rank": sl.stop - sl.start,
                   "d": args.d, "k": args.k, "row_search_ms": round(t_rows, 4), "logsum_ms": round(t_log, 4),
                   "backward_rows_ms": round(t_bwd, 4), "gathers": "not measured (one device)",
                   "gpu": info.get("name"), "power_limit": info.get("power.limit"),
                   "sm_clock_max": info.get("clocks.max.sm"), "sm_clock_after": clock}
            print(json.dumps(row), flush=True)
            rows.append(row)
        del x_all, x, xg, h
    if rank == 0 and args.out:
        with open(args.out, "a") as f:
            for row in rows:
                f.write(json.dumps(row) + "\n")
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
