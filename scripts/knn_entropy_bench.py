"""k-NN entropy estimator on the B200: forward, backward and both, for N in {25,000, 1e5, 1e6}, d in {2, 4, 6}, k = 5.

The forward is the all-pairs k-th neighbour search (ops.knn_kth: transpose, pair kernel, merge, log-sum); the
backward is the stable sort of the neighbour indices plus the gradient kernel.  Times are CUDA events around each
call (best of --reps after warm-up; a batch of N = 1e6, d = 6 is 24 MB, so the inputs stay in L2 -- the kernel is bound
by arithmetic, not memory).  Pair evaluations/s counts N (N - 1) ordered pairs per forward.  The card's name, power
limit and maximum SM clock are read in the same run, and the SM clock right after each case.  Prints one JSON line
per case; with --out, also writes them to that file.

    python scripts/knn_entropy_bench.py [--reps 5] [--out results.jsonl]
"""
import argparse
import json
import math
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from mentflow_b200 import ops                                   # noqa: E402
from mentflow_b200.entropy import KNNEntropyEstimator          # noqa: E402


def card(q="name,power.limit,clocks.max.sm"):
    try:
        row = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        return dict(zip(q.split(","), [v.strip() for v in row.split(",")]))
    except (OSError, IndexError, subprocess.SubprocessError):
        return {"name": torch.cuda.get_device_name()}


def best_ms(fn, reps, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    best = float("inf")
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        best = min(best, a.elapsed_time(b))
    return best


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--k", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("knn_entropy_bench.py needs a CUDA device")
    dev = torch.device("cuda")
    info = card()
    print(json.dumps({"card": info}))
    rows = []
    for n in (25_000, 100_000, 1_000_000):
        for d in (2, 4, 6):
            torch.manual_seed(n + d)
            x = torch.randn(n, d, device=dev)
            xg = x.clone().requires_grad_(True)
            est = KNNEntropyEstimator(k=args.k)
            reps = args.reps if n < 1_000_000 else max(2, args.reps // 2)

            def fwd():
                with torch.no_grad():
                    ops.knn_kth(x, args.k)

            h = est(xg)

            def bwd():
                xg.grad = None
                h.backward(retain_graph=True)

            def both():
                xg.grad = None
                est(xg).backward()

            t_f, t_b, t_fb = best_ms(fwd, reps), best_ms(bwd, reps), best_ms(both, reps)
            clock = card("clocks.sm").get("clocks.sm")        # right after the timed calls, while the card is busy
            pairs = float(n) * (n - 1)
            row = {"n": n, "d": d, "k": args.k, "forward_ms": round(t_f, 4), "backward_ms": round(t_b, 4),
                   "forward_backward_ms": round(t_fb, 4), "pairs_per_s": float(f"{pairs / (t_f * 1e-3):.4g}"),
                   "neg_entropy": float(h.detach()), "gpu": info.get("name"), "power_limit": info.get("power.limit"),
                   "sm_clock_max": info.get("clocks.max.sm"), "sm_clock_after": clock}
            assert math.isfinite(row["neg_entropy"])
            print(json.dumps(row), flush=True)
            rows.append(row)
    if args.out:
        with open(args.out, "w") as f:
            f.write(json.dumps({"card": info}) + "\n")
            for row in rows:
                f.write(json.dumps(row) + "\n")


if __name__ == "__main__":
    main()
