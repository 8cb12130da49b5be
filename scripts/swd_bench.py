"""Sliced Wasserstein distance on the B200: the kernels against a plain torch composition, for N in {5e4, 1e6} model
samples against M = 1e6 reference samples, d = 6, P in {50, 512} directions, p = 2.

Timed (CUDA events, best of --reps after warm-up):
  - reference: building SlicedWassersteinDistance(y) (directions + projection and stable sort of y);
  - forward: one call of the built object without a gradient;
  - forward_backward: one call with x requiring grad, then backward;
  - torch_*: the same three with an fp32 matmul, torch.sort(stable=True) on both sides and the interval sum
    (exact int64 breakpoints i M and j N, index arithmetic, float64 sum), differentiated by autograd.
The torch values are compared with the kernels' (relative difference of the distance, and of the gradient to its
largest entry).  Bytes per (direction, particle) come from the byte model in `model_bytes`; GB/s = that traffic over
the kernel time.  Inputs of 1e6 x 6 floats are 24 MB, but the sort's keys and indices for P directions are 16 P MB,
far beyond the 126 MB of L2 at P = 50.  The card's name, power limit and maximum SM clock are read in the same run.
Prints one JSON line per case; with --out, also writes them to that file.

    python scripts/swd_bench.py [--reps 5] [--out results.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from mentflow_b200 import loss                                  # noqa: E402


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


def model_bytes(n, m, grad, reference=False):
    """HBM bytes per (direction, particle) of the kernels (swd.cu): keys written (4); pass 0 reads keys (4) and writes
    keys + indices (8); passes 1 and 2 count (4), read (8) and write (8); the last pass counts (4) and reads (8).
    The model side then reads the sorted reference, M / N values per particle (4 M / N), and with a gradient writes
    one coefficient (4) that the backward reads again (4).  The reference side writes the sorted value and index (8)
    and re-reads the particle's row (24 at d = 6).  Rows of x, histograms and scans are below 1 %."""
    b = 4 + 12 + 2 * 20 + 12
    if reference:
        return b + 8 + 24
    return b + 4 * m / n + (8 if grad else 0)


def torch_swd(x, y, theta, p=2.0):
    n, m = x.shape[0], y.shape[0]
    u, _ = torch.sort(theta @ x.t(), dim=1, stable=True)
    v, _ = torch.sort(theta @ y.t(), dim=1, stable=True)
    dev = x.device
    b = torch.unique(torch.cat([torch.arange(n + 1, device=dev) * m, torch.arange(m + 1, device=dev) * n]))
    lens = (b[1:] - b[:-1]).to(torch.float64)
    i, j = b[:-1] // m, b[:-1] // n
    wpp = ((u[:, i] - v[:, j]).abs().to(torch.float64) ** p * lens).sum(dim=1) / (float(n) * float(m))
    return (wpp.mean() ** (1.0 / p)).to(torch.float32)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("swd_bench.py needs a CUDA device")
    dev = torch.device("cuda")
    info = card()
    print(json.dumps({"card": info}))
    rows = []
    m, d = 1_000_000, 6
    for nproj in (50, 512):
        for n in (50_000, 1_000_000):
            gen = torch.Generator(device=dev).manual_seed(n + nproj)
            x = torch.randn(n, d, device=dev, generator=gen)
            y = torch.randn(m, d, device=dev, generator=gen) * 1.2 + 0.3
            proj = loss.random_projections(d, nproj, seed=nproj)
            theta = proj.t().float().contiguous().to(dev)
            est = loss.SlicedWassersteinDistance(y, projections=proj)
            xg = x.clone().requires_grad_(True)

            def build():
                loss.SlicedWassersteinDistance(y, projections=proj)

            def fwd():
                with torch.no_grad():
                    est(x)

            def both():
                xg.grad = None
                est(xg).backward()

            def t_fwd():
                with torch.no_grad():
                    torch_swd(x, y, theta)

            def t_both():
                xg.grad = None
                torch_swd(xg, y, theta).backward()

            def t_build():
                torch.sort(theta @ y.t(), dim=1, stable=True)

            times = {k: best_ms(f, args.reps) for k, f in (("reference_ms", build), ("forward_ms", fwd),
                                                            ("forward_backward_ms", both), ("torch_reference_ms", t_build),
                                                            ("torch_forward_ms", t_fwd),
                                                            ("torch_forward_backward_ms", t_both))}
            clock = card("clocks.sm").get("clocks.sm")        # right after the timed calls, while the card is busy
            xg.grad = None
            s = est(xg)
            s.backward()
            g = xg.grad.clone()
            xg.grad = None
            st = torch_swd(xg, y, theta)
            st.backward()
            s, st = s.detach(), st.detach()
            rel = abs(float(s) - float(st)) / abs(float(st))
            grel = float((g - xg.grad).abs().max() / xg.grad.abs().max())
            cells = float(nproj) * n
            row = {"n": n, "m": m, "d": d, "nproj": nproj, "p": 2, **{k: round(v, 4) for k, v in times.items()},
                   "bytes_per_cell_forward": round(model_bytes(n, m, False), 2),
                   "bytes_per_cell_forward_backward": round(model_bytes(n, m, True), 2),
                   "bytes_per_cell_reference": model_bytes(m, m, False, reference=True),
                   "forward_GBps": round(model_bytes(n, m, False) * cells / (times["forward_ms"] * 1e6), 1),
                   "forward_backward_GBps": round(model_bytes(n, m, True) * cells / (times["forward_backward_ms"] * 1e6),
                                                  1),
                   "reference_GBps": round(model_bytes(m, m, False, True) * float(nproj) * m /
                                           (times["reference_ms"] * 1e6), 1),
                   "swd": float(s), "torch_swd": float(st), "rel_diff": float(f"{rel:.3g}"),
                   "grad_rel_diff": float(f"{grel:.3g}"), "gpu": info.get("name"),
                   "power_limit": info.get("power.limit"), "sm_clock_max": info.get("clocks.max.sm"),
                   "sm_clock_after": clock}
            assert rel < 1e-5 and grel < 1e-4, row
            print(json.dumps(row), flush=True)
            rows.append(row)
            del est, xg, g
            torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            f.write(json.dumps({"card": info}) + "\n")
            for row in rows:
                f.write(json.dumps(row) + "\n")


if __name__ == "__main__":
    main()
