"""Classical MENT behind thin multipole kicks against the same maps without the kick (B200).

  1. density on the C5 sampler grid (6-D, K = 25 one-dimensional screens, 16^6 cells): linear maps M_k against
     CompositeTransform(MultipoleTransform(3), LinearTransform(M_k)), each with the tables of its own measurements;
  2. one sample-mode Gauss-Seidel sweep at that size (grid density, draws, fused projection + KDE, table update);
  3. one integrate-mode sweep of rec_2d/nonlinear (six kicks -> rotation, 85-bin screens, 250 integration points),
     against the same set-up with the kicks removed.

The two variants of each case are timed alternately in one process with CUDA events (best of the repetitions).  The
card's name, power limit and clocks are read in the same run.  Prints one JSON line per case; with --out, also writes
them to that file.

    python scripts/ment_multipole_bench.py [--reps 10] [--samples 1000000] [--out results.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import mentflow_b200 as mf                         # noqa: E402
from mentflow_b200 import workloads                # noqa: E402
from mentflow_b200.simulate.transform import CompositeTransform, LinearTransform, MultipoleTransform  # noqa: E402

GOLDEN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "multipole.npz")


def card():
    q = "name,power.limit,clocks.max.sm,clocks.sm"
    try:
        row = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        return dict(zip(q.split(","), [v.strip() for v in row.split(",")]))
    except (OSError, IndexError, subprocess.SubprocessError):
        return {"name": torch.cuda.get_device_name()}


def alternate(fns, reps, warm=2):
    """Best time in ms of each callable, the callables run alternately."""
    for f in fns:
        for _ in range(warm):
            f()
    torch.cuda.synchronize()
    best = [float("inf")] * len(fns)
    for _ in range(reps):
        for i, f in enumerate(fns):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            f()
            b.record()
            b.synchronize()
            best[i] = min(best[i], a.elapsed_time(b))
    return best


def c5_models(kick: bool, n_samples: int, res: int = 16, num: int = 25, bins: int = 64, xmax: float = 3.5):
    d = 6
    wl = workloads.isotropic_1d(d, num, bins, xmax)
    if kick:
        tfs = [CompositeTransform(MultipoleTransform(order=3, strength=0.2), LinearTransform(m.cuda()))
               for m in wl["matrices"]]
    else:
        tfs = [LinearTransform(m.cuda()) for m in wl["matrices"]]
    diag = mf.diagnostics.Histogram1D(axis=0, edges=wl["edges"], bandwidth=0.5).to("cuda")
    diags = [[diag] for _ in tfs]
    truth = workloads.gaussian_mixture(200_000, ndim=d, seed=1, device="cuda")
    with torch.no_grad():
        meas = [[p[0]] for p in mf.simulate.forward(truth, tfs, diags)]
    sampler = mf.sample.GridSampler(limits=d * [(-xmax, xmax)], shape=tuple(d * [res]), device="cuda")
    model = mf.ment.MENT(ndim=d, transforms=tfs, diagnostics=diags, measurements=meas,
                         prior=mf.prior.Gaussian(ndim=d, scale=3.0), mode="sample", sampler=sampler,
                         n_samples=n_samples, device="cuda")
    torch.manual_seed(77)
    model.gauss_seidel_update(lr=0.9)            # tables of a model one sweep in: realistic supports
    return model


def nonlinear_model(kick: bool, points: int = 250):
    g = np.load(GOLDEN)
    matrix = torch.from_numpy(g["nl_matrix"]).cuda()
    if kick:
        tfs = [CompositeTransform(MultipoleTransform(order=int(g["nl_order"]), strength=float(s)),
                                  LinearTransform(matrix)) for s in g["nl_strengths"]]
    else:
        tfs = [LinearTransform(matrix) for _ in g["nl_strengths"]]
    diag = mf.diagnostics.Histogram1D(axis=0, edges=torch.from_numpy(g["nl_edges"]), bandwidth=0.5).to("cuda")
    return mf.ment.MENT(ndim=2, transforms=tfs, diagnostics=[[diag] for _ in tfs],
                        measurements=[[torch.from_numpy(m).cuda()] for m in g["nl_meas"]],
                        prior=mf.prior.Gaussian(ndim=2, scale=1.5), mode="integrate",
                        integration_limits=[[[(-4.0, 4.0)]] for _ in tfs],
                        integration_shape=[[(points,)] for _ in tfs], device="cuda")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--samples", type=int, default=1_000_000, help="particles per measurement update (sample mode)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the GPU kernels only")
    info = card()
    rows = []

    lin, mp = c5_models(False, args.samples), c5_models(True, args.samples)
    t_lin, t_mp = alternate([lambda: lin.prob_on_grid(lin.sampler), lambda: mp.prob_on_grid(mp.sampler)], args.reps)
    rows.append({"case": "C5 MENT density on the 16^6 grid, 25 tables", "linear_ms": t_lin, "kick_ms": t_mp,
                 "ratio": t_mp / t_lin, "cells_per_s_kick": 16 ** 6 / t_mp * 1e3})
    sweeps = max(2, args.reps // 4)
    t_lin, t_mp = alternate([lambda: lin.gauss_seidel_update(lr=0.9), lambda: mp.gauss_seidel_update(lr=0.9)],
                            sweeps, warm=1)
    rows.append({"case": f"C5 MENT sample-mode sweep: 25 updates, {args.samples} particles each", "linear_ms": t_lin,
                 "kick_ms": t_mp, "ratio": t_mp / t_lin, "kick_ms_per_update": t_mp / 25})
    del lin, mp

    lin, mp = nonlinear_model(False), nonlinear_model(True)
    t_lin, t_mp = alternate([lambda: lin.gauss_seidel_update(lr=1.0), lambda: mp.gauss_seidel_update(lr=1.0)],
                            args.reps)
    rows.append({"case": "rec_2d/nonlinear integrate-mode sweep: 6 screens x 85 bins x 250 points",
                 "linear_ms": t_lin, "kick_ms": t_mp, "ratio": t_mp / t_lin})

    for r in rows:
        r.update({"gpu": info})
        print(json.dumps(r))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
