"""Metropolis-Hastings chains over the classical-MENT density against explicit-point density evaluation and grid
sampling (B200).

  1. chain steps per second of the fused kernel, 1e6 chains x 100 proposals, on the C5 model (6-D, K = 25 one-
     dimensional screens, tables one sweep in) and on a 6-D model of 2-D screens;
  2. ops.ment_prob at 1e8 explicit points, the 1e6 states of those chains 100 times, in the same run (points inside
     the support: the grid's rate profits from the early exit on empty cells, which chains rarely visit);
  3. one sample-mode Gauss-Seidel update of the C5 model (draw 1e6 particles, fused projection + KDE of one screen,
     table update) with the MH sampler against GridSampler at 16^6 and 24^6 cells.

Times are the best of the repetitions, CUDA events around work that ends in a synchronise.  The card's name, power
limit and clocks are read in the same run.  Prints one JSON line per case; with --out, also writes them to that file.

    python scripts/ment_mh_bench.py [--reps 5] [--out profiles/ment_mh_bench.jsonl]
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import mentflow_b200 as mf                                  # noqa: E402
from mentflow_b200 import workloads                         # noqa: E402
from ment_multipole_bench import alternate, c5_models, card  # noqa: E402

MH = mf.sample.MetropolisHastingsSampler


def screens_2d_model(d: int = 6, num: int = 12, bins: int = 48, xmax: float = 3.5):
    """d-D model with `num` 2-D screens (axes (0, 1) behind random rotations), tables one sweep in."""
    gen = torch.Generator().manual_seed(3)
    tfs = []
    for _ in range(num):
        q, _ = torch.linalg.qr(torch.randn(d, d, generator=gen))
        tfs.append(mf.simulate.LinearTransform(q.float().cuda()))
    e = torch.linspace(-xmax, xmax, bins + 1)
    diag = mf.diagnostics.Histogram2D(axis=(0, 1), edges=(e, e), bandwidth=(0.5, 0.5)).to("cuda")
    diags = [[diag] for _ in tfs]
    truth = workloads.gaussian_mixture(200_000, ndim=d, seed=1, device="cuda")
    with torch.no_grad():
        meas = [[p[0]] for p in mf.simulate.forward(truth, tfs, diags)]
    sampler = mf.sample.GridSampler(limits=d * [(-xmax, xmax)], shape=(16,) * d, device="cuda")
    model = mf.ment.MENT(ndim=d, transforms=tfs, diagnostics=diags, measurements=meas,
                         prior=mf.prior.Gaussian(ndim=d, scale=3.0), mode="sample", sampler=sampler,
                         n_samples=1_000_000, device="cuda")
    torch.manual_seed(77)
    model.gauss_seidel_update(lr=0.9)
    return model


def chain_rates(name, model, reps, chains=1_000_000, proposals=100):
    mh = MH(model.ndim, burnin=proposals, steps=1, start_scale=1.0)
    x = mh(model.prob, chains, seed=1)
    rate = float(mh.acceptance_rate)
    pts = x.repeat(proposals, 1)             # as many explicit points as the chains take steps
    t_mh, t_pts = alternate([lambda: mh(model.prob, chains, seed=2), lambda: model.prob(pts)], reps)
    positive = float((model.prob(pts) > 0).float().mean())
    steps_per_s = chains * proposals / t_mh * 1e3
    points_per_s = pts.shape[0] / t_pts * 1e3
    return {"case": f"{name}: fused MH chains, {chains} chains x {proposals} proposals", "chain_ms": t_mh,
            "chain_steps_per_s": steps_per_s, "acceptance": rate, "ment_prob_points_ms": t_pts,
            "ment_prob_points_per_s": points_per_s, "points_with_positive_density": positive,
            "steps_over_points": steps_per_s / points_per_s}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the GPU kernels only")
    info = card()
    rows = []

    c5 = c5_models(False, 1_000_000)
    rows.append(chain_rates("C5 (6-D, 25 1-D screens of 64 bins)", c5, args.reps))
    rows.append(chain_rates("6-D, 12 2-D screens of 48 x 48 bins", screens_2d_model(), args.reps))

    mh = MH(6, burnin=50, steps=10, thin=5, start_scale=1.0)
    grids = {res: mf.sample.GridSampler(limits=6 * [(-3.5, 3.5)], shape=(res,) * 6, device="cuda") for res in (16, 24)}

    def update(sampler):
        c5.sampler = sampler
        lf = c5.lagrange_functions[0][0]
        saved = lf.values.clone()
        pred = c5.simulate(0, 0)
        mf.ops.gs_update(lf.values.view(-1), c5.measurements[0][0].reshape(-1), pred.reshape(-1), 0.9, 1e-10)
        lf.set_values(saved)

    t_mh, t16, t24 = alternate([lambda: update(mh), lambda: update(grids[16]), lambda: update(grids[24])],
                               args.reps, warm=1)
    rows.append({"case": "C5 sample-mode Gauss-Seidel update: 1e6 particles, one screen's KDE and table update",
                 "mh_ms": t_mh, "mh_config": "1e5 chains, burnin 50, steps 10, thin 5 (95 proposals per chain)",
                 "grid16_ms": t16, "grid24_ms": t24})

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
