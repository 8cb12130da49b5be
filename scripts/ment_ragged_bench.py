"""Classical MENT through the ragged Lagrange tables against the uniform ones (B200).

C5 (6-D, 25 one-dimensional screens, 16^6 sampler grid, tables one sweep in) three ways in one process:
  1. uniform: 64 bins per screen, the uniform kernels;
  2. the same model through the ragged entry points (offsets k * 64): the cost of the offset loads alone;
  3. a model whose 25 screens have 48 - 85 bins drawn at random: the ragged kernels on a real ragged model.
For each: ms per density pass (prob on the 16^6 grid) and per sample-mode Gauss-Seidel update of one screen (draw
1e6 particles from the grid, fused projection + KDE, table update).  Times are the best of the repetitions, the
three models alternated, CUDA events around work that ends in a synchronise.  The card's name, power limit and
clocks are read in the same run.  Prints one JSON line per case; with --out, also writes them to that file.

    python scripts/ment_ragged_bench.py [--reps 10] [--out profiles/ment_ragged_bench.jsonl]
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import mentflow_b200 as mf                          # noqa: E402
from mentflow_b200 import ops, workloads            # noqa: E402
from ment_multipole_bench import alternate, c5_models, card  # noqa: E402


def through_ragged_entry_points(model):
    """Route the model's (uniform) tables to the ragged entry points, with offsets k * B."""
    uniform = model._groups

    def groups(device):
        g1, g2 = uniform(device)
        k, b = g1[2].shape
        return ops.RaggedTables1D(g1[0], g1[1].reshape(-1), g1[2].reshape(-1), [i * b for i in range(k + 1)]), g2

    model._groups = groups
    return model


def ragged_c5(n_samples, res=16, num=25, xmax=3.5):
    """C5 with screens of 48 - 85 bins (a fixed draw)."""
    d = 6
    gen = torch.Generator().manual_seed(5)
    wl = workloads.isotropic_1d(d, num, 64, xmax)
    tfs = [mf.simulate.LinearTransform(m.cuda()) for m in wl["matrices"]]
    bins = [int(b) for b in torch.randint(48, 86, (num,), generator=gen)]
    diags = [[mf.diagnostics.Histogram1D(axis=0, edges=torch.linspace(-xmax, xmax, b + 1), bandwidth=0.5).to("cuda")]
             for b in bins]
    truth = workloads.gaussian_mixture(200_000, ndim=d, seed=1, device="cuda")
    with torch.no_grad():
        meas = mf.simulate.forward(truth, tfs, diags)
    sampler = mf.sample.GridSampler(limits=d * [(-xmax, xmax)], shape=(res,) * d, device="cuda")
    model = mf.ment.MENT(ndim=d, transforms=tfs, diagnostics=diags, measurements=meas,
                         prior=mf.prior.Gaussian(ndim=d, scale=3.0), mode="sample", sampler=sampler,
                         n_samples=n_samples, device="cuda")
    torch.manual_seed(77)
    model.gauss_seidel_update(lr=0.9)
    return model, bins


def update(model):
    lf = model.lagrange_functions[0][0]
    saved = lf.values.clone()
    pred = model.simulate(0, 0)
    ops.gs_update(lf.values.view(-1), model.measurements[0][0].reshape(-1), pred.reshape(-1), 0.9, 1e-10)
    lf.set_values(saved)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the GPU kernels only")
    info = card()
    uniform = c5_models(False, 1_000_000)
    via_ragged = through_ragged_entry_points(c5_models(False, 1_000_000))
    ragged, bins = ragged_c5(1_000_000)
    models = [uniform, via_ragged, ragged]
    assert isinstance(ragged._groups(torch.device("cuda"))[0], ops.RaggedTables1D)

    rho_u, rho_r = (m.prob_on_grid(m.sampler) for m in (uniform, via_ragged))
    identical = bool(torch.equal(rho_u, rho_r))
    del rho_u, rho_r
    t_density = alternate([lambda m=m: m.prob_on_grid(m.sampler) for m in models], args.reps)
    t_update = alternate([lambda m=m: update(m) for m in models], args.reps, warm=1)
    names = ["C5 uniform (25 screens of 64 bins)", "C5 through the ragged entry points (offsets k * 64)",
             f"C5 ragged (25 screens of {min(bins)} - {max(bins)} bins, {sum(bins)} in all)"]
    rows = []
    for i, name in enumerate(names):
        rows.append({"case": name, "density_pass_ms": t_density[i], "sample_update_ms": t_update[i],
                     "density_over_uniform": t_density[i] / t_density[0],
                     "update_over_uniform": t_update[i] / t_update[0]})
    rows[1]["bit_identical_to_uniform"] = identical
    rows[2]["bins"] = bins
    for r in rows:
        r.update({"gpu": info, "grid": "16^6 cells", "particles_per_update": 1_000_000, "reps": args.reps})
        print(json.dumps(r))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
