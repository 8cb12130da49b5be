"""NNGenerator on the B200: the fused tanh-MLP kernels against a torch eager nn.Sequential, and against NSFGenerator
sampling, at H = 64, L = 3 hidden layers, (Din, Dout) in {(6, 6), (2, 2)}, N in {25,000, 1e6}.

Timed (CUDA events, median of --reps after warm-up):
  - forward: gen(z) without a gradient (nn_fwd_kernel);
  - forward_backward: gen(z) with the parameters requiring grad, then backward of a linear functional
    (nn_fwd_kernel, then nn_bwd_kernel + nn_reduce_kernel);
  - torch_*: the same with an fp32 nn.Sequential on the same weights, TF32 off; its output is compared with the
    kernels' (largest |difference| over max(1, |x|));
  - nsf_sample: NSFGenerator(Dout).sample(N) (5 transforms, 64 hidden units, 3 hidden layers, 20 bins, the reference's
    flow), the paper's NN-vs-flow sampling comparison restated for this library;
  - train_step: one GraphedTrainStep replay (fused capturable AdamW) of the NN generator on C1 (2-D, 7 rotations,
    25,000 particles, covariance entropy), (Din, Dout) = (2, 2) only.
fma_floor_ms is the forward's multiply-adds, N (64 Din + 64 * 64 (L - 1) + 64 Dout), over 148 SMs x 128 FMA/clk at the
card's maximum SM clock: a bound, not a result.  The card's name, power limit and SM clocks are read in the same run
(sm_clock is the current clock at start-up, before any timed work, so it shows the idle clock).
Prints one JSON line per case; with --out, also writes them to that file.

    python scripts/nn_generator_bench.py [--reps 20] [--out results.jsonl]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import mentflow_b200 as mf                                       # noqa: E402
from mentflow_b200 import workloads                              # noqa: E402
from mentflow_b200.generate import NNGenerator, NSFGenerator      # noqa: E402
from mentflow_b200.graphs import GraphedTrainStep                 # noqa: E402


def card(q="name,power.limit,clocks.max.sm,clocks.sm"):
    try:
        row = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        return dict(zip(q.split(","), [v.strip() for v in row.split(",")]))
    except (OSError, IndexError, subprocess.SubprocessError):
        return {"name": torch.cuda.get_device_name()}


def median_ms(fn, reps, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return statistics.median(times)


def sequential_like(gen):
    H, L = gen.hidden_units, gen.hidden_layers
    mods = [torch.nn.Linear(gen.input_features, H), torch.nn.Tanh()]
    for _ in range(L - 1):
        mods += [torch.nn.Linear(H, H), torch.nn.Tanh()]
    seq = torch.nn.Sequential(*mods, torch.nn.Linear(H, gen.output_features)).to(gen.w_in.device)
    seq.load_state_dict({k[len("_network."):]: v for k, v in gen.state_dict().items()})
    return seq


def c1_train_step_ms(reps):
    dev = torch.device("cuda")
    torch.manual_seed(0)
    gen = NNGenerator(2, 2, 3, 64, device=dev)
    wl = workloads.rotations_2d(7, 64, 3.5)
    tfs = [mf.simulate.LinearTransform(m.to(dev)) for m in wl["matrices"]]
    diag = mf.diagnostics.Histogram1D(axis=0, edges=wl["edges"], bandwidth=0.5).to(dev)
    diags = [[diag] for _ in tfs]
    truth = workloads.gaussian_mixture(50_000, ndim=2, seed=1, device=dev)
    with torch.no_grad():
        meas = [[p[0]] for p in mf.simulate.forward(truth, tfs, diags)]
    model = mf.MENTFlow(transforms=tfs, diagnostics=diags, measurements=meas, generator=gen, prior=None,
                        entropy_estimator=mf.entropy.CovarianceEntropyEstimator(),
                        discrepancy_function=mf.loss.kl_divergence, penalty_parameter=50.0)
    opt = torch.optim.AdamW(model.parameters(), lr=1e-3, weight_decay=0.0, capturable=True, fused=True)
    step = GraphedTrainStep(model, opt, 25_000)
    return median_ms(step, reps, warm=5)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    dev = torch.device("cuda")
    info = card()
    clock_mhz = float(str(info.get("clocks.max.sm", "1965")).split()[0])
    L, H = 3, 64
    rows = []
    for din, dout in ((6, 6), (2, 2)):
        for n in (25_000, 1_000_000):
            torch.manual_seed(0)
            gen = NNGenerator(din, dout, L, H, device=dev)
            seq = sequential_like(gen)
            z = torch.randn(n, din, device=dev)
            c = torch.randn(n, dout, device=dev)
            with torch.no_grad():
                x, xt = gen(z), seq(z)
            err = float(((x - xt).abs() / xt.abs().clamp_min(1.0)).max())

            def fwd():
                with torch.no_grad():
                    gen(z)

            def fwd_bwd():
                (gen(z) * c).sum().backward()

            def t_fwd():
                with torch.no_grad():
                    seq(z)

            def t_fwd_bwd():
                (seq(z) * c).sum().backward()

            nsf = NSFGenerator(dout, hidden_units=64, hidden_layers=3, transforms=5, bins=20, device=dev) \
                if dout >= 2 else None

            def nsf_sample():
                with torch.no_grad():
                    nsf.sample(n)

            fma = n * (H * din + H * H * (L - 1) + H * dout)
            row = {"din": din, "dout": dout, "hidden_units": H, "hidden_layers": L, "n": n,
                   "forward_ms": round(median_ms(fwd, args.reps), 4),
                   "forward_backward_ms": round(median_ms(fwd_bwd, args.reps), 4),
                   "torch_forward_ms": round(median_ms(t_fwd, args.reps), 4),
                   "torch_forward_backward_ms": round(median_ms(t_fwd_bwd, args.reps), 4),
                   "nsf_sample_ms": round(median_ms(nsf_sample, args.reps), 4) if nsf is not None else None,
                   "fma_per_particle": fma // n,
                   "fma_floor_ms": round(fma / (148 * 128 * clock_mhz * 1e6) * 1e3, 4),
                   "max_rel_diff_vs_torch": err}
            if (din, dout) == (2, 2) and n == 25_000:
                row["c1_train_step_ms"] = round(c1_train_step_ms(args.reps), 4)
            row.update({"gpu": info.get("name"), "power_limit": info.get("power.limit"),
                        "sm_clock_max": info.get("clocks.max.sm"), "sm_clock": info.get("clocks.sm")})
            rows.append(row)
            print(json.dumps(row), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            for row in rows:
                f.write(json.dumps(row) + "\n")


if __name__ == "__main__":
    main()
