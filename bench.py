#!/usr/bin/env python
"""Benchmark of the MENT-Flow hot path on B200 (see DESIGN.md "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

One *step* = one pass of the hot path over one batch of particles on every rank:
flow sample + log-density (5 fused NSF layers) -> Monte-Carlo entropy -> fused projection + KDE
for all K screens -> KL discrepancies -> loss  (MENTFlow.loss, forward).  Workload = BASELINE
config C3: 6D, K=100 random 1-D projections, 64 bins, `--particles` (default 1e6) per GPU.

Prints ONE JSON line (rank 0).  `value` = particles/s over all ranks with the base-noise z
already resident in HBM, timed with CUDA events (max over ranks); `e2e` = the same through the
public API with z arriving from pinned host memory and the loss read back every step.

`--dump-outputs DIR` writes what the last step of `value`'s timed loop returned -- loss.npy,
entropy.npy and discrepancies.npy (one per projection) -- so that two builds run with the same
arguments (hence the same seeded weights, measurements and base noise) can be compared.
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# algorithmic work per particle, D=6, K=100, B=64 (SURVEY.md 8d / DESIGN.md)
FLOP_MASK_AWARE = {6: 165_520, 4: 132_000, 2: 120_320}
FLOP_DENSE = {6: 312_320, 4: 235_520, 2: 158_720}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--particles", type=int, default=1_000_000, help="particles per GPU per step")
    ap.add_argument("--ndim", type=int, default=6)
    ap.add_argument("--num-proj", type=int, default=100)
    ap.add_argument("--bins", type=int, default=64)
    ap.add_argument("--cpu-particles", type=int, default=25_000, help="sample size of the CPU baseline step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--host-chunks", type=int, default=3, help="pieces the pinned-host input is copied in (e2e leg)")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel eagerly instead of replaying a CUDA graph")
    ap.add_argument("--no-extra", action="store_true", help="skip the secondary configurations (C1, C3/25, C4, training steps)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the loss, entropy and discrepancies of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs records the CUDA path (--impl b200)")
    return args


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"],
                "bf16_tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


# ----------------------------------------------------------------------------------------
# clocks during the timed region
# ----------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop_evt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        while not self._stop_evt.is_set():
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                mask = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.05)

    def finish(self):
        self._stop_evt.set()
        self.join(timeout=2)
        med = statistics.median(self.samples) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ----------------------------------------------------------------------------------------
# workload
# ----------------------------------------------------------------------------------------
def trained_like_(module, factor=3.0):
    """Default initialisation leaves the flow close to the identity; scaling the weights makes
    particles spread over the screens and over the spline bins (SURVEY.md 8d)."""
    with torch.no_grad():
        for p in module.parameters():
            p.mul_(factor)


def build_model(args, device):
    import mentflow_b200 as mf
    from mentflow_b200 import workloads
    wl = workloads.isotropic_1d(ndim=args.ndim, num=args.num_proj, bins=args.bins, xmax=3.5, seed=0)
    torch.manual_seed(0)
    gen = mf.generate.build_generator("nsf", input_features=args.ndim, output_features=args.ndim, hidden_layers=3,
                                      hidden_units=64, transforms=5, bins=20)
    trained_like_(gen)
    gen = gen.to(device)
    tfs = [mf.simulate.LinearTransform(m.to(device)) for m in wl["matrices"]]
    diag = mf.diagnostics.Histogram1D(axis=0, edges=wl["edges"], bandwidth=0.5).to(device)
    diags = [[diag] for _ in tfs]
    # measurements: exact histograms of a synthetic 6-D Gaussian mixture (experiments/setup.py:52-73)
    truth = workloads.gaussian_mixture(200_000, ndim=args.ndim, seed=1, device=device)
    diag.kde = False
    meas = mf.simulate.forward(truth, tfs, diags)
    diag.kde = True
    width = float(wl["edges"][1] - wl["edges"][0])
    meas = [[m[0] / m[0].sum() / width] for m in meas]
    prior = mf.prior.Gaussian(ndim=args.ndim, scale=3.0)
    model = mf.MENTFlow(transforms=tfs, diagnostics=diags, measurements=meas, generator=gen, prior=prior,
                        entropy_estimator=mf.entropy.MonteCarloEntropyEstimator(prior=prior),
                        discrepancy_function=mf.loss.kl_divergence, penalty_parameter=25.0)
    return model, wl


def cpu_step_factory(args):
    """The same step through the CPU oracle (torch-CPU port of the reference's dense arithmetic
    + restatement of zuko's NSF), all host threads."""
    from mentflow_b200 import workloads
    from oracle import hotpath as hp
    from oracle.zuko_nsf import NSFOracle
    torch.set_num_threads(os.cpu_count() or 1)
    wl = workloads.isotropic_1d(ndim=args.ndim, num=args.num_proj, bins=args.bins, xmax=3.5, seed=0)
    torch.manual_seed(0)
    flow = NSFOracle(args.ndim)
    trained_like_(flow)
    screens = [[hp.Screen1D(edges=wl["edges"], bandwidth=0.5)] for _ in wl["matrices"]]
    truth = workloads.gaussian_mixture(200_000, ndim=args.ndim, seed=1)
    width = wl["edges"][1] - wl["edges"][0]
    meas = []
    for m in wl["matrices"]:
        h = hp.hist_density_1d(hp.linear_map(truth, m)[:, 0], wl["edges"])
        meas.append([h / h.sum() / width])
    n = args.cpu_particles

    def step():
        with torch.no_grad():
            x, logq = flow.sample_and_log_prob(n)
            L, H, D = hp.mentflow_loss(x, logq, wl["matrices"], screens, meas, 3.0, 25.0)
        return float(L)

    return step, n


def time_cpu(step, n, reps, warmup=1, budget_s=12.0):
    """Best step time over at least `reps` steps and about `budget_s` seconds of CPU work."""
    for _ in range(warmup):
        step()
    ts = []
    while len(ts) < reps or (sum(ts) < budget_s and len(ts) < 200):
        t0 = time.perf_counter()
        step()
        ts.append(time.perf_counter() - t0)
    return n / min(ts), ts


# ncu --set full capture of ONE nsf_tc_layer_kernel<6,3,20> launch of this workload (profiles/, this round)
NCU_PROFILE = {
    "file": "profiles/r2_full_metrics.txt",
    "dram_bytes_per_launch": 28.18e6 + 0.20e6,          # dram__bytes_read.sum + dram__bytes_write.sum
    "pipes": {"issue_active_pct": 62.8, "xu_mufu_pct": 40.6, "tensor_pct": 40.4, "fma_pct": 29.3, "lsu_pct": 8.1,
              "dram_pct": 1.8, "warps_active_pct": 25.0,
              "note": "no pipe is saturated: three compute warps per scheduler at the latency-bound issue rate"},
}


def shard_parity_check(model, reducer, gen, n, d, rank, world, device):
    """N > 1: the sharded step against ONE GPU doing the union batch on the same particles, outside every timed
    region.  Each rank pushes its own base noise through the flow; rank 0 gathers the particles of all ranks and
    evaluates profiles and loss unsharded.  {max_rel_profile, rel_loss}; the run fails beyond 1e-5."""
    import torch.distributed as dist

    import mentflow_b200 as mf
    with torch.no_grad():
        z = gen.sample_base(n)
        x, logq = gen.forward_and_log_prob(z)
        preds = mf.simulate.forward(x, model.transforms, model.diagnostics, reducer=reducer)
        prof = torch.stack([p[0] for p in preds])
        L = model.loss_from_particles(x, logq)[0]
        xs = [torch.empty_like(x) for _ in range(world)] if rank == 0 else None
        ls = [torch.empty_like(logq) for _ in range(world)] if rank == 0 else None
        dist.gather(x, xs, dst=0)
        dist.gather(logq, ls, dst=0)
        out = None
        if rank == 0:
            x_all, l_all = torch.cat(xs), torch.cat(ls)
            saved, saved_e = model.reducer, model.entropy_estimator.reducer
            model.reducer = model.entropy_estimator.reducer = None
            try:
                preds_u = mf.simulate.forward(x_all, model.transforms, model.diagnostics)
                prof_u = torch.stack([p[0] for p in preds_u])
                L_u = model.loss_from_particles(x_all, l_all)[0]
            finally:
                model.reducer, model.entropy_estimator.reducer = saved, saved_e
            rel_p = float(((prof - prof_u).abs().amax(dim=1) / prof_u.abs().amax(dim=1)).max())
            rel_l = float((L - L_u).abs() / L_u.abs())
            out = {"max_rel_profile": rel_p, "rel_loss": rel_l, "particles": int(x_all.shape[0]),
                   "ok": bool(rel_p <= 1e-5 and rel_l <= 1e-5),
                   "what": "sharded step (NCCL all-reduce of the unnormalised sums) vs the union batch on one GPU, same particles"}
        dist.barrier()
        torch.cuda.synchronize()
    return out


def _timed(fn, reps=5, warm=2, flush=None):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        if flush is not None:
            flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return statistics.median(ts)


def extras(args, device, pk):
    """The other BASELINE configurations on one GPU, after (and outside) the headline measurement: each entry
    is one forward step (or training step) through the public API, median of CUDA-event timings after warm-up,
    256 MB L2 flush between repeats, with the roofline that bounds its dominant kernel."""
    import math

    import mentflow_b200 as mf
    from mentflow_b200 import workloads
    from mentflow_b200.graphs import GraphedLoss, GraphedTrainStep
    N = args.particles
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=device)
    out = []

    def model_for(wl, d, kind, n_truth=200_000):
        torch.manual_seed(0)
        gen = mf.generate.NSFGenerator(d)
        trained_like_(gen)
        gen = gen.to(device)
        tfs = [mf.simulate.LinearTransform(m.to(device)) for m in wl["matrices"]]
        if kind == "1d":
            diag = mf.diagnostics.Histogram1D(axis=0, edges=wl["edges"], bandwidth=0.5).to(device)
        else:
            diag = mf.diagnostics.Histogram2D(axis=wl["axis"], edges=wl["edges"], bandwidth=(0.5, 0.5)).to(device)
        diags = [[diag] for _ in tfs]
        truth = workloads.gaussian_mixture(n_truth, ndim=d, seed=1, device=device)
        with torch.no_grad():
            meas = [[m[0].detach()] for m in mf.simulate.forward(truth, tfs, diags)]
        prior = mf.prior.Gaussian(ndim=d, scale=3.0)
        return mf.MENTFlow(transforms=tfs, diagnostics=diags, measurements=meas, generator=gen, prior=prior,
                           entropy_estimator=mf.entropy.MonteCarloEntropyEstimator(prior=prior),
                           discrepancy_function=mf.loss.kl_divergence, penalty_parameter=25.0)

    def tensor_roof(flop_per_particle, n, ms, kernel):
        a = flop_per_particle * n / (ms * 1e-3) / 1e12
        return {"bound": "tensor", "kernel": kernel, "achieved": a, "peak": pk["bf16_tflops_sustained"], "unit": "TFLOP/s",
                "frac": a / pk["bf16_tflops_sustained"], "traffic": None,
                "note": "whole step time as divisor (kernel inside a step: sustained peak); mask-aware algorithmic FLOP"}

    def entry(case, n, ms, roof, **kw):
        out.append({"case": case, "particles_per_step": n, "ms_per_step": ms, "value": n / ms * 1e3, "unit": "particles/s",
                    "roofline": roof, **kw})

    # C1 rec_2d/linear: 2-D flow, 7 rotations, 85 bins
    m1 = model_for(workloads.rotations_2d(7, 85, 3.5), 2, "1d")
    g1 = GraphedLoss(m1, N)
    ms = _timed(lambda: g1(None), flush=flush)
    hbm_bytes = 5 * (2 * 2 * 4 + 8) + 2 * 4 + 2 * 2 * 4      # flow layers (v in, y out, log q) + draw + one read by entropy and KDE each
    roof = tensor_roof(FLOP_MASK_AWARE[2], N, ms, "nsf_tc_layer_kernel<2,3,20> x5")
    roof["hbm"] = {"bound": "hbm", "achieved": hbm_bytes * N / (ms * 1e-3) / 1e9, "peak": pk["hbm_gbs"], "unit": "GB/s",
                   "frac": hbm_bytes * N / (ms * 1e-3) / 1e9 / pk["hbm_gbs"], "algorithmic_bytes_per_particle": hbm_bytes}
    entry("C1 rec_2d/linear: 2-D NSF + 7 x KDE-1D(85) + KL, forward (graph replay, draw inside)", N, ms, roof)
    del g1, m1
    # C3 with 25 projections
    m25 = model_for(workloads.isotropic_1d(6, 25, 64, 3.5), 6, "1d")
    g25 = GraphedLoss(m25, N)
    ms = _timed(lambda: g25(None), flush=flush)
    entry("C3 rec_nd_1d, 25 projections: 6-D NSF + 25 x KDE-1D(64) + KL, forward (graph replay)", N, ms,
          tensor_roof(FLOP_MASK_AWARE[6], N, ms, "nsf_tc_layer_kernel<6,3,20> x5"))
    del g25, m25
    # C3 at the reference's batch sizes (100 projections)
    m3 = model_for(workloads.isotropic_1d(6, args.num_proj, args.bins, 3.5), 6, "1d")
    for nb in (25_000, 100_000):
        g3 = GraphedLoss(m3, nb)
        ms = _timed(lambda: g3(None), reps=9, flush=flush)
        entry(f"C3 rec_nd_1d, {args.num_proj} projections at the reference batch size, forward (graph replay)", nb, ms,
              tensor_roof(FLOP_MASK_AWARE[6], nb, ms, "nsf_tc_layer_kernel<6,3,20> x5"))
        del g3
    # optimisation steps: zero_grad + loss + backward + AdamW as one graph replay
    for nb in (25_000, N):
        opt = torch.optim.AdamW(m3.parameters(), lr=1e-5, weight_decay=0.0, capturable=True, fused=True)
        gts = GraphedTrainStep(m3, opt, nb)
        ms = _timed(gts, reps=5, flush=flush)
        entry("C3 optimisation step (zero_grad + loss + backward + fused AdamW) as one CUDA-graph replay", nb, ms,
              tensor_roof(3 * FLOP_MASK_AWARE[6], nb, ms, "nsf_tc_layer_kernel<6,3,20,bwd> + dgrad + wgrad x5"))
        del gts, opt
    # density direction: log_prob(x) of the flow (generate/flows/zuko.py:21-22), tensor-core inverse kernel, default-init
    # x 1.5 weights (the inverse of a x3 flow is ill-conditioned in any fp32 arithmetic)
    torch.manual_seed(0)
    ginv = mf.generate.NSFGenerator(6)
    with torch.no_grad():
        for p_ in ginv.parameters():
            p_.mul_(1.5)
        ginv = ginv.to(device)
        xi, lqi = ginv.sample_and_log_prob(N)
        ms = _timed(lambda: ginv.log_prob(xi), reps=5, flush=flush)
        dev_lp = float((ginv.log_prob(xi) - lqi).abs().max())
    entry("flow log_prob(x), density direction: 6-D NSF inverse x5 (tcgen05 inverse kernel, eager launches)", N, ms,
          tensor_roof(5 * 5 * 2 * (16 * 64 + 2 * 64 * 64 + 64 * 64), N, ms,
                      "nsf_tc_inverse_kernel<6,3,20> x5 (dense-equivalent FLOP of 5 conditioner passes per layer)"),
          max_abs_round_trip_error=dev_lp)
    del ginv, xi, lqi
    del m3
    # C4 rec_nd_2d: 15 two-dimensional screens 85 x 85
    m4 = model_for(workloads.corner_2d(6, 85, 3.5), 6, "2d", n_truth=100_000)
    g4 = GraphedLoss(m4, N)
    ms = _timed(lambda: g4(None), reps=3, warm=1, flush=flush)
    with torch.no_grad():
        x4 = m4.generator.forward(torch.randn(N, 6, device=device))
        ms_scr = _timed(lambda: mf.simulate.forward(x4, m4.transforms, m4.diagnostics), reps=3, warm=1, flush=flush)
    flop_scr = 15 * 2 * 85 * 85      # the screens as a GEMM: K_x^T K_y per screen, 2 * Bx * By per particle
    entry("C4 rec_nd_2d: 6-D NSF + 15 x KDE-2D(85x85) + KL, forward (graph replay)", N, ms,
          tensor_roof(FLOP_MASK_AWARE[6] + flop_scr, N, ms, "kde2d_tc_kernel + nsf_tc_layer_kernel<6,3,20> x5"),
          screens_only_ms=ms_scr,
          screens_roofline=tensor_roof(flop_scr, N, ms_scr, "kde2d_tc_kernel (tcgen05 split-bf16, accumulators in TMEM)"))
    del g4

    def train4():
        for p_ in m4.parameters():
            p_.grad = None
        m4.loss(N)[0].backward()

    ms = _timed(train4, reps=3, warm=1, flush=flush)
    entry("C4 training step: forward + backward to all flow parameters (eager)", N, ms,
          tensor_roof(3 * FLOP_MASK_AWARE[6] + 2 * flop_scr, N, ms, "nsf backward kernels + kde2d_bwd_kernel"))
    del m4, x4, flush
    torch.cuda.empty_cache()
    out.append(ment_step_measure(device, 0, 1))
    return out


def ment_step_measure(device, rank, world, n_per_gpu=12_500_000, num_proj=25, res=16, bins=64, reps=2, parity=True):
    """BASELINE config 5: classical MENT, 6-D, `num_proj` 1-D screens, density on a res^6 sampler grid, one
    gauss_seidel_step = num_proj measurement updates, each drawing n_per_gpu x world particles (sample mode,
    ment.py:319-371).  Particles are sharded: every rank draws its slice of one Philox stream and the unnormalised
    profile sums are all-reduced (NCCL) before the update.  Timed with CUDA events, max over ranks."""
    import torch.distributed as dist

    import mentflow_b200 as mf
    from mentflow_b200 import distributed as mfd
    from mentflow_b200 import workloads
    d, xmax = 6, 3.5
    wl = workloads.isotropic_1d(d, num_proj, bins, xmax)
    tfs = [mf.simulate.LinearTransform(m.to(device)) for m in wl["matrices"]]
    diag = mf.diagnostics.Histogram1D(axis=0, edges=wl["edges"], bandwidth=0.5).to(device)
    diags = [[diag] for _ in tfs]
    truth = workloads.gaussian_mixture(200_000, ndim=d, seed=1, device=device)
    with torch.no_grad():
        meas = [[p[0]] for p in mf.simulate.forward(truth, tfs, diags)]

    def make(n_total, shard):
        sampler = mf.sample.GridSampler(limits=d * [(-xmax, xmax)], shape=tuple(d * [res]), device=device)
        m = mf.ment.MENT(ndim=d, transforms=tfs, diagnostics=diags, measurements=meas,
                         prior=mf.prior.Gaussian(ndim=d, scale=3.0), mode="sample", sampler=sampler, n_samples=n_total,
                         device=device)
        if shard and world > 1:
            mfd.shard_model(m)
        return m

    n_total = n_per_gpu * world
    model = make(n_total, True)
    torch.manual_seed(77)                    # the same sampler seeds on every rank
    model.gauss_seidel_update(lr=0.9)        # warm-up sweep
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        model.gauss_seidel_update(lr=0.9)
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    t = torch.tensor([min(ms)], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    step_ms = float(t[0])
    out = {"case": f"C5 classical MENT gauss_seidel_step: 6-D, {num_proj} x KDE-1D({bins}), sampler grid {res}^6, "
                   f"{n_per_gpu} sampled particles per GPU and measurement update",
           "n_gpus": world, "particles_per_step": n_total * num_proj, "ms_per_step": step_ms,
           "value": n_total * num_proj / step_ms * 1e3, "unit": "sampled particles/s",
           "grid_points_per_s": res ** d * num_proj / step_ms * 1e3}
    if parity and world > 1:
        # One measurement update, sharded, against the same update on ONE GPU from the same tables and sampler seed:
        # the ranks' slices are the particles one GPU draws, so the predicted profile differs by fp32 summation
        # order only.  (A whole sweep cannot be compared this way: a 1e-7 change of a table moves the inverse-CDF
        # cell of a sizeable fraction of the next update's particles, i.e. the later updates see a different --
        # statistically equivalent -- sample.)
        start = [lf[0].values.clone() for lf in model.lagrange_functions]
        torch.manual_seed(78)
        got = model.simulate(0, 0)
        rel = None
        if rank == 0:
            single = make(n_total, False)
            for lf, v in zip(single.lagrange_functions, start):
                lf[0].set_values(v.clone())
            torch.manual_seed(78)
            want = single.simulate(0, 0)
            rel = float((got - want).abs().max() / want.abs().max())
        dist.barrier()
        if rank == 0:
            out["shard_parity"] = {"max_rel_profile": rel, "ok": bool(rel <= 1e-5), "particles": n_total,
                                   "what": "predicted profile of one sharded measurement update (slices of one Philox "
                                           "stream + NCCL all-reduce of the sums) vs the same update on one GPU"}
    return out


# ----------------------------------------------------------------------------------------
def run_reference(args, rank):
    if rank != 0:
        return
    step, n = cpu_step_factory(args)
    for _ in range(max(1, min(args.warmup, 2))):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    value = n * args.steps / dt
    cores = torch.get_num_threads()
    sample = f"{n} particles per step (reference batch size, experiments/rec_nd_1d/run_gmm.sh:21)"
    line = {
        "impl": "reference", "metric": "particles/sec/GPU for flow sample+log_prob+project+KDE (6D, 100 proj)",
        "value": value, "unit": "particles/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"rec_nd_1d C3: D={args.ndim}, K={args.num_proj} 1-D projections, B={args.bins}, "
                               f"NSF 5x[64,64,64] bins=20; CPU oracle port on {cores} host threads",
                   "particles_per_step": n},
        "cpu_baseline": {"value": value, "unit": "particles/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "particles/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: mentflow_b200 has no CPU fallback "
                         "(use --impl reference for the CPU baseline)")
    import torch.distributed as dist

    import mentflow_b200 as mf
    from mentflow_b200 import distributed as mfd
    from mentflow_b200 import ops

    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        # NCCL prints its version banner on stdout when the communicator comes up; rank 0 must print ONE
        # JSON line there, so stdout points at stderr until the first collective has run
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=device)
            dist.all_reduce(torch.zeros(1, device=device))
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
    model, wl = build_model(args, device)
    reducer = mfd.shard_model(model, equal_shards=True) if world > 1 else None
    gen = model.generator
    n, d = args.particles, args.ndim

    torch.cuda.manual_seed(1234 + rank)      # a distinct Philox stream per rank for the draws inside the step
    # base noise resident in HBM / pinned host memory for the legs that are handed z (a distinct block per rank)
    g = torch.Generator(device=device).manual_seed(1234 + rank)
    z_dev = torch.randn(n, d, generator=g, device=device)
    z_host = torch.empty(n, d, dtype=torch.float32).pin_memory()
    z_host.copy_(z_dev.cpu())
    z_in = torch.empty_like(z_dev)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=device)  # 256 MB > 126 MB L2

    ev = lambda: torch.cuda.Event(enable_timing=True)
    nsf_ms, kde_ms = [], []

    def step(z, timers=None):
        with torch.no_grad():
            if timers:
                timers[0].record()
            x, logq = gen.forward_and_log_prob(z)
            if timers:
                timers[1].record()
            L, H, D = model.loss_from_particles(x, logq)
            if timers:
                timers[2].record()
        return L, H, D

    params = list(model.parameters())

    def train_step(z):
        """forward + hand-written backward (+ gradient all-reduce): what one optimiser step costs"""
        for p_ in params:
            p_.grad = None
        x, logq = gen.forward_and_log_prob(z)
        L, H, D = model.loss_from_particles(x, logq)
        L.backward()
        if world > 1:
            mfd.allreduce_gradients(params)
        return L

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # One step = one replay of the captured CUDA graph of the public forward pass
    # (mentflow_b200.graphs.GraphedLoss: generator.forward_and_log_prob + MENTFlow.loss_from_particles);
    # at N > 1 the NCCL all-reduce of the unnormalised profile sums is one node of the graph.  The timed
    # loop does not synchronise between steps, so the host runs ahead of the device in either mode.
    use_graph = not args.no_graph
    graphed = None
    if use_graph:
        from mentflow_b200.graphs import GraphedLoss
        graphed = GraphedLoss(model, n, warmup=2, host_chunks=args.host_chunks)

    def run_step(z):
        """(L, H, [D_k]) of one step"""
        if graphed is not None:
            return graphed(z)
        if z is None:
            z = gen.sample_base(n)
        return step(z)

    for _ in range(max(args.warmup, 3)):
        flush.zero_()
        run_step(None)
        run_step(z_dev)
        run_step(z_host if graphed is not None else z_dev)   # binds the pinned buffer to the host-input graph
        step(z_dev)
    barrier()

    sampler = ClockSampler(local_rank)
    sampler.start()
    # ---- per-section timing (eager launches): the NSF layer kernels vs the rest of the step --------
    for _ in range(args.steps):
        flush.zero_()
        tm = [ev() for _ in range(3)]
        step(z_dev, tm)
        tm[2].synchronize()
        nsf_ms.append(tm[0].elapsed_time(tm[1]))
        kde_ms.append(tm[1].elapsed_time(tm[2]))
    barrier()
    # ---- device-resident timing -------------------------------------------------------
    total_ms = 0.0
    losses = []
    z_res = z_dev
    if graphed is not None:
        graphed.z.copy_(z_dev)             # the graph's own input buffer: z is resident, nothing is copied
        z_res = graphed.z
    barrier()
    marks = []
    for _ in range(args.steps):
        flush.zero_()                      # evict L2 between timed iterations (outside the [e0, e1] bracket)
        e0, e1 = ev(), ev()
        e0.record()
        L, H, D = run_step(None)           # the base noise is drawn on the device inside the step (Philox)
        e1.record()
        marks.append((e0, e1))
        losses.append(L.clone())
    barrier()
    total_ms = sum(a.elapsed_time(b) for a, b in marks)
    if args.dump_outputs and rank == 0:
        # a graph replay returns its static output tensors: save them before the next leg replays the graph
        os.makedirs(args.dump_outputs, exist_ok=True)
        outputs = {"loss": L, "entropy": torch.as_tensor(H), "discrepancies": torch.stack(D)}
        for name, t in outputs.items():
            t = t.detach().cpu()
            np.save(os.path.join(args.dump_outputs, name + ".npy"),
                    t.numpy().astype(np.float64 if t.dtype == torch.float64 else np.float32))
    # ---- end to end through the public API: model.loss(batch_size) as GraphedLoss(model, n)() -------
    # The step's only host-side inputs are the batch size (a constant of the captured graph) and the state
    # of torch's random generator.  Every step re-seeds the generator the way a reproducible training loop
    # does (torch.cuda.manual_seed(step)), so the 16-byte (seed, offset) pair crosses from pinned host
    # memory inside the timed region; the loss is read back to the host (4 bytes) every step.
    def e2e_step(it):
        torch.cuda.manual_seed(10_000 + 1_000_003 * rank + it)
        if graphed is not None:
            L = graphed(None)[0]
        else:
            L = step(gen.sample_base(n))[0]
        return float(L.item())

    e2e_s = 0.0
    for it in range(-2, args.steps):       # two untimed passes of this very loop first
        flush.zero_()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        lval = e2e_step(it)
        if it < 0:
            continue
        e2e_s += time.perf_counter() - t0
    barrier()
    # ---- the same with the base noise handed over in pinned HOST memory (round-1 e2e leg): 24 B per
    #      particle cross PCIe every step, copied in pieces that overlap the flow layers
    host_s = 0.0
    for it in range(-2, args.steps):
        flush.zero_()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        if graphed is not None:
            L = run_step(z_host)[0]        # pinned host -> device copy, then the replay
        else:
            z_in.copy_(z_host, non_blocking=True)
            L = step(z_in)[0]
        lval = float(L.item())
        if it < 0:
            continue
        host_s += time.perf_counter() - t0
    barrier()
    # ---- training step (forward + backward), reported beside the headline ----------------------
    tsteps = max(2, args.steps // 4)
    train_step(z_dev)
    barrier()
    train_ms = 0.0
    for _ in range(tsteps):
        flush.zero_()
        e0, e1 = ev(), ev()
        e0.record()
        train_step(z_dev)
        e1.record()
        e1.synchronize()
        train_ms += e0.elapsed_time(e1)
    barrier()
    clocks = sampler.finish()

    shard_parity = shard_parity_check(model, reducer, gen, n, d, rank, world, device) if world > 1 else None
    ment_line = None
    if world > 1 and not args.no_extra:
        # BASELINE config 5 (classical MENT, particles sharded over the ranks), after and outside the headline timing
        ment_line = ment_step_measure(device, rank, world)

    t = torch.tensor([total_ms, e2e_s * 1e3, train_ms, host_s * 1e3], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, e2e_ms, train_ms, host_ms = float(t[0]), float(t[1]), float(t[2]), float(t[3])
    value = n * world * args.steps / (total_ms * 1e-3)
    e2e_value = n * world * args.steps / (e2e_ms * 1e-3)

    if rank == 0:
        pk = peaks()
        nsf_step_ms = statistics.mean(nsf_ms)
        flops = FLOP_MASK_AWARE.get(d, 0) * n
        achieved = flops / (nsf_step_ms * 1e-3) / 1e12
        layers = gen.transforms
        tc = ops.nsf_tc_supported(d, gen.hidden_units, gen.hidden_layers, gen.bins)
        nsf_kernel = (f"nsf_tc_layer_kernel<{d},3,20> x{layers} (tcgen05 split-fp16 conditioner, TMEM accumulators, "
                      f"register-resident spline epilogue)" if tc else
                      f"nsf_layer_fwd_kernel<{d}> x{layers} (fp32 CUDA-core kernel)")
        # the operand images are cached while the weights do not change: no prepare kernel in a forward-only step
        nsf_launches = {"nsf_tc_layer_kernel": layers} if tc else {"nsf_layer_fwd_kernel": layers}
        rest = {"randn_philox + advance": 2, "moments": 2, "mc_entropy": 1, "kde1d deposit + merge/normalise/KL": 2,
                "loss_tail": 1}
        if world > 1 and getattr(reducer, "peer", None) is None:
            rest["f64 split/join (packed all-reduce)"] = 2
        pieces = len(graphed._chunk_bounds()) if graphed is not None else 1
        prof = NCU_PROFILE if (tc and d == 6 and n == 1_000_000) else {}
        line = {
            "metric": "particles/sec/GPU for flow sample+log_prob+project+KDE (6D, 100 proj)",
            "value": value, "unit": "particles/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"rec_nd_1d C3: D={d}, K={args.num_proj} random 1-D projections, B={args.bins}, "
                                   f"NSF 5 layers x MaskedMLP[{d},64,64,64,{59 * d}] 20-bin RQ spline, forward "
                                   f"(base-noise draw + sample + log_prob + entropy + project + KDE + KL loss)",
                       "particles_per_gpu_per_step": n, "parallelism": f"particles sharded x{world}",
                       "cross_rank_sum": ("none (one GPU)" if world == 1 else
                                          "inside kde1d_finish_p2p_kernel: NVLink peer loads, epoch barrier in the kernel"
                                          if getattr(reducer, "peer", None) is not None else "NCCL all-reduce (packed)"),
                       "l2": "256 MB flush write between timed iterations",
                       "launch": ("CUDA graph replay of the forward step, base-noise draw (Philox) inside the graph "
                                  "(mentflow_b200.graphs.GraphedLoss)" if use_graph else "eager launches"),
                       "weights": "default init x3 (trained-like), seed 0", "value_per_gpu": value / world},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "particles/s", "h2d_bytes_per_step": 16,
                    "d2h_bytes_per_step": 4, "ms_per_step": e2e_ms / args.steps,
                    "api": ("torch.cuda.manual_seed(step); GraphedLoss(model, n)() [= model.loss(n): the base noise is drawn "
                            "on the device from torch's generator state, 16 B (seed, offset) from pinned host memory]; "
                            "loss.item()" if use_graph else
                            "torch.cuda.manual_seed(step); model.loss(n) eager; loss.item()")},
            # round-1 definition of the e2e leg, kept for comparison: z handed over in pinned host memory
            "e2e_host_z": {"value": n * world * args.steps / (host_ms * 1e-3), "unit": "particles/s",
                           "h2d_bytes_per_step": n * d * 4, "d2h_bytes_per_step": 4, "ms_per_step": host_ms / args.steps,
                           "api": "GraphedLoss(model, n)(z_pinned_host): chunked H2D copies overlapped with the flow; loss.item()"},
            # this library's kernels inside the timed region of `value` (one graph replay per step holds them all)
            "gpu_launches": args.steps * (sum(nsf_launches.values()) + sum(rest.values())),
            "gpu_launches_per_step": {**nsf_launches, **rest},
            "gpu_launches_per_e2e_host_z_step": {**{k: v * pieces for k, v in nsf_launches.items()}, "moments": 2,
                                                 "kde1d deposit + merge/normalise/KL": 2},
            "roofline": {"bound": "tensor", "kernel": nsf_kernel,
                         "achieved": achieved, "peak": pk["bf16_tflops"], "unit": "TFLOP/s",
                         "frac": achieved / pk["bf16_tflops"],
                         # dram__bytes_read.sum + dram__bytes_write.sum of one layer launch at this workload, from
                         # the ncu --set full capture named in `profile`
                         "traffic": prof.get("dram_bytes_per_launch"),
                         "traffic_unit": "bytes per layer launch (ncu)",
                         "peak_source": pk["source"] + " bf16 burst (the five layer launches are timed by CUDA events "
                                                       "around eager launches, i.e. alone)",
                         "frac_of_sustained_peak": achieved / pk["bf16_tflops_sustained"],
                         "algorithmic_flop_per_particle": FLOP_MASK_AWARE.get(d), "dense_equivalent_flop": FLOP_DENSE.get(d),
                         "kernel_ms_per_step": nsf_step_ms, "share_of_step": nsf_step_ms / (total_ms / args.steps),
                         "entropy_project_kde_loss_ms_per_step": statistics.mean(kde_ms),
                         "hbm_gbs_nsf": (n * (2 * d * 4 + 8) * layers) / (nsf_step_ms * 1e-3) / 1e9,
                         # the kernel is bound by instruction issue and the MUFU pipe, not by the tensor pipe: the
                         # pipe fractions ncu reports for the same launch (profile named below)
                         "pipe_fractions_ncu": prof.get("pipes"), "profile": prof.get("file")},
            "loss": float(losses[-1]),
            "train_step": {"value": n * world * tsteps / (train_ms * 1e-3), "unit": "particles/s",
                           "ms_per_step": train_ms / tsteps, "steps": tsteps,
                           "what": "loss forward + hand-written backward to all flow parameters"
                                   + (" + gradient all-reduce" if world > 1 else "")},
        }
        if shard_parity is not None:
            line["shard_parity"] = shard_parity
        if ment_line is not None:
            line["extra"] = [ment_line]
        if world == 1 and not args.no_cpu_baseline:
            stepf, ncpu = cpu_step_factory(args)
            v, ts = time_cpu(stepf, ncpu, reps=5)
            line["cpu_baseline"] = {"value": v, "unit": "particles/s", "cores": torch.get_num_threads(), "kind": "port",
                                    "sample": f"{ncpu} particles per step (the reference's batch size; NOT the GPU arm's "
                                              f"{n}: the dense (N, B) temporaries of the reference formulation need tens of "
                                              f"GB there), best of {len(ts)} after 1 warm-up "
                                              f"({sum(ts):.1f} s of CPU work); flow = oracle restatement of zuko NSF"}
        if world == 1 and not args.no_extra:
            del graphed
            line["extra"] = extras(args, device, pk)
        print(json.dumps(line), flush=True)
        if shard_parity is not None and not shard_parity["ok"]:
            print("shard parity violated: " + json.dumps(shard_parity), file=sys.stderr, flush=True)
            os._exit(3)
    if world > 1:
        # captured graphs hold NCCL work: drop them before the communicator goes away, and leave without
        # the (blocking) communicator teardown -- every rank is past its last collective here
        if graphed is not None:
            graphed.graph = graphed._host_graph = None
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
