"""k-NN entropy of a sharded MENTFlow on two GPUs (two spawned processes, NCCL): the entropy is bit for bit that of one
GPU on the union particles, the loss and the generator gradients agree with one GPU to the shard-parity bar, and a
sharded GraphedLoss replay equals the eager step.  Skipped when fewer than two devices are visible."""
import os
import socket

import pytest
import torch
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu

WORLD = 2
N_LOCAL = 12_000


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _model(device):
    import mentflow_b200 as mf
    from mentflow_b200 import workloads
    wl = workloads.isotropic_1d(ndim=6, num=6, bins=48, xmax=3.5, seed=2)
    tfs = [mf.simulate.LinearTransform(m.to(device)) for m in wl["matrices"]]
    diag = mf.diagnostics.Histogram1D(axis=0, edges=wl["edges"], bandwidth=0.5).to(device)
    diags = [[diag] for _ in tfs]
    truth = workloads.gaussian_mixture(50_000, ndim=6, seed=1, device=device)
    with torch.no_grad():
        meas = [[p[0]] for p in mf.simulate.forward(truth, tfs, diags)]
    torch.manual_seed(5)
    gen = mf.generate.NNGenerator(6, 6, 3, 64, device=device)
    return mf.MENTFlow(transforms=tfs, diagnostics=diags, measurements=meas, generator=gen, prior=None,
                       entropy_estimator=mf.entropy.KNNEntropyEstimator(k=5),
                       discrepancy_function=mf.loss.kl_divergence, penalty_parameter=20.0)


def _worker(rank, port, equal, out):
    import torch.distributed as dist

    from mentflow_b200 import distributed as mfd
    from mentflow_b200.graphs import GraphedLoss
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    device = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=WORLD, device_id=device)
    try:
        model = _model(device)
        gen, est = model.generator, model.entropy_estimator
        params = list(gen.parameters())
        reducer = mfd.shard_model(model, equal_shards=equal)
        n_total = WORLD * N_LOCAL + (0 if equal else 1)
        sl = mfd.shard_slice(n_total, rank, WORLD)
        z_all = torch.randn(n_total, 6, generator=torch.Generator(device=device).manual_seed(7), device=device)
        z = z_all[sl].contiguous()

        res = {}
        # sharded: this rank's particles, loss of the union batch, gradients summed over ranks
        for p in params:
            p.grad = None
        x, lq = gen.forward_and_log_prob(z)
        L, H, D = model.loss_from_particles(x, lq)
        L.backward()
        mfd.allreduce_gradients(params)
        grads = [p.grad.clone() for p in params]
        hs = [torch.empty_like(H) for _ in range(WORLD)]
        dist.all_gather(hs, H.detach())
        res["h_same_on_every_rank"] = all(torch.equal(h, hs[0]) for h in hs)

        # one GPU on the union particles: no reducer anywhere
        model.reducer = est.reducer = None
        for p in params:
            p.grad = None
        xu, lqu = gen.forward_and_log_prob(z_all)
        res["x_rows_equal"] = torch.equal(xu[sl].detach(), x.detach())
        Lu, Hu, Du = model.loss_from_particles(xu, lqu)
        Lu.backward()
        res["h_bitwise"] = torch.equal(H.detach(), Hu.detach())
        res["h"], res["h_union"] = float(H), float(Hu)
        res["rel_loss"] = float((L.detach() - Lu.detach()).abs() / Lu.detach().abs())
        gmax = max(float(p.grad.abs().max()) for p in params)
        res["rel_grad"] = max(float((g - p.grad).abs().max()) for g, p in zip(grads, params)) / gmax
        model.reducer = est.reducer = reducer

        # a sharded GraphedLoss replay against the eager step (equal shards: nothing waits for the host)
        if equal:
            graphed = GraphedLoss(model, N_LOCAL)
            Lg, Hg, Dg = graphed(z)
            Lg, Hg, Dg = graphed(z)
            with torch.no_grad():
                xe, lqe = gen.forward_and_log_prob(z)
                Le, He, De = model.loss_from_particles(xe, lqe)
            res["graph_bitwise"] = (torch.equal(Lg, Le) and torch.equal(Hg, He)
                                    and torch.equal(torch.stack(Dg), torch.stack(De)))
            res["graph_h_bitwise_to_union"] = torch.equal(Hg, Hu.detach())
        torch.cuda.synchronize()
        out.put((rank, res))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("equal", [True, False], ids=["equal_shards", "ragged_shards"])
def test_sharded_knn_entropy_matches_one_gpu(equal):
    if torch.cuda.device_count() < WORLD:
        pytest.skip(f"needs {WORLD} CUDA devices, {torch.cuda.device_count()} visible")
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, port, equal, out)) for r in range(WORLD)]
    for p in procs:
        p.start()
    try:
        for p in procs:
            p.join(timeout=600)
        assert all(p.exitcode == 0 for p in procs), [p.exitcode for p in procs]
        results = dict(out.get(timeout=30) for _ in procs)
    finally:
        for p in procs:
            if p.is_alive():
                p.kill()
                p.join(timeout=30)
    for rank, res in results.items():
        assert res["h_same_on_every_rank"] and res["x_rows_equal"], (rank, res)
        assert res["h_bitwise"], (rank, res)
        assert res["rel_loss"] <= 1e-5, (rank, res)
        assert res["rel_grad"] <= 1e-5, (rank, res)
        if equal:
            assert res["graph_bitwise"] and res["graph_h_bitwise_to_union"], (rank, res)
