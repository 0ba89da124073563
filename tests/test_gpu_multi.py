"""Multi-GPU (K sharded over ranks, SURVEY.md §8e): needs >= 2 CUDA devices (gpurun --gpus 2).
Each rank rolls out its slice; the (beta, eta, V) records are exchanged (a) inside the kernel over
NVLink peer mailboxes — the cluster records of every rank straight to every peer (direct mode) or one
combined record per rank —, (b) with an NCCL all-gather + mppi_apply_partials; all must reproduce the
unsharded update, identically on every rank — on the fused route, the stepped route (arbitrary callables) and the
tcgen05 route of the MLP model.  The log of a 2-GPU run is kept under profiles/."""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu


def _worker(rank, world, port, out, mode):
    import torch.distributed as dist
    split_mode, direct, cluster = mode
    os.environ["MPPI_B200_SPLIT_COST"] = split_mode      # "1": split-cost rollout (also on the shards), "0": single loop
    os.environ["MPPI_B200_XCHG_DIRECT"] = direct         # "1": cluster records straight to the peers, "0": one rank record
    os.environ["MPPI_B200_CLUSTER"] = cluster            # thread-block-cluster size limit of the warp-fold tail
    os.environ["MPPI_B200_XCHG_TIMEOUT_S"] = "3"
    import pytorch_mppi_b200 as eng
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        g = torch.Generator().manual_seed(11)
        K, T = 4096 + 64, 25            # 4160 splits evenly over 2 ranks; K + 1 below exercises the remainder path
        results = {}
        for variant in ("mppi", "kmppi", "smppi"):
            for K_ in (K, K + 1):
                S = 5
                rows = (S if variant == "kmppi" else T)
                z = torch.randn(K_, rows, 2, generator=g)
                U0 = torch.randn(T, 2, generator=g) * 0.3
                nav = eng.LinearPoint.toy2d_nav()

                def make(pg, exchange):
                    kw = dict(num_samples=K_, horizon=T, device=dev, terminal_state_cost=nav.terminal_cost,
                              u_max=torch.tensor([1.0, 1.0]), process_group=pg, exchange=exchange, rng_seed=3)
                    if variant == "mppi":
                        return eng.MPPI(nav.dynamics, nav.running_cost, 2, torch.eye(2), U_init=U0.clone(), **kw)
                    if variant == "smppi":
                        return eng.SMPPI(nav.dynamics, nav.running_cost, 2, torch.eye(2), w_action_seq_cost=5.0,
                                         action_max=torch.tensor([1.0, 1.0]), **kw)
                    return eng.KMPPI(nav.dynamics, nav.running_cost, 2, torch.eye(2), U_init=U0.clone(), num_support_pts=S,
                                     kernel=eng.RBFKernel(sigma=2), **kw)
                single = make(None, "p2p")
                single.inject_noise(z)
                a_ref = single.command([-3.0, -2.0]).cpu()
                U_ref = single.U.cpu()
                for exchange in ("p2p", "nccl"):
                    c = make(dist.group.WORLD, exchange)
                    for rep in range(2):     # two commands: exercises the double-buffered mailboxes
                        c.inject_noise(z)
                        if rep == 1:
                            c.U = U0 if variant != "smppi" else torch.zeros_like(U0)
                            if variant == "smppi":
                                c.action_sequence = torch.zeros_like(U0)
                            if variant == "kmppi":
                                c.theta = torch.zeros(S, 2)
                        a = c.command([-3.0, -2.0]).cpu()
                    torch.cuda.synchronize()
                    err = float((c.U.cpu() - U_ref).abs().max())
                    aerr = float((a - a_ref).abs().max())
                    # all ranks must hold bit-identical U
                    Ucat = c.U.detach().clone().contiguous()
                    lst = [torch.zeros_like(Ucat) for _ in range(world)]
                    dist.all_gather(lst, Ucat)
                    same = all(torch.equal(lst[0], t) for t in lst)
                    results[f"{variant}/{K_}/{exchange}"] = (err, aerr, same)
        # Philox mode: the sample set is keyed by the global index -> sharded == unsharded
        pend = eng.Pendulum()
        one = eng.MPPI(pend.dynamics, pend.running_cost, 2, torch.tensor(10.0), num_samples=8192, horizon=30, device=dev,
                       u_min=torch.tensor(-2.0), u_max=torch.tensor(2.0), U_init=torch.zeros(30, 1), rng_seed=99)
        many = eng.MPPI(pend.dynamics, pend.running_cost, 2, torch.tensor(10.0), num_samples=8192, horizon=30, device=dev,
                        u_min=torch.tensor(-2.0), u_max=torch.tensor(2.0), U_init=torch.zeros(30, 1), rng_seed=99,
                        process_group=dist.group.WORLD)
        for _ in range(3):
            one.command([3.0, 0.5])
            many.command([3.0, 0.5])
        results["philox"] = (float((one.U - many.U).abs().max()), 0.0, True)
        results["philox_geometry"] = (0.0, 0.0, many.launch_info.split_cost == (1 if split_mode == "1" else 0)
                                      and many.launch_info.xchg_records >= 1
                                      and (many.launch_info.xchg_records > 1) == (direct == "1")
                                      and many.launch_info.cluster_size <= int(cluster))
        # BASELINE config 2 per rank (K = 16384 x world) and a config-5-sized shard (multi-tile grid, rank-record mode)
        for K_, T_, name in ((16384 * world, 30, "c2_weak"), (131072 * world, 50, "c5_shard")):
            U0p = torch.randn(T_, 1, generator=g) * 2
            kwp = dict(num_samples=K_, horizon=T_, device=dev, u_min=torch.tensor(-2.0), u_max=torch.tensor(2.0), rng_seed=7)
            one = eng.MPPI(pend.dynamics, pend.running_cost, 2, torch.tensor(10.0), U_init=U0p.clone(), **kwp)
            many = eng.MPPI(pend.dynamics, pend.running_cost, 2, torch.tensor(10.0), U_init=U0p.clone(), process_group=dist.group.WORLD, **kwp)
            worst = 0.0
            for _ in range(3):
                a1 = one.command([3.0, 0.5])
                a2 = many.command([3.0, 0.5])
                worst = max(worst, float((a1 - a2).abs().max()))
            lst = [torch.zeros_like(many.U) for _ in range(world)]
            dist.all_gather(lst, many.U.detach().clone().contiguous())
            results[name] = (float((one.U - many.U).abs().max()), worst, all(torch.equal(lst[0], t) for t in lst))
            results[name + f"/records={many.launch_info.xchg_records}/cluster={many.launch_info.cluster_size}"] = (0.0, 0.0, True)
        # the stepped route (plain callables: no registered model is detected) and the tcgen05 route of the MLP model,
        # sharded: their softmin tail exchanges one record per rank (in the kernel, or through the library collective)
        torch.manual_seed(25)
        mlp = eng.PendulumMLP(torch.nn.Sequential(torch.nn.Linear(3, 32), torch.nn.Tanh(), torch.nn.Linear(32, 32), torch.nn.Tanh(),
                                                  torch.nn.Linear(32, 2)).to(dev))
        nav = eng.LinearPoint.toy2d_nav()

        def routed(route, variant, K_, U0, pg, exchange):
            if route == "tc":        # fp32 with the default tensor_cores: the tcgen05 kernel
                return eng.MPPI(mlp.dynamics, mlp.running_cost, 2, torch.tensor(1.0), num_samples=K_, horizon=T, device=dev,
                                u_min=torch.tensor(-2.0), u_max=torch.tensor(2.0), U_init=U0.clone(), process_group=pg,
                                exchange=exchange, rng_seed=3)
            dyn, cost = (lambda s, a: nav.dynamics(s, a)), (lambda s, a: nav.running_cost(s, a))
            kw = dict(num_samples=K_, horizon=T, device=dev, u_max=torch.tensor([1.0, 1.0]), process_group=pg, exchange=exchange,
                      rng_seed=3)
            if variant == "mppi":
                return eng.MPPI(dyn, cost, 2, torch.eye(2), U_init=U0.clone(), **kw)
            if variant == "smppi":
                return eng.SMPPI(dyn, cost, 2, torch.eye(2), w_action_seq_cost=5.0, action_max=torch.tensor([1.0, 1.0]), **kw)
            return eng.KMPPI(dyn, cost, 2, torch.eye(2), U_init=U0.clone(), num_support_pts=5, kernel=eng.RBFKernel(sigma=2), **kw)

        def on_route(c, route):
            tc = c._model is not None and (c.launch_info.block_threads, c.launch_info.threads_per_sample) == (256, 2)
            return tc if route == "tc" else c._model is None

        x_of = {"tc": [3.0, 0.5], "stepped": [-3.0, -2.0]}
        for route, variant in (("stepped", "mppi"), ("stepped", "smppi"), ("stepped", "kmppi"), ("tc", "mppi")):
            nu_ = 1 if route == "tc" else 2
            U0 = torch.randn(T, nu_, generator=g) * 0.3
            z = torch.randn(K, 5 if variant == "kmppi" else T, nu_, generator=g)
            single = routed(route, variant, K, U0, None, "p2p")
            single.inject_noise(z)
            a_ref = single.command(x_of[route]).cpu()
            for exchange in ("p2p", "nccl"):
                c = routed(route, variant, K, U0, dist.group.WORLD, exchange)
                c.inject_noise(z)
                a = c.command(x_of[route]).cpu()
                torch.cuda.synchronize()
                lst = [torch.zeros_like(c.U) for _ in range(world)]
                dist.all_gather(lst, c.U.detach().clone().contiguous())
                results[f"{route}/{variant}/{exchange}"] = (float((c.U.cpu() - single.U.cpu()).abs().max()), float((a - a_ref).abs().max()),
                                                            on_route(c, route) and all(torch.equal(lst[0], t) for t in lst))
        # a nominal drawn at random (no U_init; reset()) is one draw for the whole controller, whatever the ranks' torch seeds
        torch.manual_seed(1000 + rank)
        rnd = eng.MPPI(pend.dynamics, pend.running_cost, 2, torch.tensor(10.0), num_samples=4096, horizon=12, device=dev,
                       u_min=torch.tensor(-2.0), u_max=torch.tensor(2.0), rng_seed=5, process_group=dist.group.WORLD)
        same = True
        for step in range(2):
            a = rnd.command([3.0, 0.5])
            lst = [torch.zeros_like(rnd.U) for _ in range(world)]
            dist.all_gather(lst, rnd.U.detach().clone().contiguous())
            acts = [torch.zeros_like(a) for _ in range(world)]
            dist.all_gather(acts, a.contiguous())
            same = same and all(torch.equal(lst[0], t) for t in lst) and all(torch.equal(acts[0], t) for t in acts)
            rnd.reset()
        results["random_nominal_is_shared"] = (0.0, 0.0, same)
        # a peer that never delivers: the waiting rank gives up after the timeout, returns the un-updated nominal as
        # the action, and its NEXT command raises (ADVICE r1: the timeout used to be silent)
        if mode == MODES[0]:
            os.environ["MPPI_B200_XCHG_TIMEOUT_S"] = "0.3"
            lone = eng.MPPI(pend.dynamics, pend.running_cost, 2, torch.tensor(10.0), num_samples=4096, horizon=20, device=dev,
                            u_min=torch.tensor(-2.0), u_max=torch.tensor(2.0), U_init=torch.ones(20, 1), rng_seed=1,
                            process_group=dist.group.WORLD)
            lone.command([3.0, 0.5])                      # both ranks: fine
            torch.cuda.synchronize()
            dist.barrier()
            ok = True
            if rank == 0:
                U_before = lone.U.clone()
                a = lone.command([3.0, 0.5], shift_nominal_trajectory=False)     # rank 1 stays away
                torch.cuda.synchronize()
                ok = bool(torch.equal(lone.U, U_before)) and bool(torch.equal(a.reshape(-1), U_before[0].reshape(-1)))
                try:
                    lone.command([3.0, 0.5])
                    ok = False
                except eng.mppi._cabi.MppiLibraryError:
                    pass
            dist.barrier()
            results["timeout_is_reported"] = (0.0, 0.0, ok)
            for route in ("stepped", "tc"):
                nu_ = 1 if route == "tc" else 2
                lone = routed(route, "mppi", 4096, torch.ones(T, nu_), dist.group.WORLD, "p2p")
                lone.command(x_of[route])                 # both ranks: fine
                torch.cuda.synchronize()
                dist.barrier()
                ok = on_route(lone, route)
                if rank == 0:
                    U_before = lone.U.clone()
                    a = lone.command(x_of[route], shift_nominal_trajectory=False)     # rank 1 stays away
                    torch.cuda.synchronize()
                    ok = ok and bool(torch.equal(lone.U, U_before)) and bool(torch.equal(a.reshape(-1), U_before[0].reshape(-1)))
                    try:
                        lone.command(x_of[route])
                        ok = False
                    except eng.mppi._cabi.MppiLibraryError:
                        pass
                dist.barrier()
                results[f"timeout_is_reported/{route}"] = (0.0, 0.0, ok)
        out[rank] = results
    finally:
        dist.destroy_process_group()


# (split-cost rollout, direct exchange of cluster records, cluster size limit): the default first
MODES = [("1", "1", "8"), ("0", "0", "1"), ("1", "1", "1"), ("1", "0", "8")]


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("mode", MODES, ids=lambda m: f"split{m[0]}-direct{m[1]}-cluster{m[2]}")
def test_two_gpu_sharding_matches_single_gpu(mode):
    import torch.multiprocessing as mp
    mgr = mp.Manager()
    out = mgr.dict()
    port = 29700 + (os.getpid() % 1000) + 37 * MODES.index(mode)
    mp.spawn(_worker, args=(2, port, out, mode), nprocs=2, join=True)
    assert len(out) == 2
    for rank in range(2):
        for key, (err, aerr, same) in out[rank].items():
            assert err < 2e-6 and aerr < 2e-6, (rank, key, err, aerr)
            assert same, (rank, key)
