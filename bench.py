#!/usr/bin/env python
"""bench.py — the MPPI command() hot path on B200, BASELINE.json's metric.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl engine|reference] [--workload NAME] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Every timed loop (per-step events, back-to-back, e2e) runs exactly K steps.  `--dump-outputs DIR` writes what the last
timed command() handed its caller (see `command_outputs`) as DIR/<name>.npy; the inputs are seeded, so two builds run
with the same arguments can be compared output for output.

One "step" = one `command()` (shift + sample K x T noise + T-step rollout + softmin reweight + nominal update).
Workloads (BASELINE.json `configs`; the default is configs[1], the north star):
    pendulum_c2   pendulum analytic, MPPI,  K=16384 T=30 fp32                       (configs[1])
    nav2d_c3      2-D navigation,    KMPPI RBF(sigma=2) S=5, K=8192 T=40 fp32       (configs[2])
    mlp_c4        learned pendulum (3-32-32-2 tanh MLP), MPPI, K=32768 T=30, tcgen05 tensor-core rollout   (configs[3])
    pendulum_c5   pendulum analytic, MPPI,  K=131072 per GPU T=50 fp32 (= K=2^20 on 8 GPUs)   (configs[4] shard)

Printed JSON line (rank 0):
  value / metric : K*T rollout-steps per second (whole job), inputs resident in HBM, per-step CUDA events on the
                   launching stream, L2 flushed between timed iterations; `value` uses the 10 %-trimmed mean of the
                   per-step times (the reference's own harness, tests/benchmark_mppi.py:84-113, reports exactly that);
                   mean / median / min are in `config.step_stats_ms`
  e2e            : the same metric through the public host API `command_host(state)`, every step inside the timed
                   region (state from host memory, action back into pinned host memory); at N=1 for the analytic
                   models also on a resident grid (`start_resident()`), the faster of the two is `e2e`
  roofline       : the dominant kernel against the roof that bounds it — analytic rollouts are issue/latency-bound
                   (frac = lane-op fraction, the HBM figures beside it), the MLP rollout is a tensor-core contraction
  cpu_baseline   : the reference's own implementation (oracle/_ref: the unmodified Python package on torch CPU ops;
                   the oracle port if that copy is absent) on this host's cores, bounded sample
`--impl reference` times that CPU implementation alone, on the same config/metric.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

WORKLOADS = {
    "pendulum_c2": dict(K=16384, T=30, nx=2, nu=1, variant="mppi", model="pendulum", sigma=10.0, x0=[math.pi, 1.0],
                        lane_ops=55.0, desc="pendulum analytic K=16384 T=30 fp32 (BASELINE configs[1])"),
    "nav2d_c3": dict(K=8192, T=40, nx=2, nu=2, variant="kmppi", model="nav2d", sigma=1.0, x0=[-3.0, -2.0], S=5, rbf_sigma=2.0,
                     lane_ops=110.0, desc="2D-nav KMPPI RBF(sigma=2) num_support_pts=5 K=8192 T=40 fp32 (BASELINE configs[2])"),
    "mlp_c4": dict(K=32768, T=30, nx=2, nu=1, variant="mppi", model="mlp", sigma=1.0, x0=[math.pi, 1.0],
                   flop_per_step=2368.0, lane_ops=2368.0 / 2 + 200.0,
                   desc="pendulum_approximate 2-layer MLP dynamics K=32768 T=30 tensor-core rollout (BASELINE configs[3])"),
    "pendulum_c5": dict(K=131072, T=50, nx=2, nu=1, variant="mppi", model="pendulum", sigma=10.0, x0=[math.pi, 1.0],
                        lane_ops=55.0, desc="pendulum analytic K=2^20/8 per GPU T=50 fp32 (BASELINE configs[4] shard)"),
}
LAMBDA, UMAX = 1.0, 2.0


def algorithmic_bytes(wl, K, es=4):
    """SURVEY.md §8(d): B_min = es*(nx + 2*R + K) (state in, nominal in/out, cost_total out; R = T*nu, or S*nu control
    points + T*nu trajectory for KMPPI); B_full = B_min + es*K (omega) + es*K*T*nu (noise) — what the reference's
    API-visible tensors cost."""
    T, nu, nx = wl["T"], wl["nu"], wl["nx"]
    rows = T * nu + (wl["S"] * nu if wl["variant"] == "kmppi" else 0)
    b_min = es * (nx + 2 * rows + K)
    b_full = b_min + es * K + es * K * T * nu
    return b_min, b_full


# ------------------------------------------------------------------------------------------------
def start_clock_sampler():
    try:
        f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        p = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "50"],
                             stdout=f, stderr=subprocess.DEVNULL)
        return p, f
    except Exception:
        return None, None


def stop_clock_sampler(p, f, gpu_index, t_begin, t_end):
    out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
    if p is None:
        return out
    try:
        p.terminate()
        p.wait(timeout=5)
    except Exception:
        pass
    try:
        f.flush()
        f.seek(0)
        import datetime
        clocks, maxs, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 10 or not c[1].isdigit() or int(c[1]) != gpu_index:
                continue
            try:
                ts = datetime.datetime.strptime(c[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
            except Exception:
                ts = None
            if ts is not None and not (t_begin - 0.15 <= ts <= t_end + 0.15):
                continue
            clocks.append(float(c[2]))
            maxs.append(float(c[3]))
            for name, v in zip(names, c[6:10]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if clocks:
            clocks.sort()
            out.update(sm_mhz=clocks[len(clocks) // 2], sm_max_mhz=max(maxs), reasons=sorted(reasons), samples=len(clocks))
    except Exception:
        pass
    finally:
        try:
            os.unlink(f.name)
        except Exception:
            pass
    return out


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        d = json.load(open(path))
        return dict(hbm=float(d["hbm_gbs"]), tf_burst=float(d["bf16_tflops"]), tf_sustained=float(d["bf16_tflops_sustained"]),
                    src="measured (MEASURED_PEAKS.json)")
    except Exception:
        return dict(hbm=6650.0, tf_burst=1500.0, tf_sustained=1500.0, src="fallback (B200_PROFILING.md)")


def load_traffic(workload):
    """dram bytes per launch from the committed `ncu --set full` capture (profiles/traffic.json)."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))[workload]["dram_bytes_per_launch"]
    except Exception:
        return None


def trimmed_stats(ms):
    """tests/benchmark_mppi.py:84-113: sort, drop 10 % on each side, mean; median and min beside it."""
    s = sorted(ms)
    n = len(s)
    cut = n // 10
    core = s[cut:n - cut] if n - 2 * cut > 0 else s
    return dict(trimmed_mean=sum(core) / len(core), mean=sum(s) / n, median=s[n // 2], min=s[0], max=s[-1], n=n)


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's own implementation (oracle/_ref) or the oracle port
# ------------------------------------------------------------------------------------------------
def make_mlp_net(dtype=torch.float32):
    """pendulum_approximate.py:31, 47-53: the network as torch initialises it right after manual_seed(25)."""
    torch.manual_seed(25)
    net = torch.nn.Sequential(torch.nn.Linear(3, 32), torch.nn.Tanh(), torch.nn.Linear(32, 32), torch.nn.Tanh(),
                              torch.nn.Linear(32, 2)).to(dtype)
    for p_ in net.parameters():
        p_.requires_grad_(False)
    return net


class CpuArm:
    """One workload on the CPU.  kind "reference": the unmodified reference classes from oracle/_ref driven through
    their public API (command(state) draws its own randn); kind "port": the oracle's restatement + torch.randn."""

    def __init__(self, wl, K):
        from oracle import make_ref
        from oracle import mppi_oracle as orc
        self.wl, self.K, self.orc = wl, K, orc
        T, dt = wl["T"], torch.float32
        sigma = torch.tensor(wl["sigma"]) if wl["nu"] == 1 else torch.eye(wl["nu"]) * wl["sigma"]
        if wl["model"] == "pendulum":
            model = orc.PendulumModel()          # numpy sin, exactly as tests/pendulum.py runs on the CPU
            term = None
            bounds = dict(u_min=torch.tensor(-UMAX), u_max=torch.tensor(UMAX))
        elif wl["model"] == "mlp":
            model = orc.MlpPendulumModel(make_mlp_net(dt))
            term = None
            bounds = dict(u_min=torch.tensor(-UMAX), u_max=torch.tensor(UMAX))
        else:                                    # Toy2D navigation, tests/smooth_mppi.py:79-142, 539-560
            model = orc.LinearPointModel(B=[[0.5, 0.0], [0.0, -0.5]], goal=[2.0, 2.0], R=[[0.01, 0.0], [0.0, 0.01]],
                                         hills=[([[0.25, 0.125], [0.125, 0.25]], [-0.5, -1.0], 200.0)], terminal_scale=10.0, dtype=dt)
            term = model.terminal_cost
            bounds = dict(u_max=torch.tensor([1.0, 1.0]))
        self.model = model
        self.x = torch.tensor(wl["x0"], dtype=dt)
        torch.manual_seed(0)
        ref = make_ref.import_reference()
        self.kind = "reference" if ref is not None else "port"
        if ref is not None:
            kw = dict(num_samples=K, horizon=T, lambda_=LAMBDA, device="cpu", terminal_state_cost=term, **bounds)
            if wl["variant"] == "kmppi":
                self.ctrl = ref.KMPPI(model.dynamics, model.running_cost, wl["nx"], sigma, num_support_pts=wl["S"],
                                      kernel=ref.RBFKernel(sigma=wl["rbf_sigma"]), **kw)
            else:
                self.ctrl = ref.MPPI(model.dynamics, model.running_cost, wl["nx"], sigma, **kw)
        else:
            self.prob = orc.Problem(model.dynamics, model.running_cost, wl["nx"], sigma, K=K, T=T, lambda_=LAMBDA,
                                    terminal_state_cost=term, **bounds)
            self.U = self.prob.colour(torch.randn(T, wl["nu"]))
            if wl["variant"] == "kmppi":
                S = wl["S"]
                self.theta = torch.zeros(S, wl["nu"])
                self.W, self.Wshift = orc.kernel_matrices(T, S, lambda a, b: orc.rbf_kernel(a, b, wl["rbf_sigma"]), dt)

    def step(self):
        """One closed-loop command(): plan from the current state, then step the same model with the action."""
        wl, orc = self.wl, self.orc
        if self.kind == "reference":
            a = self.ctrl.command(self.x)
        else:
            rows = wl["S"] if wl["variant"] == "kmppi" else wl["T"]
            z = torch.randn(self.K, rows, wl["nu"])                          # mppi.py:203
            if wl["variant"] == "kmppi":
                r = orc.kmppi_command(self.prob, self.U, self.theta, self.x, z, self.W, self.Wshift)
                self.theta = r["theta"]
            else:
                r = orc.mppi_command(self.prob, self.U, self.x, z)
            self.U = r["U"]
            a = r["action"]
        self.x = self.model.dynamics(self.x.view(1, -1), a.view(1, -1)).view(-1)[: wl["nx"]]
        return a


def pick_cpu_threads(wl, K):
    """The path is ~2,400 small ATen dispatches per command: more threads is not always faster.  Give the CPU arm its
    best case: try the full core count and a few smaller pools, keep the fastest."""
    arm = CpuArm(wl, K)
    best, best_t = torch.get_num_threads(), None
    ncpu = os.cpu_count() or 1
    for nt in sorted({ncpu, max(ncpu // 2, 1), 32, 16, 8, 4, 1}):
        if nt > ncpu:
            continue
        torch.set_num_threads(nt)
        arm.step()
        t0 = time.perf_counter()
        for _ in range(2):
            arm.step()
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = nt, dt
    torch.set_num_threads(best)
    return best


def cpu_sample_text(arm, n, el, cores):
    what = ("the unmodified reference package (oracle/_ref, torch CPU ops, its own torch.randn)" if arm.kind == "reference"
            else "the oracle port (torch CPU ops, randn included)")
    return (f"{n} closed-loop command() calls of {what} in {el:.1f}s, {cores} threads "
            f"(fastest pool of 1..{os.cpu_count()} logical cores)")


def run_reference(args, wl):
    """`--impl reference`: the reference's CPU implementation of the path on this host's cores, same config/metric."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # same problem as the engine arm launched with the same flags: under weak scaling the job is K per GPU x N GPUs
    K, T = wl["K"] * (args.gpus if args.scaling == "weak" else 1), wl["T"]
    cores = pick_cpu_threads(wl, K)
    arm = CpuArm(wl, K)
    n_warm = max(min(args.warmup, 5), 1)
    for _ in range(n_warm):
        arm.step()
    steps = args.steps
    t0 = time.perf_counter()
    for _ in range(steps):
        arm.step()
    dt = time.perf_counter() - t0
    value = K * T * steps / dt
    line = {
        "impl": "reference", "metric": "K*T rollout-steps/s through command()", "value": value, "unit": "rollout-steps/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": n_warm, "ms_per_step": dt / steps * 1e3,
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl["desc"], "K_global": K, "T": T, "nx": wl["nx"], "nu": wl["nu"], "noise_sigma": wl["sigma"],
                   "lambda": LAMBDA, "device": "cpu", "commands_per_s": steps / dt},
        "cpu_baseline": {"value": value, "unit": "rollout-steps/s", "cores": cores, "kind": arm.kind,
                         "sample": cpu_sample_text(arm, steps, dt, cores)},
        "e2e": {"value": value, "unit": "rollout-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
def make_engine(eng, wl, K_global, dev, pg, exchange, seed=1234):
    """The engine controller of a workload (synthetic inputs of SURVEY.md §8d)."""
    T = wl["T"]
    torch.manual_seed(0)
    kw = dict(num_samples=K_global, horizon=T, lambda_=LAMBDA, device=dev, rng_seed=seed, process_group=pg, exchange=exchange)
    if wl["model"] == "pendulum":
        m = eng.Pendulum()
        U0 = torch.randn(T, 1) * wl["sigma"] ** 0.5
        return eng.MPPI(m.dynamics, m.running_cost, 2, torch.tensor(wl["sigma"]), u_min=torch.tensor(-UMAX),
                        u_max=torch.tensor(UMAX), U_init=U0, **kw)
    if wl["model"] == "mlp":
        m = eng.PendulumMLP(make_mlp_net().to(dev), tensor_cores=wl.get("tensor_cores", "auto"))
        torch.manual_seed(0)
        U0 = torch.randn(T, 1)
        return eng.MPPI(m.dynamics, m.running_cost, 2, torch.tensor(wl["sigma"]), u_min=torch.tensor(-UMAX),
                        u_max=torch.tensor(UMAX), U_init=U0, **kw)
    m = eng.LinearPoint.toy2d_nav()
    return eng.KMPPI(m.dynamics, m.running_cost, 2, torch.eye(2) * wl["sigma"], terminal_state_cost=m.terminal_cost,
                     u_max=torch.tensor([1.0, 1.0]), num_support_pts=wl["S"], kernel=eng.RBFKernel(sigma=wl["rbf_sigma"]), **kw)


def command_outputs(ctrl, action):
    """What one command() hands its caller, copied to the host: the returned action, the updated nominal sequence U,
    the per-sample total cost (this rank's shard of the K samples) and, for KMPPI, the updated control points."""
    out = {"action": action, "U": ctrl.U, "cost_total": ctrl.cost_total}
    if hasattr(ctrl, "theta"):
        out["theta"] = ctrl.theta
    out = {k: v.detach().to("cpu", torch.float64 if v.dtype == torch.float64 else torch.float32).numpy()
           for k, v in out.items()}
    assert sum(a.nbytes for a in out.values()) <= 64 << 20
    return out


def run_engine(args, wl):
    import torch.distributed as dist
    from pytorch_mppi_b200 import build as _build
    if int(os.environ.get("LOCAL_RANK", "0")) == 0 and _build.needs_build() and not os.path.exists(_build.OUT):
        _build.build()      # normally the in-tree .so travels with the snapshot; build only if it is absent
    import pytorch_mppi_b200 as eng

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus > 1 and world == 1:
        raise SystemExit("--gpus N>1 must be launched with torch.distributed.run (one rank per GPU)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    pg = None
    saved_stdout = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL's own output (its version banner, NCCL_DEBUG logs if the caller asked for them) goes to stderr: stdout is
        # pointed at stderr until the JSON line is printed, so it carries that one line only
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=dev)
        pg = dist.group.WORLD

    if wl["model"] == "mlp":
        wl = dict(wl, tensor_cores=args.mlp_mode)
    K_gpu, T, NX, NU = wl["K"], wl["T"], wl["nx"], wl["nu"]
    K_global = K_gpu * world if args.scaling == "weak" else K_gpu
    ctrl = make_engine(eng, wl, K_global, dev, pg, args.exchange)
    assert ctrl._model is not None, "fused route not selected"
    x_dev = torch.tensor(wl["x0"], dtype=torch.float32, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- sharded == unsharded: the same commands on ONE GPU must give the same plan -----------------
    # Philox is keyed by the GLOBAL sample index, so the sharded job and a single-GPU controller with the same seed draw
    # the same K_global samples; what differs is the order of the fp32 per-tile partial sums (the cross-tile and
    # cross-GPU combinations are fp64 in both).  Five closed-loop commands from identical nominals, compared on rank 0.
    shard_check = None
    if world > 1 and not args.no_shard_check:
        solo = make_engine(eng, wl, K_global, dev, None, "p2p") if rank == 0 else None
        for _ in range(5):
            ctrl.command(x_dev)
            if solo is not None:
                solo.command(x_dev)
        barrier()
        if rank == 0:
            diff = float((solo.U - ctrl.U).abs().max())
            scale = float(solo.U.abs().max())
            shard_check = {"commands": 5, "max_abs_diff_U": diff, "max_abs_U": scale, "tol": 2e-5,
                           "ok": bool(diff <= 2e-5 and math.isfinite(diff))}
        del solo
        barrier()

    sampler, sfile = (start_clock_sampler() if rank == 0 else (None, None))
    n_warm = max(args.warmup, 3)
    for _ in range(n_warm):
        flush.zero_()
        ctrl.command(x_dev)
    barrier()

    # ---- device-resident timing: per-step CUDA events, L2 flushed between iterations ---------------
    stream = torch.cuda.current_stream(dev)
    t_begin = time.time()
    step_ms = []
    done = 0
    CH = 512
    while done < args.steps:
        n = min(CH, args.steps - done)
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
        for e0, e1 in evs:
            flush.zero_()
            e0.record(stream)
            action = ctrl.command(x_dev)
            e1.record(stream)
        torch.cuda.synchronize()
        step_ms += [e0.elapsed_time(e1) for e0, e1 in evs]
        done += n
    barrier()
    t_end = time.time()
    if args.dump_outputs and rank == 0:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in command_outputs(ctrl, action).items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
    stats = trimmed_stats(step_ms)
    # max over ranks of the per-rank figures (every rank times the same K steps)
    agg = torch.tensor([stats["trimmed_mean"], stats["mean"], stats["median"], stats["min"]], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(agg, op=dist.ReduceOp.MAX)
    stats.update(trimmed_mean=float(agg[0]), mean=float(agg[1]), median=float(agg[2]), min=float(agg[3]))
    ms_per_step = stats["trimmed_mean"] if args.steps >= 10 else stats["mean"]
    value = K_global * T / (ms_per_step * 1e-3)

    # ---- back-to-back launches (no flush): the steady-state command rate ---------------------------
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    nb2b = args.steps
    barrier()
    e0.record(stream)
    for _ in range(nb2b):
        ctrl.command(x_dev)
    e1.record(stream)
    torch.cuda.synchronize()
    b2b_t = torch.tensor([e0.elapsed_time(e1) / nb2b], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(b2b_t, op=dist.ReduceOp.MAX)
    b2b_ms = float(b2b_t.item())

    # ---- end to end through the host API: state from host memory, action back to pinned host memory
    x_host = list(wl["x0"])
    for _ in range(20):
        ctrl.command_host(x_host)
    barrier()
    n_e2e = args.steps
    t0 = time.perf_counter()
    for _ in range(n_e2e):
        a_host = ctrl.command_host(x_host)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    e2e_t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_s = float(e2e_t.item())
    e2e_value = K_global * T * n_e2e / e2e_s
    # ---- the same host loop served by a resident grid (csrc/mppi_resident.cuh; single GPU, analytic models) ------
    # command_host() with the command's grid kept on the GPU: per step the state record is pulled from pinned host
    # memory by the grid and the action is stored back to pinned host memory — both inside the timed region.  The grid
    # is dismissed AFTER the clock stops (its idle timeout is far above the loop's period, so no relaunch inside).
    e2e_res, res_err = None, None
    if world == 1 and not args.no_resident and wl["model"] != "mlp":
        try:
            ctrl.start_resident(idle_us=200000)
            for _ in range(100):
                ctrl.command_host(x_host)
            l0 = ctrl.resident_launches
            t0 = time.perf_counter()
            for _ in range(n_e2e):
                a_res = ctrl.command_host(x_host)
            res_s = time.perf_counter() - t0           # every action has arrived in host memory: the loop is synchronous
            launches = ctrl.resident_launches - l0
            ctrl.stop_resident()
            torch.cuda.synchronize()
            e2e_res = {"value": K_global * T * n_e2e / res_s, "unit": "rollout-steps/s",
                       "h2d_bytes_per_step": 8 * (3 + NX), "d2h_bytes_per_step": NU * 8 + 8,
                       "ms_per_step": res_s / n_e2e * 1e3, "steps": n_e2e,
                       "api": "MPPI.start_resident(); MPPI.command_host(state)  [resident grid, no launch per step]",
                       "kernel_launches_in_timed_region": launches,
                       "last_action": [float(v) for v in a_res.reshape(-1)]}
        except Exception as e:      # noqa: BLE001 — the bench line must survive; the launch-route e2e stands
            res_err = repr(e)[:300]
            try:
                ctrl.stop_resident()
            except Exception:       # noqa: BLE001
                pass
    clocks = stop_clock_sampler(sampler, sfile, local_rank, t_begin, t_end) if rank == 0 else None
    ranks_agree = True
    if world > 1:      # every rank must hold the bit-identical nominal sequence (no broadcast is ever issued)
        mine = ctrl.U.detach().clone().contiguous()
        allU = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allU, mine)
        ranks_agree = all(torch.equal(allU[0], u) for u in allU) and bool(torch.isfinite(mine).all())

    if rank == 0:
        info = ctrl.launch_info
        K_loc = ctrl._K_local
        b_min, b_full = algorithmic_bytes(wl, K_loc)
        peaks = load_peaks()
        t_s = ms_per_step * 1e-3
        hbm_achieved = b_full / t_s / 1e9
        lane_ops = wl["lane_ops"] * K_loc * T / t_s
        lane_peak = info.sm_count * 128 * (clocks["sm_max_mhz"] or 1965.0) * 1e6
        if wl["model"] == "mlp":
            tf = wl["flop_per_step"] * K_loc * T / t_s / 1e12
            roofline = {"bound": "tensor", "achieved": tf, "peak": peaks["tf_sustained"], "unit": "TFLOP/s",
                        "frac": tf / peaks["tf_sustained"], "traffic": load_traffic(args.workload),
                        "peak_source": peaks["src"] + " bf16_tflops_sustained (kernel timed inside a long step)",
                        "algorithmic_flop_per_launch": wl["flop_per_step"] * K_loc * T,
                        "note": "useful MLP math only (2,368 flop per rollout-step, SURVEY 8a); bf16x3 issues 7 MMAs per "
                                "layer-triple for fp32-grade layer outputs, N=32 tiles: the step is bound by the "
                                "tanh/convert epilogue and the MMA round trips, not by tensor throughput",
                        "hbm_achieved_GBps": hbm_achieved, "hbm_frac": hbm_achieved / peaks["hbm"], "lane_ops_frac": lane_ops / lane_peak}
        else:
            roofline = {"bound": "latency/issue", "achieved": lane_ops / 1e12, "peak": lane_peak / 1e12, "unit": "Tlane-op/s",
                        "frac": lane_ops / lane_peak, "traffic": load_traffic(args.workload),
                        "peak_source": "SMs x 128 FP32 lanes x max SM clock (nvidia-smi); HBM peak: " + peaks["src"] + " hbm_gbs",
                        "lane_ops_per_rollout_step": wl["lane_ops"],
                        "hbm": {"achieved": hbm_achieved, "peak": peaks["hbm"], "unit": "GB/s", "frac": hbm_achieved / peaks["hbm"],
                                "algorithmic_bytes_per_launch": b_full, "algorithmic_bytes_min_per_launch": b_min,
                                "frac_min_bytes": b_min / t_s / 1e9 / peaks["hbm"]},
                        "note": "the fused analytic rollout moves ~B_min bytes per launch (traffic) and is bound by FP32/SFU "
                                "issue and dependent-issue latency, not HBM (SURVEY 8d); frac = lane-op fraction"}
        line = {
            "metric": "K*T rollout-steps/s through command()", "value": value, "unit": "rollout-steps/s",
            "n_gpus": world, "steps": args.steps, "warmup": n_warm, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f32" if wl["model"] != "mlp" else ("bf16x3 (hi/lo-split bf16 operands, fp32 accumulate)" if wl["tensor_cores"] != "bf16" else "bf16"),
            "data": "synthetic",
            "config": {"workload": wl["desc"], "K_global": K_global, "K_per_gpu": K_loc, "T": T, "nx": NX, "nu": NU,
                       "noise_sigma": wl["sigma"], "lambda": LAMBDA, "rng": "in-kernel Philox4x32-10",
                       "commands_per_s": 1e3 / ms_per_step, "back_to_back_ms_per_step": b2b_ms, "step_stats_ms": stats,
                       "value_from": "10%-trimmed mean of per-step CUDA events" if args.steps >= 10 else "mean of per-step CUDA events",
                       "l2": "flushed between timed iterations (256 MiB memset), per-step CUDA events on the launch stream",
                       "parallelism": f"K sharded over {world} GPU(s), exchange={args.exchange if world > 1 else 'none'}",
                       "ranks_hold_identical_U": ranks_agree, "sharded_equals_unsharded": shard_check,
                       "grid": info.grid_blocks, "block": info.block_threads, "threads_per_sample": info.threads_per_sample,
                       "smem_bytes": info.smem_bytes, "regs": info.regs_per_thread, "split_cost": info.split_cost,
                       "cluster": info.cluster_size, "reduction_records": info.xchg_records},
            "roofline": roofline,
            "e2e": {"value": e2e_value, "unit": "rollout-steps/s", "h2d_bytes_per_step": NX * 8, "d2h_bytes_per_step": NU * 4 + 8,
                    "ms_per_step": e2e_s / n_e2e * 1e3, "steps": n_e2e, "api": "MPPI.command_host(state)  [one launch per step]",
                    "last_action": [float(v) for v in a_host.reshape(-1)]},
            "gpu_launches": args.steps,
            "clocks": clocks,
        }
        if e2e_res is not None and e2e_res["value"] > line["e2e"]["value"]:
            line["e2e_launch_route"] = line["e2e"]           # kept beside it: the same loop with one launch per step
            line["e2e"] = e2e_res
        elif e2e_res is not None:
            line["e2e_resident"] = e2e_res
        if res_err is not None:
            line["config"]["resident_error"] = res_err
        # ---- CPU baseline on this host's cores, bounded sample ------------------------------------
        if world == 1 and not args.no_cpu_baseline:
            cores = pick_cpu_threads(wl, K_gpu)
            arm = CpuArm(wl, K_gpu)
            for _ in range(2):
                arm.step()
            t0 = time.perf_counter()
            n = 0
            while True:
                arm.step()
                n += 1
                el = time.perf_counter() - t0
                if (el >= args.cpu_seconds and n >= 10) or n >= 5000 or el > 6 * args.cpu_seconds:
                    break
            line["cpu_baseline"] = {"value": K_gpu * T * n / el, "unit": "rollout-steps/s", "cores": cores, "kind": arm.kind,
                                    "sample": cpu_sample_text(arm, n, el, cores), "ms_per_step": el / n * 1e3}
        sys.stdout.flush()
        if saved_stdout is not None:
            os.dup2(saved_stdout, 1)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10000)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--workload", default="pendulum_c2", choices=sorted(WORKLOADS))
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--exchange", default="p2p", choices=["p2p", "nccl"])
    ap.add_argument("--mlp-mode", default="auto", choices=["auto", "bf16x3", "bf16"],
                    help="mlp_c4 operand precision on the tensor cores: hi/lo-split bf16 (fp32-grade layer outputs, the parity "
                         "route) or plain bf16")
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-shard-check", action="store_true")
    ap.add_argument("--no-resident", action="store_true",
                    help="e2e on the launch route only (default at N=1: also time the host loop on a resident grid, "
                         "csrc/mppi_resident.cuh, and report the faster one as e2e)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed command() (action, U, cost_total; theta for KMPPI) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "engine":
        ap.error("--dump-outputs writes the engine's outputs (--impl engine)")
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, wl)
    else:
        run_engine(args, wl)


if __name__ == "__main__":
    main()
