"""GPU: every path of the softmin reduction, the wide user models (nu 3-4, nx up to 8) and infinite sample costs, each
against the fp64 oracle (oracle/mppi_oracle.py) on the same injected noise, over two commands with the nominal kept in
step with the oracle.  Every check covers U, the action, cost_total and omega (and theta / action_sequence).

Tolerances:
  fp64  1e-10 on U, the action, A and theta; cost_total to 1e-10 relative; omega to 1e-10.
  fp32  max |engine - oracle_f64| <= 2 max |oracle_f32 - oracle_f64| + 1e-5: the fp32 oracle's own distance from fp64 on
        the same draws is the yardstick (as in test_large_k_grid_stride_and_block_sizes); costs are compared relative to
        max(1, |cost|) with a 1e-6 floor.

Which reduction path a fused command takes follows from its launch_info (csrc/mppi_fused_host.cuh, mppi_fused.cuh
`warp_tail`): a tile of samples_per_tile = block_threads / threads_per_sample samples has samples_per_tile / 32 warp
records; a cluster combines cluster_size of those tiles' records (combine_narrow up to 64 records, combine_records above);
NC = grid_blocks / cluster_size cluster records then reach the finisher: none when NC == 1, as flagged words staged in
shared memory (LL mode, xchg_records == NC) or through the L2 workspace and a ticket (combine_global) otherwise.
"""
import fnmatch
import math

import numpy as np
import pytest
import torch

import pytorch_mppi_b200 as eng
from oracle import mppi_oracle as orc
from tests import user_models as um

pytestmark = pytest.mark.gpu

CLS = {"mppi": eng.MPPI, "smppi": eng.SMPPI, "kmppi": eng.KMPPI}
DTYPES = {"f64": torch.float64, "f32": torch.float32}


def rbf_sigma(T, S):
    """KMPPI's RBF width: 0.6 x the support-point spacing keeps k(Tk, Tk) well conditioned at every S the tests use, so
    the interpolation operator W is not itself a source of fp32 error."""
    return 0.6 * (T - 1) / (S - 1)


# ---- problems: the engine's model (fused route), its torch twin (stepped route, device-generic) and the oracle's -------
class Problem:
    def __init__(self, kind, nu, model, gpu_fns, cpu_fns, nx, sigma, terminal=False, **kw):
        self.kind, self.nu, self.model, self.nx = kind, nu, model, nx
        self.gpu_fns = gpu_fns                                  # (dynamics, running_cost, terminal_cost or None)
        self.cpu_fns = cpu_fns                                  # dtype -> the oracle's (dynamics, running_cost, terminal)
        self.sigma = sigma                                      # fp64; 0-dim for nu = 1
        self.terminal = terminal
        self.kw = kw                                            # lambda_, u_min, u_max, noise_mu, u_init, u_scale (fp64)


def pendulum():
    m = eng.Pendulum()
    o = orc.PendulumModel(numpy_sin=False)
    return Problem("pendulum", 1, m, (m.dynamics, m.running_cost, None), lambda dt: (o.dynamics, o.running_cost, None), 2,
                   torch.tensor(4.0, dtype=torch.float64), lambda_=1.0,
                   u_min=torch.tensor([-2.0], dtype=torch.float64), u_max=torch.tensor([2.0], dtype=torch.float64))


def linear_point():
    m = eng.LinearPoint.unit_test_env()

    def oracle_fns(dt):
        o = orc.LinearPointModel(B=m.B, goal=m.goal, dtype=dt)
        return o.dynamics, o.running_cost, None
    return Problem("linear", 2, m, (m.dynamics, m.running_cost, None), oracle_fns, 2,
                   torch.tensor([[0.8, 0.2], [0.2, 0.6]], dtype=torch.float64), lambda_=2.0,
                   u_max=torch.tensor([1.5, 1.2], dtype=torch.float64))


def wide(name, terminal=True):
    """arm4 (nx 8, nu 4) or lin6 (nx 6, nu 3, 68 parameters, a terminal cost unless `terminal` is False): full covariance,
    per-component bounds, noise_mu, u_init and u_scale != 1."""
    if name == "arm4":
        m = um.arm4_user_model()
        fns = (um.arm_dyn, um.arm_cost, None)
        L = torch.tensor([[0.9, 0, 0, 0], [0.3, 0.7, 0, 0], [-0.2, 0.25, 0.8, 0], [0.1, -0.3, 0.2, 0.6]], dtype=torch.float64)
        bounds = dict(u_min=torch.tensor([-1.5, -1.0, -2.0, -1.2], dtype=torch.float64),
                      u_max=torch.tensor([1.2, 1.4, 1.6, 0.9], dtype=torch.float64))
        mu, uinit = [0.05, -0.1, 0.0, 0.08], [0.1, 0.0, -0.05, 0.02]
    else:
        m = um.lin6_user_model(terminal)
        fns = (um.lin6_dyn, um.lin6_cost, um.lin6_term if terminal else None)
        L = torch.tensor([[0.8, 0, 0], [-0.35, 0.6, 0], [0.2, 0.3, 0.9]], dtype=torch.float64)
        bounds = dict(u_min=torch.tensor([-1.0, -0.8, -1.5], dtype=torch.float64),
                      u_max=torch.tensor([1.3, 0.9, 1.1], dtype=torch.float64))
        mu, uinit = [-0.05, 0.1, 0.03], [0.0, 0.2, -0.1]
    nu = m.nu
    return Problem(name, nu, m, fns, lambda dt: fns, m.nx, L @ L.T, terminal=m.has_terminal, lambda_=0.7,
                   noise_mu=torch.tensor(mu, dtype=torch.float64), u_init=torch.tensor(uinit, dtype=torch.float64),
                   u_scale=1.3, **bounds)


def flagged(threshold=float("inf")):
    """x = (pos, vel, flag, steps): running cost +inf while the flag is set (tests/user_models.py)."""
    m = um.flag_user_model(threshold)
    fns = (um.flag_dyn_for(threshold), um.flag_cost, None)
    return Problem("flag", 1, m, fns, lambda dt: fns, 4, torch.tensor(1.0, dtype=torch.float64), lambda_=0.5,
                   u_max=torch.tensor([3.0], dtype=torch.float64))


def _cast(v, dt):
    return v.to(dt) if torch.is_tensor(v) else v


# ---- engine and oracle ---------------------------------------------------------------------------------------------
def make_engine(pb, variant, dtype, K, T, route, S=None, U0=None, A0=None, theta0=None, batched_envs=0, **ctor):
    dyn, cost, term = pb.model.dynamics, pb.model.running_cost, (pb.model.terminal_cost if pb.terminal else None)
    if route == "stepped":
        g = pb.gpu_fns
        dyn, cost = (lambda s, a: g[0](s, a)), (lambda s, a: g[1](s, a))
        term = (lambda s, a: g[2](s, a)) if pb.terminal else None
    kw = {k: _cast(v, dtype) for k, v in pb.kw.items()}
    sigma = pb.sigma.to(dtype)
    if batched_envs:
        assert term is None                                     # MPPI_Batched takes no terminal cost (mppi.py:691-873)
        c = eng.MPPI_Batched(dyn, cost, pb.nx, sigma, num_envs=batched_envs, num_samples=K, horizon=T, device="cuda",
                             **kw, **ctor)
        c.U = U0.to(dtype)
    else:
        extra = {}
        if variant == "smppi":
            extra = dict(w_action_seq_cost=0.5, delta_t=0.8, action_max=torch.full((pb.nu,), 2.5, dtype=dtype), U_init=A0.to(dtype))
        elif variant == "kmppi":
            extra = dict(num_support_pts=S, kernel=eng.RBFKernel(sigma=rbf_sigma(T, S)), U_init=U0.to(dtype))
        else:
            extra = dict(U_init=U0.to(dtype))
        c = CLS[variant](dyn, cost, pb.nx, sigma, num_samples=K, horizon=T, device="cuda", terminal_state_cost=term,
                         **kw, **extra, **ctor)
        if variant == "kmppi":
            c.theta = theta0.to(dtype)
            c.U = U0.to(dtype)
    assert (c._model is not None) == (route == "fused")
    return c


class Oracle:
    def __init__(self, pb, variant, dtype, K, T, S=None, batched=False):
        self.variant, self.batched, self.dt = variant, batched, dtype
        dyn, cost, term = pb.cpu_fns(dtype)
        self.prob = orc.Problem(dyn, cost, pb.nx, pb.sigma.to(dtype), K=K, T=T, terminal_state_cost=term,
                                **{k: _cast(v, dtype) for k, v in pb.kw.items()})
        if variant == "smppi":
            self.sp = orc.SmoothParams(w_action_seq_cost=0.5, delta_t=0.8, action_max=torch.full((pb.nu,), 2.5, dtype=dtype))
        if variant == "kmppi":
            self.W, self.Wshift = orc.kernel_matrices(T, S, lambda a, b: orc.rbf_kernel(a, b, rbf_sigma(T, S)), dtype)

    def step(self, nom, x, z):
        d = self.dt
        nom = {k: v.to(d) for k, v in nom.items()}
        x, z = x.to(d), z.to(d)
        if self.batched:
            return orc.mppi_batched_command(self.prob, nom["U"], x, z)
        if self.variant == "mppi":
            return orc.mppi_command(self.prob, nom["U"], x, z)
        if self.variant == "smppi":
            return orc.smppi_command(self.prob, self.sp, nom["U"], nom["A"], x, z)
        return orc.kmppi_command(self.prob, nom["U"], nom["theta"], x, z, self.W, self.Wshift)


def _nominal_of(variant, r):
    out = {"U": r["U"]}
    if variant == "smppi":
        out["A"] = r["action_sequence"]
    if variant == "kmppi":
        out["theta"] = r["theta"]
    return out


def _err(a, b):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    assert a.shape == b.shape, (a.shape, b.shape)
    return float((a - b).abs().max()) if a.numel() else 0.0


def compare(tag, dtype, got, r64, r32, infeasible=None):
    """got: the engine's values; r64 / r32: the oracle in fp64 / fp32 (r32 None for fp64 controllers)."""
    for key in ("U", "action", "action_sequence", "theta"):
        if key not in got:
            continue
        e = _err(got[key], r64[key])
        assert math.isfinite(e), f"{tag}: {key} is not finite"
        bound = 1e-10 if r32 is None else 2 * _err(r32[key], r64[key]) + 1e-5
        assert e <= bound, f"{tag}: |{key} - oracle| = {e:.3e} > {bound:.3e}"
    c, c64 = got["cost_total"].double().cpu(), r64["cost_total"].double()
    assert torch.equal(torch.isinf(c), torch.isinf(c64)), f"{tag}: cost_total has infs where the oracle does not (or not)"
    fin = torch.isfinite(c64)
    assert torch.isfinite(c[fin]).all()
    rel = lambda a, b: float(((a - b).abs() / b.abs().clamp_min(1.0)).max()) if fin.any() else 0.0
    e = rel(c[fin], c64[fin])
    bound = 1e-10 if r32 is None else 2 * rel(r32["cost_total"].double()[fin], c64[fin]) + 1e-6
    assert e <= bound, f"{tag}: cost_total relative error {e:.3e} > {bound:.3e}"
    om, om64 = got["omega"].double().cpu(), r64["omega"].double()
    e = _err(om, om64)
    bound = 1e-10 if r32 is None else 2 * _err(r32["omega"], om64) + 1e-5
    assert e <= bound, f"{tag}: |omega - oracle| = {e:.3e} > {bound:.3e}"
    sums = om.sum(dim=-1)
    assert float((sums - 1).abs().max()) < 1e-5, f"{tag}: omega sums to {sums}"
    if torch.isinf(c64).any():
        assert float(om[torch.isinf(c64)].abs().max()) == 0.0, f"{tag}: an infeasible sample has a weight"
    if infeasible is not None:
        assert torch.isinf(c64[..., infeasible]).all()


def run_parity(pb, variant, dtype, K, T, route="fused", S=None, steps=2, x0=None, N=0, seed=0, infeasible=None, **ctor):
    """`steps` commands of a fresh controller against the oracle; returns the controller."""
    g = torch.Generator().manual_seed(seed)
    nu = pb.nu
    S = S or max(2, T // 2)
    rows = S if variant == "kmppi" else T
    U0 = 0.3 * torch.randn((N, T, nu) if N else (T, nu), generator=g, dtype=torch.float64)
    nom = {"U": U0}
    A0 = theta0 = None
    if variant == "smppi":
        A0 = 0.3 * torch.randn(T, nu, generator=g, dtype=torch.float64)
        nom = {"U": torch.zeros(T, nu, dtype=torch.float64), "A": A0}
    if variant == "kmppi":
        theta0 = 0.3 * torch.randn(S, nu, generator=g, dtype=torch.float64)
        nom["theta"] = theta0
    ctrl = make_engine(pb, variant, dtype, K, T, route, S=S, U0=U0, A0=A0, theta0=theta0, batched_envs=N, **ctor)
    o64 = Oracle(pb, variant, torch.float64, K, T, S, batched=bool(N))
    o32 = Oracle(pb, variant, torch.float32, K, T, S, batched=bool(N)) if dtype == torch.float32 else None
    if x0 is None:
        x0 = 0.5 * torch.randn((N, pb.nx) if N else (pb.nx,), generator=g, dtype=torch.float64)
    for step in range(steps):
        z = torch.randn(K, rows, nu, generator=g, dtype=torch.float64)
        ctrl.inject_noise(z.to(dtype))
        a = ctrl.command(x0.to(dtype).cuda())
        r64 = o64.step(nom, x0, z)
        r32 = o32.step(nom, x0, z) if o32 else None
        got = {"U": ctrl.U, "action": a, "cost_total": ctrl.cost_total, "omega": ctrl.omega}
        if variant == "smppi" and not N:
            got["action_sequence"] = ctrl.action_sequence
        if variant == "kmppi" and not N:
            got["theta"] = ctrl.theta
        compare(f"{pb.kind}/{variant}/{route}/K={K}/T={T} step {step}", dtype, got, r64, r32, infeasible)
        # keep the engine's nominal in step with the fp64 oracle
        nom = _nominal_of("mppi" if N else variant, r64)
        ctrl.U = nom["U"].to(dtype)
        if "A" in nom:
            ctrl.action_sequence = nom["A"].to(dtype)
        if "theta" in nom:
            ctrl.theta = nom["theta"].to(dtype)
    return ctrl


# ---- A. the fused reduction paths, asserted from launch_info ------------------------------------------------------
def path_of(info):
    cs = info.cluster_size
    tile = info.block_threads // info.threads_per_sample
    nc = info.grid_blocks // cs
    in_cluster = "narrow" if cs * (tile // 32) <= 64 else "records"
    if nc == 1:
        fin = "none"
    elif info.xchg_records == nc:
        fin = "ll-narrow" if nc <= 64 else "ll-records"
    else:
        fin = "ticket"
    return f"c{cs}-{in_cluster}-{fin}"


def fused_path_case(monkeypatch, variant, dtype, K, T, want, env=(), split=True, S=None, pb=None, **ctor):
    for k, v in env:
        monkeypatch.setenv(k, v)
    monkeypatch.setenv("MPPI_B200_SPLIT_COST", "1" if split else "0")
    pb = pb or pendulum()
    ctrl = run_parity(pb, variant, dtype, K, T, S=S, seed=K + T, **ctor)
    info = ctrl.launch_info
    path = path_of(info)
    assert fnmatch.fnmatch(path, want), (path, want, info.block_threads, info.threads_per_sample, info.grid_blocks)
    if ctor.get("block_threads"):
        assert info.block_threads // info.threads_per_sample == ctor["block_threads"]      # samples per tile
    assert info.split_cost == (1 if split and info.threads_per_sample > 1 else 0)
    return ctrl, info


# (id, K, T, KMPPI support points, constructor, environment, expected path, helper threads expected)
# K = 1000 at the default geometry plans 16 tiles of 64 (two clusters); 128-sample tiles make it one cluster.
# K = 16384 at the default geometry is BASELINE config 2's plan on a B200: 128 CTAs of 128 samples (4 helper threads
# each) in clusters of 4 — 16 warp records per cluster, 32 cluster records.  The single-loop kernel needs less shared
# memory and gets clusters of 8 (32 warp records, 16 cluster records): the same combine at both levels.
FUSED_PATHS = [
    ("one-cluster", 1000, 20, None, dict(block_threads=128), (), "c8-narrow-none", True),
    ("one-cluster-records", 4096, 20, None, dict(block_threads=512), (), "c8-records-none", False),
    ("config2", 16384, 20, None, {}, (), "c[48]-narrow-ll-narrow", True),
    ("cluster-records", 16384, 20, None, dict(block_threads=512), (), "c8-records-ll-narrow", False),
    # 148 one-CTA "clusters" of 64-sample tiles: 148 records of R + 2 <= 41 doubles fit the 48 KB staging
    ("ll-records", 148 * 64, 20, None, dict(block_threads=64), (("MPPI_B200_CLUSTER", "1"),), "c1-narrow-ll-records", True),
    ("ticket-knob", 16384, 20, None, {}, (("MPPI_B200_XCHG_DIRECT", "0"),), "c[48]-narrow-ticket", True),
    # 148 x (R + 2) x 8 bytes > 48 KB at R = 50 (KMPPI: 42 support points): ticket mode without the knob
    ("ticket-wide-R", 148 * 64, 50, 42, dict(block_threads=64), (("MPPI_B200_CLUSTER", "1"),), "c1-narrow-ticket", True),
    # 4689 tiles of 64 over at most 2368 CTAs: several passes, a last tile of 5 samples (its second warp has none)
    ("grid-stride", 300000 + 37, 20, None, dict(block_threads=64), (), "c*-narrow-ticket", False),
]
_FUSED_PARAMS = [pytest.param(r, split, id=f"{r[0]}[{r[6]}]" + ("" if split else "-single-loop"))
                 for r in FUSED_PATHS for split in ((True, False) if r[7] else (True,))]


@pytest.mark.parametrize("dtype", ["f64", "f32"])
@pytest.mark.parametrize("variant", ["mppi", "smppi", "kmppi"])
@pytest.mark.parametrize("row,split", _FUSED_PARAMS)
def test_fused_reduction_path_matches_oracle(row, split, variant, dtype, monkeypatch):
    name, K, T, S, ctor, env, want, _ = row
    ctrl, info = fused_path_case(monkeypatch, variant, DTYPES[dtype], K, T, want, env=env, split=split, S=S, **ctor)
    if name == "grid-stride":
        tile = info.block_threads // info.threads_per_sample
        assert info.grid_blocks * tile < K and K % tile < 32


# ---- A. the stepped route: softmin_update_kernel -> warp_fold -> warp_tail (no cluster, ticket) -----------------------
# Every CTA publishes one record; the last arrival combines the grid's nb records from the L2 workspace (combine_global).
# nb = min(n_tiles, 148 x occupancy, 2368) (plan_geometry); at 109-115 registers (ptxas) the occupancy is 8 CTAs of 64
# threads, 2 of 256.
#   few records      K = 4096: at most 4096 / 64 = 64 tiles at any tile size
#   296 records      K = 80000, 256 threads: 313 tiles, nb = min(313, 148 x 2) = 296 (two passes for some CTAs)
#   1184 records     K = 300000, 64 threads: 4688 tiles, nb = min(4688, 148 x 8) = 1184, more records than threads
STEPPED_PATHS = [("nb-le-256", 4096, {}), ("nb-gt-256", 80000, dict(block_threads=256)),
                 ("nb-gt-2BD", 300000, dict(block_threads=64))]


@pytest.mark.parametrize("dtype", ["f64", "f32"])
@pytest.mark.parametrize("variant", ["mppi", "smppi", "kmppi"])
@pytest.mark.parametrize("row", STEPPED_PATHS, ids=[r[0] for r in STEPPED_PATHS])
def test_stepped_reduction_path_matches_oracle(row, variant, dtype):
    _, K, ctor = row
    run_parity(pendulum(), variant, DTYPES[dtype], K, 20, route="stepped", seed=K, **ctor)


# ---- A. MPPI_Batched -------------------------------------------------------------------------------------------------
BATCHED = [("default", 4, 2048, 15, {}), ("large-grid", 3, 300000 + 37, 10, dict(block_threads=64))]


@pytest.mark.parametrize("dtype", ["f64", "f32"])
@pytest.mark.parametrize("route", ["fused", "stepped"])
@pytest.mark.parametrize("row", BATCHED, ids=[r[0] for r in BATCHED])
def test_batched_matches_oracle(row, route, dtype):
    _, N, K, T, ctor = row
    ctrl = run_parity(pendulum(), "mppi", DTYPES[dtype], K, T, route=route, N=N, seed=N + K, **ctor)
    if route == "fused" and ctor:
        info = ctrl.launch_info
        assert info.grid_blocks * (info.block_threads // info.threads_per_sample) < K      # grid-stride tiles


# ---- A. column boundaries: warp_fold's 32-column blocks, combine_narrow's C = R + 1 columns, the PF prefetch -----------
# R = T x nu at 31/32/33 and 63/64/65 (pendulum) and 32/64/66 (LinearPoint).  The records path uses 288-sample tiles
# (9 warp records, 72 per cluster of 8) so that a 66-row fp64 tile and the cluster's records fit in shared memory
# (about 212 KB; 512-sample tiles would need 300); its 57 tiles round up to 64 CTAs, so the last cluster carries seven
# CTAs without samples.  The one-warp paths run 32-thread CTAs (K = 6000: 188 tiles of 32 > 148 SMs, so no helper threads)
# that finish in ticket mode: combine_global's column groups must not be wider than the CTA.
COLUMN_CASES = [("pendulum", T) for T in (31, 32, 33, 63, 64, 65)] + [("linear", T) for T in (16, 32, 33)]
_ONE_WARP_TICKET = (("MPPI_B200_CLUSTER", "1"), ("MPPI_B200_XCHG_DIRECT", "0"))
COLUMN_PATHS = {"fused-narrow": (16384, {}, "c*-narrow-*", ()), "fused-records": (16384, dict(block_threads=288), "c8-records-*", ()),
                "fused-one-warp": (6000, dict(block_threads=32), "c1-narrow-ticket", _ONE_WARP_TICKET),
                "stepped-small": (4096, {}, None, ()), "stepped-large": (64000, dict(block_threads=64), None, ()),
                "stepped-one-warp": (6000, dict(block_threads=32), None, ())}


@pytest.mark.parametrize("path", sorted(COLUMN_PATHS))
@pytest.mark.parametrize("model,T", COLUMN_CASES, ids=[f"{m}-R{T * (1 if m == 'pendulum' else 2)}" for m, T in COLUMN_CASES])
def test_column_boundaries_match_oracle(model, T, path, monkeypatch):
    K, ctor, want, env = COLUMN_PATHS[path]
    pb = pendulum() if model == "pendulum" else linear_point()
    if want is None:
        run_parity(pb, "mppi", torch.float64, K, T, route="stepped", seed=T, **ctor)
    else:
        fused_path_case(monkeypatch, "mppi", torch.float64, K, T, want, env=env, pb=pb, **ctor)


# ---- B. wide models -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("split", [True, False], ids=["split-cost", "single-loop"])
@pytest.mark.parametrize("dtype", ["f64", "f32"])
@pytest.mark.parametrize("variant", ["mppi", "smppi", "kmppi"])
@pytest.mark.parametrize("model", ["arm4", "lin6"])
def test_wide_model_fused_matches_oracle(model, variant, dtype, split, monkeypatch):
    monkeypatch.setenv("MPPI_B200_SPLIT_COST", "1" if split else "0")
    ctrl = run_parity(wide(model), variant, DTYPES[dtype], 4096, 15, S=6, seed=7)
    assert ctrl.launch_info.threads_per_sample > 1 and ctrl.launch_info.split_cost == int(split)


@pytest.mark.parametrize("dtype", ["f64", "f32"])
@pytest.mark.parametrize("variant", ["mppi", "smppi", "kmppi"])
@pytest.mark.parametrize("model", ["arm4", "lin6"])
def test_wide_model_stepped_matches_oracle(model, variant, dtype):
    run_parity(wide(model), variant, DTYPES[dtype], 4096, 15, route="stepped", S=6, seed=8)


@pytest.mark.parametrize("dtype", ["f64", "f32"])
@pytest.mark.parametrize("model", ["arm4", "lin6"])
def test_wide_model_batched_fused_matches_oracle(model, dtype):
    run_parity(wide(model, terminal=False), "mppi", DTYPES[dtype], 2048, 12, N=3, seed=9)


@pytest.mark.parametrize("dtype", ["f64", "f32"])
@pytest.mark.parametrize("model", ["arm4", "lin6"])
def test_wide_model_resident_and_rollouts(model, dtype):
    """Resident commands equal launch-route commands bit for bit; the launch route equals the oracle fed the Philox
    normals it recorded; get_rollouts (the states kernel) equals the torch twin."""
    pb, dt = wide(model), DTYPES[dtype]
    K, T = 2048, 12
    U0 = 0.2 * torch.randn(T, pb.nu, generator=torch.Generator().manual_seed(3), dtype=torch.float64)
    x0 = torch.linspace(-0.4, 0.4, pb.nx, dtype=torch.float64)
    a = make_engine(pb, "mppi", dt, K, T, "fused", U0=U0, rng_seed=21)
    b = make_engine(pb, "mppi", dt, K, T, "fused", U0=U0, rng_seed=21)
    a.record_noise(True)
    o64 = Oracle(pb, "mppi", torch.float64, K, T)
    o32 = Oracle(pb, "mppi", torch.float32, K, T) if dt == torch.float32 else None
    with b.resident(idle_us=500000):
        for step in range(3):
            U_before = a.U.double().cpu().clone()
            ua = a.command_host(x0.to(dt))
            ub = b.command_host(x0.to(dt))
            assert torch.equal(ua, ub), step
            z = a.z_used.double().cpu().reshape(K, T, pb.nu)
            nom = {"U": U_before}
            r64 = o64.step(nom, x0, z)
            r32 = o32.step(nom, x0, z) if o32 else None
            compare(f"{model}/resident step {step}", dt, {"U": a.U, "action": ua, "cost_total": a.cost_total, "omega": a.omega},
                    r64, r32)
        assert b.resident_launches == 1
        assert torch.equal(a.U, b.U) and torch.equal(a.cost_total, b.cost_total)
    starts = 0.3 * torch.randn(5, pb.nx, generator=torch.Generator().manual_seed(4), dtype=torch.float64)
    seq = a.U.detach().cpu().double()
    got = a.get_rollouts(starts.to(dt), num_rollouts=5)
    assert got.shape == (5, T, pb.nx)
    want = []
    s = starts.clone()
    for t in range(T):
        s = pb.cpu_fns(torch.float64)[0](s, pb.kw["u_scale"] * seq[t].expand(5, -1))
        want.append(s)
    want = torch.stack(want, dim=1)
    assert _err(got, want) <= (1e-10 if dt == torch.float64 else 1e-4 * float(want.abs().max().clamp_min(1)))


def test_wide_model_largest_horizon_fp64():
    """nu = 4 in fp64 at the largest horizon the planner accepts (the shared-memory tile at its limit): parity with the
    oracle there; one step longer the plan is refused with MppiLibraryError before anything is launched."""
    pb = wide("arm4")

    def accepted(T):
        c = make_engine(pb, "mppi", torch.float64, 256, T, "fused", U0=torch.zeros(T, pb.nu, dtype=torch.float64))
        try:
            c.command(torch.zeros(pb.nx, dtype=torch.float64).cuda())
            return True
        except eng._cabi.MppiLibraryError:
            assert c.cost_total is None                         # refused before any launch
            assert torch.equal(c.U.cpu(), torch.zeros(T, pb.nu, dtype=torch.float64))
            return False
    lo, hi = 15, 4096
    assert accepted(lo) and not accepted(hi)
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (mid, hi) if accepted(mid) else (lo, mid)
    torch.cuda.synchronize()
    ctrl = run_parity(pb, "mppi", torch.float64, 256, lo, seed=10)
    assert not accepted(lo + 1)
    print(f"largest fp64 nu=4 horizon: T = {lo} (R = {4 * lo}), smem {ctrl.launch_info.smem_bytes} B")


# ---- C. infinite sample costs ---------------------------------------------------------------------------------------
# (id, K, constructor, infeasible mask of K).  128-sample tiles on both routes, so "the last tile" is known: K = 16421
# leaves a ragged last tile of 37 samples.
def _mask(case, K):
    m = torch.zeros(K, dtype=torch.bool)
    if case == "first-60pct":
        m[: int(0.6 * K)] = True
    elif case == "last-tile-only":
        m[: (K // 128) * 128] = True
    elif case == "random-99pct":
        m = torch.rand(K, generator=torch.Generator().manual_seed(99)) < 0.99
        m[-1] = False
    elif case == "cluster8-first-4096":
        m[:4096] = True
    return m


INF_CASES = [("first-60pct", 16384 + 37, dict(block_threads=128)), ("last-tile-only", 16384 + 37, dict(block_threads=128)),
             ("random-99pct", 16384 + 37, dict(block_threads=128)),
             # fused: 32 CTAs of 512 samples, cluster 8, 128 warp records per cluster -> combine_records over a cluster
             # whose samples are all infinite
             ("cluster8-first-4096", 16384, dict(block_threads=512))]


@pytest.mark.parametrize("dtype", ["f64", "f32"])
@pytest.mark.parametrize("variant", ["mppi", "smppi", "kmppi"])
@pytest.mark.parametrize("route", ["fused", "stepped"])
@pytest.mark.parametrize("case", INF_CASES, ids=[c[0] for c in INF_CASES])
def test_infinite_costs_match_oracle(case, route, variant, dtype):
    name, K, ctor = case
    mask = _mask(name, K)
    x0 = torch.zeros(K, 4, dtype=torch.float64)
    x0[:, 0] = torch.linspace(-1.0, 1.0, K, dtype=torch.float64)
    x0[:, 2] = mask.double()
    ctrl = run_parity(flagged(), variant, DTYPES[dtype], K, 15, route=route, S=5, x0=x0, seed=11, infeasible=mask, **ctor)
    assert torch.isinf(ctrl.cost_total.cpu()[mask]).all()
    if route == "fused" and name == "cluster8-first-4096":
        assert path_of(ctrl.launch_info) == "c8-records-ll-narrow"


@pytest.mark.parametrize("dtype", ["f64", "f32"])
@pytest.mark.parametrize("route", ["fused", "stepped"])
def test_infinite_costs_batched_match_oracle(route, dtype):
    """One start state per environment: the cost is +inf when the first perturbed action exceeds -2.5, which about
    99 % of the N(0, 1) draws around a nominal of |U| < 1 do."""
    ctrl = run_parity(flagged(threshold=-2.5), "mppi", DTYPES[dtype], 4096, 12, route=route, N=3, seed=12,
                      x0=torch.zeros(3, 4, dtype=torch.float64))
    inf = torch.isinf(ctrl.cost_total.cpu())
    assert float(inf.double().mean()) > 0.95 and not inf.all(dim=1).any()
