"""MPPI / SMPPI / KMPPI controllers with the reference's constructor + ``command()`` API
(/root/reference/src/pytorch_mppi/mppi.py:35-688), executing on hand-written sm_100a kernels.

Two execution routes, chosen at construction:

* fused  — dynamics / running_cost (/ terminal cost) are bound methods of one registered analytic
           model (pytorch_mppi_b200.models): ONE kernel launch per ``command()`` does sampling,
           rollout, softmin and the nominal update (csrc/mppi_fused.cuh `fused_command_kernel`).
* stepped — arbitrary Python callables (a torch MLP, step-dependent functions, M>1 rollouts, a
           SpecificActionSampler): the T-loop stays in Python exactly like mppi.py:312-322, with the
           sampling (`mppi_sample_perturb`), cost accumulation (`mppi_cost_accumulate`) and softmin
           update (`mppi_softmin_update`) as kernels.

There is no CPU / eager-PyTorch fallback: a missing CUDA library or a non-CUDA device raises.
PyTorch is used for device memory, streams and (multi-GPU) torch.distributed only.
"""
from __future__ import annotations

import ctypes as C
import logging
import os
import math
import time
import typing

import torch

from . import _cabi
from .models import AnalyticModel, resolve_fused_model

logger = logging.getLogger(__name__)

_DT = {torch.float32: _cabi.F32, torch.float64: _cabi.F64}
_ES = {torch.float32: 4, torch.float64: 8}


class SpecificActionSampler:
    """Same hook as the reference's (mppi.py:16-32)."""

    def __init__(self):
        self.start_idx = 0
        self.end_idx = 0
        self.slice = slice(0, 0)

    def sample_trajectories(self, state, info):
        raise NotImplementedError

    def specific_dynamics(self, next_state, state, action, t):
        return next_state

    def register_sample_start_end(self, start_idx, end_idx):
        self.start_idx = start_idx
        self.end_idx = end_idx
        self.slice = slice(start_idx, end_idx)


def _vec(x, n, name):
    """nu-vector of python floats from a float / 0-dim / (n,) tensor."""
    if x is None:
        return None
    t = torch.as_tensor(x).detach().to("cpu", torch.float64).reshape(-1)
    if t.numel() == 1:
        t = t.repeat(n)
    if t.numel() != n:
        raise ValueError(f"{name} must have {n} entries, got {t.numel()}")
    return t.tolist()


def _pad16(n_elems, es):
    return (n_elems * es + 15) // 16 * 16 // es


class MPPI:
    """Model Predictive Path Integral control (Williams et al. 2017, alg. 2), B200 engine.
    Constructor and methods mirror the reference (mppi.py:45-61, 208-290, 425-448)."""

    _VARIANT = _cabi.VARIANT_MPPI

    def __init__(self, dynamics, running_cost, nx, noise_sigma, num_samples=100, horizon=15, device="cuda",
                 terminal_state_cost=None,
                 lambda_=1.,
                 noise_mu=None,
                 u_min=None,
                 u_max=None,
                 u_init=None,
                 U_init=None,
                 u_scale=1,
                 u_per_command=1,
                 step_dependent_dynamics=False,
                 rollout_samples=1,
                 rollout_var_cost=0,
                 rollout_var_discount=0.95,
                 sample_null_action=False,
                 specific_action_sampler: typing.Optional[SpecificActionSampler] = None,
                 noise_abs_cost=False,
                 *,
                 rng_seed: typing.Optional[int] = None,
                 rng: str = "philox",
                 block_threads: int = 0,
                 threads_per_sample: int = 0,
                 process_group=None,
                 exchange: str = "p2p"):
        self._lib = _cabi.load()          # raises if the CUDA library is not built
        self.d = torch.device(device)
        if self.d.type != "cuda":
            raise ValueError("pytorch_mppi_b200 runs on CUDA devices only (pass device='cuda'); "
                             "there is no CPU fallback")
        if self.d.index is None:
            self.d = torch.device("cuda", torch.cuda.current_device())
        if not torch.is_tensor(noise_sigma):
            noise_sigma = torch.tensor(noise_sigma)
        self.dtype = noise_sigma.dtype                                         # mppi.py:88
        if self.dtype not in _DT:
            raise ValueError(f"dtype {self.dtype} is not supported (float32 / float64)")
        self.K = int(num_samples)
        self.T = int(horizon)
        self.nx = int(nx)
        self.nu = 1 if noise_sigma.dim() == 0 else noise_sigma.shape[0]        # mppi.py:94
        if self.nu > _cabi.MPPI_MAX_NU:
            raise ValueError(f"nu={self.nu} exceeds the engine's MPPI_MAX_NU={_cabi.MPPI_MAX_NU}")
        self._dirty = True
        self._lambda = float(lambda_)
        if noise_mu is None:
            noise_mu = torch.zeros(self.nu, dtype=self.dtype)
        if u_init is None:
            u_init = torch.zeros_like(torch.as_tensor(noise_mu))
        noise_mu = torch.as_tensor(noise_mu)
        if self.nu == 1:                                                       # mppi.py:104-106
            noise_mu = noise_mu.reshape(-1)
            noise_sigma = noise_sigma.reshape(-1, 1)
        self._u_scale = u_scale
        self.u_per_command = int(u_per_command)
        # bounds (mppi.py:112-126)
        if u_max is not None and u_min is None:
            u_max = torch.as_tensor(u_max)
            u_min = -u_max
        if u_min is not None and u_max is None:
            u_min = torch.as_tensor(u_min)
            u_max = -u_min
        if u_min is not None:
            self._u_min = torch.as_tensor(u_min).to(self.d)
            self._u_max = torch.as_tensor(u_max).to(self.d)
        else:
            self._u_min = torch.tensor(float("-inf"), device=self.d)
            self._u_max = torch.tensor(float("inf"), device=self.d)
        self._noise_mu = noise_mu.to(self.d, self.dtype)
        self._set_sigma(noise_sigma.to(self.d, self.dtype))
        self._u_init = torch.as_tensor(u_init).to(self.d, self.dtype).reshape(-1)

        # plugins (mppi.py:147-163)
        self.step_dependency = step_dependent_dynamics
        if step_dependent_dynamics:
            self._dynamics_fn = dynamics
            self._running_cost_fn = running_cost
        else:
            self._dynamics_fn = lambda state, u, t: dynamics(state, u)
            self._running_cost_fn = lambda state, u, t: running_cost(state, u)
        self.F = dynamics
        self.running_cost = running_cost
        self.terminal_state_cost = terminal_state_cost
        self.sample_null_action = sample_null_action
        self.specific_action_sampler = specific_action_sampler
        self.noise_abs_cost = noise_abs_cost
        self.state = None
        self.info = None
        self.M = int(rollout_samples)
        self.rollout_var_cost = rollout_var_cost
        self.rollout_var_discount = rollout_var_discount

        # route selection
        self._model: typing.Optional[AnalyticModel] = None
        if (self.M == 1 and specific_action_sampler is None and not step_dependent_dynamics):
            m = resolve_fused_model(dynamics, running_cost, terminal_state_cost)
            if m is not None and m.nx == self.nx and m.nu == self.nu:
                self._model = m
                # user model: its kernels are compiled at run time with NVRTC and registered with the stock library
                # (_pack); MPPI_B200_USER_MODEL_BUILD=nvcc builds a variant library with the toolkit instead
                self._user_model_nvcc = hasattr(m, "library_path") and os.environ.get("MPPI_B200_USER_MODEL_BUILD", "rtc") == "nvcc"
                if self._user_model_nvcc:
                    self._lib = _cabi.load(m.library_path())
        if rng not in ("philox", "torch"):
            raise ValueError("rng must be 'philox' (one subsequence per sample) or 'torch' (the stream torch.randn draws on CUDA)")
        self._rng_mode = rng
        self._block_threads = int(block_threads)
        self._pdl = os.environ.get("MPPI_B200_PDL", "1") != "0"
        # split-cost rollout for problems that run with helper threads: measured 17.1 -> 14.8 us per command back to
        # back at K=16384, T=30 (bit-identical results); MPPI_B200_SPLIT_COST=0 selects the single-loop kernel
        self._split_cost = os.environ.get("MPPI_B200_SPLIT_COST", "1") != "0"
        self._threads_per_sample = int(threads_per_sample)

        # multi-GPU: K is the GLOBAL sample count, sharded over the group (SURVEY.md §8e)
        self._pg = process_group
        self._exchange = exchange
        self._rank, self._world = 0, 1
        if process_group is not None:
            import torch.distributed as dist
            self._rank = dist.get_rank(process_group)
            self._world = dist.get_world_size(process_group)
        from .distributed import shard_bounds
        self._k_offset, self._K_local = shard_bounds(self.K, self._rank, self._world)
        self._epoch = 0
        self._mailboxes = None

        # RNG: own (seed, counter) if rng_seed is given, else the torch CUDA generator protocol
        self._rng_seed = None if rng_seed is None else int(rng_seed) & 0xFFFFFFFFFFFFFFFF
        self._rng_counter = 0
        if self._world > 1 and self._rng_seed is None:
            import torch.distributed as dist
            s = torch.empty(1, dtype=torch.int64, device=self.d)
            if self._rank == 0:
                s.fill_(torch.initial_seed() & 0x7FFFFFFFFFFFFFFF)
            dist.broadcast(s, src=dist.get_global_rank(process_group, 0) if hasattr(dist, "get_global_rank") else 0,
                           group=process_group)
            self._rng_seed = int(s.item())
        self._z_inject = None
        self._z_out = None
        self._host_box = None
        self._host_epoch = 0            # launch-route command_host() calls so far: the mailbox tag, carried across re-plans
        self._plan = None
        self._last = None
        self._resident = False          # a resident grid is armed for command_host (start_resident)
        self._resident_wanted = 0       # idle_us to re-enter resident mode with, after something made the grid leave

        # device state
        self._alloc_nominal(U_init)
        self._alloc_results()
        self._p = _cabi.MppiFusedParams()
        self._cmd_count = 0
        self._materialized_at = {}

        # sampled results from last command (mppi.py:179-184)
        self.cost_total = None
        self._states = None
        self._actions = None

    # ------------------------------------------------------------------------------------------
    # configuration that feeds kernel constants; setters mark the packed struct dirty
    # (fixes the reference's stale-cache gotcha when autotune mutates these: SURVEY.md §5)
    # ------------------------------------------------------------------------------------------
    def _set_sigma(self, sigma):
        self._noise_sigma = sigma
        self._diagonal_sigma = bool(torch.equal(sigma, torch.diag(torch.diag(sigma))))     # mppi.py:131
        if self._diagonal_sigma:
            diag = torch.diag(sigma)
            self._noise_sigma_inv_diag = 1.0 / diag
            self._noise_sigma_sqrt_diag = torch.sqrt(diag)
            self._noise_sigma_inv = torch.diag(self._noise_sigma_inv_diag)
            self._chol = torch.diag(self._noise_sigma_sqrt_diag)
        else:
            self._noise_sigma_inv = torch.linalg.inv(sigma)                                  # mppi.py:138-139
            self._chol = torch.linalg.cholesky(sigma)
        self._dirty = True

    noise_sigma = property(lambda self: self._noise_sigma, lambda self, v: self._set_sigma(torch.as_tensor(v).to(self.d, self.dtype).reshape(self.nu, self.nu)))

    @property
    def noise_sigma_inv(self):
        return self._noise_sigma_inv

    @noise_sigma_inv.setter
    def noise_sigma_inv(self, v):
        """The reference's tuner writes this next to `noise_sigma` (autotune.py:160-162).  The engine always derives the
        inverse from `noise_sigma`, so a consistent value is accepted as a no-op and an inconsistent one is an error
        (it would otherwise be silently ignored)."""
        v = torch.as_tensor(v).to(self.d, self.dtype).reshape(self.nu, self.nu)
        if not torch.allclose(v, self._noise_sigma_inv, rtol=1e-4, atol=1e-6):
            raise ValueError("noise_sigma_inv is derived from noise_sigma; assign noise_sigma (the given inverse does not "
                             "match the current covariance)")

    def _mk(name):   # noqa: N805  (tiny property factory)
        def get(self):
            return getattr(self, "_" + name)

        def set_(self, v):
            setattr(self, "_" + name, v)
            self._dirty = True
        return property(get, set_)

    lambda_ = _mk("lambda")
    u_scale = _mk("u_scale")
    u_min = _mk("u_min")
    u_max = _mk("u_max")
    noise_mu = _mk("noise_mu")
    u_init = _mk("u_init")
    del _mk

    # ------------------------------------------------------------------------------------------
    # buffers
    # ------------------------------------------------------------------------------------------
    def _rows(self):
        return self.T * self.nu

    def _alloc_nominal(self, U_init):
        es = _ES[self.dtype]
        tn = self.T * self.nu
        self._Ubuf = torch.zeros(_pad16(tn, es), device=self.d, dtype=self.dtype)
        if U_init is None:
            self.U = self._one_draw_for_all_ranks(self._sample_noise((self.T,)))            # mppi.py:144-145
        else:
            self.U = U_init

    def _one_draw_for_all_ranks(self, t):
        """A nominal drawn at random (U_init=None, reset()) has to be ONE draw for a sharded controller: every rank adds
        the same update to its copy of U, so the copies must start equal.  Rank 0's draw is broadcast."""
        if self._world > 1:
            import torch.distributed as dist
            t = t.to(self.d, self.dtype).contiguous()
            src = dist.get_global_rank(self._pg, 0) if hasattr(dist, "get_global_rank") else 0
            dist.broadcast(t, src=src, group=self._pg)
        return t

    def _alloc_results(self):
        K, tn = self._K_local, self.T * self.nu
        self._cost_buf = torch.empty(K, device=self.d, dtype=self.dtype)
        self._nominal_used = torch.zeros(3 * tn + 4, device=self.d, dtype=self.dtype)
        self._stats = torch.zeros(4, device=self.d, dtype=torch.float64)
        self._workspace = None
        self._partial = None

    @property
    def U(self):
        self._resident_sync()
        return self._Ubuf[: self.T * self.nu].view(self.T, self.nu)

    @U.setter
    def U(self, value):
        value = torch.as_tensor(value).to(self.d, self.dtype).reshape(-1, self.nu)
        if value.shape[0] != self.T:
            raise ValueError(f"U must have T={self.T} rows, got {value.shape[0]}")
        self._leave_resident()
        self._Ubuf[: self.T * self.nu].copy_(value.reshape(-1))

    @property
    def cost_total(self):
        """(K) total cost per sample of the last command (mppi.py:180, 416)"""
        self._resident_sync()
        return self._cost_total

    @cost_total.setter
    def cost_total(self, value):
        self._cost_total = value

    def _sample_noise(self, shape):
        """N(noise_mu, noise_sigma) draws for U initialisation / reset (mppi.py:201-206).  Off the hot
        path: plain torch on the device."""
        z = torch.randn(*shape, self.nu, device=self.d, dtype=self.dtype)
        if self._diagonal_sigma:
            return z * self._noise_sigma_sqrt_diag + self._noise_mu
        return z @ self._chol.T + self._noise_mu

    # ------------------------------------------------------------------------------------------
    # packing the C-ABI struct
    # ------------------------------------------------------------------------------------------
    def _variant_pack(self, p):
        pass

    def _pack(self):
        p = self._p
        nu = self.nu
        p.struct_size = C.sizeof(_cabi.MppiFusedParams)
        p.variant = self._VARIANT
        p.model = self._model.model_id if self._model is not None else 0
        p.user_model = None
        if self._model is not None and hasattr(self._model, "rtc_handle") and not getattr(self, "_user_model_nvcc", False):
            with torch.cuda.device(self.d):
                p.user_model = self._model.rtc_handle(self._lib, self.dtype, self._VARIANT)
        p.dtype = _DT[self.dtype]
        p.K, p.T, p.nx, p.nu = self._K_local, self.T, self.nx, nu
        p.S = 0
        p.u_per_command = self.u_per_command
        p.block_threads = self._block_threads
        p.threads_per_sample = self._threads_per_sample
        p.grid_blocks = 0
        p.k_offset = self._k_offset
        # sharded controllers plan their launch for the LARGEST shard: every rank then launches the same grid and
        # publishes the same number of records per command (the shards differ by at most one sample)
        p.K_geom = -(-self.K // self._world) if self._world > 1 else 0
        p.lambda_ = float(self._lambda)
        p.u_scale = float(self._u_scale)
        mu = _vec(self._noise_mu, nu, "noise_mu")
        umin = _vec(self._u_min, nu, "u_min")
        umax = _vec(self._u_max, nu, "u_max")
        uinit = _vec(self._u_init, nu, "u_init")
        L = self._chol.detach().to("cpu", torch.float64)
        Si = self._noise_sigma_inv.detach().to("cpu", torch.float64)
        for i in range(_cabi.MPPI_MAX_NU):
            p.noise_mu[i] = mu[i] if i < nu else 0.0
            p.u_min[i] = umin[i] if i < nu else 0.0
            p.u_max[i] = umax[i] if i < nu else 0.0
            p.u_init[i] = uinit[i] if i < nu else 0.0
            p.action_min[i] = -math.inf
            p.action_max[i] = math.inf
            for j in range(_cabi.MPPI_MAX_NU):
                inside = i < nu and j < nu
                p.chol[i * _cabi.MPPI_MAX_NU + j] = float(L[i, j]) if inside else 0.0
                p.sigma_inv[i * _cabi.MPPI_MAX_NU + j] = float(Si[i, j]) if inside else 0.0
        p.w_action_seq_cost = 0.0
        p.delta_t = 1.0
        blob = self._model.param_blob() if self._model is not None else []
        for i in range(_cabi.MPPI_MODEL_PARAM_DOUBLES):
            p.model_params[i] = float(blob[i]) if i < len(blob) else 0.0
        ext = self._model.param_blob_ext() if self._model is not None else []
        if ext:
            self._ext_arr = (C.c_double * len(ext))(*ext)      # host memory, read by the library at plan creation / launch
            p.model_params_ext = C.cast(self._ext_arr, C.c_void_p)
            p.n_model_params_ext = len(ext)
        else:
            p.model_params_ext = None
            p.n_model_params_ext = 0
        self._base_flags = ((_cabi.FLAG_NULL_ACTION if self.sample_null_action else 0)
                            | (_cabi.FLAG_ABS_COST if self.noise_abs_cost else 0)
                            | (_cabi.FLAG_DIAG_SIGMA if self._diagonal_sigma else 0)
                            | _cabi.FLAG_NOMINAL_PADDED
                            | (_cabi.FLAG_PDL if (self._pdl and self._model is not None) else 0)
                            | (_cabi.FLAG_SPLIT_COST if (self._split_cost and self._model is not None) else 0))
        p.U = self._Ubuf.data_ptr()
        p.A = None
        p.theta = None
        p.W = None
        p.Wshift = None
        p.cost_total = self._cost_buf.data_ptr()
        p.nominal_used = self._nominal_used.data_ptr()
        p.stats = self._stats.data_ptr()
        p.z = None
        p.z_out = None
        p.rank, p.world = self._rank, self._world
        for g in range(_cabi.MPPI_MAX_RANKS):
            p.peer_slots[g] = None
        p.partial_out = None
        dbg = getattr(self, "_debug_clocks", None)
        p.debug_clocks = None if dbg is None else dbg.data_ptr()
        p.n_env, p.env_u_stride, p.env_ws_stride = 0, 0, 0
        p.torch_rng_total = 0
        if self._rng_mode == "torch":
            # launch policy of ATen's distribution kernel (DistributionTemplates.h:50-62) for K*T*nu elements
            props = torch.cuda.get_device_properties(self.d)
            numel = self.K * self._noise_rows()
            grid = min(props.multi_processor_count * (props.max_threads_per_multi_processor // 256), (numel + 255) // 256)
            unroll = 4 if self.dtype == torch.float32 else 2
            self._torch_counter_offset = ((numel - 1) // (256 * grid * unroll) + 1) * 4
            p.torch_rng_total = 256 * grid
        od = getattr(self, "_offset_dev", None)
        p.offset_dev = None if od is None else od.data_ptr()
        per = 4 if self.dtype == torch.float32 else 2
        p.offset_inc = (self._noise_rows() + per - 1) // per
        p.host_mailbox = None
        p.host_epoch = 0
        p.xchg_status_host = None
        if self._world > 1 and self._exchange == "p2p":
            if getattr(self, "_xchg_status", None) is None:
                self._xchg_status = torch.zeros(1, dtype=torch.int64).pin_memory()     # written by the kernel on a peer timeout
                # read on every command: through ctypes (0.07 us), not int(tensor[0]) (2.2 us)
                self._xchg_status_word = C.c_longlong.from_address(self._xchg_status.data_ptr())
            p.xchg_status_host = self._xchg_status.data_ptr()
        self._variant_pack(p)
        # workspace sized for the worst-case geometry of these dimensions
        if self._model is not None:
            info = _cabi.MppiLaunchInfo()
            p.flags = self._base_flags
            _cabi.check(self._lib.mppi_fused_query(C.byref(p), C.byref(info)), "mppi_fused_query")
            self.launch_info = info
            need = int(info.workspace_bytes)
        else:
            need = 32 + 148 * 16 * (4 + self._noise_rows()) * 8 + 256 + 2 * 12288 * 8
        if self._workspace is None or self._workspace.numel() < need:
            self._workspace = torch.zeros(need, device=self.d, dtype=torch.uint8)
        p.workspace = self._workspace.data_ptr()
        p.workspace_bytes = self._workspace.numel()
        if self._world > 1:
            self._setup_exchange(p)
            if self._model is not None:       # the exchange mode depends on the peers: report the geometry of the real plan
                info = _cabi.MppiLaunchInfo()
                _cabi.check(self._lib.mppi_fused_query(C.byref(p), C.byref(info)), "mppi_fused_query")
                self.launch_info = info
        self._dirty = False
        if self._model is not None:
            self._make_plan(p)

    def _make_plan(self, p):
        """Freeze the launch state in the C library (`mppi_plan_create`): per command only the state,
        RNG counter, flags and action destination cross the boundary."""
        self._drop_plan()
        p.flags = self._base_flags | (_cabi.FLAG_EXPORT_PARTIAL if (self._world > 1 and self._exchange != "p2p") else 0)
        p.z_out = None if self._z_out is None else self._z_out.data_ptr()
        p.epoch = self._epoch
        p.host_epoch = self._host_epoch      # the new plan continues the mailbox tags where the old one stopped
        plan = C.c_void_p()
        _cabi.check(self._lib.mppi_plan_create(C.byref(p), C.byref(plan)), "mppi_plan_create")
        self._plan = plan
        self._state_arr = (C.c_double * _cabi.MPPI_MAX_NX)()
        self._scratch_action = torch.empty((self.u_per_command, self.nu), device=self.d, dtype=self.dtype)
        # command_host() hands every action back in a fresh CPU tensor the C side writes into directly
        # ((nu,) or (u_per_command, nu), mppi.py:273-274): `torch.empty_like(template)` + `data_ptr` costs 1.3 us in the
        # build container, a clone + index of a staging tensor 4.1 us, `torch.empty(shape_tuple)` 2.7 us
        self._host_out_shape = (self.nu,) if self.u_per_command == 1 else (self.u_per_command, self.nu)
        self._host_template = torch.empty(self._host_out_shape, dtype=self.dtype)

    def _drop_plan(self):
        plan = getattr(self, "_plan", None)
        if plan is not None:
            if getattr(self, "_resident", False):        # mppi_plan_destroy sends the resident grid away
                self._resident, self._resident_wanted = False, self._resident_idle_us
            # the next plan continues this one's command epochs (the tags of the reduction / exchange records)
            self._epoch = max(self._epoch, int(self._lib.mppi_plan_epoch(plan)))
            self._lib.mppi_plan_destroy(plan)
            self._plan = None

    def __del__(self):
        try:
            self._drop_plan()
        except Exception:
            pass

    def _noise_rows(self):
        return self.T * self.nu

    def _setup_exchange(self, p):
        from . import distributed as D
        if self._exchange == "p2p":
            if self._mailboxes is None:
                self._mailboxes = D.PeerMailboxes(self._lib, self._pg, self.d)
            for g in range(self._world):
                p.peer_slots[g] = self._mailboxes.ptrs[g]
        else:
            rows = self._noise_rows()
            if self._partial is None:
                self._partial = torch.zeros(rows + 2, device=self.d, dtype=torch.float64)
                self._gathered = torch.zeros(self._world * (rows + 2), device=self.d, dtype=torch.float64)
            p.partial_out = self._partial.data_ptr()

    # ------------------------------------------------------------------------------------------
    # RNG stream
    # ------------------------------------------------------------------------------------------
    def _next_rng(self):
        """(seed, counter base) for this command; the counter advances by the Philox calls one
        sample makes.  With rng_seed=None the stream is the torch CUDA generator's
        (torch.manual_seed reseeds it), consumed with the same (seed, offset) protocol ATen ops use."""
        per = 4 if self.dtype == torch.float32 else 2
        chunks = (self._noise_rows() + per - 1) // per
        if self._rng_mode == "torch":      # consume the torch CUDA generator exactly as torch.randn(K,T,nu) would
            gen = torch.cuda.default_generators[self.d.index]
            seed = gen.initial_seed() & 0xFFFFFFFFFFFFFFFF
            off = gen.get_offset()
            gen.set_offset(off + self._torch_counter_offset)
            return seed, off // 4
        if self._rng_seed is not None:
            base = self._rng_counter
            self._rng_counter += chunks
            return self._rng_seed, base
        gen = torch.cuda.default_generators[self.d.index]
        seed = gen.initial_seed() & 0xFFFFFFFFFFFFFFFF
        try:
            off = gen.get_offset()
            gen.set_offset(off + 4 * chunks)
        except (AttributeError, RuntimeError):   # very old torch: private counter keyed by the seed
            if getattr(self, "_rng_last_seed", None) != seed:
                self._rng_last_seed, self._rng_counter = seed, 0
            off = 4 * self._rng_counter
            self._rng_counter += chunks
        return seed, off // 4

    def refresh(self):
        """Re-read everything that feeds kernel constants (e.g. after retraining a PendulumMLP's network)."""
        self._dirty = True

    def inject_noise(self, z):
        """Parity hook: the next command consumes these standard normals — shape (K,T,nu)
        (KMPPI: (K,S,nu)) — instead of drawing from Philox.  This is how the engine and the
        reference/oracle are fed identical draws (SURVEY.md §8c)."""
        rows = self._noise_rows()
        z = torch.as_tensor(z).to(self.d, self.dtype).contiguous()
        if z.numel() != self._K_local * rows:
            if z.numel() == self.K * rows:   # global tensor given to a shard
                z = z.reshape(self.K, rows)[self._k_offset:self._k_offset + self._K_local].contiguous()
            else:
                raise ValueError(f"injected noise must have {self._K_local * rows} elements, got {z.numel()}")
        self._z_inject = z

    def record_noise(self, enable=True):
        """Keep the standard normals each command actually used in `self.z_used`."""
        self._z_out = torch.empty(self._K_local * self._noise_rows(), device=self.d, dtype=self.dtype) if enable else None
        self._dirty = True

    @property
    def z_used(self):
        return None if self._z_out is None else self._z_out.view(self._K_local, -1, self.nu)

    # ------------------------------------------------------------------------------------------
    # resident mode: command_host() without a kernel launch (csrc/mppi_resident.cuh)
    # ------------------------------------------------------------------------------------------
    def start_resident(self, idle_us=1000):
        """Keep the command's grid on the GPU between `command_host()` calls: each command becomes a record in
        pinned host memory that the grid polls, and the action comes back the same way — no kernel launch on the
        control loop's critical path, and the next command's noise / perturbed actions are prepared while the host
        turns around.  Results are bit-identical to the launch route.  The grid leaves by itself after `idle_us`
        microseconds without a command (the next command relaunches it), so `torch.cuda.synchronize()` never waits
        longer than that — choose `idle_us` above the control period (a 100 Hz loop wants idle_us > 10000), or every
        command pays a relaunch, which is slower than the launch route.  While resident: reading `U` / `cost_total` / `omega` / ... waits for the last command
        to finish; anything that writes controller state or launches (`command()`, setting `U`, `reset()`, parameter
        setters) makes the grid leave first and the next `command_host()` brings it back.  Write through the
        setters, not through views obtained earlier.
        Requires a registered analytic model on the split-cost rollout (a problem of at most one tile per SM, e.g.
        BASELINE config 2), host states and a single-GPU controller."""
        if self._dirty:
            self._pack()
        if self._model is None or self._plan is None:
            raise _cabi.MppiLibraryError("resident mode needs a registered model (the fused route)")
        if self._z_out is not None:
            raise _cabi.MppiLibraryError("resident mode does not record noise; call record_noise(False) first")
        words = 64 + self.u_per_command * self.nu * (2 if self.dtype == torch.float64 else 1)
        if getattr(self, "_res_box", None) is None or self._res_box.numel() != words:
            self._res_box = torch.zeros(words, dtype=torch.int64).pin_memory()
            self._res_board = torch.zeros(128, dtype=torch.int64, device=self.d)
            self._res_stream = torch.cuda.Stream(device=self.d)       # non-blocking, used for nothing else
        torch.cuda.synchronize(self.d)     # whatever wrote U / parameters on other streams is complete
        _cabi.check(self._lib.mppi_resident_start(self._plan, self._res_box.data_ptr(), self._res_board.data_ptr(),
                                                  self._scratch_action.data_ptr(), int(idle_us), self._res_stream.cuda_stream),
                    "mppi_resident_start")
        self._resident, self._resident_wanted, self._resident_idle_us = True, 0, int(idle_us)

    def stop_resident(self):
        """Send the resident grid away and stay on the launch route."""
        if self._resident and self._plan is not None:
            _cabi.check(self._lib.mppi_resident_stop(self._plan), "mppi_resident_stop")
        self._resident, self._resident_wanted = False, 0

    def resident(self, idle_us=1000):
        """`with ctrl.resident(): ... ctrl.command_host(x) ...`"""
        import contextlib

        @contextlib.contextmanager
        def cm():
            self.start_resident(idle_us)
            try:
                yield self
            finally:
                self.stop_resident()
        return cm()

    @property
    def resident_launches(self):
        """Kernel launches resident mode has made on the current plan (first command + wake-ups after idle exits)."""
        return 0 if self._plan is None else int(self._lib.mppi_resident_launches(self._plan))

    def _resident_sync(self):
        """Reads of device-side results: wait until the resident grid finished writing the last command's."""
        if getattr(self, "_resident", False):
            _cabi.check(self._lib.mppi_resident_sync(self._plan), "mppi_resident_sync")

    def _leave_resident(self):
        """Writes to controller state / launch-route commands: the grid leaves now, the next command_host() re-enters."""
        if getattr(self, "_resident", False):
            _cabi.check(self._lib.mppi_resident_stop(self._plan), "mppi_resident_stop")
            self._resident, self._resident_wanted = False, self._resident_idle_us

    def _command_resident(self, shift):
        flags = self._base_flags | (_cabi.FLAG_SHIFT if shift else 0)
        _, seed, off = self._noise_source()
        self._last = (flags, seed, off, None, None)
        self._cmd_count += 1
        out = torch.empty_like(self._host_template)
        rc = self._lib.mppi_resident_command(self._plan, self._state_arr, flags, seed, off, out.data_ptr())
        if rc != 0:
            _cabi.check(rc, "mppi_resident_command")
        if self._world > 1:
            self._epoch += 1           # mirrors the plan's exchange epoch, as on the launch route
        self._cost_total = self._cost_buf
        self._states = None
        self._actions = None
        return out

    # ------------------------------------------------------------------------------------------
    # public API (mppi.py:208-290)
    # ------------------------------------------------------------------------------------------
    def compile(self, **kwargs):
        """The reference wraps the plugins in torch.compile (mppi.py:208-215).  Here: the fused route is
        already one kernel; on the stepped route the WHOLE command — sampling kernel, the T-loop of the
        user's callables, cost accumulation, softmin update — is captured once into a CUDA graph and
        replayed (the Philox counter lives in device memory so every replay draws fresh noise).  The
        callables must be capture-safe (no host syncs, no data-dependent Python control flow)."""
        self._compile_kwargs = kwargs
        self._graph_mode = self._model is None
        self._graphs = {}

    # ---- CUDA-graph replay of the stepped route ---------------------------------------------------
    def _graph_eligible(self, state):
        return (getattr(self, "_graph_mode", False) and self._z_inject is None and self._z_out is None and self._world == 1
                and self.specific_action_sampler is None)

    def _command_graphed(self, state, shift):
        st = torch.as_tensor(state).to(self.d, self.dtype)
        key = (bool(shift), tuple(st.shape))
        if key not in self._graphs:
            try:
                self._capture_graph(key, st, shift)
            except Exception as e:     # plugin not capture-safe (host sync, H2D copy, ...): stay on the eager route
                logger.warning("compile(): CUDA-graph capture failed (%s); continuing without graphs", e)
                self._graph_mode = False
                torch.cuda.synchronize(self.d)
                try:
                    # a capture that died in the plugin leaves torch's default CUDA generator flagged as "capturing"
                    # (its next use would raise): give it a fresh state object with the same seed / offset
                    gen = torch.cuda.default_generators[self.d.index]
                    gen.graphsafe_set_state(gen.clone_state())
                except Exception:      # noqa: BLE001 — best effort; older torch has no graph-safe generator states
                    pass
                return self._command_stepped(state, shift)
        g, st_static, action_static, cost_buf = self._graphs[key]
        st_static.copy_(st)
        g.replay()
        self._cmd_count += 1
        self._materialized_at["noise"] = self._cmd_count
        self._last = None
        self._cost_buf = cost_buf                      # the buffer THIS graph writes (several keys = several graphs)
        self._p.cost_total = cost_buf.data_ptr()
        self.cost_total = self._cost_buf
        out = action_static.clone()
        return out[0] if self.u_per_command == 1 else out

    def _nominal_snapshot(self):
        snap = {"U": self._Ubuf.clone()}
        if getattr(self, "_Abuf", None) is not None:
            snap["A"] = self._Abuf.clone()
        if getattr(self, "_theta", None) is not None:
            snap["theta"] = self._theta.clone()
        return snap

    def _nominal_restore(self, snap):
        self._Ubuf.copy_(snap["U"])
        if "A" in snap:
            self._Abuf.copy_(snap["A"])
        if "theta" in snap:
            self._theta.copy_(snap["theta"])

    def _capture_graph(self, key, st, shift):
        if getattr(self, "_offset_dev", None) is None:
            # continue the host-side stream on the device: same seed, counter where the host counter stands
            if self._rng_seed is not None:
                self._graph_seed, start = self._rng_seed, self._rng_counter
            else:
                self._graph_seed, start = self._next_rng()
            self._offset_dev = torch.full((1,), start, dtype=torch.int64, device=self.d)
            self._dirty = True
        if self._dirty:
            self._pack()
        st_static = st.clone()
        snap = self._nominal_snapshot()
        off0 = self._offset_dev.clone()
        count0 = self._cmd_count
        try:
            cur = torch.cuda.current_stream(self.d)
            side = torch.cuda.Stream(device=self.d)
            side.wait_stream(cur)
            with torch.cuda.stream(side):                       # warm-up: allocator, geometry cache, lazy module loads
                for _ in range(2):
                    self._command_stepped(st_static, shift)
            cur.wait_stream(side)
            torch.cuda.synchronize(self.d)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                p, action = self._begin_command(st_static, shift)
                action = self._stepped_body(p, action, st_static)
            cost_buf = self._cost_buf                           # this graph's own result buffer
        finally:
            # the warm-up (and a failed capture) ran real commands: undo them whatever happened, so that the caller's
            # command() — replayed from the graph, or re-run eagerly after a capture failure — is the only one applied
            torch.cuda.synchronize(self.d)
            self._nominal_restore(snap)
            self._offset_dev.copy_(off0)
            self._cmd_count = count0
        self._graphs[key] = (g, st_static, action, cost_buf)

    def get_params(self):
        return f"K={self.K} T={self.T} M={self.M} lambda={self.lambda_} noise_mu={self.noise_mu.cpu().numpy()} noise_sigma={self.noise_sigma.cpu().numpy()}".replace(
            "\n", ",")

    def get_action_sequence(self):
        return self.U

    def shift_nominal_trajectory(self):
        """mppi.py:232-238.  (command() folds the shift into the kernel; this explicit form is for
        callers that shift by hand.)"""
        U = torch.roll(self.U, -1, dims=0)
        U[-1] = self._u_init
        self.U = U

    def reset(self):
        """mppi.py:286-290"""
        self.U = self._one_draw_for_all_ranks(self._sample_noise((self.T,)))

    def change_horizon(self, horizon):
        """mppi.py:277-284"""
        U = self.U.clone()
        if horizon < U.shape[0]:
            U = U[:horizon]
        elif horizon > U.shape[0]:
            U = torch.cat((U, self._u_init.repeat(horizon - U.shape[0], 1)))
        self._resize_horizon(horizon, U)

    def _resize_horizon(self, horizon, U):
        self._leave_resident()              # the buffers the resident grid reads are about to be replaced
        self.T = int(horizon)
        self._alloc_nominal(U)
        self._alloc_results()
        self._dirty = True

    def command(self, state, shift_nominal_trajectory=True, info=None):
        """mppi.py:240-252: returns the first `u_per_command` actions of the updated sequence."""
        self.info = info
        self._leave_resident()
        if self._dirty:
            self._pack()
        if self._model is not None:
            return self._command_fused(state, shift_nominal_trajectory)
        if self._graph_eligible(state):
            return self._command_graphed(state, shift_nominal_trajectory)
        return self._command_stepped(state, shift_nominal_trajectory)

    # ------------------------------------------------------------------------------------------
    # fused route
    # ------------------------------------------------------------------------------------------
    def _host_state(self, state):
        """(flags, state_dev_ptr) — host states go by value into the launch (no H2D copy); CUDA tensors
        and one-state-per-sample batches are read from device memory."""
        if torch.is_tensor(state) and state.is_cuda:
            if state.dim() == 1 and state.dtype == self.dtype and state.is_contiguous() and state.shape[0] >= self.nx:
                self.state = state                     # fast path: no torch ops on the hot path
                return _cabi.FLAG_STATE_DEVICE, state.data_ptr()
            st = state.to(self.dtype)
            if st.dim() == 2 and st.shape == (self.K, self.nx) and self.K != 1:
                st = st[self._k_offset:self._k_offset + self._K_local].contiguous()
                self.state = st
                return _cabi.FLAG_STATE_DEVICE | _cabi.FLAG_STATE_PER_SAMPLE, st.data_ptr()
            st = st.reshape(-1).contiguous()
            self.state = st
            return _cabi.FLAG_STATE_DEVICE, st.data_ptr()
        vals = state.tolist() if hasattr(state, "tolist") else list(state)
        if len(vals) and isinstance(vals[0], (list, tuple)):
            if len(vals) == self.K and self.K != 1:   # (K,nx) host states -> upload once
                return self._host_state(torch.as_tensor(state).to(self.d))
            vals = vals[0]
        if len(vals) < self.nx:
            raise ValueError(f"state has {len(vals)} entries, nx={self.nx}")
        self._state_arr[: self.nx] = vals[: self.nx]
        self.state = state
        return 0, None

    def _check_exchange_status(self):
        """A peer exchange that timed out inside an earlier command left this rank's nominal one update behind its
        peers (the kernel returned the un-updated nominal as the action and flagged a pinned status word): refuse to
        continue silently."""
        st = getattr(self, "_xchg_status_word", None)
        if st is not None and st.value != 0:
            code = int(st.value)
            st.value = 0
            raise _cabi.MppiLibraryError(
                f"a peer exchange of an earlier command() timed out on rank {self._rank} (status {code}): this rank's nominal "
                "sequence is now out of step with its peers; reset() / re-synchronise U across ranks before continuing "
                "(MPPI_B200_XCHG_TIMEOUT_S sets the wait, default 20 s)")

    def _noise_source(self):
        """(z_ptr, seed, offset) for this command."""
        if self._z_inject is not None:
            self._z_keep = self._z_inject          # stays alive for lazy materialisation
            self._z_inject = None
            return self._z_keep.data_ptr(), 0, 0
        self._z_keep = None
        if getattr(self, "_offset_dev", None) is not None:     # counter lives on the device (CUDA-graph mode)
            return None, self._graph_seed, 0
        seed, off = self._next_rng()
        return None, seed, off

    def _command_fused(self, state, shift):
        if self._world > 1:
            self._check_exchange_status()
        sflags, sdev = self._host_state(state)
        flags = self._base_flags | sflags | (_cabi.FLAG_SHIFT if shift else 0)
        zptr, seed, off = self._noise_source()
        action = torch.empty((self.u_per_command, self.nu), device=self.d, dtype=self.dtype)
        stream = torch._C._cuda_getCurrentRawStream(self.d.index)
        self._last = (flags, seed, off, zptr, sdev)
        self._cmd_count += 1
        rc = self._lib.mppi_plan_command(self._plan, None if sdev is not None else self._state_arr, sdev, flags, seed, off,
                                         zptr, action.data_ptr(), stream)
        if rc != 0:
            _cabi.check(rc, "mppi_plan_command")
        if self._world > 1:
            self._epoch += 1
            if self._exchange != "p2p":
                self._finish_exported(action, stream)
        self.cost_total = self._cost_buf
        self._states = None
        self._actions = None
        return action[0] if self.u_per_command == 1 else action                            # mppi.py:273-274

    def _finish_exported(self, action, stream):
        """NCCL route: all-gather the per-rank records, then `mppi_apply_partials` finishes the update."""
        import torch.distributed as dist
        p = self._p
        dist.all_gather_into_tensor(self._gathered, self._partial, group=self._pg)
        p.flags = self._base_flags
        p.action_out = action.data_ptr()
        _cabi.check(self._lib.mppi_apply_partials(C.byref(p), self._gathered.data_ptr(), stream), "mppi_apply_partials")

    def _sync_params_for_materialize(self):
        """Write the last command's per-call values back into the parameter struct (the plan path does not)."""
        p = self._p
        flags, seed, off, zptr, sdev = self._last
        p.flags = flags & ~_cabi.FLAG_SHIFT
        p.seed, p.offset = seed, off
        p.z = zptr
        p.state_dev = sdev
        for i in range(self.nx):
            p.state[i] = self._state_arr[i]

    # -- struct-based command setup used by the stepped route ------------------------------------
    def _begin_command(self, state, shift):
        p = self._p
        flags = self._base_flags | (_cabi.FLAG_SHIFT if shift else 0)
        zptr, seed, off = self._noise_source()
        p.z = zptr
        p.seed, p.offset = seed, off
        p.state_dev = None
        p.z_out = None if self._z_out is None else self._z_out.data_ptr()
        if self._world > 1:
            self._epoch += 1
            p.epoch = self._epoch
            if self._exchange != "p2p":
                flags |= _cabi.FLAG_EXPORT_PARTIAL
        p.flags = flags
        action = torch.empty((self.u_per_command, self.nu), device=self.d, dtype=self.dtype)
        p.action_out = action.data_ptr()
        self._cmd_count += 1
        self._last = None
        return p, action

    def _finish_command(self, p, action, stream):
        if self._world > 1 and self._exchange != "p2p":
            self._finish_exported(action, stream)
        self.cost_total = self._cost_buf
        self._states = None
        self._actions = None
        if self.u_per_command == 1:                                                        # mppi.py:273-274
            return action[0]
        return action

    def command_host(self, state, shift_nominal_trajectory=True, info=None):
        """`command()` for a control loop that lives on the host: the start state travels in the
        kernel's parameter block (no H2D copy) and the kernel stores the action straight into pinned
        host memory followed by an epoch flag; the C library spins on that flag — no D2H memcpy call,
        no stream synchronise.  Returns a CPU tensor ((nu,) or (u_per_command, nu)); the device-side
        state (U, cost_total, ...) is exactly what `command()` leaves."""
        self.info = info
        if self._dirty:
            self._pack()
        if self._model is None or (torch.is_tensor(state) and state.is_cuda) or self._world > 1 and self._exchange != "p2p":
            out = self.command(state, shift_nominal_trajectory, info)      # stepped / device-state / NCCL route
            return out.cpu()
        if self._host_box is None:
            words = self.u_per_command * self.nu * (2 if self.dtype == torch.float64 else 1)
            self._host_box = torch.zeros(words, dtype=torch.int64).pin_memory()
        sflags, sdev = self._host_state(state)
        if sdev is not None:
            return self.command(state, shift_nominal_trajectory, info).cpu()
        if self._resident or self._resident_wanted:
            if self._z_inject is None and getattr(self, "_offset_dev", None) is None:
                if not self._resident:
                    self.start_resident(self._resident_wanted)
                return self._command_resident(shift_nominal_trajectory)
            self._leave_resident()         # injected noise / device-resident counter: a launch-route command
        if self._world > 1:
            self._check_exchange_status()
        flags = self._base_flags | (_cabi.FLAG_SHIFT if shift_nominal_trajectory else 0)
        zptr, seed, off = self._noise_source()
        stream = torch._C._cuda_getCurrentRawStream(self.d.index)
        self._last = (flags, seed, off, zptr, None)
        self._cmd_count += 1
        out = torch.empty_like(self._host_template)
        self._host_epoch += 1
        rc = self._lib.mppi_plan_command_host(self._plan, self._state_arr, flags, seed, off, zptr,
                                              self._scratch_action.data_ptr(), self._host_box.data_ptr(), out.data_ptr(), stream)
        if rc != 0:
            _cabi.check(rc, "mppi_plan_command_host")
        if self._world > 1:
            self._epoch += 1
        self._cost_total = self._cost_buf
        self._states = None
        self._actions = None
        return out

    # ------------------------------------------------------------------------------------------
    # stepped route (arbitrary callables): mppi.py:297-373 with kernels around the T-loop
    # ------------------------------------------------------------------------------------------
    def _ensure_step_buffers(self):
        K, T, nu = self._K_local, self.T, self.nu
        if getattr(self, "_pa_buf", None) is None or self._pa_buf.shape != (K, T, nu):
            self._pa_buf = torch.empty(K, T, nu, device=self.d, dtype=self.dtype)
            self._noise_buf = torch.empty(K, T, nu, device=self.d, dtype=self.dtype)
            self._cost_init = torch.empty(K, device=self.d, dtype=self.dtype)
            self._noise_theta_buf = None

    def _eps_for_update(self):
        return self._noise_buf

    def _command_stepped(self, state, shift):
        if self._world > 1:
            self._check_exchange_status()
        lib = self._lib
        self._ensure_step_buffers()
        if not torch.is_tensor(state):
            state = torch.tensor(state)
        st = state.to(dtype=self.dtype, device=self.d)                                     # mppi.py:262-264
        p, action = self._begin_command(st, shift)
        out = self._stepped_body(p, action, st)
        return out[0] if self.u_per_command == 1 else out

    def _stepped_body(self, p, action, st):
        """Everything of one stepped command that runs on the device; returns the (u_per_command, nu) action."""
        lib = self._lib
        self.state = st
        stream = torch.cuda.current_stream(self.d).cuda_stream
        K, T, nu = self._K_local, self.T, self.nu

        ovr_ptr, n_ovr, ovr_start = None, 0, 0
        if self.specific_action_sampler is not None:                                       # mppi.py:393-399
            acts = self.specific_action_sampler.sample_trajectories(self.state, self.info)
            acts = acts.reshape(-1, T, nu).to(self.d, self.dtype).contiguous()
            ovr_start = 1 if self.sample_null_action else 0
            n_ovr = acts.shape[0]
            self.specific_action_sampler.register_sample_start_end(ovr_start, ovr_start + n_ovr)
            self._ovr_keep = acts
            ovr_ptr = acts.data_ptr()
        nth = None if self._noise_theta_buf is None else self._noise_theta_buf.data_ptr()
        _cabi.check(lib.mppi_sample_perturb(C.byref(p), self._pa_buf.data_ptr(), self._noise_buf.data_ptr(), nth,
                                            self._cost_init.data_ptr(), ovr_ptr, n_ovr, ovr_start, stream),
                    "mppi_sample_perturb")
        self._materialized_at["noise"] = self._cmd_count

        if self.M == 1:
            rollout, states, actions = self._rollout_single(self._pa_buf, stream)
        else:
            rollout, states, actions = self._rollout_multi(self._pa_buf, stream)
        # cost_total = rollout + perturbation (+ smoothness), mppi.py:416 / :569
        _cabi.check(lib.mppi_cost_accumulate(rollout.data_ptr(), self._cost_init.data_ptr(), None, 1, K, 1.0,
                                             _DT[self.dtype], stream), "mppi_cost_accumulate")
        self._cost_buf = rollout
        p.cost_total = rollout.data_ptr()
        _cabi.check(lib.mppi_softmin_update(C.byref(p), rollout.data_ptr(), self._eps_for_update().data_ptr(), stream),
                    "mppi_softmin_update")
        self._finish_command(p, action, stream)
        self._states = states
        self._actions = actions / self._u_scale if actions is not None else None         # mppi.py:412
        return action

    def _rollout_single(self, perturbed_actions, stream):
        """mppi.py:297-332"""
        lib = self._lib
        K, T, nu = perturbed_actions.shape
        cost_total = torch.zeros(K, device=self.d, dtype=self.dtype)
        if self.state.shape == (self.K, self.nx) and self.K != 1:
            state = self.state[self._k_offset:self._k_offset + K].clone()
        else:
            state = self.state.view(1, -1).expand(K, -1)
        need_storage = self.terminal_state_cost is not None
        states = actions = None
        if need_storage:
            states = torch.empty(1, K, T, self.nx, device=self.d, dtype=self.dtype)
            actions = torch.empty(1, K, T, nu, device=self.d, dtype=self.dtype)
        dt = _DT[self.dtype]
        for t in range(T):
            u = self._u_scale * perturbed_actions[:, t]
            state = self._dynamics_fn(state, u, t)
            if self.specific_action_sampler is not None:
                state = self.specific_action_sampler.specific_dynamics(
                    state.unsqueeze(0), state.unsqueeze(0), u.unsqueeze(0), t).squeeze(0)
            c = self._running_cost_fn(state, u, t).reshape(K)
            if c.dtype != self.dtype or not c.is_contiguous():
                c = c.to(self.dtype).contiguous()
            rc = lib.mppi_cost_accumulate(cost_total.data_ptr(), c.data_ptr(), None, 1, K, 1.0, dt, stream)
            if rc != 0:
                _cabi.check(rc, "mppi_cost_accumulate")
            if need_storage:
                states[0, :, t] = state[:, :self.nx]
                actions[0, :, t] = u
        if need_storage:
            c = self.terminal_state_cost(states, actions)
            if torch.is_tensor(c) and c.dim() > 1:
                c = c.squeeze(0)
            if torch.is_tensor(c):
                c = c.to(self.dtype).reshape(K).contiguous()
                _cabi.check(lib.mppi_cost_accumulate(cost_total.data_ptr(), c.data_ptr(), None, 1, K, 1.0, dt, stream),
                            "mppi_cost_accumulate")
            else:
                cost_total += c
        return cost_total, states, actions

    def _rollout_multi(self, perturbed_actions, stream):
        """mppi.py:334-373 (M>1: stochastic dynamics with a discounted variance cost)"""
        lib = self._lib
        K, T, nu = perturbed_actions.shape
        M = self.M
        dt = _DT[self.dtype]
        cost_samples = torch.zeros(M, K, device=self.d, dtype=self.dtype)
        cost_var = torch.zeros(K, device=self.d, dtype=self.dtype)
        if self.state.shape == (self.K, self.nx) and self.K != 1:
            state = self.state[self._k_offset:self._k_offset + K]
        else:
            state = self.state.view(1, -1).expand(K, -1)
        state = state.repeat(M, 1, 1)
        states = torch.empty(M, K, T, self.nx, device=self.d, dtype=self.dtype)
        actions = torch.empty(M, K, T, nu, device=self.d, dtype=self.dtype)
        MK = M * K
        state_flat = state.reshape(MK, self.nx)
        # mppi.py:174-175: discount^t evaluated in the controller dtype (so fp32 controllers use the reference's factors)
        disc = (self.rollout_var_discount ** torch.arange(T, dtype=self.dtype)).tolist()
        for t in range(T):
            u = self._u_scale * perturbed_actions[:, t].expand(M, -1, -1)
            u_flat = u.reshape(MK, nu)
            state_flat = self._dynamics_fn(state_flat, u_flat, t)
            if self.specific_action_sampler is not None:
                s3 = state_flat.reshape(M, K, -1)
                s3 = self.specific_action_sampler.specific_dynamics(s3, state.reshape(M, K, -1), u, t)
                state_flat = s3.reshape(MK, -1)
            c = self._running_cost_fn(state_flat, u_flat, t).reshape(MK).to(self.dtype).contiguous()
            _cabi.check(lib.mppi_cost_accumulate(cost_samples.data_ptr(), c.data_ptr(), cost_var.data_ptr(), M, K,
                                                 disc[t], dt, stream), "mppi_cost_accumulate")
            states[:, :, t] = state_flat.reshape(M, K, -1)[:, :, :self.nx]
            actions[:, :, t] = u
        if self.terminal_state_cost is not None:
            cost_samples = cost_samples + self.terminal_state_cost(states, actions)
        cost_total = cost_samples.mean(dim=0) + cost_var * self.rollout_var_cost
        return cost_total.contiguous(), states, actions

    # ------------------------------------------------------------------------------------------
    # API-visible intermediates, materialised on demand (mppi.py:180-184, 383-385)
    # ------------------------------------------------------------------------------------------
    def _materialize(self, want_states=False):
        if self.cost_total is None:
            return False
        key = "states" if want_states else "noise"
        if self._materialized_at.get(key) == self._cmd_count:
            return True
        self._ensure_step_buffers()
        p = self._p
        if getattr(self, "_last", None) is not None:
            self._sync_params_for_materialize()
        stream = torch.cuda.current_stream(self.d).cuda_stream
        nth = None if self._noise_theta_buf is None else self._noise_theta_buf.data_ptr()
        st_ptr = None
        if want_states:
            self._states_buf = torch.empty(self._K_local, self.T, self.nx, device=self.d, dtype=self.dtype)
            st_ptr = self._states_buf.data_ptr()
        _cabi.check(self._lib.mppi_materialize(C.byref(p), self._pa_buf.data_ptr(), self._noise_buf.data_ptr(), nth,
                                               st_ptr, stream), "mppi_materialize")
        self._materialized_at["noise"] = self._cmd_count
        if want_states:
            self._materialized_at["states"] = self._cmd_count
        return True

    @property
    def noise(self):
        return self._noise_buf if self._materialize() else None

    @property
    def perturbed_action(self):
        return self._pa_buf if self._materialize() else None

    @property
    def omega(self):
        """mppi.py:258"""
        if self.cost_total is None:
            return None
        if self._materialized_at.get("omega") != self._cmd_count:
            self._omega_buf = torch.empty_like(self.cost_total)
            stream = torch.cuda.current_stream(self.d).cuda_stream
            _cabi.check(self._lib.mppi_omega(self.cost_total.data_ptr(), self._omega_buf.data_ptr(), self._stats.data_ptr(),
                                             float(self._lambda), self._K_local, _DT[self.dtype], stream), "mppi_omega")
            self._materialized_at["omega"] = self._cmd_count
        return self._omega_buf

    @property
    def cost_total_non_zero(self):
        """mppi.py:256: exp(-(c-beta)/lambda) = omega * eta"""
        om = self.omega
        return None if om is None else om * self._stats[1].to(self.dtype)

    @property
    def states(self):
        """(1,K,T,nx) iff a terminal cost is set (mppi.py:307-310, test_mppi.py:241-260)"""
        if self.cost_total is None or self.terminal_state_cost is None:
            return None
        if self._model is None:
            return self._states
        self._materialize(want_states=True)
        return self._states_buf.unsqueeze(0)

    @property
    def actions(self):
        if self.cost_total is None or self.terminal_state_cost is None:
            return None
        if self._model is None:
            return self._actions
        self._materialize()
        return self._pa_buf.unsqueeze(0)          # (u_scale * pa) / u_scale, mppi.py:412

    @property
    def beta(self):
        return None if self.cost_total is None else self._stats[0]

    @property
    def eta(self):
        return None if self.cost_total is None else self._stats[1]

    def get_rollouts(self, state, num_rollouts=1, U=None):
        """mppi.py:425-448: open-loop replay of one control sequence through the dynamics plugin."""
        state = torch.as_tensor(state).to(self.d, self.dtype).view(-1, self.nx)
        if state.size(0) == 1:
            state = state.expand(num_rollouts, -1)
        if U is None:
            U = self.get_action_sequence()
        T = U.shape[0]
        if self._model is not None and torch.is_tensor(U) and U.dim() == 2 and U.shape[1] == self.nu and T >= 1:
            # registered model: one launch of the states kernel (every rollout replays the same sequence)
            if state.size(0) != num_rollouts:
                raise ValueError(f"state has {state.size(0)} rows, expected 1 or num_rollouts={num_rollouts}")
            if self._dirty:
                self._pack()
            x0 = state.contiguous()
            seq = U.to(self.d, self.dtype).contiguous()
            out = torch.empty((num_rollouts, T, self.nx), dtype=self.dtype, device=self.d)
            stream = torch.cuda.current_stream(self.d).cuda_stream
            _cabi.check(self._lib.mppi_rollout_states(C.byref(self._p), x0.data_ptr(), seq.data_ptr(), 0, num_rollouts, T,
                                                      out.data_ptr(), stream), "mppi_rollout_states")
            return out
        states = torch.zeros((num_rollouts, T + 1, self.nx), dtype=U.dtype, device=U.device)
        states[:, 0] = state
        for t in range(T):
            nxt = self._dynamics_fn(states[:, t].view(num_rollouts, -1), self._u_scale * U[t].expand(num_rollouts, -1), t)
            states[:, t + 1] = nxt[:, :self.nx]
        return states[:, 1:]


class SMPPI(MPPI):
    """Smooth MPPI: noise is sampled on the control derivative, actions are its integral, and the
    change between consecutive actions is penalised (mppi.py:451-570, arXiv:2112.09988)."""

    _VARIANT = _cabi.VARIANT_SMPPI

    def __init__(self, *args, w_action_seq_cost=1., delta_t=1., U_init=None, action_min=None, action_max=None, **kwargs):
        self.w_action_seq_cost = w_action_seq_cost
        self.delta_t = delta_t
        self._Abuf = None
        super().__init__(*args, U_init=U_init, **kwargs)
        if action_min is not None and action_max is None:                                  # mppi.py:464-477
            action_min = torch.as_tensor(action_min)
            action_max = -action_min
        if action_max is not None and action_min is None:
            action_max = torch.as_tensor(action_max)
            action_min = -action_max
        if action_min is not None:
            self.action_min = torch.as_tensor(action_min).to(self.d)
            self.action_max = torch.as_tensor(action_max).to(self.d)
        else:
            self.action_min = torch.tensor(float("-inf"), device=self.d)
            self.action_max = torch.tensor(float("inf"), device=self.d)
        # the lifted formulation starts from zero controls (mppi.py:480-484)
        if U_init is None:
            self.action_sequence = torch.zeros_like(self.U)
        else:
            self.action_sequence = U_init
        self.U = torch.zeros_like(self.U)
        self._dirty = True

    def _alloc_nominal(self, U_init):
        super()._alloc_nominal(U_init)
        old = self._Abuf
        self._Abuf = torch.zeros_like(self._Ubuf)
        if old is not None:
            n = min(old.numel(), self._Abuf.numel())
            self._Abuf[:n].copy_(old[:n])

    @property
    def action_sequence(self):
        self._resident_sync()
        # one view object per buffer: `ctrl.get_action_sequence() is ctrl.action_sequence` holds as in the reference
        # (test_mppi.py:452-456), and the kernels update it in place
        v = getattr(self, "_A_view", None)
        if v is None or v.data_ptr() != self._Abuf.data_ptr() or v.shape != (self.T, self.nu):
            v = self._A_view = self._Abuf[: self.T * self.nu].view(self.T, self.nu)
        return v

    @action_sequence.setter
    def action_sequence(self, value):
        value = torch.as_tensor(value).to(self.d, self.dtype).reshape(-1, self.nu)
        self._leave_resident()
        self._Abuf[: self.T * self.nu].copy_(value.reshape(-1))

    def _variant_pack(self, p):
        p.A = self._Abuf.data_ptr()
        p.w_action_seq_cost = float(self.w_action_seq_cost)
        p.delta_t = float(self.delta_t)
        amin = _vec(self.action_min, self.nu, "action_min")
        amax = _vec(self.action_max, self.nu, "action_max")
        for i in range(self.nu):
            p.action_min[i] = amin[i]
            p.action_max[i] = amax[i]

    def get_params(self):
        return f"{super().get_params()} w={self.w_action_seq_cost} t={self.delta_t}"

    def shift_nominal_trajectory(self):
        """mppi.py:489-493"""
        super().shift_nominal_trajectory()
        A = torch.roll(self.action_sequence, -1, dims=0)
        A[-1] = A[-2]
        self.action_sequence = A

    def get_action_sequence(self):
        return self.action_sequence

    def reset(self):
        """mppi.py:498-500"""
        self._leave_resident()
        self._Ubuf.zero_()
        self._Abuf.zero_()

    def change_horizon(self, horizon):
        """mppi.py:502-512"""
        U = self.U.clone()
        A = self.action_sequence.clone()
        self._leave_resident()
        if horizon < U.shape[0]:
            U, A = U[:horizon], A[:horizon]
        elif horizon > U.shape[0]:
            ext = horizon - U.shape[0]
            U = torch.cat((U, self._u_init.repeat(ext, 1)))
            A = torch.cat((A, A[-1].repeat(ext, 1)))
        self._Abuf = None
        self._resize_horizon(horizon, U)
        self.action_sequence = A

    @property
    def perturbed_control(self):
        """mppi.py:546 (clamped, unused by the algorithm itself): U + coloured noise, bounded."""
        n = self.noise
        if n is None:
            return None
        tn = self.T * self.nu
        Uu = self._nominal_used[:tn].view(self.T, self.nu)
        return torch.clamp(Uu + n, self._u_min, self._u_max)


class TimeKernel:
    """Kernel acting on the time dimension of trajectories (mppi.py:573-577)."""

    def __call__(self, t, tk):
        raise NotImplementedError


class RBFKernel(TimeKernel):
    """mppi.py:580-590"""

    def __init__(self, sigma=1):
        self.sigma = sigma

    def __repr__(self):
        return f"RBFKernel(sigma={self.sigma})"

    def __call__(self, t, tk):
        d = torch.sum((t[:, None] - tk) ** 2, dim=-1)
        return torch.exp(-d / (1e-8 + 2 * self.sigma ** 2))


class KMPPI(MPPI):
    """MPPI with kernel interpolation of control points for smoothing (mppi.py:593-688).

    The reference solves a (S x S) system per sample through torch.vmap; the interpolation operator
    ``W = k(Hs,Tk) k(Tk,Tk)^-1`` is sample-independent, so it is computed once here and staged in
    shared memory by the kernel."""

    _VARIANT = _cabi.VARIANT_KMPPI

    def __init__(self, *args, num_support_pts=None, kernel: TimeKernel = RBFKernel(), **kwargs):
        self.num_support_pts = None
        self.interpolation_kernel = kernel
        self._theta = None
        super().__init__(*args, **kwargs)
        self.num_support_pts = int(num_support_pts or self.T // 2)                         # mppi.py:598
        self._theta = torch.zeros((self.num_support_pts, self.nu), dtype=self.dtype, device=self.d)
        self.prepare_vmap_interpolation()
        self._alloc_results()
        self._dirty = True

    @property
    def theta(self):
        self._resident_sync()
        return self._theta

    @theta.setter
    def theta(self, v):
        self._leave_resident()
        self._theta.copy_(torch.as_tensor(v).to(self.d, self.dtype).reshape(self.num_support_pts, self.nu))

    def _noise_rows(self):
        S = self.num_support_pts if self.num_support_pts else self.T
        return S * self.nu

    def get_params(self):
        return f"{super().get_params()} num_support_pts={self.num_support_pts} kernel={self.interpolation_kernel}"

    def prepare_vmap_interpolation(self):
        """mppi.py:636-648 reduced to its sample-independent content: Tk, Hs and the two operators."""
        S, T = self.num_support_pts, self.T
        self.Tk = torch.linspace(0, T - 1, int(S), device=self.d, dtype=self.dtype).unsqueeze(0)
        self.Hs = torch.linspace(0, T - 1, int(T), device=self.d, dtype=self.dtype).unsqueeze(0)
        tk = self.Tk[0]
        G = self.interpolation_kernel(tk.unsqueeze(-1), tk.unsqueeze(-1))
        self._W = torch.linalg.solve(G, self.interpolation_kernel(self.Hs[0].unsqueeze(-1), tk.unsqueeze(-1)), left=False).contiguous()
        self._Wshift = torch.linalg.solve(G, self.interpolation_kernel((tk + 1).unsqueeze(-1), tk.unsqueeze(-1)), left=False).contiguous()

    def do_kernel_interpolation(self, t, tk, c):
        """mppi.py:621-627"""
        K = self.interpolation_kernel(t.unsqueeze(-1), tk.unsqueeze(-1))
        Ktktk = self.interpolation_kernel(tk.unsqueeze(-1), tk.unsqueeze(-1))
        KK = torch.linalg.solve(Ktktk, K, left=False)
        return torch.matmul(KK, c), K

    def deparameterize_to_trajectory_single(self, theta):
        return self.do_kernel_interpolation(self.Hs[0], self.Tk[0], theta)

    def deparameterize_to_trajectory_batch(self, theta):
        assert theta.shape == (self.K, self.num_support_pts, self.nu)
        return torch.matmul(self._W, theta), None

    def change_horizon(self, horizon):
        """The reference inherits MPPI.change_horizon (mppi.py:277-284) and then fails on stale interpolation
        matrices; here the control points are kept, the time grids and operators are rebuilt for the new horizon, and
        the trajectory is re-derived from the control points (U = W theta, as mppi.py:682 leaves it)."""
        self._leave_resident()
        self._resize_horizon(int(horizon), torch.zeros(int(horizon), self.nu, device=self.d, dtype=self.dtype))
        self.prepare_vmap_interpolation()
        self.U = self._W @ self._theta
        self._dirty = True

    def _variant_pack(self, p):
        p.S = self.num_support_pts
        p.theta = self._theta.data_ptr()
        p.W = self._W.data_ptr()
        p.Wshift = self._Wshift.data_ptr()

    def reset(self):
        """mppi.py:613-615"""
        super().reset()
        self._leave_resident()
        self._theta.zero_()

    def shift_nominal_trajectory(self):
        """mppi.py:617-619"""
        super().shift_nominal_trajectory()
        self._leave_resident()
        self._theta.copy_(self._Wshift @ self._theta)

    def _ensure_step_buffers(self):
        super()._ensure_step_buffers()
        shape = (self._K_local, self.num_support_pts, self.nu)
        if self._noise_theta_buf is None or self._noise_theta_buf.shape != shape:
            self._noise_theta_buf = torch.empty(*shape, device=self.d, dtype=self.dtype)

    def _eps_for_update(self):
        return self._noise_theta_buf

    @property
    def noise_theta(self):
        return self._noise_theta_buf if self._materialize() else None


class MPPI_Batched(MPPI):
    """MPPI for N parallel environments (mppi.py:691-873): the K noise samples are shared across
    environments, every environment keeps its own nominal sequence and softmin.  The reference
    concatenates N*K rows into one dynamics call per step; here the N problems are the y-dimension of
    ONE launch (registered models: the fused kernel; arbitrary callables: the sampling and softmin
    kernels around the Python T-loop)."""

    def __init__(self, dynamics, running_cost, nx, noise_sigma, num_envs, num_samples=100, horizon=15, device="cuda",
                 lambda_=1., noise_mu=None, u_min=None, u_max=None, u_init=None, u_scale=1, u_per_command=1,
                 step_dependent_dynamics=False, noise_abs_cost=False, *, rng_seed=None, block_threads=0):
        self.N = int(num_envs)
        super().__init__(dynamics, running_cost, nx, noise_sigma, num_samples=num_samples, horizon=horizon, device=device,
                         lambda_=lambda_, noise_mu=noise_mu, u_min=u_min, u_max=u_max, u_init=u_init, u_scale=u_scale,
                         u_per_command=u_per_command, step_dependent_dynamics=step_dependent_dynamics,
                         noise_abs_cost=noise_abs_cost, rng_seed=rng_seed, block_threads=block_threads, threads_per_sample=0)

    # ---- (N, ...) buffers ------------------------------------------------------------------------
    def _alloc_nominal(self, U_init):
        es = _ES[self.dtype]
        self._u_stride = _pad16(self.T * self.nu, es)
        self._Ubuf = torch.zeros(self.N, self._u_stride, device=self.d, dtype=self.dtype)
        self.U = self._sample_noise((self.N, self.T)) if U_init is None else U_init          # mppi.py:807

    def _alloc_results(self):
        tn = self.T * self.nu
        self._cost_buf = torch.empty(self.N, self.K, device=self.d, dtype=self.dtype)
        self._nominal_used = torch.zeros(self.N, 3 * tn + 4, device=self.d, dtype=self.dtype)
        self._stats = torch.zeros(self.N, 4, device=self.d, dtype=torch.float64)
        self._workspace = None
        self._partial = None

    @property
    def U(self):
        return self._Ubuf[:, : self.T * self.nu].view(self.N, self.T, self.nu)

    @U.setter
    def U(self, value):
        value = torch.as_tensor(value).to(self.d, self.dtype).reshape(self.N, self.T * self.nu)
        self._Ubuf[:, : self.T * self.nu].copy_(value)

    def _variant_pack(self, p):
        rows = self.T * self.nu
        nb_max = min((self.K + 31) // 32 + 1, 148 * 16)
        stride = (16 + nb_max * (rows + 2) * 8 + 255) // 256 * 256 + 2 * 12288 * 8   # ws_bytes: ticket + records + local mailbox
        self._env_ws_stride = (stride + 255) // 256 * 256
        need = self._env_ws_stride * self.N
        if self._workspace is None or self._workspace.numel() < need:
            self._workspace = torch.zeros(need, device=self.d, dtype=torch.uint8)
        p.n_env = self.N
        p.env_u_stride = self._u_stride
        p.env_ws_stride = self._env_ws_stride

    def _pack(self):
        super()._pack()
        # super() sized the workspace for one problem; restore the per-environment slices
        p = self._p
        assert p.workspace == self._workspace.data_ptr() and p.workspace_bytes >= self._env_ws_stride * self.N

    def reset(self):
        """mppi.py:819-820"""
        self.U = self._sample_noise((self.N, self.T))

    def shift_nominal_trajectory(self):
        U = torch.roll(self.U, -1, dims=1)
        U[:, -1] = self._u_init
        self.U = U

    def change_horizon(self, horizon):
        raise NotImplementedError("MPPI_Batched has no change_horizon in the reference either")

    def command_host(self, *a, **k):
        raise NotImplementedError("use command(); N actions are returned as a device tensor")

    def command(self, states, shift_nominal_trajectory=True):
        """mppi.py:822-873: states (N, nx) -> actions (N, nu) (or (N, u_per_command, nu))."""
        if not torch.is_tensor(states):
            states = torch.tensor(states)
        states = states.to(dtype=self.dtype, device=self.d).reshape(self.N, self.nx).contiguous()
        self.state = states
        if self._dirty:
            self._pack()
        N, K, T, nu = self.N, self.K, self.T, self.nu
        action = torch.empty((N, self.u_per_command, nu), device=self.d, dtype=self.dtype)
        stream = torch._C._cuda_getCurrentRawStream(self.d.index)
        flags = self._base_flags | _cabi.FLAG_STATE_DEVICE | (_cabi.FLAG_SHIFT if shift_nominal_trajectory else 0)
        zptr, seed, off = self._noise_source()
        self._cmd_count += 1
        if self._model is not None:
            self._last = (flags, seed, off, zptr, states.data_ptr())
            _cabi.check(self._lib.mppi_plan_command(self._plan, None, states.data_ptr(), flags, seed, off, zptr,
                                                    action.data_ptr(), stream), "mppi_plan_command")
        else:
            self._last = None
            p = self._p
            p.flags = flags & ~_cabi.FLAG_STATE_DEVICE
            p.z, p.seed, p.offset = zptr, seed, off
            p.action_out = action.data_ptr()
            if getattr(self, "_pa_buf", None) is None or self._pa_buf.shape != (N, K, T, nu):
                self._pa_buf = torch.empty(N, K, T, nu, device=self.d, dtype=self.dtype)
                self._noise_buf = torch.empty(N, K, T, nu, device=self.d, dtype=self.dtype)
                self._cost_init = torch.empty(N, K, device=self.d, dtype=self.dtype)
            lib = self._lib
            _cabi.check(lib.mppi_sample_perturb(C.byref(p), self._pa_buf.data_ptr(), self._noise_buf.data_ptr(), None,
                                                self._cost_init.data_ptr(), None, 0, 0, stream), "mppi_sample_perturb")
            NK = N * K
            state = states.unsqueeze(1).expand(N, K, self.nx).reshape(NK, self.nx)                # mppi.py:846
            total = torch.zeros(N, K, device=self.d, dtype=self.dtype)
            dt = _DT[self.dtype]
            for t in range(T):                                                                    # mppi.py:849-853
                u = self._u_scale * self._pa_buf[:, :, t].reshape(NK, nu)
                state = self._dynamics_fn(state, u, t)
                c = self._running_cost_fn(state, u, t).reshape(NK).to(self.dtype).contiguous()
                _cabi.check(lib.mppi_cost_accumulate(total.data_ptr(), c.data_ptr(), None, 1, NK, 1.0, dt, stream),
                            "mppi_cost_accumulate")
            _cabi.check(lib.mppi_cost_accumulate(total.data_ptr(), self._cost_init.data_ptr(), None, 1, NK, 1.0, dt, stream),
                        "mppi_cost_accumulate")
            self._cost_buf = total
            _cabi.check(lib.mppi_softmin_update(C.byref(p), total.data_ptr(), self._noise_buf.data_ptr(), stream),
                        "mppi_softmin_update")
        self.cost_total = self._cost_buf
        return action[:, 0] if self.u_per_command == 1 else action                               # mppi.py:870-873

    # per-environment intermediates are not materialised lazily for the batched controller
    noise = property(lambda self: None)
    perturbed_action = property(lambda self: None)
    states = property(lambda self: None)
    actions = property(lambda self: None)

    @property
    def omega(self):
        if self.cost_total is None:
            return None
        beta = self._stats[:, 0:1].to(self.dtype)
        eta = self._stats[:, 1:2].to(self.dtype)
        return torch.exp(-(1.0 / self._lambda) * (self.cost_total - beta)) / eta


def run_mppi(mppi, env, retrain_dynamics, retrain_after_iter=50, iter=1000, render=True):
    """Closed-loop driver with the reference's signature (mppi.py:876-898): command -> env.step ->
    log (state, action) rows, calling `retrain_dynamics(dataset)` every `retrain_after_iter` steps.
    Host glue only; nothing here is on the measured path."""
    width = mppi.nx + mppi.nu
    dataset = torch.zeros((retrain_after_iter, width), dtype=mppi.dtype, device=mppi.d)
    total_reward = 0
    for step in range(iter):
        obs = env.unwrapped.state.copy()
        t0 = time.perf_counter()
        action = mppi.command(obs)
        dt_cmd = time.perf_counter() - t0
        out = env.step(action.cpu().numpy())
        reward = out[1]
        total_reward += reward
        logger.debug("step %d: cost %.4f, command() %.5fs", step, -reward, dt_cmd)
        if render:
            env.render()
        row = step % retrain_after_iter
        if row == 0 and step > 0:
            retrain_dynamics(dataset)
            dataset.zero_()
        dataset[row, :mppi.nx] = torch.as_tensor(obs, dtype=mppi.dtype)
        dataset[row, mppi.nx:] = action
    return total_reward, dataset
