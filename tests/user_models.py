"""User-written CUDA models used by the tests (built into variant libraries by `__graft_entry__.build()` so the
GPU box does not spend GPU time running nvcc)."""
import torch

import pytorch_mppi_b200 as eng

PEND_STEP = """
    real uc = clamp<real>(u[0], -p[4], p[4]);
    real acc = O::add(O::mul((real)(3 * 10.0 / 2), O::sin_(x[0])), O::mul((real)3.0, uc));
    real thd = clamp<real>(O::add(x[1], O::mul(acc, p[3])), -p[5], p[5]);
    x[0] = O::add(x[0], O::mul(thd, p[3]));
    x[1] = thd;
"""
PEND_COST = """
    const real pi = (real)3.141592653589793, two_pi = (real)(2 * 3.141592653589793);
    real an = O::sub(remainder<real>(O::add(x[0], pi), two_pi), pi);
    return O::add(O::mul(an, an), O::mul(p[6], O::mul(x[1], x[1])));
"""


def pendulum_user_model():
    ref = eng.Pendulum()
    return eng.CudaModel(2, 1, PEND_STEP, PEND_COST, params=[10.0, 1.0, 1.0, 0.05, 2.0, 8.0, 0.1],
                         dynamics=ref.dynamics, running_cost=ref.running_cost)


# a model that exists nowhere else: x = (pos, vel); vel' = vel + dt (u - c vel); pos' = pos + dt vel'
DT_, DRAG, GOAL, WV, WT = 0.1, 0.3, 1.5, 0.05, 4.0
INT_STEP = "real v = O::add(x[1], O::mul(p[0], O::sub(u[0], O::mul(p[1], x[1])))); x[0] = O::add(x[0], O::mul(p[0], v)); x[1] = v;"
INT_COST = "real d = O::sub(x[0], p[2]); return O::add(O::mul(d, d), O::mul(p[3], O::mul(x[1], x[1])));"
INT_TERM = "real d = O::sub(x[0], p[2]); return O::mul(p[4], O::mul(d, d));"


def int_dyn(s, a):
    v = s[:, 1] + DT_ * (a[:, 0] - DRAG * s[:, 1])
    return torch.stack((s[:, 0] + DT_ * v, v), dim=1)


def int_cost(s, a):
    return (s[:, 0] - GOAL) ** 2 + WV * s[:, 1] ** 2


def int_term(states, actions):
    return WT * (states[..., -1, 0] - GOAL) ** 2


def integrator_user_model():
    return eng.CudaModel(2, 1, INT_STEP, INT_COST, params=[DT_, DRAG, GOAL, WV, WT], terminal_code=INT_TERM,
                         dynamics=int_dyn, running_cost=int_cost, terminal_cost=int_term)


# ---- wide models: every control moves several states, every state enters the cost ---------------------------------
# ARM4: nx = 8, nu = 4.  Four damped joints q (x[0..3]) with velocities qd (x[4..7]); the torques reach the joints
# through a dense 4 x 4 mixing matrix:  qd' = qd + dt (B u - c qd - k sin q),  q' = q + dt qd'.
# cost = sum_i wq_i (q_i - g_i)^2 + wv_i qd_i^2 + r |u|^2
ARM_DT, ARM_C, ARM_K, ARM_R = 0.05, 0.4, 2.0, 0.01
ARM_B = [[1.0, 0.3, -0.2, 0.1], [0.25, 0.9, 0.3, -0.15], [-0.1, 0.35, 1.1, 0.2], [0.2, -0.25, 0.15, 0.8]]
ARM_G = [0.5, -0.3, 0.8, -0.6]
ARM_WQ = [1.0, 0.7, 1.3, 0.9]
ARM_WV = [0.05, 0.08, 0.03, 0.06]
ARM_PARAMS = [ARM_DT, ARM_C, ARM_K] + [v for row in ARM_B for v in row] + ARM_G + ARM_WQ + ARM_WV + [ARM_R]   # 32
ARM_STEP = """
    real qd[4];
    for (int i = 0; i < 4; ++i) {
        real acc = O::add(O::mul(p[1], x[4 + i]), O::mul(p[2], O::sin_(x[i])));
        real bu = O::mul(p[3 + 4 * i], u[0]);
        for (int j = 1; j < 4; ++j) bu = O::add(bu, O::mul(p[3 + 4 * i + j], u[j]));
        qd[i] = O::add(x[4 + i], O::mul(p[0], O::sub(bu, acc)));
    }
    for (int i = 0; i < 4; ++i) {
        x[i] = O::add(x[i], O::mul(p[0], qd[i]));
        x[4 + i] = qd[i];
    }
"""
ARM_COST = """
    real c = (real)0;
    for (int i = 0; i < 4; ++i) {
        real d = O::sub(x[i], p[19 + i]);
        c = O::add(c, O::add(O::mul(p[23 + i], O::mul(d, d)), O::mul(p[27 + i], O::mul(x[4 + i], x[4 + i]))));
    }
    real uu = (real)0;
    for (int j = 0; j < 4; ++j) uu = O::add(uu, O::mul(u[j], u[j]));
    return O::add(c, O::mul(p[31], uu));
"""


def _consts(like, *vals):
    return [torch.tensor(v, dtype=like.dtype, device=like.device) for v in vals]


def arm_dyn(s, a):
    B, = _consts(s, ARM_B)
    q, qd = s[:, :4], s[:, 4:]
    acc = ARM_C * qd + ARM_K * torch.sin(q)
    qd = qd + ARM_DT * (a @ B.T - acc)
    return torch.cat((q + ARM_DT * qd, qd), dim=1)


def arm_cost(s, a):
    g, wq, wv = _consts(s, ARM_G, ARM_WQ, ARM_WV)
    return ((s[:, :4] - g) ** 2 * wq).sum(1) + (s[:, 4:] ** 2 * wv).sum(1) + ARM_R * (a ** 2).sum(1)


def arm4_user_model():
    return eng.CudaModel(8, 4, ARM_STEP, ARM_COST, params=ARM_PARAMS, dynamics=arm_dyn, running_cost=arm_cost)


# LIN6: nx = 6, nu = 3, a discrete linear system x' = A x + B u with dense A (6 x 6) and B (6 x 3), quadratic running and
# terminal costs.  68 parameters: everything from B's last row on arrives through `model_params_ext`.
def _lin6_mats():
    g = torch.Generator().manual_seed(61)
    A = torch.eye(6, dtype=torch.float64) + 0.06 * torch.randn(6, 6, generator=g, dtype=torch.float64)
    B = 0.1 * torch.randn(6, 3, generator=g, dtype=torch.float64) + 0.05
    return A.tolist(), B.tolist()


LIN6_A, LIN6_B = _lin6_mats()
LIN6_G = [1.0, -0.5, 0.25, 0.75, -1.0, 0.5]
LIN6_W = [1.0, 0.5, 2.0, 0.8, 1.5, 0.3]
LIN6_R, LIN6_WT = 0.02, 3.0
LIN6_PARAMS = [v for row in LIN6_A for v in row] + [v for row in LIN6_B for v in row] + LIN6_G + LIN6_W + [LIN6_R, LIN6_WT]
LIN6_STEP = """
    real y[6];
    for (int i = 0; i < 6; ++i) {
        real s = O::mul(p[6 * i], x[0]);
        for (int j = 1; j < 6; ++j) s = O::add(s, O::mul(p[6 * i + j], x[j]));
        for (int j = 0; j < 3; ++j) s = O::add(s, O::mul(p[36 + 3 * i + j], u[j]));
        y[i] = s;
    }
    for (int i = 0; i < 6; ++i) x[i] = y[i];
"""
LIN6_COST = """
    real c = (real)0;
    for (int i = 0; i < 6; ++i) {
        real d = O::sub(x[i], p[54 + i]);
        c = O::add(c, O::mul(p[60 + i], O::mul(d, d)));
    }
    real uu = (real)0;
    for (int j = 0; j < 3; ++j) uu = O::add(uu, O::mul(u[j], u[j]));
    return O::add(c, O::mul(p[66], uu));
"""
LIN6_TERM = """
    real c = (real)0;
    for (int i = 0; i < 6; ++i) {
        real d = O::sub(x[i], p[54 + i]);
        c = O::add(c, O::mul(d, d));
    }
    return O::mul(p[67], c);
"""
assert len(LIN6_PARAMS) == 68


def lin6_dyn(s, a):
    A, B = _consts(s, LIN6_A, LIN6_B)
    return s @ A.T + a @ B.T


def lin6_cost(s, a):
    g, w = _consts(s, LIN6_G, LIN6_W)
    return ((s - g) ** 2 * w).sum(1) + LIN6_R * (a ** 2).sum(1)


def lin6_term(states, actions):
    g, = _consts(states, LIN6_G)
    return LIN6_WT * ((states[..., -1, :] - g) ** 2).sum(-1)


def lin6_user_model(terminal=True):
    """(MPPI_Batched takes no terminal cost: `terminal=False` is the same model without it.)"""
    return eng.CudaModel(6, 3, LIN6_STEP, LIN6_COST, params=LIN6_PARAMS, terminal_code=LIN6_TERM if terminal else None,
                         dynamics=lin6_dyn, running_cost=lin6_cost, terminal_cost=lin6_term if terminal else None)


# ---- infeasible samples: x = (pos, vel, flag, steps taken); the running cost is +inf while the flag is set ------------
# The flag is part of the start state (per-sample start states choose the infeasible samples), or is raised by the first
# action when that exceeds the threshold p[2] (+inf: never) — MPPI_Batched has one start state per environment.
FLAG_DT, FLAG_DRAG, FLAG_GOAL, FLAG_WV = 0.1, 0.3, 1.0, 0.05
FLAG_STEP = """
    real v = O::add(x[1], O::mul(p[0], O::sub(u[0], O::mul(p[1], x[1]))));
    x[0] = O::add(x[0], O::mul(p[0], v));
    x[1] = v;
    if (x[3] == (real)0 && u[0] > p[2]) x[2] = (real)1;
    x[3] = O::add(x[3], (real)1);
"""
FLAG_COST = """
    if (x[2] > (real)0.5) return O::inf();
    real d = O::sub(x[0], p[3]);
    return O::add(O::mul(d, d), O::mul(p[4], O::mul(x[1], x[1])));
"""


def flag_dyn_for(threshold):
    def dyn(s, a):
        v = s[:, 1] + FLAG_DT * (a[:, 0] - FLAG_DRAG * s[:, 1])
        raise_ = (s[:, 3] == 0) & (a[:, 0] > threshold)
        flag = torch.where(raise_, torch.ones_like(s[:, 2]), s[:, 2])
        return torch.stack((s[:, 0] + FLAG_DT * v, v, flag, s[:, 3] + 1), dim=1)
    return dyn


def flag_cost(s, a):
    d = s[:, 0] - FLAG_GOAL
    c = d * d + FLAG_WV * (s[:, 1] * s[:, 1])
    return torch.where(s[:, 2] > 0.5, torch.full_like(c, float("inf")), c)


def flag_user_model(threshold=float("inf")):
    return eng.CudaModel(4, 1, FLAG_STEP, FLAG_COST, params=[FLAG_DT, FLAG_DRAG, threshold, FLAG_GOAL, FLAG_WV],
                         dynamics=flag_dyn_for(threshold), running_cost=flag_cost)


# every (model, dtype, variant) the tests load: `__graft_entry__.build()` compiles these ahead of the GPU run
def precompiled():
    out = [(pendulum_user_model, torch.float32, 0), (integrator_user_model, torch.float64, 0)]
    for make in (arm4_user_model, lin6_user_model, flag_user_model):
        for dtype in (torch.float32, torch.float64):
            for variant in (0, 1, 2):
                out.append((make, dtype, variant))
    for dtype in (torch.float32, torch.float64):
        out.append((lambda: lin6_user_model(terminal=False), dtype, 0))
    return out
