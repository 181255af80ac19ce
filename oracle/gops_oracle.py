"""CPU oracle for the GOPS batched model-rollout + ADP-update hot path.

TEST INFRASTRUCTURE -- NOT THE PRODUCT.  Only `tests/`, `__graft_entry__.smoke()` and the
`cpu_baseline` / `--impl reference` legs of `bench.py` may import this module.  The product
(`gops_b200/`) never imports it and has no CPU fallback.

What it is: a compact, functional PyTorch-fp32 (optionally fp64) restatement of the reference's
algorithm for this path, written op-for-op in the reference's vectorised style so that (a) results
agree with the reference to fp32 round-off and (b) its CPU timing is representative of the
reference's own CPU path.  Gradients come from torch autograd exactly as in the reference.

Parity pin: `oracle/make_golden.py` runs the UNMODIFIED reference (through `oracle/ref_shim.py`)
in the build container and stores inputs / losses / gradients / post-Adam weights under
`tests/golden/`; `tests/test_oracle_vs_golden.py` and `tests/test_oracle_vs_reference.py` check
this file against those vectors.  Reference file:line citations are given per function (paths relative to the GOPS tree).
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.nn.functional as F

Tensor = torch.Tensor

# --------------------------------------------------------------------------------------
# MLP apprfuncs            gops/apprfunc/mlp.py:36-41 (mlp), :50-77 (DetermPolicy),
#                          :80-111 (FiniteHorizonPolicy), :309-329 (StateValue)
#                          gops/utils/common_utils.py:26-55 (activation table)
# --------------------------------------------------------------------------------------
_ACTS = {
    "relu": F.relu,
    "elu": F.elu,                      # alpha = 1
    "gelu": F.gelu,                    # exact erf form (nn.GELU default)
    "selu": F.selu,
    "sigmoid": torch.sigmoid,
    "tanh": torch.tanh,
    "linear": lambda x: x,
}


def mlp_forward(layers: Sequence[Tuple[Tensor, Tensor]], x: Tensor, hidden_act: str,
                out_act: str = "linear") -> Tensor:
    """nn.Sequential(Linear, act, ..., Linear, out_act); W is torch layout [out, in]."""
    n = len(layers)
    for j, (w, b) in enumerate(layers):
        x = torch.addmm(b, x, w.t())
        x = _ACTS[hidden_act if j < n - 1 else out_act](x)
    return x


def policy_forward(layers, obs: Tensor, act_high: Tensor, act_low: Tensor, hidden_act: str,
                   out_act: str = "linear", virtual_t: Optional[float] = None) -> Tensor:
    """DetermPolicy.forward (mlp.py:73-77) when virtual_t is None, FiniteHorizonPolicy.forward
    (mlp.py:103-111) otherwise (the time feature is appended as the last input column)."""
    if virtual_t is not None:
        tcol = virtual_t * torch.ones((obs.shape[0], 1), dtype=obs.dtype)
        obs = torch.cat((obs, tcol), 1)
    z = mlp_forward(layers, obs, hidden_act, out_act)
    return (act_high - act_low) / 2 * torch.tanh(z) + (act_high + act_low) / 2


def value_forward(layers, obs: Tensor, hidden_act: str, out_act: str = "linear") -> Tensor:
    """StateValue.forward (mlp.py:327-329)."""
    return torch.squeeze(mlp_forward(layers, obs, hidden_act, out_act), -1)


def init_mlp(sizes: Sequence[int], gen: torch.Generator, dtype=torch.float32):
    """torch.nn.Linear default init (kaiming-uniform a=sqrt(5) == U(-1/sqrt(in), 1/sqrt(in)))."""
    layers = []
    for i, o in zip(sizes[:-1], sizes[1:]):
        bound = 1.0 / math.sqrt(i)
        w = (torch.rand(o, i, generator=gen, dtype=torch.float64) * 2 - 1) * bound
        b = (torch.rand(o, generator=gen, dtype=torch.float64) * 2 - 1) * bound
        layers.append((w.to(dtype), b.to(dtype)))
    return layers


def angle_normalize(x):
    """gops/utils/math_utils.py:8-11 (python % == torch.remainder semantics)."""
    return ((x + math.pi) % (2 * math.pi)) - math.pi


# --------------------------------------------------------------------------------------
# Base dynamics models
# --------------------------------------------------------------------------------------
class BaseModel:
    obs_dim: int
    action_dim: int
    dt: float

    def _bounds(self, obs_lo=None, obs_hi=None, act_lo=None, act_hi=None, dtype=torch.float32):
        # gops/env/env_ocp/env_model/pyth_base_model.py:21-57
        inf = float("inf")
        self.obs_lower_bound = torch.tensor(obs_lo if obs_lo is not None else [-inf] * self.obs_dim, dtype=dtype)
        self.obs_upper_bound = torch.tensor(obs_hi if obs_hi is not None else [inf] * self.obs_dim, dtype=dtype)
        self.action_lower_bound = torch.tensor(act_lo if act_lo is not None else [-inf] * self.action_dim, dtype=dtype)
        self.action_upper_bound = torch.tensor(act_hi if act_hi is not None else [inf] * self.action_dim, dtype=dtype)

    def step(self, obs, action, done, info):
        raise NotImplementedError


class IdPendulumModel(BaseModel):
    """gops/env/env_ocp/env_model/pyth_idpendulum_model.py: Dynamics.f_xu :31-124,
    compute_rewards :126-149, get_done :151-172, PythInvertedpendulum.forward :199-216."""

    def __init__(self, dtype=torch.float32, **_):
        self.obs_dim, self.action_dim, self.dt, self.discrete_num = 6, 1, 0.01, 5
        self._bounds(act_lo=[-1.0], act_hi=[1.0], dtype=dtype)
        self.m, self.m1, self.m2 = 9.42477796, 4.1033127, 4.1033127
        self.l1, self.l2, self.g = 0.6, 0.6, 9.81

    def f_xu(self, s, u, tau):
        m, m1, m2, l1, l2, g = self.m, self.m1, self.m2, self.l1, self.l2, self.g
        th1, th2, pd, th1d, th2d = s[:, 1], s[:, 2], s[:, 3], s[:, 4], s[:, 5]
        u = u[:, 0]
        ones = torch.ones_like(th1)
        M = torch.stack([
            (m + m1 + m2) * ones,
            l1 * (0.5 * m1 + m2) * torch.cos(th1),
            0.5 * m2 * l2 * torch.cos(th2),
            l1 * (0.5 * m1 + m2) * torch.cos(th1),
            l1 * l1 * (0.3333 * m1 + m2) * ones,
            0.5 * l1 * l2 * m2 * torch.cos(th1 - th2),
            0.5 * l2 * m2 * torch.cos(th2),
            0.5 * l1 * l2 * m2 * torch.cos(th1 - th2),
            0.3333 * l2 * l2 * m2 * ones,
        ], dim=1).reshape(-1, 3, 3)
        f = torch.stack([
            l1 * (0.5 * m1 + m2) * torch.square(th1d) * torch.sin(th1)
            + 0.5 * m2 * l2 * torch.square(th2d) * torch.sin(th2) - 0.0 * pd + u,
            -0.5 * l1 * l2 * m2 * torch.square(th2d) * torch.sin(th1 - th2)
            + g * (0.5 * m1 + m2) * l1 * torch.sin(th1) - 0.0 * th1d,
            0.5 * l1 * l2 * m2 * torch.square(th1d) * torch.sin(th1 - th2)
            + g * 0.5 * l2 * m2 * torch.sin(th2),
        ], dim=1).reshape(-1, 3, 1)
        acc = torch.matmul(torch.linalg.inv(M), f).squeeze(-1)
        return s + tau * torch.cat([s[:, 3:], acc], dim=-1)

    def step(self, obs, action, done, info):
        for _ in range(self.discrete_num):
            obs = self.f_xu(obs, 500 * action, self.dt / self.discrete_num)
        a = action.squeeze(-1)
        th1, th2, pd, th1d, th2d = obs[:, 1], obs[:, 2], obs[:, 3], obs[:, 4], obs[:, 5]
        dist = 0 * torch.square(obs[:, 0]) + 5 * torch.square(th1) + 10 * torch.square(th2)
        vel = 0.5 * torch.square(pd) + 0.5 * torch.square(th1d) + 1 * torch.square(th2d)
        reward = 10 - dist - vel - 1 * torch.square(a)
        tip_y = self.l1 * torch.cos(th1) + self.l2 * torch.cos(th2)
        isdone = torch.logical_or(tip_y <= 1.0, torch.abs(obs[:, 0]) >= 15)
        return obs, reward, isdone, {"constraint": None}


LQ_CONFIGS: Dict[str, dict] = {
    # gops/env/env_ocp/resources/lq_configs.py:15-116 (numerical data)
    "s2a1": dict(A=[[0.0, 1.0], [0.0, 0.0]], B=[[0.0], [1.0]], Q=[2, 1], R=[1.0], dt=0.05,
                 init_mean=[0.0, 0.0], init_std=[1.0, 1.0], state_high=[20.0, 20.0], state_low=[-20.0, -20.0],
                 action_high=[5.0], action_low=[-5.0], max_step=200, reward_scale=1, reward_shift=0),
    "s3a1": dict(A=[[-1.01887, 0.90506, -0.00215], [0.82225, -1.07741, -0.17555], [0.0, 0.0, -1.0]],
                 B=[[0.0], [0.0], [5.0]], Q=[50.0, 1, 1], R=[1.0], dt=0.1, init_mean=[0, 0, 0],
                 init_std=[2, 2, 2], state_high=[20, 20, 20], state_low=[-20, -20, -20],
                 action_high=[5.0], action_low=[-5.0], max_step=200, reward_scale=1.0, reward_shift=0),
    "s4a2": dict(A=[[0, 1, 0, 0], [0, 1, 0, 0], [0.1, -0.2, 0, 0.5], [-0.2, 0.1, 0.1, 0]],
                 B=[[0, 0], [-2, -1], [0.0, 0], [1, 1.5]], Q=[1, 2, 2, 1], R=[1.0, 1.0], dt=0.1,
                 init_mean=[0, 0, 0, 0], init_std=[0.7, 0.3, 0.7, 0.3], state_high=[15] * 4,
                 state_low=[-15] * 4, action_high=[8.0, 8.0], action_low=[-8.0, -8.0], max_step=200,
                 reward_scale=1, reward_shift=0),
}


class LqModel(BaseModel):
    """gops/env/env_ocp/resources/lq_base.py: LQDynamics ctor :36-59, prediction :89-108,
    compute_reward :110-141, LqModel.forward :343-354; creator pyth_lq_model.py:18-34."""

    def __init__(self, lq_config="s3a1", dtype=torch.float32, **_):
        cfg = LQ_CONFIGS[lq_config] if isinstance(lq_config, str) else lq_config
        self.cfg = cfg
        self.A = torch.as_tensor(cfg["A"], dtype=torch.float32)
        self.B = torch.as_tensor(cfg["B"], dtype=torch.float32)
        self.Q = torch.as_tensor(cfg["Q"], dtype=torch.float32)
        self.R = torch.as_tensor(cfg["R"], dtype=torch.float32)
        self.dt = cfg["dt"]
        self.obs_dim, self.action_dim = self.A.shape[0], self.B.shape[1]
        IA = torch.eye(self.obs_dim) - self.A * self.dt
        self.inv_IA = torch.linalg.pinv(IA)          # fp32 pinv, as the reference
        self.reward_scale, self.reward_shift = cfg["reward_scale"], cfg["reward_shift"]
        self._bounds(cfg["state_low"], cfg["state_high"], cfg["action_low"], cfg["action_high"], dtype)
        if dtype != torch.float32:
            for k in ("A", "B", "Q", "R", "inv_IA"):
                setattr(self, k, getattr(self, k).to(dtype))

    def step(self, obs, action, done, info):
        tmp = torch.mm(self.B, action.T) * self.dt + obs.T
        nxt = torch.mm(self.inv_IA, tmp).T
        rs = torch.sum(torch.pow(obs, 2) * self.Q, dim=-1)
        ra = torch.sum(torch.pow(action, 2) * self.R, dim=-1)
        reward = self.reward_scale * (self.reward_shift - 1.0 * (rs + ra))
        isdone = torch.full([obs.shape[0]], False, dtype=torch.bool)
        return nxt, reward.reshape(-1), isdone, {"constraint": None}


# ---- analytic reference trajectories ------------------------------------------------
@dataclass
class RefTraj:
    """gops/env/env_ocp/resources/ref_traj_model.py:27-232, defaults ref_traj_data.py:19-37.
    path_num: 0 sine, 1 double_lane, 2 triangle, 3 circle;  speed_num: 0 sine, 1 constant."""
    sine_A: float = 1.5
    sine_omega: float = 2 * np.pi / 10
    sine_phi: float = 0.0
    dl_t: Tuple[float, float, float, float] = (5.0, 9.0, 14.0, 18.0)
    dl_y: Tuple[float, float] = (0.0, 3.5)
    tri_A: float = 3.0
    tri_T: float = 10.0
    circ_r: float = 100.0
    sp_A: float = 1.0
    sp_omega: float = 2 * np.pi / 10
    sp_phi: float = 0.0
    sp_b: float = 5.0
    sp_const: float = 5.0

    def _int_u(self, t, speed_num):
        sine = (-self.sp_A / self.sp_omega * torch.cos(self.sp_omega * t + self.sp_phi)
                + self.sp_b * t + self.sp_A / self.sp_omega * np.cos(self.sp_phi))
        const = self.sp_const * t
        return torch.zeros_like(t) + (speed_num == 0) * sine + (speed_num == 1) * const

    def _u(self, t, speed_num):
        sine = self.sp_A * torch.sin(self.sp_omega * t + self.sp_phi) + self.sp_b
        const = self.sp_const * torch.ones_like(t)
        return torch.zeros_like(t) + (speed_num == 0) * sine + (speed_num == 1) * const

    def _path_x(self, i, t, sp):
        if i == 3:
            return self.circ_r * torch.sin(self._int_u(t, sp) / self.circ_r)
        return self._int_u(t, sp)

    def _path_y(self, i, t, sp):
        if i == 0:
            return self.sine_A * torch.sin(self.sine_omega * t + self.sine_phi)
        if i == 1:
            t1, t2, t3, t4 = self.dl_t
            y1, y2 = self.dl_y
            ya = (y2 - y1) / (t2 - t1) * (t - t1) + y1
            yb = (y1 - y2) / (t4 - t3) * (t - t3) + y2
            return (y1 * (t <= t1) + ya * ((t > t1) & (t <= t2)) + y2 * ((t > t2) & (t <= t3))
                    + yb * ((t > t3) & (t <= t4)) + y1 * (t > t4))
        if i == 2:
            s = torch.remainder(t, self.tri_T)
            ya = 2 * self.tri_A / self.tri_T * s
            yb = -2 * self.tri_A / self.tri_T * (s - self.tri_T)
            return ya * (s <= self.tri_T / 2) + yb * ((s > self.tri_T / 2) & (s < self.tri_T))
        return self.circ_r * (torch.cos(self._int_u(t, sp) / self.circ_r) - 1)

    def _path_phi(self, i, t, sp):
        dt = 0.001
        dx = self._path_x(i, t + dt, sp) - self._path_x(i, t, sp)
        dy = self._path_y(i, t + dt, sp) - self._path_y(i, t, sp)
        return torch.atan2(dy, dx)

    def _select(self, fn, t, path_num, sp):
        out = torch.zeros_like(t)
        for i in range(4):
            out = out + (path_num == i) * fn(i, t, sp)
        return out

    def x(self, t, p, s):
        return self._select(self._path_x, t, p, s)

    def y(self, t, p, s):
        return self._select(self._path_y, t, p, s)

    def phi(self, t, p, s):
        return self._select(self._path_phi, t, p, s)

    def u(self, t, p, s):
        return self._select(lambda i, tt, ss: self._u(tt, ss), t, p, s)


VEH = dict(k_f=-128915.5, k_r=-85943.6, l_f=1.06, l_r=1.85, m=1412.0, I_z=1536.7)


def veh3dof_next_state(state, action, dt, normalize_phi=True):
    """VehicleDynamicsModel.f_xu, pyth_veh3dofconti_model.py:24-61 (params pyth_veh3dofconti.py:24-33);
    identical physics in env_gen_ocp/robot/veh3dof_model.py:24-58."""
    x, y, phi, u, v, w = (state[:, i] for i in range(6))
    steer, a_x = action[:, 0], action[:, 1]
    k_f, k_r, l_f, l_r, m, I_z = (VEH[k] for k in ("k_f", "k_r", "l_f", "l_r", "m", "I_z"))
    nxt = [
        x + dt * (u * torch.cos(phi) - v * torch.sin(phi)),
        y + dt * (u * torch.sin(phi) + v * torch.cos(phi)),
        phi + dt * w,
        u + dt * a_x,
        (m * v * u + dt * (l_f * k_f - l_r * k_r) * w - dt * k_f * steer * u - dt * m * torch.square(u) * w)
        / (m * u - dt * (k_f + k_r)),
        (I_z * w * u + dt * (l_f * k_f - l_r * k_r) * v - dt * l_f * k_f * steer * u)
        / (I_z * u - dt * (l_f ** 2 * k_f + l_r ** 2 * k_r)),
    ]
    nxt[2] = angle_normalize(nxt[2])
    return torch.stack(nxt, 1)


def ego_transform(ego_x, ego_y, ego_phi, rx, ry, rphi):
    """ego_vehicle_coordinate_transform, pyth_veh3dofconti_model.py:189-203."""
    ego_x, ego_y, ego_phi = ego_x.unsqueeze(1), ego_y.unsqueeze(1), ego_phi.unsqueeze(1)
    c, s = torch.cos(-ego_phi), torch.sin(-ego_phi)
    return ((rx - ego_x) * c - (ry - ego_y) * s, (rx - ego_x) * s + (ry - ego_y) * c,
            angle_normalize(rphi - ego_phi))


def veh_obs(state, ref_points):
    """Veh3dofcontiModel.get_obs :147-159 (same layout in veh3dof_tracking_model.py:37-57)."""
    rx, ry, rphi = ego_transform(state[:, 0], state[:, 1], state[:, 2],
                                 ref_points[..., 0], ref_points[..., 1], ref_points[..., 2])
    ru = ref_points[..., 3] - state[:, 3].unsqueeze(1)
    ego = torch.cat((torch.stack((rx[:, 0], ry[:, 0], rphi[:, 0], ru[:, 0]), dim=1), state[:, 4:]), dim=1)
    ref = torch.stack((rx, ry, rphi, ru), 2)[:, 1:].reshape(ego.shape[0], -1)
    return torch.cat((ego, ref), 1)


class Veh3dofContiModel(BaseModel):
    """pyth_veh3dofconti_model.py: Veh3dofcontiModel.forward :91-145, compute_reward :161-177,
    judge_done :179-186."""

    def __init__(self, pre_horizon=10, max_steer=np.pi / 6, dtype=torch.float32, **_):
        self.pre_horizon = pre_horizon
        self.obs_dim, self.action_dim, self.dt = 6 + 4 * pre_horizon, 2, 0.1
        self._bounds(act_lo=[-max_steer, -3], act_hi=[max_steer, 3], dtype=dtype)
        self.ref = RefTraj()

    def step(self, obs, action, done, info):
        state, ref_points = info["state"], info["ref_points"]
        path_num, u_num, t = info["path_num"], info["u_num"], info["ref_time"]
        dx, dy, dphi, du, w = obs[:, 0], obs[:, 1], obs[:, 2], obs[:, 3], obs[:, 5]
        steer, a_x = action[:, 0], action[:, 1]
        reward = -(0.04 * dx ** 2 + 0.04 * dy ** 2 + 0.02 * dphi ** 2 + 0.02 * du ** 2
                   + 0.01 * w ** 2 + 0.01 * steer ** 2 + 0.01 * a_x ** 2)
        nstate = veh3dof_next_state(state, action, self.dt)
        nt = t + self.dt
        tq = nt + self.pre_horizon * self.dt
        nref = ref_points.clone()
        nref[:, :-1] = ref_points[:, 1:]
        nref[:, -1] = torch.stack((self.ref.x(tq, path_num, u_num), self.ref.y(tq, path_num, u_num),
                                   self.ref.phi(tq, path_num, u_num), self.ref.u(tq, path_num, u_num)), dim=1)
        nobs = veh_obs(nstate, nref)
        isdone = (torch.abs(nobs[:, 0]) > 10) | (torch.abs(nobs[:, 1]) > 10) | (torch.abs(nobs[:, 2]) > np.pi)
        ninfo = {"state": nstate, "ref_points": nref, "path_num": path_num, "u_num": u_num, "ref_time": nt}
        return nobs, reward, isdone, ninfo


class Veh3dofContiErrCstrModel(Veh3dofContiModel):
    """pyth_veh3dofconti_errcstr_model.py:19-55: the same model, plus info["constraint"] =
    (|y_err| - y_error_tol, |u_err| - u_error_tol) of the INCOMING observation."""

    def __init__(self, pre_horizon=10, y_error_tol=0.2, u_error_tol=2.0, **kw):
        super().__init__(pre_horizon=pre_horizon, **kw)
        self.y_error_tol, self.u_error_tol = y_error_tol, u_error_tol

    def step(self, obs, action, done, info):
        nobs, reward, isdone, ninfo = super().step(obs, action, done, info)
        ninfo["constraint"] = torch.stack((obs[:, 1].abs() - self.y_error_tol, obs[:, 3].abs() - self.u_error_tol), dim=1)
        return nobs, reward, isdone, ninfo


class Veh3dofTrackingModel(BaseModel):
    """env_gen_ocp/env_model/veh3dof_tracking_model.py:11-102 via EnvModel.forward
    env_gen_ocp/env_model/pyth_base_model.py:109-119.  info = {"state": (robot_state[B,6],
    reference[B,2P+1,4], t:int)} (a plain tuple stands in for State/ContextState)."""

    def __init__(self, pre_horizon=10, max_acc=3.0, max_steer=math.pi / 6, dtype=torch.float32, **_):
        self.pre_horizon = pre_horizon
        self.obs_dim, self.action_dim, self.dt = 6 + 4 * pre_horizon, 2, 0.1
        self._bounds(act_lo=[-max_steer, -max_acc], act_hi=[max_steer, max_acc], dtype=dtype)

    def get_obs(self, robot, reference, t):
        return veh_obs(robot, reference[:, t:t + self.pre_horizon + 1])

    def step(self, obs, action, done, info):
        robot, reference, t = info["state"]
        nrobot = veh3dof_next_state(robot, action, self.dt)
        nobs = self.get_obs(nrobot, reference, t + 1)
        r = reference[:, t]
        steer, a_x = action[:, 0], action[:, 1]
        reward = -(0.04 * (robot[:, 0] - r[:, 0]) ** 2 + 0.04 * (robot[:, 1] - r[:, 1]) ** 2
                   + 0.02 * angle_normalize(robot[:, 2] - r[:, 2]) ** 2 + 0.02 * (robot[:, 3] - r[:, 3]) ** 2
                   + 0.01 * robot[:, 5] ** 2 + 0.01 * steer ** 2 + 0.01 * a_x ** 2)
        rn = reference[:, t + 1]
        isdone = ((torch.abs(nrobot[:, 0] - rn[:, 0]) > 5) | (torch.abs(nrobot[:, 1] - rn[:, 1]) > 2)
                  | (torch.abs(angle_normalize(nrobot[:, 2] - rn[:, 2])) > math.pi))
        return nobs, reward, isdone, {"state": (nrobot, reference, t + 1)}


class Veh3dofTrackingDetourModel(BaseModel):
    """env_gen_ocp/env_model/veh3dof_tracking_detour_model.py:13-176 via EnvModel.forward
    env_gen_ocp/env_model/pyth_base_model.py:109-119: veh3dof_tracking plus ONE surrounding vehicle -- its ego-frame
    pose (and raw speed) as four more observation entries (:62-76), the bicircle collision constraint 2 r - min dist of
    the INCOMING state (:78-131, pyth_base_model.py:117-118), other reward weights / offset (:133-150) and a wider lateral
    termination bound (:152-163).  info = {"state": (robot[B,6], reference[B,L,4], t:int, surr[B,P+1,n,5])}."""

    def __init__(self, pre_horizon=10, max_steer=math.pi / 6, veh_length=4.8, veh_width=2.0, dtype=torch.float32, **_):
        self.pre_horizon = pre_horizon
        self.obs_dim, self.action_dim, self.dt = 6 + 4 * pre_horizon + 4, 2, 0.1
        self.veh_length, self.veh_width = veh_length, veh_width
        self._bounds(act_lo=[-max_steer, -3], act_hi=[max_steer, 3], dtype=dtype)

    def get_obs(self, robot, reference, t, surr):
        base = veh_obs(robot, reference[:, t:t + self.pre_horizon + 1])
        c = surr[:, t]
        sx, sy, sphi = ego_transform(robot[:, 0], robot[:, 1], robot[:, 2], c[..., 0], c[..., 1], c[..., 2])
        so = torch.stack((sx, sy, sphi, c[..., 3]), 2).reshape(base.shape[0], -1)
        return torch.cat((base, so), 1)

    y_done, radius_factor = 3, 0.5

    def reward(self, robot, r, steer, a_x):
        return -0.01 * (10.0 * (robot[:, 0] - r[:, 0]) ** 2 + 10.0 * (robot[:, 1] - r[:, 1]) ** 2
                        + 500 * angle_normalize(robot[:, 2] - r[:, 2]) ** 2 + 5.0 * (robot[:, 3] - r[:, 3]) ** 2
                        + 1000 * robot[:, 5] ** 2 + 1000 * steer ** 2 + 50 * a_x ** 2) + 2.0

    def get_constraint(self, robot, surr_t):
        d, r = (self.veh_length - self.veh_width) / 2, self.radius_factor * self.veh_width
        x, y, phi = robot[:, 0:1], robot[:, 1:2], robot[:, 2:3]
        ego = [torch.cat((x + s * d * torch.cos(phi), y + s * d * torch.sin(phi)), 1) for s in (1.0, -1.0)]
        sx, sy, sphi = surr_t[..., 0], surr_t[..., 1], surr_t[..., 2]
        sur = [torch.stack((sx + s * d * torch.cos(sphi), sy + s * d * torch.sin(sphi)), 2) for s in (1.0, -1.0)]
        min_dist = torch.full_like(x, float(np.finfo(np.float32).max))
        for e in ego:
            for q in sur:
                dist = torch.linalg.norm(e.unsqueeze(1) - q, dim=2)
                min_dist = torch.minimum(min_dist, dist.min(dim=1, keepdim=True).values)
        return 2 * r - min_dist

    def step(self, obs, action, done, info):
        robot, reference, t, surr = info["state"]
        nrobot = veh3dof_next_state(robot, action, self.dt)
        nobs = self.get_obs(nrobot, reference, t + 1, surr)
        r = reference[:, t]
        steer, a_x = action[:, 0], action[:, 1]
        reward = self.reward(robot, r, steer, a_x)
        rn = reference[:, t + 1]
        isdone = ((torch.abs(nrobot[:, 0] - rn[:, 0]) > 5) | (torch.abs(nrobot[:, 1] - rn[:, 1]) > self.y_done)
                  | (torch.abs(angle_normalize(nrobot[:, 2] - rn[:, 2])) > math.pi))
        return nobs, reward, isdone, {"state": (nrobot, reference, t + 1, surr),
                                      "constraint": self.get_constraint(robot, surr[:, t])}


class Veh3dofTrackingSurrCstrModel(Veh3dofTrackingDetourModel):
    """env_gen_ocp/env_model/veh3dof_tracking_surrcstr_model.py:13-181: the detour model's structure with the tracking
    model's reward (:138-158) and lateral bound (:160-171) and circle radius sqrt(2)/2 * veh_width (:88)."""
    y_done, radius_factor = 2, math.sqrt(2) / 2

    def reward(self, robot, r, steer, a_x):
        return -(0.04 * (robot[:, 0] - r[:, 0]) ** 2 + 0.04 * (robot[:, 1] - r[:, 1]) ** 2
                 + 0.02 * angle_normalize(robot[:, 2] - r[:, 2]) ** 2 + 0.02 * (robot[:, 3] - r[:, 3]) ** 2
                 + 0.01 * robot[:, 5] ** 2 + 0.01 * steer ** 2 + 0.01 * a_x ** 2)


MODEL_REGISTRY = {
    "pyth_idpendulum": IdPendulumModel,
    "pyth_lq": LqModel,
    "pyth_veh3dofconti": Veh3dofContiModel,
    "veh3dof_tracking": Veh3dofTrackingModel,
                  "pyth_veh3dofconti_errcstr": Veh3dofContiErrCstrModel,
                  "veh3dof_tracking_detour": Veh3dofTrackingDetourModel,
                  "veh3dof_tracking_surrcstr": Veh3dofTrackingSurrCstrModel}


# --------------------------------------------------------------------------------------
# Wrapper chain            gops/create_pkg/create_env_model.py:104-126 (assembly order)
# --------------------------------------------------------------------------------------
class WrappedModel:
    """ScaleAction -> ClipAction -> ClipObservation -> [ScaleObservation] -> [ShapingReward] ->
    [ActionRepeat] -> MaskAtDone -> base model, fused into one `forward`.

    wrapper/scale_action.py:75-83, clip_action.py:27-40, clip_observation.py:27-44,
    scale_observation.py:104-116, shaping_reward.py:77-88, action_repeat.py:71-87,
    mask_at_done.py:26-40."""

    def __init__(self, model: BaseModel, *, reward_shift=None, reward_scale=None, obs_shift=None,
                 obs_scale=None, clip_obs=True, clip_action=True, mask_at_done=True, repeat_num=None,
                 sum_reward=True, action_scale=True, min_action=-1.0, max_action=1.0):
        self.model = model
        dt = model.action_lower_bound.dtype
        self.mask_at_done, self.clip_obs, self.clip_action = mask_at_done, clip_obs, clip_action
        self.action_scale = action_scale
        self.repeat_num, self.sum_reward = repeat_num, sum_reward
        self.shaping = reward_scale is not None or reward_shift is not None
        self.reward_scale = 1.0 if reward_scale is None else reward_scale
        self.reward_shift = 0.0 if reward_shift is None else reward_shift
        self.obs_scaling = obs_shift is not None or obs_scale is not None
        osc = 1.0 if obs_scale is None else obs_scale
        osh = 0.0 if obs_shift is None else obs_shift
        self.obs_scale = torch.as_tensor(osc, dtype=dt) if isinstance(osc, (list, np.ndarray)) else osc
        self.obs_shift = torch.as_tensor(osh, dtype=dt) if isinstance(osh, (list, np.ndarray)) else osh
        self.min_action = torch.zeros_like(model.action_lower_bound) + torch.as_tensor(min_action, dtype=dt)
        self.max_action = torch.zeros_like(model.action_upper_bound) + torch.as_tensor(max_action, dtype=dt)
        self.obs_dim, self.action_dim, self.dt = model.obs_dim, model.action_dim, model.dt

    def _masked(self, obs, action, done, info):
        nobs, r, nd, ninfo = self.model.step(obs, action, done, info)
        if self.mask_at_done:
            d = done.bool()
            nobs = ~d.unsqueeze(1) * nobs + d.unsqueeze(1) * obs
            r = ~d * r
            nd = nd.bool() | d
        return nobs, r, nd, ninfo

    def _repeated(self, obs, action, done, info):
        if self.repeat_num is None:
            return self._masked(obs, action, done, info)
        total = 0
        for _ in range(self.repeat_num):
            nobs, r, nd, ninfo = self._masked(obs, action, done, info)
            total = total + r
            obs = nobs                      # reference quirk: done / info are NOT advanced
        return nobs, (total if self.sum_reward else r), nd, ninfo

    def forward(self, obs, action, done, info):
        m = self.model
        if self.action_scale:
            lo, hi = m.action_lower_bound, m.action_upper_bound
            action = torch.clip(action, self.min_action, self.max_action)
            action = lo + (hi - lo) * ((action - self.min_action) / (self.max_action - self.min_action))
            action = torch.clip(action, lo, hi)
        if self.clip_action:
            action = action.clip(m.action_lower_bound, m.action_upper_bound)
        inner_obs = obs / self.obs_scale - self.obs_shift if self.obs_scaling else obs
        nobs, r, nd, ninfo = self._repeated(inner_obs, action, done, info)
        if self.shaping:
            r = (r + self.reward_shift) * self.reward_scale
        if self.obs_scaling:
            nobs = (nobs + self.obs_shift) * self.obs_scale
        if self.clip_obs:
            nobs = nobs.clip(m.obs_lower_bound, m.obs_upper_bound)
        return nobs, r, nd, ninfo


def create_env_model(env_id: str, dtype=torch.float32, **kwargs) -> WrappedModel:
    wrap_keys = ("reward_shift", "reward_scale", "obs_shift", "obs_scale", "clip_obs", "clip_action",
                 "mask_at_done", "repeat_num", "sum_reward", "action_scale", "min_action", "max_action")
    wk = {k: kwargs[k] for k in wrap_keys if k in kwargs}
    mk = {k: v for k, v in kwargs.items() if k not in wrap_keys}
    if env_id not in MODEL_REGISTRY:
        raise KeyError(f"No registered env with id: {env_id}_model")
    return WrappedModel(MODEL_REGISTRY[env_id](dtype=dtype, **mk), **wk)


# --------------------------------------------------------------------------------------
# Algorithms
# --------------------------------------------------------------------------------------
@dataclass
class NetSpec:
    layers: List[Tuple[Tensor, Tensor]]
    hidden_act: str
    out_act: str = "linear"
    act_high: Optional[Tensor] = None
    act_low: Optional[Tensor] = None
    time_input: bool = False           # FiniteHorizonPolicy

    def params(self):
        return [p for wb in self.layers for p in wb]

    def clone(self, requires_grad=False, dtype=None):
        ls = [(w.detach().clone().to(dtype or w.dtype).requires_grad_(requires_grad),
               b.detach().clone().to(dtype or b.dtype).requires_grad_(requires_grad)) for w, b in self.layers]
        cast = lambda t: None if t is None else t.to(dtype or t.dtype)
        return NetSpec(ls, self.hidden_act, self.out_act, cast(self.act_high), cast(self.act_low), self.time_input)

    def act(self, obs, t=None):
        return policy_forward(self.layers, obs, self.act_high, self.act_low, self.hidden_act, self.out_act,
                              virtual_t=t if self.time_input else None)

    def value(self, obs):
        return value_forward(self.layers, obs, self.hidden_act, self.out_act)


def fhadp_loss(policy: NetSpec, env: WrappedModel, data: dict, pre_horizon: int, gamma: float = 1.0,
               trace: Optional[list] = None):
    """FHADP._compute_loss_policy, gops/algorithm/fhadp.py:113-125."""
    o, d = data["obs"], data["done"]
    info = data
    v_pi = 0
    for step in range(pre_horizon):
        a = policy.act(o, step + 1)
        o, r, d, info = env.forward(o, a, d, info)
        v_pi = v_pi + r * (gamma ** step)
        if trace is not None:
            trace.append((o.detach().clone(), a.detach().clone(), r.detach().clone(), d.clone()))
    return -v_pi.mean()


def fhadp_constrained_loss(mode: str, policy: NetSpec, env: WrappedModel, data: dict, pre_horizon: int, gamma: float,
                           coef: float):
    """_compute_loss_policy of fhadp_exterior.py:55-70 ("exterior", coef = penalty), fhadp_lagrangian.py:59-71
    ("lagrangian", coef = multiplier) and fhadp_interior.py:55-84 ("interior", coef = penalty).
    Returns (loss_policy, loss_reward, loss_constraint, feasible_ratio)."""
    o, d, info = data["obs"], data["done"], data
    v_r, v_c, v_int, cs = 0, 0, 0, []
    for step in range(pre_horizon):
        a = policy.act(o, step + 1)
        o, r, d, info = env.forward(o, a, d, info)
        c = info["constraint"]
        cs.append(c)
        v_r = v_r + r * (gamma ** step)
        if mode == "lagrangian":
            v_c = v_c + torch.clamp_min(c, 0).sum(1) * (gamma ** step)
        else:
            v_c = v_c + (torch.clamp_min(c, 0) ** 2).sum(1) * (gamma ** step)
        v_int = v_int + (-torch.clamp_max(c, 0) + 1e-8).log().sum(1) * (gamma ** step)
    loss_reward = -v_r.mean()
    feasible = (torch.stack(cs, dim=1) < 0).all(2).all(1)
    if mode == "interior":
        l_int, l_ext = (v_int * feasible).mean(), (v_c * ~feasible).mean()
        return loss_reward + 1 / coef * l_int + coef * l_ext, loss_reward, l_ext, feasible.float().mean()
    l_c = v_c.mean()
    return loss_reward + coef * l_c, loss_reward, l_c, feasible.float().mean()


def _rollout(policy: NetSpec, env, data, n, gamma):
    o, d, info = data["obs"], data["done"], data
    total = None
    for step in range(n):
        a = policy.act(o)
        o, r, d, info = env.forward(o, a, d, info)
        total = r if step == 0 else total + gamma ** step * r
    return total, o, d


def infadp_loss_policy(policy: NetSpec, v_target: NetSpec, env, data, forward_step=10, gamma=0.99):
    """INFADP.__compute_loss_policy, gops/algorithm/infadp.py:188-213."""
    v_pi, o2, d = _rollout(policy, env, data, forward_step, gamma)
    v_pi = v_pi + (~d) * gamma ** forward_step * v_target.value(o2)
    return -v_pi.mean()


def infadp_loss_value(v: NetSpec, policy: NetSpec, v_target: NetSpec, env, data, forward_step=10, gamma=0.99):
    """INFADP.__compute_loss_v, gops/algorithm/infadp.py:159-186. Returns (loss, mean v)."""
    val = v.value(data["obs"])
    with torch.no_grad():
        backup, o2, d = _rollout(policy, env, data, forward_step, gamma)
        backup = backup + (~d) * gamma ** forward_step * v_target.value(o2)
    return ((val - backup) ** 2).mean(), torch.mean(val)


def adam_step(params: Sequence[Tensor], grads: Sequence[Tensor], state: dict, lr: float,
              betas=(0.9, 0.999), eps=1e-8):
    """torch.optim.Adam single-tensor update rule (no weight decay / amsgrad), as used at
    fhadp.py:45-47 and infadp.py:52-55."""
    state["step"] = state.get("step", 0) + 1
    t = state["step"]
    b1, b2 = betas
    out = []
    for i, (p, g) in enumerate(zip(params, grads)):
        m = state.setdefault(("m", i), torch.zeros_like(p))
        v = state.setdefault(("v", i), torch.zeros_like(p))
        m.mul_(b1).add_(g, alpha=1 - b1)
        v.mul_(b2).addcmul_(g, g, value=1 - b2)
        bc1, bc2 = 1 - b1 ** t, 1 - b2 ** t
        denom = (v.sqrt() / math.sqrt(bc2)).add_(eps)
        out.append(p.detach() - (lr / bc1) * (m / denom))
    return out


def polyak(target: Sequence[Tensor], src: Sequence[Tensor], tau: float):
    """INFADP.__update target update, infadp.py:126-133: p_targ = (1-tau) p_targ + tau p."""
    return [pt * (1 - tau) + tau * p for pt, p in zip(target, src)]


# --------------------------------------------------------------------------------------
# Synthetic inputs (SURVEY.md §8(d)): seeded draws from the data envs' initial-state laws
# --------------------------------------------------------------------------------------
def sample_inputs(env_id: str, batch: int, seed: int, *, pre_horizon: int = 10, lq_config: str = "s4a2",
                  ref_len: Optional[int] = None) -> dict:
    g = torch.Generator().manual_seed(seed)
    U = lambda *s: torch.rand(*s, generator=g, dtype=torch.float32)
    if env_id == "pyth_idpendulum":
        # pyth_idpendulum.py:36-38 (init box), pyth_base_env.py:61-65
        h = torch.tensor([5, 0.1, 0.1, 0.3, 0.3, 0.3])
        return {"obs": (U(batch, 6) * 2 - 1) * h, "done": torch.zeros(batch)}
    if env_id == "pyth_lq":
        cfg = LQ_CONFIGS[lq_config]
        mean, std = torch.tensor(cfg["init_mean"], dtype=torch.float32), torch.tensor(cfg["init_std"], dtype=torch.float32)
        return {"obs": mean + std * torch.randn(batch, len(cfg["init_mean"]), generator=g), "done": torch.zeros(batch)}
    if env_id in ("pyth_veh3dofconti", "veh3dof_tracking", "veh3dof_tracking_detour", "veh3dof_tracking_surrcstr"):
        # pyth_veh3dofconti.py:144-191 ; env_gen_ocp/context/ref_traj.py:25-53
        ref = RefTraj()
        P = pre_horizon
        n_pts = (P + 1) if env_id == "pyth_veh3dofconti" else (ref_len or 2 * P + 1)
        t0 = 20.0 * U(batch)
        path = torch.randint(0, 4, (batch,), generator=g).float()
        spd = torch.randint(0, 2, (batch,), generator=g).float()
        pts = []
        for i in range(n_pts):
            tt = t0 + i * 0.1
            pts.append(torch.stack((ref.x(tt, path, spd), ref.y(tt, path, spd), ref.phi(tt, path, spd),
                                    ref.u(tt, path, spd)), 1))
        ref_points = torch.stack(pts, 1)
        h = torch.tensor([2, 1, math.pi / 6, 2, 0.1, 0.1])
        delta = (U(batch, 6) * 2 - 1) * h
        state = torch.cat((ref_points[:, 0] + delta[:, :4], delta[:, 4:]), 1)
        state[:, 2] = angle_normalize(state[:, 2])
        obs = veh_obs(state, ref_points[:, :P + 1])
        if env_id == "pyth_veh3dofconti":
            return {"obs": obs, "done": torch.zeros(batch), "state": state, "ref_points": ref_points,
                    "path_num": path, "u_num": spd, "ref_time": t0}
        if env_id in ("veh3dof_tracking_detour", "veh3dof_tracking_surrcstr"):
            # env_gen_ocp/context/ref_traj_with_static_obstacle.py:76-127: one surrounding vehicle predicted over P + 1
            # points (x, y, phi, u, delta); here ahead of the ego vehicle near the path (some samples start infeasible)
            # and moving slowly along its heading
            sp = ref_points[:, 0]
            ahead, side = 4.0 + 12.0 * U(batch), (U(batch) * 2 - 1) * 3.0
            sphi = sp[:, 2] + (U(batch) * 2 - 1) * 0.3
            su = 2.0 * U(batch)
            x0 = sp[:, 0] + ahead * torch.cos(sp[:, 2]) - side * torch.sin(sp[:, 2])
            y0 = sp[:, 1] + ahead * torch.sin(sp[:, 2]) + side * torch.cos(sp[:, 2])
            steps = torch.arange(P + 1, dtype=torch.float32).unsqueeze(0) * 0.1
            surr = torch.stack((x0.unsqueeze(1) + su.unsqueeze(1) * torch.cos(sphi).unsqueeze(1) * steps,
                                y0.unsqueeze(1) + su.unsqueeze(1) * torch.sin(sphi).unsqueeze(1) * steps,
                                sphi.unsqueeze(1).expand(-1, P + 1), su.unsqueeze(1).expand(-1, P + 1),
                                torch.zeros(batch, P + 1)), 2).unsqueeze(2).contiguous()
            model = Veh3dofTrackingDetourModel(pre_horizon=P)
            return {"obs": model.get_obs(state, ref_points, 0, surr), "done": torch.zeros(batch),
                    "state": (state, ref_points, 0, surr)}
        return {"obs": obs, "done": torch.zeros(batch), "state": (state, ref_points, 0)}
    raise KeyError(env_id)
