"""Generate golden vectors by running the UNMODIFIED reference (GOPS @ /root/reference) on CPU.

TEST INFRASTRUCTURE.  Run in the build container only (`python oracle/make_golden.py`); the
outputs under `tests/golden/*.npz` are committed and travel to the GPU box, the reference does
not.  Every case stores: inputs, the initial `state_dict`, the loss the reference reports
(`tb_info`), the gradients left in `p.grad` by `local_update`, and the post-update `state_dict`
(one Adam step, plus Polyak targets for INFADP).

Reference entry points exercised (all through the reference's own factories):
  create_alg                      gops/create_pkg/create_alg.py:60-97
  FHADP.local_update              gops/algorithm/fhadp.py:87-125 (+ base.py:94-98)
  INFADP.local_update             gops/algorithm/infadp.py:101-213
  create_env_model wrapper chain  gops/create_pkg/create_env_model.py:51-128
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import ref_shim  # noqa: E402
from oracle import gops_oracle as orc  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def _np(t):
    return t.detach().cpu().numpy()


def _sd(alg):
    return {k: _np(v).copy() for k, v in alg.state_dict().items()}


def base_kwargs(env_id, algorithm, obs_dim, act_dim, hidden, act, policy_name, **extra):
    kw = dict(
        env_id=env_id, algorithm=algorithm, seed=0, trainer="off_serial_trainer", cnn_shared=False,
        use_gpu=False, action_type="continu", obsv_dim=obs_dim, action_dim=act_dim,
        action_high_limit=np.ones(act_dim, dtype=np.float32), action_low_limit=-np.ones(act_dim, dtype=np.float32),
        policy_func_name=policy_name, policy_func_type="MLP", policy_hidden_sizes=list(hidden),
        policy_hidden_activation=act, policy_act_distribution="default", policy_learning_rate=1e-3,
        value_func_name="StateValue", value_func_type="MLP", value_hidden_sizes=list(hidden),
        value_hidden_activation=act, value_learning_rate=1e-3,
    )
    kw.update(extra)
    return kw


def to_ref_data(env_id, data):
    """Oracle input dict -> the dict the reference trainer would hand to local_update."""
    gen_ocp = env_id in ("veh3dof_tracking", "veh3dof_tracking_detour", "veh3dof_tracking_surrcstr")
    out = {k: v for k, v in data.items() if k != "state" or not gen_ocp}
    B = data["obs"].shape[0]
    if gen_ocp:
        from gops.env.env_gen_ocp.pyth_base import ContextState, State
        robot, reference, t = data["state"][:3]
        surr = data["state"][3].clone() if len(data["state"]) > 3 else None
        out["state"] = State(robot_state=robot.clone(),
                             context_state=ContextState(reference=reference.clone(), constraint=surr, t=t))
    out.setdefault("act", torch.zeros(B, 1))
    out.setdefault("rew", torch.zeros(B))
    out.setdefault("obs2", data["obs"].clone())
    return out


def flat_inputs(env_id, data):
    d = {}
    for k, v in data.items():
        if k == "state" and env_id in ("veh3dof_tracking", "veh3dof_tracking_detour", "veh3dof_tracking_surrcstr"):
            d["in_robot_state"], d["in_reference"] = _np(v[0]), _np(v[1])
            d["in_t"] = np.int64(v[2])
            if len(v) > 3:
                d["in_surr"] = _np(v[3])
        else:
            d["in_" + k] = _np(v)
    return d


def run_case(name, kw, data, iterations, trace_n=0, set_params=None, load_ckpt=None):
    from gops.create_pkg.create_alg import create_alg

    torch.manual_seed(1234)
    alg = create_alg(**kw)
    if load_ckpt:
        alg.load_state_dict(torch.load(load_ckpt, map_location="cpu"))
    if set_params:
        alg.set_parameters(set_params)
    env_id = kw["env_id"]
    rec = flat_inputs(env_id, data)
    for k, v in _sd(alg).items():
        rec["init/" + k] = v
    if trace_n and kw["algorithm"] == "FHADP":
        with torch.no_grad():
            rd = to_ref_data(env_id, data)
            o, d, info = rd["obs"], rd["done"], rd
            tr = {"obs": [], "act": [], "rew": [], "done": []}
            for step in range(kw["pre_horizon"]):
                a = alg.networks.policy(o, step + 1)
                o, r, d, info = alg.envmodel.forward(o, a, d, info)
                tr["obs"].append(_np(o[:trace_n])); tr["act"].append(_np(a[:trace_n]))
                tr["rew"].append(_np(r[:trace_n])); tr["done"].append(_np(d[:trace_n]))
            for k, v in tr.items():
                rec["trace_" + k] = np.stack(v, 0)
    for it in iterations:
        tb = alg.local_update(to_ref_data(env_id, data), it)
        for k, v in tb.items():
            if "Time" not in k:
                rec[f"it{it}/tb/{k}"] = np.float64(v)
        for nm in ("policy", "v"):
            net = getattr(alg.networks, nm, None)
            if net is None:
                continue
            for pn, p in net.named_parameters():
                if p.grad is not None:
                    rec[f"it{it}/grad/{nm}.{pn}"] = _np(p.grad).copy()
        for k, v in _sd(alg).items():
            rec[f"it{it}/post/{k}"] = v
    os.makedirs(OUT, exist_ok=True)
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **rec)
    print(name, {k: float(v) for k, v in rec.items() if "/tb/" in k})


def run_trajectory(name, kw, batches, n_updates, remote_every=0):
    """K consecutive updates on a rotating set of fixed batches (incl. LR scheduler steps, base.py:94-98): stores the
    loss of every update and the weights after updates 1, K/2 and K.  `remote_every` = m > 0 routes every m-th update
    through get_remote_update_info + remote_update (base.py:100-104, fhadp.py:92-102), the Ray-replica entry points."""
    from gops.create_pkg.create_alg import create_alg

    torch.manual_seed(4321)
    alg = create_alg(**kw)
    env_id = kw["env_id"]
    rec = {}
    for j, data in enumerate(batches):
        for k, v in flat_inputs(env_id, data).items():
            rec[f"b{j}/{k}"] = v
    for k, v in _sd(alg).items():
        rec["init/" + k] = v
    losses, lrs = [], []
    keep = {1, n_updates // 2, n_updates}
    for it in range(n_updates):
        data = to_ref_data(env_id, batches[it % len(batches)])
        if remote_every and it % remote_every == remote_every - 1:
            tb, upd = alg.get_remote_update_info(data, it)
            alg.remote_update(upd)
        else:
            tb = alg.local_update(data, it)
        key = "Loss/Critic loss-RL iter" if (kw["algorithm"] == "INFADP" and it % 2 == 0) else "Loss/Actor loss-RL iter"
        losses.append(tb[key])
        lrs.append(alg.networks.policy_optimizer.param_groups[0]["lr"])
        if it + 1 in keep:
            for k, v in _sd(alg).items():
                rec[f"after{it + 1}/{k}"] = v
    rec["losses"], rec["lrs"] = np.asarray(losses, np.float64), np.asarray(lrs, np.float64)
    # trained-policy actions: what the evaluator would see after the K updates
    with torch.no_grad():
        o = batches[0]["obs"][:64]
        rec["final_actions"] = _np(alg.networks.policy(o, 1) if kw["policy_func_name"] == "FiniteHorizonPolicy"
                                   else alg.networks.policy(o))
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **rec)
    print(name, "losses", losses[0], losses[-1], "lr", lrs[0], lrs[-1])


def run_dsac(name, n_iter=4, B=128, hidden=(64, 64, 64)):
    """DSAC.local_update (dsac.py:121-290) on a fixed synthetic replay batch.  The reference draws its Gaussian noise from
    torch's global generator inside the update; the draws are RECORDED here (wrappers around torch.normal and
    torch.distributions.normal._standard_normal -- instrumentation of the generator script, the reference is untouched)
    so that the parity tests can replay exactly the same noise: per update [eps_new, eps_next, z(unused), z_next, z(unused)]."""
    from gops.create_pkg.create_alg import create_alg
    import torch.distributions.normal as tdn

    kw = base_kwargs("pyth_idpendulum", "DSAC", 6, 1, hidden, "gelu", "StochaPolicy",
                     value_func_name="ActionValueDistri", policy_act_distribution="TanhGaussDistribution",
                     value_learning_rate=3e-4, policy_learning_rate=3e-4, alpha_learning_rate=5e-3, gamma=0.99, tau=0.005,
                     auto_alpha=True, alpha=0.2, delay_update=2, TD_bound=10, bound=True,
                     policy_min_log_std=-20, policy_max_log_std=1, value_hidden_sizes=list(hidden),
                     policy_hidden_sizes=list(hidden))
    torch.manual_seed(777)
    alg = create_alg(**kw)
    g = torch.Generator().manual_seed(5)
    obs = orc.sample_inputs("pyth_idpendulum", B, 60)["obs"]
    data = {"obs": obs, "act": torch.rand(B, 1, generator=g) * 2 - 1, "rew": torch.randn(B, generator=g) * 3 + 5,
            "obs2": obs + 0.05 * torch.randn(B, 6, generator=g), "done": (torch.rand(B, generator=g) < 0.05).float()}
    rec = {"in_" + k: _np(v) for k, v in data.items()}
    for k, v in _sd(alg).items():
        rec["init/" + k] = v
    noise = []
    o_sn, o_nm = tdn._standard_normal, torch.normal

    def sn(*a, **k):
        x = o_sn(*a, **k); noise.append(x.clone()); return x

    def nm(*a, **k):
        x = o_nm(*a, **k); noise.append(x.clone()); return x
    tdn._standard_normal, torch.normal = sn, nm
    try:
        torch.manual_seed(4242)
        for it in range(n_iter):
            noise.clear()
            tb = alg.local_update({k: v.clone() for k, v in data.items()}, it)
            assert len(noise) == 5, len(noise)
            rec[f"it{it}/eps_new"], rec[f"it{it}/eps_next"], rec[f"it{it}/z_next"] = _np(noise[0]), _np(noise[1]), _np(noise[3])
            for k, v in tb.items():
                if "Time" not in k:
                    rec[f"it{it}/tb/{k}"] = np.float64(v)
            for nm_ in ("policy", "q"):
                for pn, p in getattr(alg.networks, nm_).named_parameters():
                    rec[f"it{it}/grad/{nm_}.{pn}"] = _np(p.grad).copy()
            rec[f"it{it}/grad/log_alpha"] = _np(alg.networks.log_alpha.grad).copy()
            for k, v in _sd(alg).items():
                rec[f"it{it}/post/{k}"] = v
    finally:
        tdn._standard_normal, torch.normal = o_sn, o_nm
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **rec)
    print(name, {k: float(v) for k, v in rec.items() if "it0/tb/" in k})


def run_constrained():
    """fhadp_exterior / fhadp_lagrangian / fhadp_interior on the constraint-providing pyth_veh3dofconti_errcstr model:
    two consecutive updates (penalty_delay = 1 / multiplier_delay = 1, so the second one runs with the annealed
    coefficient), tolerances chosen so that the batch mixes feasible and infeasible samples."""
    extra = {"FHADPExterior": dict(penalty=2.0, penalty_increase=1.5, penalty_delay=1),
             "FHADPInterior": dict(penalty=2.0, penalty_increase=1.5, penalty_delay=1),
             "FHADPLagrangian": dict(multiplier=1.5, multiplier_lr=5e-2, multiplier_delay=1)}
    for algname, ex in extra.items():
        kw = base_kwargs("pyth_veh3dofconti_errcstr", algname, 46, 2, (64, 64), "elu", "FiniteHorizonPolicy", pre_horizon=10,
                         gamma=0.97, y_error_tol=1.2, u_error_tol=2.2, **ex)
        d = orc.sample_inputs("pyth_veh3dofconti", 160, 70, pre_horizon=10)
        d["done"][::9] = 1.0
        run_case("cstr_" + algname.lower(), kw, d, [0, 1])


def run_detour():
    """env_gen_ocp veh3dof_tracking_detour (the model of example_train/fhadp/fhadp_mlp_veh3ddetour_serial.py): plain FHADP
    and the three constrained variants, two consecutive updates each, a batch that mixes feasible and colliding rollouts
    and samples that arrive done (their state keeps evolving behind the frozen observation, mask_at_done.py:26-40)."""
    extra = {"FHADP": {}, "FHADPExterior": dict(penalty=2.0, penalty_increase=1.5, penalty_delay=1),
             "FHADPInterior": dict(penalty=2.0, penalty_increase=1.5, penalty_delay=1),
             "FHADPLagrangian": dict(multiplier=1.5, multiplier_lr=5e-2, multiplier_delay=1)}
    for algname, ex in extra.items():
        kw = base_kwargs("veh3dof_tracking_detour", algname, 50, 2, (64, 64), "elu", "FiniteHorizonPolicy", pre_horizon=10,
                         gamma=0.97, **ex)
        d = orc.sample_inputs("veh3dof_tracking_detour", 160, 71, pre_horizon=10)
        d["done"][::9] = 1.0
        run_case("detour_" + algname.lower(), kw, d, [0, 1])
    # veh3dof_tracking_surrcstr: same structure, other radius / reward / bound -- one constrained case
    kw = base_kwargs("veh3dof_tracking_surrcstr", "FHADPExterior", 50, 2, (64, 64), "elu", "FiniteHorizonPolicy", pre_horizon=10,
                     gamma=0.97, **extra["FHADPExterior"])
    d = orc.sample_inputs("veh3dof_tracking_surrcstr", 160, 72, pre_horizon=10)
    d["done"][::9] = 1.0
    run_case("surrcstr_fhadpexterior", kw, d, [0, 1])


def run_fresh_fhadp(H, B, seed):
    """The reference's FHADP idpendulum update from its own initial weights on oracle-sampled inputs (a ninth of the
    batch arriving done): initial policy, inputs, loss and gradients (tests/test_oracle_vs_reference.py)."""
    from oracle import ref_runner
    torch.set_num_threads(4)
    torch.manual_seed(seed)
    alg = ref_runner.create_reference_alg(ref_runner.c1_kwargs(H))
    data = orc.sample_inputs("pyth_idpendulum", B, seed=seed)
    data["done"][::9] = 1.0
    rec = flat_inputs("pyth_idpendulum", data)
    for k, v in _sd(alg).items():
        rec["init/" + k] = v
    tb = alg.local_update({k: v.clone() for k, v in data.items()}, 0)
    rec["loss"] = np.float64(tb["Loss/Actor loss-RL iter"])
    for pn, p in alg.networks.policy.named_parameters():
        rec["grad/policy." + pn] = _np(p.grad).copy()
    name = f"fresh_fhadp_idp_h{H}_b{B}_s{seed}"
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **rec)
    print(name, float(rec["loss"]))


def run_trainer_steps(n_steps=3, H=30, minibatch=512):
    """Three OffSerialTrainer steps of the reference FHADP fed by the reference's own ReplayBuffer: initial state_dict,
    the sampled minibatches, the loss of every step, and the policy's actions on 32 buffered observations after the
    last step (tests/test_gpu_reference_integration.py)."""
    from gops.trainer.buffer.replay_buffer import ReplayBuffer
    from oracle import ref_runner
    torch.manual_seed(11)
    alg = ref_runner.create_reference_alg(ref_runner.c1_kwargs(H))
    rec = {"init/" + k: v for k, v in _sd(alg).items()}
    buf = ReplayBuffer(trainer="off_serial_trainer", seed=0, obsv_dim=6, action_dim=1, buffer_max_size=4096,
                       additional_info={})
    g = torch.Generator().manual_seed(3)
    h = torch.tensor([5, 0.1, 0.1, 0.3, 0.3, 0.3])
    obs = ((torch.rand(2048, 6, generator=g) * 2 - 1) * h).numpy()
    buf.add_batch([(o, np.zeros(1, np.float32), 0.0, False, {}, o, {}, 0.0) for o in obs])
    for it in range(n_steps):
        replay = buf.sample_batch(minibatch)
        for k, v in replay.items():
            rec[f"it{it}/batch/{k}"] = _np(v).copy()
        tb = alg.local_update({k: v.clone() for k, v in replay.items()}, it)
        rec[f"it{it}/loss"] = np.float64(tb["Loss/Actor loss-RL iter"])
    rec["act_obs"] = obs[:32].copy()
    with torch.no_grad():
        rec["act"] = _np(alg.networks.policy(torch.from_numpy(obs[:32]), 1)).copy()
    np.savez_compressed(os.path.join(OUT, "trainer_steps_fhadp_idp_h30.npz"), **rec)
    print("trainer_steps_fhadp_idp_h30", [float(rec[f"it{i}/loss"]) for i in range(n_steps)])


def main():
    ref_shim.install()
    torch.set_num_threads(4)
    if "--detour" in sys.argv:
        run_detour()
        return
    if "--integration" in sys.argv:
        run_fresh_fhadp(30, 64, 101)
        run_fresh_fhadp(7, 33, 102)
        run_trainer_steps()
        return
    run_dsac("dsac_idp")
    run_constrained()
    run_detour()

    # K = 20 consecutive updates, LinearLR scheduler, every 5th through the remote-update entry points
    kw = base_kwargs("pyth_idpendulum", "FHADP", 6, 1, (64, 64), "gelu", "FiniteHorizonPolicy", pre_horizon=30,
                     reward_scale=1.0, policy_learning_rate=3e-4,
                     policy_scheduler={"name": "LinearLR", "params": {"start_factor": 1.0, "end_factor": 0.25,
                                                                      "total_iters": 16}})
    run_trajectory("traj_fhadp_idp_k20", kw, [orc.sample_inputs("pyth_idpendulum", 512, 40 + j) for j in range(3)], 20,
                   remote_every=5)
    kw = base_kwargs("pyth_lq", "INFADP", 4, 2, (64, 64), "gelu", "DetermPolicy", lq_config="s4a2",
                     reward_scale=1.0, reward_shift=0.0, policy_learning_rate=8e-4, value_learning_rate=3e-4)
    run_trajectory("traj_infadp_lq_k20", kw, [orc.sample_inputs("pyth_lq", 256, 50 + j, lq_config="s4a2")
                                              for j in range(2)], 20)
    # long horizon with every sample alive to the end (MaskAtDone off): the h80 case above is degenerate, every sample
    # of an untrained policy terminates by step ~24 and the tail of the tape / reverse sweep is masked out
    kw = base_kwargs("pyth_idpendulum", "FHADP", 6, 1, (64, 64), "gelu", "FiniteHorizonPolicy",
                     pre_horizon=80, reward_scale=1.0, policy_learning_rate=1e-4, mask_at_done=False)
    d = orc.sample_inputs("pyth_idpendulum", 128, 22)
    d["obs"] = d["obs"] * torch.tensor([1.0, 0.2, 0.2, 0.2, 0.2, 0.2])     # near upright: finite 80-step rollouts
    run_case("fhadp_idp_h80_nomask", kw, d, [0])
    # FHADP2 / FiniteHorizonFullPolicy (open-loop policy, fhadp2.py:98-121, mlp.py:114-145)
    kw = base_kwargs("pyth_idpendulum", "FHADP2", 6, 1, (64, 64), "gelu", "FiniteHorizonFullPolicy", pre_horizon=20,
                     reward_scale=1.0, policy_learning_rate=1e-3)
    d = orc.sample_inputs("pyth_idpendulum", 256, 23)
    d["obs"] = d["obs"] * torch.tensor([1.0, 0.3, 0.3, 0.3, 0.3, 0.3])
    run_case("fhadp2_idp", kw, d, [0])
    rec = dict(np.load(os.path.join(OUT, "fhadp2_idp.npz")))
    rec["pre_horizon"] = np.int64(20)
    np.savez_compressed(os.path.join(OUT, "fhadp2_idp.npz"), **rec)
    if "--only-new" in sys.argv:
        return

    # C1: FHADP idpendulum, FiniteHorizonPolicy [64,64] gelu (fhadp_mlp_idpendulum_serial.py:34-75)
    for H in (30, 80):
        kw = base_kwargs("pyth_idpendulum", "FHADP", 6, 1, (64, 64), "gelu", "FiniteHorizonPolicy",
                         pre_horizon=H, reward_scale=1.0, policy_learning_rate=1e-4)
        run_case(f"fhadp_idp_h{H}", kw, orc.sample_inputs("pyth_idpendulum", 256, 11), [0],
                 trace_n=32 if H == 30 else 0)
    # gamma != 1, relu, and half the batch arriving already done
    kw = base_kwargs("pyth_idpendulum", "FHADP", 6, 1, (64, 64), "relu", "FiniteHorizonPolicy",
                     pre_horizon=12, reward_scale=0.5, reward_shift=1.0, gamma=0.97)
    d = orc.sample_inputs("pyth_idpendulum", 128, 12)
    d["done"][::2] = 1.0
    run_case("fhadp_idp_relu_done", kw, d, [0])

    # C5: INFADP LQ s4a2 (infadp_mlp_lqs4a2_offserial.py), PEV then PIM
    kw = base_kwargs("pyth_lq", "INFADP", 4, 2, (64, 64), "gelu", "DetermPolicy", lq_config="s4a2",
                     reward_scale=1.0, reward_shift=0.0, policy_learning_rate=8e-4, value_learning_rate=3e-4)
    run_case("infadp_lq_s4a2", kw, orc.sample_inputs("pyth_lq", 256, 13, lq_config="s4a2"), [0, 1])
    run_case("infadp_lq_s4a2_n40", kw, orc.sample_inputs("pyth_lq", 128, 14, lq_config="s4a2"), [0, 1],
             set_params={"forward_step": 40, "tau": 0.2, "gamma": 0.97})
    # FHADP on LQ s3a1 wide initial box so that ClipObservation is active
    kw = base_kwargs("pyth_lq", "FHADP", 3, 1, (64, 64), "elu", "FiniteHorizonPolicy", lq_config="s3a1",
                     pre_horizon=20, reward_scale=0.1)
    d = orc.sample_inputs("pyth_lq", 128, 15, lq_config="s3a1")
    d["obs"] = d["obs"] * 4.0
    run_case("fhadp_lq_s3a1_clip", kw, d, [0])

    # INFADP idpendulum (infadp_mlp_idpendulum_serial.py)
    kw = base_kwargs("pyth_idpendulum", "INFADP", 6, 1, (64, 64), "relu", "DetermPolicy", reward_scale=1.0)
    run_case("infadp_idp", kw, orc.sample_inputs("pyth_idpendulum", 256, 16), [0, 1])

    # optional wrappers of the chain: ScaleObservation, ActionRepeat (create_env_model.py:109-122)
    scale6 = [0.5, 2.0, 2.0, 1.0, 0.25, 0.5]
    shift6 = [0.1, 0.0, -0.05, 0.0, 0.2, 0.0]
    kw = base_kwargs("pyth_idpendulum", "FHADP", 6, 1, (64, 64), "gelu", "FiniteHorizonPolicy", pre_horizon=15,
                     reward_scale=0.2, obs_scale=scale6, obs_shift=shift6)
    d = orc.sample_inputs("pyth_idpendulum", 128, 31)
    d["obs"] = (d["obs"] + torch.tensor(shift6)) * torch.tensor(scale6)
    d["done"][::5] = 1.0
    run_case("fhadp_idp_obsscale", kw, d, [0])
    kw = base_kwargs("pyth_lq", "INFADP", 4, 2, (64, 64), "tanh", "DetermPolicy", lq_config="s4a2", reward_scale=0.1,
                     obs_scale=[2.0, 0.5, 1.5, 1.0], repeat_num=3)
    d = orc.sample_inputs("pyth_lq", 128, 32, lq_config="s4a2")
    d["obs"] = d["obs"] * torch.tensor([2.0, 0.5, 1.5, 1.0]) * 6.0       # wide enough for ClipObservation to bite
    run_case("infadp_lq_obsscale_repeat3", kw, d, [0, 1])
    kw = base_kwargs("pyth_idpendulum", "FHADP", 6, 1, (64, 64), "elu", "FiniteHorizonPolicy", pre_horizon=6,
                     reward_scale=1.0, repeat_num=2, sum_reward=False)
    run_case("fhadp_idp_repeat2_last", kw, orc.sample_inputs("pyth_idpendulum", 128, 33), [0])
    sc46 = (1.0 + 0.5 * torch.rand(46, generator=torch.Generator().manual_seed(7))).tolist()
    sh46 = (0.2 * torch.rand(46, generator=torch.Generator().manual_seed(8)) - 0.1).tolist()
    kw = base_kwargs("pyth_veh3dofconti", "INFADP", 46, 2, (64, 64), "relu", "DetermPolicy", pre_horizon=10,
                     obs_scale=sc46, obs_shift=sh46)
    d = orc.sample_inputs("pyth_veh3dofconti", 128, 34, pre_horizon=10)
    d["obs"] = (d["obs"] + torch.tensor(sh46)) * torch.tensor(sc46)
    run_case("infadp_veh3dofconti_obsscale", kw, d, [0, 1])

    # C2: INFADP veh3dofconti [64,64] relu, P=10 (infadp_mlp_veh3dofconti_offserial.py:34-81)
    kw = base_kwargs("pyth_veh3dofconti", "INFADP", 46, 2, (64, 64), "relu", "DetermPolicy", pre_horizon=10)
    run_case("infadp_veh3dofconti", kw, orc.sample_inputs("pyth_veh3dofconti", 256, 17, pre_horizon=10), [0, 1])
    # FHADP veh3dofconti (fhadp_mlp_veh3dofconti_serial.py:58-71), small P=H
    kw = base_kwargs("pyth_veh3dofconti", "FHADP", 6 + 4 * 12, 2, (64, 64), "elu", "FiniteHorizonPolicy", pre_horizon=12)
    run_case("fhadp_veh3dofconti_p12", kw, orc.sample_inputs("pyth_veh3dofconti", 128, 18, pre_horizon=12), [0])

    # C3: FHADP env_gen_ocp veh3dof_tracking, FiniteHorizonPolicy elu
    kw = base_kwargs("veh3dof_tracking", "FHADP", 6 + 4 * 10, 2, (64, 64), "elu", "FiniteHorizonPolicy", pre_horizon=10)
    run_case("fhadp_veh3dof_tracking_p10", kw, orc.sample_inputs("veh3dof_tracking", 128, 19, pre_horizon=10), [0])
    kw = base_kwargs("veh3dof_tracking", "FHADP", 6 + 4 * 60, 2, (256, 256), "elu", "FiniteHorizonPolicy", pre_horizon=60)
    run_case("fhadp_veh3dof_tracking_p60_w256", kw, orc.sample_inputs("veh3dof_tracking", 32, 20, pre_horizon=60), [0])

    # Known answer from a checkpoint the reference ships (results/FHADP/idpendulum)
    ck = os.path.join(ref_shim.REFERENCE_ROOT, "results", "FHADP", "idpendulum", "apprfunc", "apprfunc_100000.pkl")
    if os.path.exists(ck):
        kw = base_kwargs("pyth_idpendulum", "FHADP", 6, 1, (64, 64), "gelu", "FiniteHorizonPolicy",
                         pre_horizon=80, reward_scale=1.0, policy_learning_rate=1e-4)
        run_case("fhadp_idp_trained_h80", kw, orc.sample_inputs("pyth_idpendulum", 256, 21), [0], load_ckpt=ck)
        from gops.create_pkg.create_alg import create_alg
        kw = base_kwargs("pyth_idpendulum", "FHADP", 6, 1, (64, 64), "gelu", "FiniteHorizonPolicy",
                         pre_horizon=80, reward_scale=1.0)
        alg = create_alg(**kw)
        alg.load_state_dict(torch.load(ck, map_location="cpu"))
        rec = {"sd/" + k: v for k, v in _sd(alg).items()}
        obs = torch.tensor([[-1, 0.05, 0.05, 0, 0.1, 0.1]], dtype=torch.float32)  # example_run/run_idp_fhadp.py:19-20
        acts = []
        with torch.no_grad():
            o, d, info = obs, torch.zeros(1), {}
            for _ in range(5):
                a = alg.networks.policy(o)          # evaluator convention: virtual_t = 1
                acts.append(_np(a)[0])
                o, r, d, info = alg.envmodel.forward(o, a, d, info)
            data = {"obs": obs, "done": torch.zeros(1)}
            loss, _ = alg._compute_loss_policy(data)
        rec["obs0"], rec["closed_loop_actions"], rec["loss_h80"] = _np(obs), np.stack(acts), np.float64(loss.item())
        np.savez_compressed(os.path.join(OUT, "ckpt_fhadp_idp.npz"), **rec)
        print("ckpt_fhadp_idp", rec["closed_loop_actions"].ravel(), rec["loss_h80"])


if __name__ == "__main__":
    main()
