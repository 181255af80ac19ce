#!/usr/bin/env python
"""bench.py -- batched env-steps/s of the FHADP rollout+update hot path (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            (N>1: launched under torch.distributed.run)
  python bench.py --impl reference --gpus N --steps K --warmup W

Workload (config.workload): FHADP on pyth_idpendulum, FiniteHorizonPolicy [64,64] gelu, horizon 30, synthetic initial
states from the data env's reset box.  N = 1: batch 2^18 on the GPU (the configuration BASELINE.json quotes).
N > 1: STRONG scaling by default -- the north-star configuration itself, GLOBAL batch 2^18 sharded over the N GPUs
(2^18 / N samples each) with one NCCL all-reduce of the flat gradient per update; the weak-scaling figure (2^18 per
GPU) is measured in the same run and reported in the `weak` sub-object (`--scaling weak` swaps the two).
One step = one `alg.local_update(data, it)` through the plugin API: weight packing, fused rollout forward+backward,
partial reduction, (all-reduce), fused Adam, and the host read of the loss scalar.

value : inputs resident in HBM when the timed region starts (a rotating set of input batches whose total size exceeds
        L2, so no step finds its inputs in L2);
e2e   : same call with PINNED HOST tensors -- H2D copy of the batch and D2H read of the loss inside the timed region.
        Loss read-back mode (config.loss_readback): every step copies its 4-float result tail to pinned host memory and
        the host reads it; "pipelined" = the host reads step i-1's loss while step i runs (alg.loss_lag = 1; the last
        loss is read before the closing synchronize), "synchronous" = it waits for step i's own loss (reference
        semantics; reported beside it as `sync_loss`).
roofline : the fused rollout kernel alone, timed with CUDA events on its launch stream inside the library
        (gops_b200_plan_enable_timing).  Compute bound by design (SURVEY.md 8(d)): `achieved` = algorithmic TFLOP/s,
        `peak` = tensor roof for FP32-accurate (BF16x3) GEMMs = measured BURST bf16 peak / 6 (the kernel is timed alone);
        FP32-FFMA, HBM, raw-bf16 and sustained-peak fractions beside it.
cpu_baseline : the UNMODIFIED reference's `alg.local_update` (oracle/_ref, kind "reference") on the host cores, on a
        bounded sample of the same workload -- or the oracle port (kind "port") if the reference tree is absent.
gpu_eager_baseline : the unmodified reference with use_gpu=True on the same B200 (PyTorch eager; SURVEY 8(d)'s
        "existing Blackwell path").
configs : the other BASELINE.json configurations, each one timed update (device-resident inputs, L2 flushed between
        iterations) with its own kernel path and roofline line.
"""
import argparse
import ctypes as C
import json
import math
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H = 30
OBS_DIM, ACT_DIM, HID = 6, 1, 64
MAC = (OBS_DIM + 1) * HID + HID * HID + HID * ACT_DIM          # 4608
FLOP_PER_ENV_STEP = 6 * MAC + 1500                             # SURVEY.md 8(d): MLP fwd+bwd + dynamics
BYTES_PER_ENV_STEP = (OBS_DIM * 4 + 4) / H                     # obs + done read once per sample
L2_BYTES = 126 * 1024 * 1024
GLOBAL_BATCH = 1 << 18


def alg_kwargs(env_id="pyth_idpendulum", algorithm="FHADP", hid=HID, act="gelu", obs_dim=OBS_DIM, act_dim=ACT_DIM, **kw):
    import numpy as np
    base = dict(env_id=env_id, algorithm=algorithm, seed=0, trainer="off_serial_trainer",
                use_gpu=True, action_type="continu", obsv_dim=obs_dim, action_dim=act_dim,
                action_high_limit=np.ones(act_dim, dtype=np.float32), action_low_limit=-np.ones(act_dim, dtype=np.float32),
                policy_func_name="FiniteHorizonPolicy" if algorithm.startswith("FHADP") else "DetermPolicy",
                policy_func_type="MLP", policy_hidden_sizes=[hid, hid],
                policy_hidden_activation=act, policy_act_distribution="default", policy_learning_rate=1e-4,
                value_func_name="StateValue", value_func_type="MLP", value_hidden_sizes=[hid, hid],
                value_hidden_activation=act, value_learning_rate=1e-3)
    base.update(kw)
    return base


class ClockSampler:
    """nvidia-smi sampling DURING the timed region (B200_PROFILING.md clocks line): one `nvidia-smi -lms 100`
    child process started before and killed after the region."""

    QUERY = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc = index, None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            time.sleep(0.4)          # let the first samples arrive before the timed region starts
        except Exception:
            self.proc = None

    def stop(self):
        rows = []
        if self.proc is not None:
            try:
                self.proc.terminate()
                out, _ = self.proc.communicate(timeout=5)
                rows = [[x.strip() for x in ln.split(",")] for ln in out.strip().splitlines() if ln.count(",") >= 6]
            except Exception:
                pass
        sm = [float(r[0]) for r in rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in rows if r[1].replace(".", "").isdigit()]
        pw = [float(r[2]) for r in rows if r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "reasons": sorted(reasons), "samples": len(rows)}


def usable_cores():
    """Host cores this process may really use: min(affinity, cgroup cpu quota)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(float(quota) / float(period))))
    except Exception:
        pass
    return n


def idp_init_batch(batch, seed):
    """Synthetic inputs of the GPU arm: the initial-state box of pyth_idpendulum (reference pyth_idpendulum.py:36-38,
    pyth_base_env.py:61-65): obs ~ U(-h, h), nobody done.  (The oracle is only imported by the CPU legs below.)"""
    import torch
    g = torch.Generator().manual_seed(seed)
    h = torch.tensor([5, 0.1, 0.1, 0.3, 0.3, 0.3])
    return {"obs": (torch.rand(batch, 6, generator=g, dtype=torch.float32) * 2 - 1) * h, "done": torch.zeros(batch)}


# ----------------------------------------------------------------------------------------------------------------
# CPU legs (the only places that import oracle/)
# ----------------------------------------------------------------------------------------------------------------
def port_update_rate(batch, steps, warmup, threads):
    """env-steps/s of the CPU oracle port: loss + autograd backward + Adam, as FHADP.local_update."""
    import torch
    torch.set_num_threads(threads)
    from oracle import gops_oracle as orc
    gen = torch.Generator().manual_seed(0)
    layers = [(w.requires_grad_(True), b.requires_grad_(True))
              for w, b in orc.init_mlp([OBS_DIM + 1, HID, HID, ACT_DIM], gen)]
    pol = orc.NetSpec(layers, "gelu", "linear", torch.ones(ACT_DIM), -torch.ones(ACT_DIM), time_input=True)
    env = orc.create_env_model("pyth_idpendulum", reward_scale=1.0)
    opt = torch.optim.Adam(pol.params(), lr=1e-4)
    data = orc.sample_inputs("pyth_idpendulum", batch, seed=1)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        opt.zero_grad()
        loss = orc.fhadp_loss(pol, env, data, H)
        loss.backward()
        opt.step()
        loss.item()
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    total = sum(times)
    return batch * H * len(times) / total, total / len(times)


def cpu_reference_leg(batch, steps, warmup):
    """The reference's own CPU implementation on the host cores: at all usable cores (the headline `value`) and at
    the reference's own default of 4 torch threads for `*serial*` trainers (init_args.py:29-35)."""
    cores = usable_cores()
    try:
        from oracle import ref_runner
        have_ref = ref_runner.available()
    except Exception:
        have_ref = False
    if have_ref:
        rate, sec = ref_runner.time_reference_updates(batch, steps, warmup, threads=cores, H=H)
        rate4, _ = ref_runner.time_reference_updates(batch, min(steps, 2), 1, threads=min(4, cores), H=H)
        kind, what = "reference", "unmodified gops FHADP.local_update (oracle/_ref via oracle/ref_shim.py)"
    else:
        rate, sec = port_update_rate(batch, steps, warmup, cores)
        rate4, _ = port_update_rate(batch, min(steps, 2), 1, min(4, cores))
        kind, what = "port", "oracle/gops_oracle.py (reference tree not reachable)"
    return {"value": rate, "unit": "env-steps/s", "cores": cores, "kind": kind, "sec_per_update": sec,
            "sample": f"B={batch}, H={H}, {steps} updates after {warmup} warm-up: {what}",
            "at_reference_default_threads": {"threads": min(4, cores), "value": rate4}}


def run_reference(args, rank):
    """Reference arm: the reference's own CPU implementation of the path, bounded sample per step."""
    if rank != 0:
        return
    cpu = cpu_reference_leg(args.cpu_batch, args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": "batched env-steps/sec (FHADP rollout+update)", "value": cpu["value"],
        "unit": "env-steps/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": cpu["sec_per_update"] * 1e3, "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"FHADP pyth_idpendulum H={H} FiniteHorizonPolicy[64,64] gelu",
                   "sample": f"batch {args.cpu_batch} per step on the host CPU ({cpu['cores']} threads)"},
        "cpu_baseline": cpu,
        "e2e": {"value": cpu["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------------------------
class Harness:
    def __init__(self, rank, local_rank, world):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank, self.world = rank, world
        self.dev = torch.device("cuda", local_rank)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def timed(self, alg, sets, steps, plan=None):
        """K steps between barrier+synchronize pairs; device time by CUDA events, max over ranks."""
        from gops_b200 import _lib
        torch = self.torch
        kms = []
        self.barrier()
        n0 = _lib.lib().gops_b200_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            alg.local_update(sets[i % len(sets)], i)
            if plan is not None:
                ms = C.c_float()
                _lib.check(_lib.lib().gops_b200_plan_last_kernel_ms(plan.handle, C.byref(ms)))
                kms.append(ms.value)
        e1.record()
        self.barrier()
        launches = _lib.lib().gops_b200_launch_count() - n0
        ms = torch.tensor([e0.elapsed_time(e1)], device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(ms, op=self.dist.ReduceOp.MAX)
        return float(ms.item()), kms, launches


def measure_c1(hx, batch_per_gpu, K, W, want_kernel=True, want_e2e=True, want_sync=True, dump_dir=None):
    """The C1 update on this rank's shard: returns dict(value-side timings, kernel ms, e2e timings, launches).
    With `dump_dir`, rank 0 writes the outputs of its last step there (dump_outputs)."""
    import torch
    from gops_b200.create_pkg.create_alg import create_alg
    from gops_b200 import _lib
    torch.manual_seed(0)                       # identical replicas on every rank
    alg = create_alg(**alg_kwargs(pre_horizon=H, reward_scale=1.0))
    alg.loss_lag = 1
    batch_bytes = batch_per_gpu * (OBS_DIM + 1) * 4
    n_sets = max(2, math.ceil(1.5 * L2_BYTES / batch_bytes))
    host_sets = [{k: v.pin_memory() for k, v in idp_init_batch(batch_per_gpu, seed=1000 * hx.rank + i).items()}
                 for i in range(n_sets)]
    dev_sets = [{k: v.to(hx.dev) for k, v in d.items()} for d in host_sets]
    out = {"batch_bytes": batch_bytes, "n_sets": n_sets}
    hx.timed(alg, dev_sets, W)                                    # warm-up (creates the plan)
    plan = next(iter(alg._plans.values()))
    if want_kernel:
        _lib.check(_lib.lib().gops_b200_plan_enable_timing(plan.handle, 1))
        hx.timed(alg, dev_sets, 1)
        _, out["kernel_ms"], _ = hx.timed(alg, dev_sets, K, plan=plan)
        _lib.check(_lib.lib().gops_b200_plan_enable_timing(plan.handle, 0))
        hx.timed(alg, dev_sets, 2)
    sampler = ClockSampler(hx.dev.index)
    sampler.start()
    out["ms_total"], _, out["launches"] = hx.timed(alg, dev_sets, K)
    out["clocks"] = sampler.stop()
    if want_sync:
        alg.loss_lag = 0
        hx.timed(alg, dev_sets, 2)
        out["ms_total_sync"], _, _ = hx.timed(alg, dev_sets, K)
        alg.loss_lag = 1
    if want_e2e:
        hx.timed(alg, host_sets, W)
        out["ms_e2e"], _, _ = hx.timed(alg, host_sets, K)
    info = (C.c_int32 * 4)()
    _lib.check(_lib.lib().gops_b200_plan_launch_info(plan.handle, info))
    out["launch"] = {"grid": info[0], "block": info[1], "tile_samples": info[2], "smem_bytes": info[3],
                     "kernel_path": alg.last_kernel_path()}
    if dump_dir and hx.rank == 0:
        dump_outputs(alg, dump_dir)
    return out


def dump_outputs(alg, out_dir):
    """What the last timed `local_update` left its caller, as float32 .npy files: the loss it computed (`loss.npy`;
    with loss_lag = 1 the returned tb_info still carries the step before), every policy gradient
    (`grad.<param>.npy`) and every updated policy parameter (`param.<param>.npy`).  All of it is a few KiB."""
    import numpy as np
    from gops_b200.utils.flat_params import GRAD_TAIL
    os.makedirs(out_dir, exist_ok=True)
    pol = alg.networks.policy
    tail = pol.flat_params.gbuf[-GRAD_TAIL:].detach().cpu().numpy()
    np.save(os.path.join(out_dir, "loss.npy"), tail[:1].astype(np.float32))
    for name, p in pol.named_parameters():
        np.save(os.path.join(out_dir, f"param.{name}.npy"), p.detach().cpu().numpy().astype(np.float32))
        np.save(os.path.join(out_dir, f"grad.{name}.npy"), p.grad.detach().cpu().numpy().astype(np.float32))


PATH_TEXT = {"tc": "tcgen05: BF16x3 UMMA for every dense product, weight gradients accumulate in TMEM",
             "mma": "mma.sync 3xTF32 (64-wide nets) / FP32 FFMA (256-wide nets)"}


def secondary_configs(hx, peaks, K=10, W=3):
    """The other BASELINE.json configurations on one GPU: one timed update each (device-resident inputs, L2 flushed by a
    256 MiB memset between iterations, per-iteration CUDA events), kernel-only time, path, roofline."""
    import numpy as np
    import torch
    from gops_b200.create_pkg.create_alg import create_alg
    from gops_b200 import _lib
    from gops_b200.trainer import device_sampler as ds
    dev = hx.dev
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    burst = peaks.get("bf16_tflops", 1700.0)
    n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
    ffma_peak = n_sm * 128 * 2 * peaks.get("sm_max_mhz", 1965.0) * 1e6 / 1e12
    rows = []

    def run(name, kw, data, horizon, flop_pev, flop_pim, set_params=None):
        torch.manual_seed(0)
        alg = create_alg(**kw)
        if set_params:
            alg.set_parameters(set_params)
        infadp = kw["algorithm"] == "INFADP"
        B = data["obs"].shape[0]
        for phase in ((0, 1) if infadp else (0,)):
            it_of = (lambda i: 2 * i + phase) if infadp else (lambda i: i)
            for i in range(W):
                alg.local_update(data, it_of(i))
            torch.cuda.synchronize()
            plan = next(reversed(alg._plans.values()))
            _lib.check(_lib.lib().gops_b200_plan_enable_timing(plan.handle, 1))
            tot, kms = 0.0, []
            for i in range(K):
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                alg.local_update(data, it_of(i))
                e1.record()
                torch.cuda.synchronize()
                tot += e0.elapsed_time(e1)
                ms = C.c_float()
                _lib.check(_lib.lib().gops_b200_plan_last_kernel_ms(plan.handle, C.byref(ms)))
                kms.append(ms.value)
            _lib.check(_lib.lib().gops_b200_plan_enable_timing(plan.handle, 0))
            path = alg.last_kernel_path()
            flop = (flop_pev if phase == 0 else flop_pim) if infadp else flop_pim
            k_ms = statistics.mean(kms)
            ach = B * horizon * flop / (k_ms * 1e-3) / 1e12
            wide_ffma = kw["policy_hidden_sizes"][0] > 64 and path != "tc"
            peak = ffma_peak if wide_ffma else burst / 6.0
            rows.append({
                "name": name + ((" PEV" if phase == 0 else " PIM") if infadp else ""), "batch": B, "horizon": horizon,
                "value": B * horizon * K / (tot * 1e-3), "unit": "env-steps/s", "ms_per_step": tot / K,
                "kernel_ms": k_ms, "kernel_path": path,
                "roofline": {"bound": "fp32_ffma" if wide_ffma else "tensor", "achieved": ach, "peak": peak,
                             "unit": "TFLOP/s", "frac": ach / peak, "algorithmic_flop_per_env_step": flop}})
        del alg

    # C1 at the reference's own CPU-runnable size
    run("C1 FHADP idpendulum B=256", alg_kwargs(pre_horizon=H, reward_scale=1.0),
        {k: v.to(dev) for k, v in idp_init_batch(256, 5).items()}, H, None, FLOP_PER_ENV_STEP)
    # C2 INFADP veh3dofconti, B=4096, P=10, forward_step=10, [64,64] relu
    d = ds.sample_veh3dofconti(4096, 10, dev, seed=3)
    run("C2 INFADP veh3dofconti B=4096", alg_kwargs("pyth_veh3dofconti", "INFADP", 64, "relu", 46, 2, pre_horizon=10,
                                                    policy_learning_rate=1e-3), d, 10, 2.0e4, 4.6e4)
    # C3 FHADP veh3dof_tracking P=H=60 [256,256] elu, one GPU's shard (8192) of the 65 536 batch
    d = ds.sample_veh3dof_tracking(8192, 60, dev, seed=4)
    run("C3 FHADP veh3dof_tracking H=60 [256,256] B=8192/GPU",
        alg_kwargs("veh3dof_tracking", "FHADP", 256, "elu", 6 + 4 * 60, 2, pre_horizon=60, policy_learning_rate=1e-3),
        d, 60, None, 7.8e5)
    # C4 DSAC idpendulum, [256,256,256] gelu, minibatch 8192 from the on-device replay buffer: one update = 5 network
    # evaluations + 3 back-propagations on the layer-wise tcgen05 MLP (2.7 MFLOP algorithmic per sample, SURVEY 8(f) N1)
    try:
        from gops_b200.trainer.device_buffer import DeviceReplayBuffer
        torch.manual_seed(0)
        dkw = alg_kwargs("pyth_idpendulum", "DSAC", 256, "gelu", 6, 1, policy_func_name="StochaPolicy",
                         policy_hidden_sizes=[256, 256, 256], value_hidden_sizes=[256, 256, 256],
                         policy_act_distribution="TanhGaussDistribution", policy_min_log_std=-20, policy_max_log_std=1,
                         value_func_name="ActionValueDistri", value_learning_rate=3e-4, policy_learning_rate=3e-4,
                         alpha_learning_rate=5e-5, gamma=0.99, tau=0.005, auto_alpha=True, alpha=0.2, delay_update=2,
                         TD_bound=10, bound=True)
        dsac = create_alg(**dkw)
        buf = DeviceReplayBuffer(6, 1, 1 << 20, device=dev, seed=1)
        o = ds.sample_idpendulum(1 << 18, dev, seed=2)["obs"]
        buf.add_batch({"obs": o, "act": torch.rand(1 << 18, 1, device=dev) * 2 - 1, "rew": torch.randn(1 << 18, device=dev),
                       "obs2": o + 0.01 * torch.randn_like(o), "done": torch.zeros(1 << 18, device=dev)})
        MB = 8192
        for i in range(W):
            dsac.local_update(buf.sample_batch(MB), i)
        torch.cuda.synchronize()
        n0 = _lib.lib().gops_b200_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(K):
            dsac.local_update(buf.sample_batch(MB), i)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / K
        flop = 2.7e6
        ach = MB * flop / (ms * 1e-3) / 1e12
        rows.append({"name": "C4 DSAC idpendulum [256,256,256] minibatch 8192 (on-device replay buffer)", "batch": MB,
                     "value": MB / (ms * 1e-3), "unit": "samples/s", "ms_per_step": ms, "kernel_path": "tc",
                     "launches_per_update": (_lib.lib().gops_b200_launch_count() - n0) / K,
                     "roofline": {"bound": "tensor", "achieved": ach, "peak": burst / 6.0, "unit": "TFLOP/s",
                                  "frac": ach / (burst / 6.0), "algorithmic_flop_per_sample": flop}})
        del dsac, buf
    except Exception as e:      # a secondary config must never take the bench down
        rows.append({"name": "C4 DSAC", "error": repr(e)[:300]})
    # C5 INFADP LQ s4a2 batch sweep
    for e in (10, 12, 14, 16, 18, 20):
        B = 1 << e
        d = ds.sample_lq(B, "s4a2", dev, seed=e)
        run(f"C5 INFADP lq s4a2 B=2^{e}",
            alg_kwargs("pyth_lq", "INFADP", 64, "gelu", 4, 2, lq_config="s4a2", reward_scale=1.0, reward_shift=0.0,
                       policy_learning_rate=8e-4, value_learning_rate=3e-4), d, 10, 1.25e4, 2.9e4)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"])
    ap.add_argument("--global-batch", type=int, default=GLOBAL_BATCH)
    ap.add_argument("--cpu-batch", type=int, default=32768)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true")
    ap.add_argument("--no-eager", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the loss, policy gradient and updated policy parameters of the "
                         "last step as DIR/<name>.npy (inputs and initial weights are seeded: same arguments, same inputs)")
    args = ap.parse_args()

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    torch.set_num_threads(usable_cores())      # the box reports 128 cpus under a 16-core cgroup quota
    import torch.distributed as dist
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    hx = Harness(rank, local_rank, world)
    W, K = max(args.warmup, 3), args.steps

    Bglobal = args.global_batch
    per_gpu_strong = Bglobal // world
    main_b = per_gpu_strong if args.scaling == "strong" else Bglobal
    m = measure_c1(hx, main_b, K, W, dump_dir=args.dump_outputs)
    other = None
    if world > 1:      # the other scaling mode, same run (value side only)
        other_b = Bglobal if args.scaling == "strong" else per_gpu_strong
        other = measure_c1(hx, other_b, K, W, want_kernel=True, want_e2e=False, want_sync=False)
        other["batch_per_gpu"] = other_b

    if rank == 0:
        peaks = {}
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                peaks = json.load(f)
        except Exception:
            pass
        peak_src = "MEASURED_PEAKS.json" if peaks else "fallback (B200_PROFILING.md)"
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        burst = peaks.get("bf16_tflops", 1700.0)
        sustained = peaks.get("bf16_tflops_sustained", 1400.0)
        env_steps = main_b * world * H
        value = env_steps * K / (m["ms_total"] * 1e-3)
        e2e = env_steps * K / (m["ms_e2e"] * 1e-3)
        k_ms = statistics.mean(m["kernel_ms"])
        clocks = m["clocks"]
        sm_mhz = clocks["sm_mhz"] or peaks.get("sm_max_mhz", 1965.0)
        n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
        fp32_peak = n_sm * 128 * 2 * sm_mhz * 1e6 / 1e12
        ach_tflops = main_b * H * FLOP_PER_ENV_STEP / (k_ms * 1e-3) / 1e12
        ach_gbs = main_b * H * BYTES_PER_ENV_STEP / (k_ms * 1e-3) / 1e9
        traffic = None
        tfile = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tfile):
            try:
                traffic = json.load(open(tfile)).get("rollout_kernel_dram_bytes_per_launch")
            except Exception:
                pass
        path = m["launch"]["kernel_path"]
        # FP32-accurate tensor roof: BF16x3 = six bf16 MMAs per product (tc path), 3xTF32 = three TF32 MMAs at half the
        # bf16 rate (mma path): both = bf16 peak / 6.  The kernel is event-timed alone -> burst peak.
        tens_roof = burst / 6.0
        m["launch"]["kernel_path_text"] = PATH_TEXT.get(path, path)
        roof = {"bound": "tensor", "achieved": ach_tflops, "peak": tens_roof, "unit": "TFLOP/s",
                "frac": ach_tflops / tens_roof, "traffic": traffic,
                "peak_source": f"{peak_src} bf16_tflops (burst: kernel timed alone) / 6 (six bf16 MMAs per FP32-accurate product)",
                "frac_of_sustained_peak": ach_tflops / (sustained / 6.0),
                "kernel_ms": k_ms, "kernel_share_of_step": k_ms * K / m["ms_total"],
                "non_kernel_ms_per_step": m["ms_total"] / K - k_ms,
                "algorithmic_flop_per_env_step": FLOP_PER_ENV_STEP, "algorithmic_bytes_per_env_step": BYTES_PER_ENV_STEP,
                "fp32_ffma": {"achieved_tflops": ach_tflops, "peak_tflops": fp32_peak, "frac": ach_tflops / fp32_peak,
                              "of": f"{n_sm} SM x 128 lanes x 2 x {sm_mhz:.0f} MHz sampled under load"},
                "hbm": {"achieved_gbs": ach_gbs, "peak_gbs": hbm_peak, "frac": ach_gbs / hbm_peak, "of": peak_src},
                "tensor_bf16": {"achieved_tflops": ach_tflops, "peak_tflops": burst, "frac": ach_tflops / burst,
                                "of": peak_src + " bf16 burst"},
                "launch": m["launch"]}
        cpu = None
        if not args.no_cpu_baseline and world == 1:
            cpu = cpu_reference_leg(args.cpu_batch, 3, 1)
        eager = None
        if not args.no_eager and world == 1:
            try:
                from oracle import ref_runner
                if ref_runner.available():
                    eb = 1 << 16
                    rate, sec = ref_runner.time_reference_updates(eb, 3, 2, H=H, device=f"cuda:{local_rank}")
                    eager = {"value": rate, "unit": "env-steps/s", "ms_per_step": sec * 1e3,
                             "what": f"unmodified gops FHADP.local_update with use_gpu=True (PyTorch eager) on this GPU, "
                                     f"B={eb}, H={H}, 3 updates after 2 warm-ups (oracle/_ref)"}
                    torch.cuda.empty_cache()
            except Exception as e:          # the eager leg must never take the bench down
                eager = {"unavailable": repr(e)[:200]}
        configs = None
        if not args.no_configs and world == 1:
            try:
                configs = secondary_configs(hx, peaks)
            except Exception as e:
                configs = [{"error": repr(e)[:300]}]
        line = {
            "metric": "batched env-steps/sec (FHADP rollout+update)", "value": value, "unit": "env-steps/s",
            "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": m["ms_total"] / K, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"FHADP pyth_idpendulum H={H} FiniteHorizonPolicy[64,64] gelu, "
                                   f"batch {main_b} per GPU (global {main_b * world})",
                       "parallelism": f"dp{world}", "l2_policy": f"{m['n_sets']} rotating input batches "
                       f"({m['n_sets'] * m['batch_bytes'] / 2**20:.0f} MiB total > L2)",
                       "loss_readback": "pipelined: every step's 4-float tail is copied to pinned memory and read by "
                                        "the host one step later (alg.loss_lag=1); sync_loss = same with loss_lag=0"},
            "clocks": clocks, "roofline": roof, "cpu_baseline": cpu,
            "e2e": {"value": e2e, "unit": "env-steps/s", "h2d_bytes_per_step": m["batch_bytes"], "d2h_bytes_per_step": 16,
                    "ms_per_step": m["ms_e2e"] / K},
            "sync_loss": {"value": env_steps * K / (m["ms_total_sync"] * 1e-3), "ms_per_step": m["ms_total_sync"] / K},
            "gpu_launches": m["launches"],
        }
        if other is not None:
            ob = other["batch_per_gpu"]
            line["weak" if args.scaling == "strong" else "strong"] = {
                "value": ob * world * H * K / (other["ms_total"] * 1e-3), "unit": "env-steps/s",
                "batch_per_gpu": ob, "global_batch": ob * world, "ms_per_step": other["ms_total"] / K,
                "kernel_ms": statistics.mean(other["kernel_ms"]), "launch": other["launch"]}
        if eager is not None:
            line["gpu_eager_baseline"] = eager
        if configs is not None:
            line["configs"] = configs
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
