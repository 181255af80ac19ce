"""INTEGRATION.md's binding: `create_alg.register` puts the fused B200 algorithm into a GOPS-style registry, the factory
builds it from the reference's C1 keyword arguments, and three OffSerialTrainer-style steps (off_serial_trainer.py:79-105:
sample_batch -> .cuda() -> alg.local_update) replay what the unmodified reference did on the same minibatches
(tests/golden/trainer_steps_fhadp_idp_h30.npz, oracle/make_golden.py run_trainer_steps): the reference's initial
state_dict, the minibatches its own ReplayBuffer sampled, its loss at every step and its policy's actions afterwards."""
import numpy as np
import pytest
import torch

from golden_util import load
from oracle import ref_runner

pytestmark = pytest.mark.gpu


def test_register_binding_and_three_trainer_steps():
    from gops_b200.algorithm import fhadp as b200_fhadp
    from gops_b200.create_pkg import create_alg as ca

    rec = load("trainer_steps_fhadp_idp_h30")
    ref_sd = {k[len("init/"):]: torch.from_numpy(v) for k, v in rec.items() if k.startswith("init/")}
    kw = ref_runner.c1_kwargs(30)
    saved = ca.registry["FHADP"]
    try:
        ca.register("FHADP", b200_fhadp.FHADP, b200_fhadp.ApproxContainer)   # INTEGRATION.md section 1
        alg = ca.create_alg(**dict(kw, use_gpu=True))
    finally:
        ca.registry["FHADP"] = saved
    assert type(alg).__module__ == "gops_b200.algorithm.fhadp"
    alg.load_state_dict(ref_sd)                                          # identical start (reference checkpoint keys)

    for it in range(3):
        prefix = f"it{it}/batch/"
        replay = {k[len(prefix):]: torch.from_numpy(v) for k, v in rec.items() if k.startswith(prefix)}
        gpu_batch = {k: v.cuda() for k, v in replay.items()}          # off_serial_trainer.py:92-94
        alg.networks.train()
        tb = alg.local_update(gpu_batch, it)
        alg.networks.eval()
        assert set(tb) >= {"Loss/Actor loss-RL iter", "Time/Algorithm time [ms]-RL iter"}
        ref_loss = float(rec[f"it{it}/loss"])
        assert abs(tb["Loss/Actor loss-RL iter"] - ref_loss) <= (1e-4 if it == 0 else 5e-4) * max(1.0, abs(ref_loss))
    # the sampler / evaluator side: the trained policies act alike
    o = torch.from_numpy(rec["act_obs"])
    a = alg.networks.policy(o.cuda(), 1).cpu()
    assert float((a - torch.from_numpy(rec["act"])).abs().max()) < 1e-3
    # and the checkpoint the fused algorithm writes loads back into the reference (a strict load: same keys and shapes)
    sd = alg.state_dict()
    assert set(sd) == set(ref_sd)
    for k, v in ref_sd.items():
        assert sd[k].shape == v.shape, k
