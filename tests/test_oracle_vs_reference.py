"""CPU: the oracle restatement against the unmodified reference's FHADP idpendulum update on inputs the other goldens do
not cover (tests/golden/fresh_fhadp_idp_*.npz, oracle/make_golden.py run_fresh_fhadp): the reference's own initial
weights, a ninth of the batch arriving done, the loss and policy gradients its `local_update` produced."""
import numpy as np
import pytest
import torch

from golden_util import load, rel_l2
from oracle import gops_oracle as orc


@pytest.mark.parametrize("H,B,seed", [(30, 64, 101), (7, 33, 102)])
def test_fhadp_idpendulum_fresh_inputs(H, B, seed):
    torch.set_num_threads(4)
    rec = load(f"fresh_fhadp_idp_h{H}_b{B}_s{seed}")
    data = orc.sample_inputs("pyth_idpendulum", B, seed=seed)
    data["done"][::9] = 1.0
    np.testing.assert_array_equal(data["obs"].numpy(), rec["in_obs"])      # the oracle's sampler is unchanged
    np.testing.assert_array_equal(data["done"].numpy(), rec["in_done"])
    layers = [(torch.tensor(rec[f"init/policy.pi.{j}.weight"]).requires_grad_(True),
               torch.tensor(rec[f"init/policy.pi.{j}.bias"]).requires_grad_(True)) for j in (0, 2, 4)]
    pol = orc.NetSpec(layers, "gelu", "linear", torch.ones(1), -torch.ones(1), time_input=True)
    loss = orc.fhadp_loss(pol, orc.create_env_model("pyth_idpendulum", reward_scale=1.0), data, H)
    loss.backward()
    ref_loss = float(rec["loss"])
    assert abs(loss.item() - ref_loss) <= 2e-6 * max(1.0, abs(ref_loss))
    ref_g = [rec[f"grad/policy.pi.{j}.{w}"] for j in (0, 2, 4) for w in ("weight", "bias")]
    assert rel_l2([p.grad.numpy() for p in pol.params()], ref_g) < 1e-5
