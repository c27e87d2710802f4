"""The JRPO oracle (tests/jrpo_oracle.py: the multi-agent oracle of oracle/loop_ma.py with the joint-action loss,
cfg.use_joint_action_loss) against traces of the unmodified reference running examples/mpe/mpe_jrpo.yaml on
simple_spread (4 envs x 3 agents, T = 25, GRU, ValueNorm, advantage normalisation), recorded by tools/gen_golden_jrpo.py:
  trace_mpe_jrpo      data_chunk_length 2, one minibatch: chunks over g = n*T + t straddle two envs
  trace_mpe_jrpo_mb2  data_chunk_length 5, two minibatches: ValueNorm / loss weights from per-minibatch agent-0 moments
Same bars as the MAPPO traces in tests/test_oracle_loop.py."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from oracle import TRACE_THREADS


@pytest.fixture(autouse=True)
def trace_threads():
    """Replay with the thread count the traces were recorded with (bit-exact results depend on it)."""
    prev = torch.get_num_threads()
    torch.set_num_threads(TRACE_THREADS)
    yield
    torch.set_num_threads(prev)


@pytest.mark.parametrize("tag,chunks", [("mpe_jrpo", 50), ("mpe_jrpo_mb2", 20)])
def test_oracle_jrpo_reproduces_reference_trace(tag, chunks):
    import jrpo_oracle

    d = np.load(os.path.join(GOLDEN, f"trace_{tag}.npz"), allow_pickle=True)
    cfg = jrpo_oracle.cfg_from_flags(str(d["meta/flags"]))
    assert cfg.use_joint_action_loss and cfg.use_recurrent_policy
    tr = jrpo_oracle.JRPOTrainer(cfg, "simple_spread", int(d["meta/env_num"]))
    for mk, prm in (("policy", tr.pol), ("critic", tr.cri)):
        for k, v in prm.items():
            np.testing.assert_allclose(v.detach().numpy(), d[f"init/{mk}.{k}"], rtol=0, atol=1e-6, err_msg=k)
            v.data.copy_(torch.from_numpy(d[f"init/{mk}.{k}"]))
    for it in range(int(d["meta/iters"])):
        tr.rollout()
        b = tr.buf
        assert np.array_equal(b.actions, d[f"it{it}/actions"])
        assert np.array_equal(b.policy_obs, d[f"it{it}/policy_obs"])
        assert np.array_equal(b.rewards, d[f"it{it}/rewards"])
        assert np.array_equal(b.masks, d[f"it{it}/masks"])
        np.testing.assert_allclose(b.rnn_states, d[f"it{it}/rnn_states"], rtol=0, atol=1e-5)
        np.testing.assert_allclose(b.rnn_states_critic, d[f"it{it}/rnn_states_critic"], rtol=0, atol=1e-5)
        tr.compute_returns()
        np.testing.assert_allclose(b.value_preds, d[f"it{it}/value_preds"], rtol=0, atol=1e-5)
        updates, perms = tr.train()
        assert perms.shape == (cfg.ppo_epoch, chunks)   # one randperm(N*T // L) per epoch
        assert np.array_equal(perms, d[f"it{it}/perms"])
        np.testing.assert_allclose(tr.last_adv, d[f"it{it}/advantages"], rtol=1e-4, atol=1e-5)
        np.testing.assert_allclose(updates, d[f"it{it}/updates"], rtol=2e-4, atol=2e-6)
        tr.after_update()
        for mk, prm in (("policy", tr.pol), ("critic", tr.cri)):
            for k, v in prm.items():
                np.testing.assert_allclose(v.detach().numpy(), d[f"it{it}/params/{mk}.{k}"], rtol=2e-4, atol=2e-6, err_msg=k)
        np.testing.assert_allclose(tr.vn.state(), d[f"it{it}/vn_after_update"], rtol=1e-6)
