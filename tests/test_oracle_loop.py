"""The full-iteration oracle (oracle/loop.py) against traces of the unmodified reference
(tests/golden/trace_*.npz, produced by oracle/gen_golden.py): same seeds -> same actions
(bit-exact), same rollout buffer, same losses / grad norms and same parameters."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from oracle import TRACE_THREADS, loop


@pytest.fixture(autouse=True)
def trace_threads():
    """Replay with the thread count the traces were recorded with (bit-exact results depend on it)."""
    prev = torch.get_num_threads()
    torch.set_num_threads(TRACE_THREADS)
    yield
    torch.set_num_threads(prev)


def _params(tr):
    out = {}
    for mk, d in (("policy", tr.pol), ("critic", tr.cri)):
        for k, v in d.items():
            out[f"{mk}.{k}"] = v.detach().numpy()
    return out


@pytest.mark.parametrize("tag,env_id", [("cartpole", "CartPole-v1"), ("cartpole_c1", "CartPole-v1"),
                                        ("identity_continuous", "IdentityEnvcontinuous")])
def test_oracle_reproduces_reference_trace(tag, env_id):
    d = np.load(os.path.join(GOLDEN, f"trace_{tag}.npz"), allow_pickle=True)
    cfg = loop.cfg_from_flags(str(d["meta/flags"]))
    tr = loop.Trainer(cfg, env_id, int(d["meta/env_num"]))
    for k, v in _params(tr).items():
        assert np.array_equal(v, d[f"init/{k}"]), k  # same init stream as the reference
    for it in range(int(d["meta/iters"])):
        tr.rollout()
        b = tr.buf
        assert np.array_equal(b.actions, d[f"it{it}/actions"])  # bit-exact sampling
        assert np.array_equal(b.obs, d[f"it{it}/policy_obs"])   # bit-exact trajectories
        assert np.array_equal(b.rewards, d[f"it{it}/rewards"])
        assert np.array_equal(b.masks, d[f"it{it}/masks"])
        np.testing.assert_allclose(b.action_log_probs, d[f"it{it}/action_log_probs"], rtol=0, atol=1e-6)
        tr.compute_returns()
        np.testing.assert_allclose(b.value_preds, d[f"it{it}/value_preds"], rtol=0, atol=1e-5)
        np.testing.assert_allclose(b.returns[:-1], d[f"it{it}/returns"][:-1], rtol=1e-5, atol=1e-5)
        updates, perms = tr.train()
        assert np.array_equal(perms, d[f"it{it}/perms"])
        np.testing.assert_allclose(tr.last_adv, d[f"it{it}/advantages"], rtol=1e-4, atol=1e-5)
        np.testing.assert_allclose(updates, d[f"it{it}/updates"], rtol=1e-4, atol=1e-6)
        tr.after_update()
        for k, v in _params(tr).items():
            np.testing.assert_allclose(v, d[f"it{it}/params/{k}"], rtol=1e-4, atol=1e-6, err_msg=k)
        np.testing.assert_allclose(tr.vn.state(), d[f"it{it}/vn_after_update"], rtol=1e-6)


@pytest.mark.parametrize("tag,env_id", [("mpe_mlp", "simple_spread"), ("mpe_gru", "simple_spread"), ("cartpole_gru", "CartPole-v1"),
                                        ("mpe_naive_gru", "simple_spread")])
def test_multi_agent_oracle_reproduces_reference_trace(tag, env_id):
    """MAPPO on simple_spread (3 agents, shared nets; feed-forward and GRU + chunked BPTT with
    data_chunk_length 2) and single-agent recurrent PPO on CartPole-v1 (episodes ending inside chunks of 4,
    two minibatches) vs the unmodified reference."""
    from oracle import loop_ma

    d = np.load(os.path.join(GOLDEN, f"trace_{tag}.npz"), allow_pickle=True)
    cfg = loop.cfg_from_flags(str(d["meta/flags"]))
    tr = loop_ma.MATrainer(cfg, env_id, int(d["meta/env_num"]))
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
        if cfg.use_recurrent_policy or cfg.use_naive_recurrent_policy:
            np.testing.assert_allclose(b.rnn_states, d[f"it{it}/rnn_states"], rtol=0, atol=1e-5)
            np.testing.assert_allclose(b.rnn_states_critic, d[f"it{it}/rnn_states_critic"], rtol=0, atol=1e-5)
        tr.compute_returns()
        np.testing.assert_allclose(b.value_preds, d[f"it{it}/value_preds"], rtol=0, atol=1e-5)
        updates, perms = tr.train()
        assert np.array_equal(perms, d[f"it{it}/perms"])
        np.testing.assert_allclose(tr.last_adv, d[f"it{it}/advantages"], rtol=1e-4, atol=1e-5)
        np.testing.assert_allclose(updates, d[f"it{it}/updates"], rtol=2e-4, atol=2e-6)
        tr.after_update()
        for mk, prm in (("policy", tr.pol), ("critic", tr.cri)):
            for k, v in prm.items():
                np.testing.assert_allclose(v.detach().numpy(), d[f"it{it}/params/{mk}.{k}"], rtol=2e-4, atol=2e-6, err_msg=k)


FLAG_TAGS = ["a2c", "dual_clip", "no_huber", "no_value_clip", "proper_time_limits", "no_gae", "no_valuenorm", "adv_norm_no_masks",
             "no_grad_clip_wd", "popart"]


@pytest.mark.parametrize("tag", FLAG_TAGS)
def test_oracle_reproduces_reference_flag_variants(tag):
    """Every loss / return option branch of the hot path (A2C, dual clip, MSE value loss, unclipped value loss,
    proper time limits, plain discounted returns, no ValueNorm, advantage normalisation without active masks,
    no gradient clip + weight decay + tanh) pinned to a trace of the unmodified reference
    (oracle/gen_golden.py FLAG_VARIANTS)."""
    d = np.load(os.path.join(GOLDEN, f"trace_flag_{tag}.npz"), allow_pickle=True)
    cfg = loop.cfg_from_flags(str(d["meta/flags"]))
    cfg.a2c = str(d["meta/algo"]) == "a2c"
    if cfg.a2c:
        cfg.num_mini_batch = 1   # A2CAlgorithm.__init__ (a2c.py:37)
    tr = loop.Trainer(cfg, "CartPole-v1", int(d["meta/env_num"]))
    for k, v in _params(tr).items():
        assert np.array_equal(v, d[f"init/{k}"]), k
    for it in range(int(d["meta/iters"])):
        tr.rollout()
        b = tr.buf
        assert np.array_equal(b.actions, d[f"it{it}/actions"])
        assert np.array_equal(b.obs, d[f"it{it}/policy_obs"])
        tr.compute_returns()
        np.testing.assert_allclose(b.value_preds, d[f"it{it}/value_preds"], rtol=0, atol=1e-5)
        np.testing.assert_allclose(b.returns[:-1], d[f"it{it}/returns"][:-1], rtol=1e-5, atol=1e-5)
        updates, perms = tr.train()
        assert np.array_equal(perms, d[f"it{it}/perms"])
        np.testing.assert_allclose(updates, d[f"it{it}/updates"], rtol=1e-4, atol=1e-6)
        tr.after_update()
        for k, v in _params(tr).items():
            np.testing.assert_allclose(v, d[f"it{it}/params/{k}"], rtol=1e-4, atol=1e-6, err_msg=k)


OPTION_TAGS = ["lr_decay", "act_leaky_relu", "act_elu", "coefs", "lrs_wd", "gamma_lambda"]


@pytest.mark.parametrize("tag", OPTION_TAGS)
def test_oracle_reproduces_reference_option_values(tag):
    """Option VALUES beyond the branch switches (oracle/gen_golden.py ORACLE_VARIANTS): the linear lr schedule
    (rl_driver.py:159-161, 3 iterations so the rate changes twice), LeakyReLU / ELU trunks, non-default clip / entropy /
    value-loss / huber / grad-norm coefficients, separate lrs + weight decay, gamma / lambda with advantage
    normalisation.  These are the settings of the device-vs-oracle flag matrix (tests/test_ppo_flags_cuda.py) and of the
    device lr-schedule test: with the oracle pinned here, those chains end at the executed reference."""
    d = np.load(os.path.join(GOLDEN, f"trace_opt_{tag}.npz"), allow_pickle=True)
    cfg = loop.cfg_from_flags(str(d["meta/flags"]))
    iters = int(d["meta/iters"])
    tr = loop.Trainer(cfg, "CartPole-v1", int(d["meta/env_num"]))
    for k, v in _params(tr).items():
        assert np.array_equal(v, d[f"init/{k}"]), k
    for it in range(iters):
        tr.rollout()
        b = tr.buf
        assert np.array_equal(b.actions, d[f"it{it}/actions"])
        assert np.array_equal(b.obs, d[f"it{it}/policy_obs"])
        if cfg.use_linear_lr_decay:
            tr.lr_decay(it, iters)
        tr.compute_returns()
        np.testing.assert_allclose(b.value_preds, d[f"it{it}/value_preds"], rtol=0, atol=1e-5)
        np.testing.assert_allclose(b.returns[:-1], d[f"it{it}/returns"][:-1], rtol=1e-5, atol=1e-5)
        updates, perms = tr.train()
        assert np.array_equal(perms, d[f"it{it}/perms"])
        np.testing.assert_allclose(updates, d[f"it{it}/updates"], rtol=1e-4, atol=1e-6)
        tr.after_update()
        for k, v in _params(tr).items():
            np.testing.assert_allclose(v, d[f"it{it}/params/{k}"], rtol=1e-4, atol=1e-6, err_msg=k)
    if tag == "lr_decay":   # the schedule really moved the parameters: the last step is a third of the first
        assert abs(tr.opt_p.param_groups[0]["lr"] - cfg.lr * (1 - 2 / 3)) < 1e-12


def test_oracle_reproduces_reference_share_model_trace():
    """cfg.use_share_model: PolicyValueNetwork (obs_prep -> common -> {act, v_out}, policy_value_network.py:33-174), one
    optimiser, both losses into the same gradients, two clip_grad_norm_ over all parameters (ppo.py:120-141)."""
    d = np.load(os.path.join(GOLDEN, "trace_share_model.npz"), allow_pickle=True)
    cfg = loop.cfg_from_flags(str(d["meta/flags"]))
    assert cfg.use_share_model
    tr = loop.Trainer(cfg, "CartPole-v1", int(d["meta/env_num"]))
    for k, v in tr.pol.items():
        assert np.array_equal(v.detach().numpy(), d[f"init/model.{k}"]), k
    for it in range(int(d["meta/iters"])):
        tr.rollout()
        b = tr.buf
        assert np.array_equal(b.actions, d[f"it{it}/actions"])
        assert np.array_equal(b.obs, d[f"it{it}/policy_obs"])
        tr.compute_returns()
        np.testing.assert_allclose(b.value_preds, d[f"it{it}/value_preds"], rtol=0, atol=1e-5)
        updates, perms = tr.train()
        assert np.array_equal(perms, d[f"it{it}/perms"])
        np.testing.assert_allclose(updates, d[f"it{it}/updates"], rtol=1e-4, atol=1e-6)
        tr.after_update()
        for k, v in tr.pol.items():
            np.testing.assert_allclose(v.detach().numpy(), d[f"it{it}/params/model.{k}"], rtol=1e-4, atol=1e-6, err_msg=k)
