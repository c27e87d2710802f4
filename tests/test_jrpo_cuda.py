"""Joint-action PPO (JRPO, cfg.use_joint_action_loss; examples/mpe/mpe_jrpo.yaml) on the device: the recurrent update
over recurrent_generator_v3 chunks (g = n*T + t, all agents of a step together), the joint log-prob ratio with agent 0's
advantage, the agent-0 critic and the all-agent entropy.

Pinned to traces of the unmodified reference (tests/golden/trace_mpe_jrpo*.npz, which also pin the torch oracle in
tests/test_oracle_jrpo.py) with the bars of tests/test_gru_cuda.py: losses 2e-4 relative, parameters 2e-3,
ValueNorm 1e-5."""
import os
import re

import numpy as np
import pytest

from conftest import GOLDEN

pytestmark = pytest.mark.gpu

JRPO = ["--episode_length", "25", "--lr", "7e-4", "--critic_lr", "7e-4", "--ppo_epoch", "2", "--use_recurrent_policy", "true",
        "--use_joint_action_loss", "true", "--use_valuenorm", "true", "--use_adv_normalize", "true"]


@pytest.mark.parametrize("tag", ["mpe_jrpo", "mpe_jrpo_mb2"])
def test_jrpo_matches_reference_trace(cuda, tag):
    """Chunks of 2 that straddle two envs with one minibatch, and chunks of 5 with two minibatches (per-minibatch
    agent-0 ValueNorm moments and loss weights)."""
    from test_gru_cuda import check_recurrent_trace

    check_recurrent_trace(tag, "simple_spread")


def _train(env_id, N, flags, iters, train_algo_class=None):
    from openrl_b200.utils.logger import Logger
    from test_rollout_cuda import _product

    cfg, env, net, agent = _product(env_id, N, flags)
    logger = Logger(quiet=True)
    kw = {} if train_algo_class is None else {"train_algo_class": train_algo_class}
    agent.train(total_time_steps=cfg.episode_length * N * iters, logger=logger, **kw)
    logs = [h[1] for h in logger.history if "value_loss" in h[1]]
    params = {f"{mk}.{k}": v.detach().cpu().numpy().copy()
              for mk in ("policy", "critic") for k, v in net.module.models[mk].state_dict().items()}
    return logs, params, agent


@pytest.mark.parametrize("mini", [1, 2])
def test_jrpo_with_one_agent_is_recurrent_ppo(cuda, mini):
    """With A = 1 the v3 flattening n*T + t is the recurrent generator's (n*A + a)*T + t and every agent-0 reduction is
    the identity: CartPole-v1 GRU in parity mode with and without the joint-action loss trains the same parameters.
    The update kernels differ only in how many chunks a warp holds, which does not change any per-row arithmetic, and
    the gradient reductions are deterministic, so the parameters agree bit for bit; the logged metrics are float
    atomics over a different number of CTAs."""
    base = ["--seed", "0", "--episode_length", "32", "--ppo_epoch", "2", "--num_mini_batch", str(mini),
            "--use_recurrent_policy", "true", "--data_chunk_length", "4"]
    logs0, p0, _ = _train("CartPole-v1", 8, base, 2)
    logs1, p1, _ = _train("CartPole-v1", 8, base + ["--use_joint_action_loss", "true"], 2)
    assert len(logs0) == len(logs1) == 2
    for a, b in zip(logs0, logs1):
        for k in a:
            np.testing.assert_allclose(b[k], a[k], rtol=2e-4, atol=1e-6, err_msg=k)
    for k in p0:
        np.testing.assert_allclose(p1[k], p0[k], rtol=1e-6, atol=0, err_msg=k)


def test_jrpo_sharded_buckets_sum_to_global_bucket(cuda):
    """Multi-GPU contract of the JRPO update on one GPU: two uneven halves of the v3 chunk list, each processed with
    norm_rows = the global joint rows and the global minibatch moments, give gradient buckets (and loss sums) whose
    SUM is the bucket of the whole chunk list."""
    import torch

    from openrl_b200 import lib
    from openrl_b200.utils.logger import Logger
    from test_rollout_cuda import _product

    d = np.load(os.path.join(GOLDEN, "trace_mpe_jrpo.npz"), allow_pickle=True)
    cfg, env, net, agent = _product("simple_spread", int(d["meta/env_num"]), str(d["meta/flags"]).split(), golden=d)
    agent.train(total_time_steps=0, logger=Logger(quiet=True))
    drv = agent.driver
    drv.actor_rollout()
    drv.compute_returns()
    tr, b = drv.trainer, drv.buffer.data
    assert tr.joint and tr.flags & lib.PPO_JOINT_ACTION
    Lc, A = cfg.data_chunk_length, b.num_agents
    chunks = b.episode_length * b.n_rollout_threads // Lc
    ids = torch.randperm(chunks).cuda()
    stats = tr.joint_minibatch_stats(b, ids, Lc).clone()
    act = b.active_masks[:-1].double()
    np.testing.assert_allclose(stats.cpu().numpy(), [float(b.returns[:-1, :, 0].double().sum()),
                                                     float((b.returns[:-1, :, 0].double() ** 2).sum()),
                                                     float(act[:, :, 0].sum()), float(act.sum())], rtol=1e-12)
    tr.tape = torch.empty(int(tr._lib.orl_rnn_workspace_floats(chunks * Lc * A, tr.rnn_stride)), dtype=torch.float32, device="cuda")

    def bucket(part, norm_rows):
        a = tr._rnn_args(b, part.contiguous(), stats)
        a.norm_rows = norm_rows
        lib.check(tr._lib.orl_rnn_fwdbwd(a, lib.current_stream()), "orl_rnn_fwdbwd")
        return tr.rnn_bucket.clone()

    whole = bucket(ids, 0)
    parts = bucket(ids[:chunks // 3], chunks * Lc) + bucket(ids[chunks // 3:], chunks * Lc)   # uneven split: odd chunk counts too
    np.testing.assert_allclose(parts.cpu().numpy(), whole.cpu().numpy(), rtol=2e-4, atol=2e-6)
    assert float(whole[:2 * tr.rnn_stride].abs().max()) > 1e-3
    # the loss sums: policy loss, entropy, joint ratio sum (~ 1 per chunk step), value loss
    assert abs(float(whole[2 * tr.rnn_stride + 2]) - chunks * Lc) < 1e-2 * chunks * Lc


def test_jrpo_runs_at_baseline_scale(cuda):
    """BASELINE configs[2] shape with the joint-action loss: simple_spread, 3 agents x 2048 envs, T = 25."""
    from openrl_b200.configs.config import create_config_parser
    from openrl_b200.envs.common import make
    from openrl_b200.modules.common import PPONet
    from openrl_b200.runners.common import PPOAgent
    from openrl_b200.utils.logger import Logger

    cfg = create_config_parser().parse_args(JRPO + ["--log_interval", "1"])
    cfg.quiet = True
    env = make("simple_spread", env_num=2048)
    agent = PPOAgent(PPONet(env, cfg=cfg, device="cuda:0"))
    logger = Logger(quiet=True)
    agent.train(total_time_steps=25 * 2048 * 2, logger=logger)
    logs = [h[1] for h in logger.history if "value_loss" in h[1]]
    assert len(logs) == 2 and all(np.isfinite(list(l.values())).all() for l in logs), logs
    assert abs(logs[0]["ratio"] - 1.0) < 1e-3 and logs[0]["dist_entropy"] > 1.5


@pytest.mark.parametrize("flags,algo", [
    (["--use_joint_action_loss", "true"], None),                                                         # MLP policy
    (["--use_joint_action_loss", "true", "--use_naive_recurrent_policy", "true", "--episode_length", "25"], None),
    (["--use_joint_action_loss", "true", "--use_recurrent_policy", "true", "--use_share_model", "true"], None),
    (["--use_joint_action_loss", "true", "--use_recurrent_policy", "true"], "a2c"),
])
def test_jrpo_limits_are_loud(cuda, flags, algo):
    from openrl_b200.algorithms import A2CAlgorithm
    from openrl_b200.configs.config import create_config_parser
    from openrl_b200.envs.common import make
    from openrl_b200.modules.common import PPONet
    from openrl_b200.runners.common import PPOAgent

    cfg = create_config_parser().parse_args(flags + ["--episode_length", "25"] if "--episode_length" not in flags else flags)
    cfg.quiet = True
    with pytest.raises(NotImplementedError, match="joint_action|recurrent|share"):
        agent = PPOAgent(PPONet(make("simple_spread", env_num=2), cfg=cfg, device="cuda:0"))
        agent.train(total_time_steps=25 * 2, **({"train_algo_class": A2CAlgorithm} if algo == "a2c" else {}))


def test_jrpo_entry_point_refuses_more_than_four_agents(cuda):
    """The JRPO policy warp holds one chunk's agent rows (at most 4); the C entry point refuses more with
    ORL_ERR_UNSUPPORTED and a message, before any launch."""
    import torch

    from openrl_b200 import lib
    from openrl_b200.utils.logger import Logger
    from test_rollout_cuda import _product

    cfg, env, net, agent = _product("simple_spread", 4, JRPO)
    agent.train(total_time_steps=0, logger=Logger(quiet=True))
    drv = agent.driver
    tr, b = drv.trainer, drv.buffer.data
    ids = torch.arange(4, device="cuda")
    tr.tape = torch.empty(int(tr._lib.orl_rnn_workspace_floats(4 * 2 * 3, tr.rnn_stride)), dtype=torch.float32, device="cuda")
    a = tr._rnn_args(b, ids, tr.mb_stats)
    a.n_agents = 5
    assert tr._lib.orl_rnn_fwdbwd(a, lib.current_stream()) == _header_defs()["ORL_ERR_UNSUPPORTED"]
    assert b"n_agents <= 4" in tr._lib.orl_last_error()
    torch.cuda.synchronize()


def _header_defs():
    with open(os.path.join(os.path.dirname(os.path.dirname(GOLDEN)), "include", "openrl_b200.h")) as f:
        return dict((k, int(v)) for k, v in re.findall(r"#define (ORL_[A-Z0-9_]+) (\d+)\b", f.read()))


def test_joint_action_flag_matches_header():
    from openrl_b200 import lib

    assert _header_defs()["ORL_PPO_JOINT_ACTION"] == lib.PPO_JOINT_ACTION == 1024
