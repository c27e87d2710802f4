#!/usr/bin/env python
"""Generate golden vectors by EXECUTING THE UNMODIFIED REFERENCE (/root/reference).

TEST INFRASTRUCTURE.  Runs only in the build container (the reference does not exist on
the GPU box); its outputs are committed under tests/golden/ and are what pins the oracle
(oracle/*.py) and, through it, the CUDA path.

    PYTHONPATH=oracle/refstubs:oracle:/root/reference python oracle/gen_golden.py

What is recorded (reference file:line of the code that produced it):
  gae_<branch>.npz   ReplayData.compute_returns, all 8 branches
                     (openrl/buffers/replay_data.py:320-423), random inputs.
  trace_<env>.npz    PPOAgent.train() on CartPole-v1 / GridWorldEnv / simple_spread, seed 0:
                     initial + per-iteration parameters, the rollout buffer
                     (onpolicy_driver.py:154-203), returns (replay_data.py:320), normalised
                     advantages (ppo.py:384-409), every torch.randperm drawn by the minibatch
                     sampler (replay_data.py:578-580), the 6 scalars of every ppo_update
                     (ppo.py:46-176) and the ValueNorm running statistics (valuenorm.py:59-76).
The reference is not modified: recording is done by wrapping bound methods at run time.
"""
import argparse
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(os.path.dirname(HERE), "tests", "golden")

import openrl.runners.common  # noqa: E402,F401  (must be imported first: circular import otherwise)
from openrl.algorithms.ppo import PPOAlgorithm  # noqa: E402
from openrl.buffers.replay_data import ReplayData  # noqa: E402
from openrl.configs.config import create_config_parser  # noqa: E402
from openrl.drivers.onpolicy_driver import OnPolicyDriver  # noqa: E402
from openrl.envs.common import make  # noqa: E402
from openrl.modules.common import PPONet  # noqa: E402
from openrl.modules.utils.valuenorm import ValueNorm  # noqa: E402
from openrl.runners.common import PPOAgent  # noqa: E402

import gymnasium  # noqa: E402  (the stand-in)


def gen_gae():
    rng = np.random.default_rng(1234)
    T, N, A = 7, 5, 2
    obs_space = gymnasium.spaces.Box(-1, 1, (3,), np.float32)
    act_space = gymnasium.spaces.Discrete(2)
    for use_gae in (True, False):
        for ptl in (True, False):
            for vn in (True, False):
                flags = [
                    "--episode_length", str(T),
                    "--use_gae", str(use_gae),
                    "--use_proper_time_limits", str(ptl),
                    "--use_valuenorm", str(vn),
                    "--gamma", "0.97", "--gae_lambda", "0.9",
                ]
                cfg = create_config_parser().parse_args(flags)
                cfg.n_rollout_threads = N
                cfg.learner_n_rollout_threads = N
                data = ReplayData(cfg, A, obs_space, act_space)
                data.rewards[:] = rng.standard_normal(data.rewards.shape)
                data.value_preds[:] = rng.standard_normal(data.value_preds.shape)
                data.masks[:] = rng.random(data.masks.shape) > 0.2
                data.bad_masks[:] = rng.random(data.bad_masks.shape) > 0.15
                next_value = rng.standard_normal((N, A, 1)).astype(np.float32)
                normalizer = None
                vn_state = np.zeros(3, np.float32)
                if vn:
                    normalizer = ValueNorm(1)
                    normalizer.update(torch.from_numpy(rng.standard_normal((64, 1)).astype(np.float32) * 3 + 1.5))
                    vn_state = np.array(
                        [normalizer.running_mean.item(), normalizer.running_mean_sq.item(), normalizer.debiasing_term.item()],
                        np.float32,
                    )
                inp = dict(
                    rewards=data.rewards.copy(), value_preds=data.value_preds.copy(),
                    masks=data.masks.copy(), bad_masks=data.bad_masks.copy(), next_value=next_value,
                )
                data.compute_returns(next_value, normalizer)
                name = f"gae_g{int(use_gae)}_p{int(ptl)}_v{int(vn)}.npz"
                np.savez_compressed(
                    os.path.join(OUT, name), returns=data.returns.copy(), vn_state=vn_state,
                    gamma=np.float64(cfg.gamma), gae_lambda=np.float64(cfg.gae_lambda),
                    value_preds_after=data.value_preds.copy(), **inp,
                )
                print("wrote", name)


def flat_params(module):
    out = {}
    for mk, model in module.models.items():
        for k, v in model.state_dict().items():
            out[f"{mk}.{k}"] = v.detach().cpu().numpy().copy()
    return out


def gen_trace(env_id, env_num, flags, iters, tag, algo="ppo", ref_flags=None):
    """`flags` is recorded in the golden (canonical `--name value` form); `ref_flags` is what the reference's own parser
    is given when it spells an option differently (its store_false switches, config.py:679-772)."""
    rec = {}
    cfg = create_config_parser().parse_args(ref_flags if ref_flags is not None else flags)
    env = make(env_id, env_num=env_num)
    net = PPONet(env, cfg=cfg)
    agent = PPOAgent(net)
    for k, v in flat_params(net.module).items():
        rec[f"init/{k}"] = v

    perms = []
    orig_randperm = torch.randperm

    def rec_randperm(*a, **k):
        p = orig_randperm(*a, **k)
        perms.append(p.numpy().copy())
        return p

    torch.randperm = rec_randperm

    state = {"it": 0}
    orig_compute_returns = OnPolicyDriver.compute_returns
    orig_ppo_update = PPOAlgorithm.ppo_update
    orig_ffg = ReplayData.feed_forward_generator
    orig_rg = ReplayData.recurrent_generator
    orig_ng = ReplayData.naive_recurrent_generator
    updates = []

    def compute_returns(self):
        orig_compute_returns(self)
        it = state["it"]
        d = self.buffer.data
        for name in ("value_preds", "returns", "masks", "active_masks", "bad_masks", "actions", "action_log_probs", "rewards"):
            rec[f"it{it}/{name}"] = getattr(d, name).copy()
        if d.action_masks is not None:
            rec[f"it{it}/action_masks"] = d.action_masks.copy()
        if isinstance(d.policy_obs, np.ndarray):
            rec[f"it{it}/policy_obs"] = d.policy_obs.copy()
            rec[f"it{it}/critic_obs"] = d.critic_obs.copy()
        else:
            rec[f"it{it}/policy_obs"] = d.policy_obs["policy"].copy()
            rec[f"it{it}/critic_obs"] = d.critic_obs["critic"].copy()
        if cfg.use_recurrent_policy or cfg.use_naive_recurrent_policy:
            rec[f"it{it}/rnn_states"] = d.rnn_states.copy()
            rec[f"it{it}/rnn_states_critic"] = d.rnn_states_critic.copy()
        vn = self.trainer.algo_module.get_critic_value_normalizer()
        if vn is not None:
            rec[f"it{it}/vn_before_update"] = np.array(
                [vn.running_mean.item(), vn.running_mean_sq.item(), vn.debiasing_term.item()], np.float32)

    def ppo_update(self, sample, turn_on=True):
        out = orig_ppo_update(self, sample, turn_on)
        value_loss, critic_grad_norm, policy_loss, dist_entropy, actor_grad_norm, ratio = out
        updates.append([
            float(value_loss.item()), float(critic_grad_norm), float(policy_loss.item()),
            float(dist_entropy.item()), float(actor_grad_norm), float(ratio.mean().item()),
        ])
        return out

    def ffg(self, advantages, *a, **k):
        rec.setdefault(f"it{state['it']}/advantages", advantages.copy())
        return orig_ffg(self, advantages, *a, **k)

    def rg(self, advantages, *a, **k):
        rec.setdefault(f"it{state['it']}/advantages", advantages.copy())
        return orig_rg(self, advantages, *a, **k)

    def ng(self, advantages, *a, **k):
        rec.setdefault(f"it{state['it']}/advantages", advantages.copy())
        return orig_ng(self, advantages, *a, **k)

    orig_inner = OnPolicyDriver._inner_loop

    def inner(self):
        r = orig_inner(self)
        it = state["it"]
        rec[f"it{it}/updates"] = np.array(updates, np.float64)
        rec[f"it{it}/perms"] = np.array(perms, dtype=object) if False else np.stack(perms) if perms else np.zeros((0,))
        updates.clear()
        perms.clear()
        for k, v in flat_params(self.trainer.algo_module).items():
            rec[f"it{it}/params/{k}"] = v
        vn = self.trainer.algo_module.get_critic_value_normalizer()
        if vn is not None:
            rec[f"it{it}/vn_after_update"] = np.array(
                [vn.running_mean.item(), vn.running_mean_sq.item(), vn.debiasing_term.item()], np.float32)
        state["it"] += 1
        return r

    OnPolicyDriver.compute_returns = compute_returns
    PPOAlgorithm.ppo_update = ppo_update
    ReplayData.feed_forward_generator = ffg
    ReplayData.recurrent_generator = rg
    ReplayData.naive_recurrent_generator = ng
    OnPolicyDriver._inner_loop = inner
    try:
        if algo == "a2c":   # the reference's A2CAgent.train == PPOAgent.train(train_algo_class=A2CAlgorithm) (a2c_agent.py:66-77)
            from openrl.algorithms.a2c import A2CAlgorithm

            agent.train(total_time_steps=cfg.episode_length * env_num * iters, train_algo_class=A2CAlgorithm)
        else:
            agent.train(total_time_steps=cfg.episode_length * env_num * iters)
    finally:
        OnPolicyDriver.compute_returns = orig_compute_returns
        PPOAlgorithm.ppo_update = orig_ppo_update
        ReplayData.feed_forward_generator = orig_ffg
        ReplayData.recurrent_generator = orig_rg
        ReplayData.naive_recurrent_generator = orig_ng
        OnPolicyDriver._inner_loop = orig_inner
        torch.randperm = orig_randperm
    env.close()
    rec["meta/flags"] = np.array(" ".join(flags))
    rec["meta/env_id"] = np.array(env_id)
    rec["meta/env_num"] = np.int64(env_num)
    rec["meta/iters"] = np.int64(iters)
    rec["meta/algo"] = np.array(algo)
    name = f"trace_{tag}.npz"
    np.savez_compressed(os.path.join(OUT, name), **rec)
    print("wrote", name, "iters", state["it"], "bytes", os.path.getsize(os.path.join(OUT, name)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default="")
    a = ap.parse_args()
    sys.path.insert(0, os.path.dirname(HERE))
    from oracle import TRACE_THREADS

    torch.set_num_threads(TRACE_THREADS)
    os.makedirs(OUT, exist_ok=True)
    if a.only in ("", "gae"):
        gen_gae()
    if a.only in ("", "cartpole"):
        gen_trace("CartPole-v1", 8,
                  ["--seed", "0", "--episode_length", "32", "--ppo_epoch", "2", "--num_mini_batch", "2", "--log_interval", "1000"],
                  3, "cartpole")
        # C1 of BASELINE.json at its own flags but few iterations
        gen_trace("CartPole-v1", 8,
                  ["--seed", "0", "--episode_length", "128", "--ppo_epoch", "4", "--log_interval", "1000"],
                  2, "cartpole_c1")
    if a.only in ("", "gridworld"):
        gen_trace("GridWorldEnv", 4,
                  ["--seed", "0", "--episode_length", "32", "--ppo_epoch", "2", "--log_interval", "1000"],
                  2, "gridworld")
    if a.only in ("", "mpe"):
        gen_trace("simple_spread", 4,
                  ["--seed", "0", "--episode_length", "25", "--ppo_epoch", "2", "--lr", "7e-4", "--critic_lr", "7e-4",
                   "--use_recurrent_policy", "true", "--use_valuenorm", "true", "--use_adv_normalize", "true",
                   "--log_interval", "1000"],
                  2, "mpe_gru")
    if a.only in ("", "cartpole_gru"):
        # single-agent recurrent PPO: episodes end mid-rollout (masks == 0 inside chunks), chunks of 4, two minibatches
        gen_trace("CartPole-v1", 8,
                  ["--seed", "0", "--episode_length", "32", "--ppo_epoch", "2", "--num_mini_batch", "2",
                   "--use_recurrent_policy", "true", "--data_chunk_length", "4", "--log_interval", "1000"],
                  2, "cartpole_gru")
    if a.only in ("", "mpe_naive_gru"):
        # whole-trajectory BPTT (naive_recurrent_generator, replay_data.py:806-946): minibatches of (env, agent) rows
        gen_trace("simple_spread", 4,
                  ["--seed", "0", "--episode_length", "25", "--ppo_epoch", "2", "--num_mini_batch", "2", "--lr", "7e-4", "--critic_lr", "7e-4",
                   "--use_naive_recurrent_policy", "true", "--use_valuenorm", "true", "--use_adv_normalize", "true", "--log_interval", "1000"],
                  2, "mpe_naive_gru")
    if a.only in ("", "gaussian"):
        gen_trace("IdentityEnvcontinuous", 4,
                  ["--seed", "0", "--episode_length", "16", "--ppo_epoch", "2", "--num_mini_batch", "2", "--log_interval", "1000"],
                  2, "identity_continuous")
    if a.only in ("", "flags"):
        gen_flag_variants()
    if a.only in ("", "oracle_variants"):
        gen_oracle_variants()
    if a.only in ("", "mpe_mlp"):
        gen_trace("simple_spread", 4,
                  ["--seed", "0", "--episode_length", "25", "--ppo_epoch", "2", "--lr", "7e-4", "--critic_lr", "7e-4",
                   "--use_valuenorm", "true", "--use_adv_normalize", "true", "--log_interval", "1000"],
                  2, "mpe_mlp")


# Loss / return option branches of the hot path (ppo.py:178-220,254-339, a2c.py:39-140, replay_data.py:320-423):
# one short CartPole trace each, so that every branch of oracle/ppo.py + oracle/gae.py is pinned to the reference.
FLAG_VARIANTS = {   # name: (canonical flags, the reference parser's spelling, algorithm)
    "a2c": (["--ppo_epoch", "1"], None, "a2c"),
    "dual_clip": (["--dual_clip_ppo", "true", "--dual_clip_coeff", "1.02"], None, "ppo"),
    "no_huber": (["--use_huber_loss", "false"], ["--use_huber_loss"], "ppo"),
    "no_value_clip": (["--use_clipped_value_loss", "false"], ["--use_clipped_value_loss"], "ppo"),
    "proper_time_limits": (["--use_proper_time_limits", "true"], None, "ppo"),
    "no_gae": (["--use_gae", "false"], None, "ppo"),
    "no_valuenorm": (["--use_valuenorm", "false"], None, "ppo"),
    "adv_norm_no_masks": (["--use_adv_normalize", "true", "--use_value_active_masks", "false", "--use_policy_active_masks", "false"],
                          ["--use_adv_normalize", "true", "--use_value_active_masks", "false", "--use_policy_active_masks"], "ppo"),
    "popart": (["--use_popart", "true", "--use_valuenorm", "false"], None, "ppo"),   # the reference asserts not (popart and valuenorm)
    "no_grad_clip_wd": (["--use_max_grad_norm", "false", "--weight_decay", "0.01", "--activation_id", "0"],
                        ["--use_max_grad_norm", "--weight_decay", "0.01", "--activation_id", "0"], "ppo"),
}


# Further option values, pinned for the ORACLE only (tests/test_oracle_loop.py): they are the settings the device-vs-oracle
# flag matrix (tests/test_ppo_flags_cuda.py) and the lr-schedule test use, so that chain ends at the executed reference too.
ORACLE_VARIANTS = {
    "lr_decay": (["--use_linear_lr_decay", "true"], 3),
    "act_leaky_relu": (["--activation_id", "2"], 2),
    "act_elu": (["--activation_id", "3"], 2),
    "coefs": (["--clip_param", "0.05", "--entropy_coef", "0.05", "--value_loss_coef", "1.0", "--huber_delta", "0.5",
               "--max_grad_norm", "0.5"], 2),
    "lrs_wd": (["--lr", "1e-3", "--critic_lr", "2e-3", "--weight_decay", "0.01"], 2),
    "gamma_lambda": (["--gamma", "0.9", "--gae_lambda", "0.8", "--use_adv_normalize", "true"], 2),
}


def gen_oracle_variants():
    base = ["--seed", "0", "--episode_length", "24", "--ppo_epoch", "2", "--num_mini_batch", "2", "--log_interval", "1000"]
    for name, (extra, iters) in ORACLE_VARIANTS.items():
        gen_trace("CartPole-v1", 6, base + extra, iters, f"opt_{name}")


def gen_flag_variants():
    base = ["--seed", "0", "--episode_length", "24", "--ppo_epoch", "2", "--num_mini_batch", "2", "--log_interval", "1000"]
    for name, (extra, ref_extra, algo) in FLAG_VARIANTS.items():
        gen_trace("CartPole-v1", 6, base + extra, 2, f"flag_{name}", algo=algo,
                  ref_flags=None if ref_extra is None else base + ref_extra)


if __name__ == "__main__":
    main()
