"""Torch-CPU oracle of the joint-action loss (JRPO, cfg.use_joint_action_loss), built on the multi-agent oracle
(oracle/loop_ma.py) without changing it.  TEST INFRASTRUCTURE: only the tests import it.  Restates, with the reference's
consumption order of the global torch generator:
  ReplayData.recurrent_generator_v3 (chunks of L over the env-major / time-minor flattening g = n*T + t, every g carrying
  all A agents; minibatch rows (l*n + j)*A + a)     openrl/buffers/replay_data.py:425-551, buffers/utils/util.py:92-101
  PPOAlgorithm.prepare_loss, joint-action branch   openrl/algorithms/ppo.py:222-224,254-321
  ACTLayer.evaluate_actions (entropy over all agent rows, before the agent-0 reshape)
                                                   openrl/modules/networks/utils/act.py:114-118
Pinned against tests/golden/trace_mpe_jrpo*.npz (tests/test_oracle_jrpo.py)."""
import numpy as np
import torch

from oracle import gae as ogae
from oracle import loop, nets, ppo
from oracle.loop_ma import MATrainer


def cfg_from_flags(flag_string):
    """oracle.loop.cfg_from_flags plus the use_joint_action_loss switch it does not know."""
    cfg = loop.cfg_from_flags(flag_string)
    toks = flag_string.split()
    flags = dict(zip(toks[::2], toks[1::2]))
    cfg.use_joint_action_loss = flags.get("--use_joint_action_loss", "false").lower() in ("true", "1")
    return cfg


def joint_ppo_update(cfg, pol, cri, opt_p, opt_c, vn, batch, A):
    """One minibatch update with the joint-action loss; rows ordered (step, agent).  The critic sees agent 0 only
    (`to_single_np`), the ratio is that of the summed log-probs of the A agents, the advantage and the policy / value
    active masks are agent 0's, the entropy is the mean over all agent rows.  Returns the six scalars of
    oracle.ppo.ppo_update."""
    single = lambda x: x.reshape(-1, A, *x.shape[1:])[:, 0]   # noqa: E731
    opt_p.zero_grad()
    opt_c.zero_grad()
    values, _ = nets.critic_forward(cri, cfg, single(batch["critic_obs"]), single(batch["rnn_states_critic"]),
                                    single(batch["masks"]))
    logp, ent = nets.policy_eval(pol, cfg, batch["policy_obs"], batch["actions"], batch["action_masks"],
                                 batch["active_masks"], batch["rnn_states"], batch["masks"])
    joint = logp.reshape(-1, A, logp.shape[-1]).sum(dim=(1, -1), keepdim=True).reshape(-1, 1)
    old = batch["old_logp"]
    old_joint = old.reshape(-1, A, old.shape[-1]).sum(dim=(1, -1), keepdim=True).reshape(-1, 1)
    adv, active = single(batch["adv"]), single(batch["active_masks"])
    ratio = torch.exp(joint - old_joint)
    if getattr(cfg, "dual_clip_ppo", False):   # ppo.py:304-305
        ratio = torch.min(ratio, torch.tensor(cfg.dual_clip_coeff))
    surr = torch.min(ratio * adv, torch.clamp(ratio, 1.0 - cfg.clip_param, 1.0 + cfg.clip_param) * adv)
    if cfg.use_policy_active_masks:
        policy_loss = (-torch.sum(surr, dim=-1, keepdim=True) * active).sum() / active.sum()
    else:
        policy_loss = -torch.sum(surr, dim=-1, keepdim=True).mean()
    value_loss = ppo.value_loss_fn(cfg, vn, values, single(batch["value_preds"]), single(batch["returns"]), active)
    (policy_loss - ent * cfg.entropy_coef).backward()
    (value_loss * cfg.value_loss_coef).backward()
    if cfg.use_max_grad_norm:
        agn = torch.nn.utils.clip_grad_norm_(list(pol.values()), cfg.max_grad_norm)
        cgn = torch.nn.utils.clip_grad_norm_(list(cri.values()), cfg.max_grad_norm)
    else:
        agn = torch.sqrt(sum(p.grad.norm() ** 2 for p in pol.values()))
        cgn = torch.sqrt(sum(p.grad.norm() ** 2 for p in cri.values()))
    opt_p.step()
    opt_c.step()
    return (value_loss.item(), float(cgn), policy_loss.item(), ent.item(), float(agn), ratio.mean().item())


class JRPOTrainer(MATrainer):
    """MATrainer whose update is JRPO (use_recurrent_policy + use_joint_action_loss)."""

    def _recurrent_batches_v3(self, adv):
        cfg, b = self.cfg, self.buf
        T, N, A = b.rewards.shape[:3]
        L = cfg.data_chunk_length
        data_chunks = N * T // L
        mb = data_chunks // cfg.num_mini_batch
        rand = torch.randperm(data_chunks).numpy()
        cast = lambda x: x.transpose(1, 0, 2, 3).reshape(-1, *x.shape[2:])   # noqa: E731  (T, N, A, d) -> (N*T, A, d)
        flat = {k: cast(getattr(b, k)[:T]) for k in ("policy_obs", "critic_obs", "actions", "action_log_probs", "value_preds",
                                                      "returns", "masks", "active_masks", "action_masks")}
        flat["adv"] = cast(adv)
        hs = b.rnn_states[:-1].transpose(1, 0, 2, 3, 4).reshape(-1, *b.rnn_states.shape[2:])
        hc = b.rnn_states_critic[:-1].transpose(1, 0, 2, 3, 4).reshape(-1, *b.rnn_states_critic.shape[2:])
        for i in range(cfg.num_mini_batch):
            idx = rand[i * mb:(i + 1) * mb]
            out = {}
            for k, v in flat.items():
                st = np.stack([v[c * L:c * L + L] for c in idx], axis=1)  # (L, n, A, d)
                out[k] = torch.from_numpy(st.reshape(L * len(idx) * A, *st.shape[3:]))
            out["rnn_states"] = torch.from_numpy(np.stack([hs[c * L] for c in idx]).reshape(len(idx) * A, *hs.shape[2:]))
            out["rnn_states_critic"] = torch.from_numpy(np.stack([hc[c * L] for c in idx]).reshape(len(idx) * A, *hc.shape[2:]))
            yield rand, out

    def train(self):
        cfg, b = self.cfg, self.buf
        assert cfg.use_recurrent_policy and cfg.use_joint_action_loss
        vn_state = self.vn.state() if self.vn is not None else None
        _, adv = ogae.advantages(b.returns, b.value_preds, b.active_masks, vn_state, cfg.use_adv_normalize)
        self.last_adv = adv
        updates, perms = [], []
        for _ in range(cfg.ppo_epoch):
            for rand, bt in self._recurrent_batches_v3(adv):
                batch = dict(critic_obs=bt["critic_obs"], policy_obs=bt["policy_obs"], actions=bt["actions"],
                             value_preds=bt["value_preds"], returns=bt["returns"], active_masks=bt["active_masks"],
                             old_logp=bt["action_log_probs"], adv=bt["adv"], action_masks=bt["action_masks"],
                             masks=bt["masks"], rnn_states=bt["rnn_states"], rnn_states_critic=bt["rnn_states_critic"])
                updates.append(joint_ppo_update(cfg, self.pol, self.cri, self.opt_p, self.opt_c, self.vn, batch, self.A))
            perms.append(rand.copy())
        return np.array(updates, np.float64), np.stack(perms)
