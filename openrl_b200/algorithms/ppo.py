"""PPOAlgorithm(cfg, init_module, agent_num, device).train(buffer_data) -> dict
(reference: openrl/algorithms/ppo.py:32-469, base_algorithm.py:24-86).

`train` runs `ppo_epoch x num_mini_batch` updates, each three asynchronous CUDA launches
(orl_ppo_fwdbwd / orl_ppo_reduce / orl_ppo_apply) plus, with >1 GPU, ONE all-reduce of the
folded gradient bucket.  Nothing is read back until the metrics are logged.

Minibatch order: the reference draws one `torch.randperm(T*N*A)` per epoch from the global CPU
generator (replay_data.py:578-580).  cfg.parity_mode=True reproduces exactly that (host draw,
H2D copy); otherwise the permutation is drawn on the device, and with num_mini_batch == 1 no
permutation is needed at all (a minibatch that is the whole buffer is a sum over all rows).
"""
import numpy as np
import torch
from .. import lib, parallel
from ..buffers.replay_data import ReplayData, chunk_row_indices, chunk_row_indices_v3


class PPOAlgorithm:
    def __init__(self, cfg, init_module, agent_num=1, device="cuda:0"):
        self.cfg = cfg
        self.algo_module = init_module
        self.agent_num = agent_num
        self.device = torch.device(device) if not isinstance(device, torch.device) else device
        self.world_size = parallel.world_size()
        self.ppo_epoch, self.num_mini_batch = cfg.ppo_epoch, cfg.num_mini_batch
        self.clip_param = cfg.clip_param
        self._lib = lib.load()
        pol, cri = init_module.models["policy"], init_module.models["critic"]
        self.d, self.dc, self.n = pol.obs_dim, cri.obs_dim, pol.n_actions
        self.stride = self._lib.orl_ppo_stride(self.d, self.dc, self.n)
        self.head_kind = pol.head_kind
        self.recurrent = bool(cfg.use_recurrent_policy or getattr(cfg, "use_naive_recurrent_policy", False))
        # naive_recurrent_generator (replay_data.py:806-946) == chunks of the WHOLE trajectory: chunk length = episode_length,
        # chunk c = buffer row c, one randperm over rows per epoch (ppo.py:363-381: taken only when use_recurrent_policy is off)
        self.naive = bool(getattr(cfg, "use_naive_recurrent_policy", False)) and not cfg.use_recurrent_policy
        # tensor-core update (tcgen05, split fp16, fp32-class accuracy): Categorical heads, obs widths <= 8
        self.use_tensor_cores = (bool(getattr(cfg, "use_tensor_cores", True)) and bool(getattr(cfg, "use_tf32", True))
                                 and max(self.d, self.dc) <= 8 and self.head_kind == lib.HEAD_CATEGORICAL and not self.recurrent)
        sm = torch.cuda.get_device_properties(self.device).multi_processor_count
        # CTAs per net: the tensor-core kernel runs two 256-thread CTAs per SM, the FFMA kernel one
        self.grid_per_net = max(1, sm if self.use_tensor_cores else sm // 2)
        dev = self.device
        self.partials = torch.zeros(2 * self.grid_per_net, self.stride, dtype=torch.float32, device=dev)
        # the gradient bucket that is all-reduced once per update (symmetric memory over NVLink when > 1 GPU)
        self.folded, self.folded_sum = parallel.symmetric_buffer((2, self.stride), torch.float32, dev)
        # > 1 GPU, feed-forward nets: the exchange is fused into the reduce / optimiser kernels over NVLink peer memory
        self.peer = None
        if self.world_size > 1 and not self.recurrent and not bool(getattr(cfg, "use_share_model", False)):
            self.peer = parallel.PeerBucket.create(self._lib.orl_ppo_peer_bucket_bytes(self.d, self.dc, self.n, self.world_size),
                                                    self.stride, dev)
        self.grads_stride = self._lib.orl_ppo_grads_stride(self.d, self.dc, self.n)
        self.grads = torch.zeros(2, self.grads_stride, dtype=torch.float32, device=dev)
        self.train_info = torch.zeros(6, dtype=torch.float32, device=dev)
        self.lrs = torch.zeros(2, dtype=torch.float32, device=dev)
        self.mb_stats = torch.zeros(4, dtype=torch.float64, device=dev)   # 3 doubles; the 4th is JRPO's all-agent active sum
        self.flags = ((lib.PPO_HUBER if cfg.use_huber_loss else 0) | (lib.PPO_CLIP_VALUE if cfg.use_clipped_value_loss else 0)
                      | (lib.PPO_VALUE_ACTIVE_MASKS if cfg.use_value_active_masks else 0)
                      | (lib.PPO_POLICY_ACTIVE_MASKS if cfg.use_policy_active_masks else 0)
                      | (lib.PPO_VALUENORM if (cfg.use_valuenorm and cri.value_normalizer is not None) else 0)
                      | (lib.PPO_ADV_NORMALIZE if cfg.use_adv_normalize else 0)
                      | (lib.PPO_MAX_GRAD_NORM if cfg.use_max_grad_norm else 0))
        if self.use_tensor_cores:
            self.flags |= lib.PPO_TENSORCORE
        if getattr(cfg, "dual_clip_ppo", False):
            self.flags |= lib.PPO_DUAL_CLIP
        assert not (getattr(cfg, "use_popart", False) and cfg.use_valuenorm), \
            "self._use_popart and self._use_valuenorm can not be set True simultaneously"   # ppo.py:40-44
        self.share = bool(getattr(init_module, "share_model", False))
        # JRPO (ppo.py:254-321, 363-369): the joint-action loss over recurrent_generator_v3 chunks; the reference takes it
        # only with use_recurrent_policy
        self.joint = bool(getattr(cfg, "use_joint_action_loss", False))
        if self.joint:
            if self.share or getattr(cfg, "use_share_model", False):
                raise NotImplementedError("use_joint_action_loss with use_share_model is not built")
            if self.naive:
                raise NotImplementedError("use_joint_action_loss with use_naive_recurrent_policy is not built (the reference "
                                          "applies the joint loss to naive_recurrent_generator batches of unrelated rows)")
            if not cfg.use_recurrent_policy:
                raise NotImplementedError("use_joint_action_loss needs use_recurrent_policy: with an MLP policy the reference's "
                                          "feed_forward_generator groups agent_num random rows into one joint action")
            self.flags |= lib.PPO_JOINT_ACTION
        if self.share:
            # one network, one optimiser: true-layout gradients + 8 loss-sum slots in ONE bucket (a single all-reduce per update)
            if self.recurrent:
                raise NotImplementedError("use_share_model with recurrent policies is not built")
            self.use_tensor_cores = False
            self.flags &= ~lib.PPO_TENSORCORE
            self.share_total = int(self._lib.orl_share_param_count(self.d, self.n))
            self.share_bucket = torch.zeros(((self.share_total + 3) & ~3) + 8, dtype=torch.float32, device=dev)
            self.share_grads = self.share_bucket[:(self.share_total + 3) & ~3]
            self.share_loss = self.share_bucket[(self.share_total + 3) & ~3:]
            self.share_ws = None
        for name in ("use_policy_vhead", "use_amp", "use_deepspeed"):
            if getattr(cfg, name, False):
                raise NotImplementedError(f"cfg.{name} is not built into the CUDA update yet (SURVEY.md §8f)")
        if self.recurrent:
            if self.head_kind != lib.HEAD_CATEGORICAL:
                raise NotImplementedError("recurrent policies are built for Discrete action spaces")
            self.chunk_length = cfg.episode_length if self.naive else cfg.data_chunk_length
            if not 1 <= self.chunk_length <= 32:
                raise NotImplementedError("the recurrent kernels take chunks of 1..32 steps (data_chunk_length, or episode_length "
                                          "with use_naive_recurrent_policy)")
            self.rnn_stride = (max(self._lib.orl_rnn_param_count(self.d, self.n), self._lib.orl_rnn_param_count(self.dc, 1)) + 3) & ~3
            # one bucket = gradients of both nets + the loss sums: a single all-reduce per update with >1 GPU
            self.rnn_bucket = torch.zeros(2 * self.rnn_stride + 8, dtype=torch.float32, device=dev)
            self.rnn_grads = self.rnn_bucket[:2 * self.rnn_stride].view(2, self.rnn_stride)
            self.loss_acc = self.rnn_bucket[2 * self.rnn_stride:]
            self.tape = None
        self.gpu_launches = 0
        self.h2d_bytes = 0
        self.d2h_bytes = 0
        self._lrs_host = None

    def prep_rollout(self):
        pass

    def prep_training(self):
        pass

    def _args(self, buf, batch_rows, indices, row_begin):
        m = self.algo_module
        pol, cri = m.models["policy"], m.models["critic"]
        op, oc = m.optimizers["policy"], m.optimizers["critic"]
        cfg = self.cfg
        a = lib.OrlPpoArgs()
        a.obs_dim, a.critic_obs_dim, a.n_actions, a.activation_id = self.d, self.dc, self.n, pol.activation_id
        a.flags, a.grid_per_net = self.flags, self.grid_per_net
        a.head_kind = self.head_kind
        a.dual_clip_coeff = float(getattr(self.cfg, "dual_clip_coeff", 3.0))
        total = buf.episode_length * buf.n_rollout_threads * buf.num_agents
        a.batch_rows, a.row_begin, a.total_rows = int(batch_rows), int(row_begin), int(total)
        # every rank holds an equal shard of the global minibatch: weights / batch moments refer to the global row count
        a.norm_rows = int(batch_rows) * self.world_size if self.world_size > 1 else 0
        a.indices = lib.ptr(indices)
        a.policy_obs, a.critic_obs = lib.ptr(buf.policy_obs), lib.ptr(buf.critic_obs)
        a.actions, a.old_log_probs = lib.ptr(buf.actions), lib.ptr(buf.action_log_probs)
        a.advantages, a.value_preds, a.returns = lib.ptr(buf.advantages), lib.ptr(buf.value_preds), lib.ptr(buf.returns)
        a.active_masks = lib.ptr(buf.active_masks)
        a.action_masks = None if (buf.action_masks_trivial or buf.continuous) else lib.ptr(buf.action_masks)
        a.gae_stats = lib.ptr(buf.gae_stats)
        vn = cri.value_normalizer
        a.vn_state = None if vn is None else lib.ptr(vn.state)
        a.policy_params, a.critic_params = lib.ptr(pol.flat_params), lib.ptr(cri.flat_params)
        a.policy_adam_m, a.policy_adam_v = lib.ptr(op.exp_avg), lib.ptr(op.exp_avg_sq)
        a.critic_adam_m, a.critic_adam_v = lib.ptr(oc.exp_avg), lib.ptr(oc.exp_avg_sq)
        a.adam_steps, a.lrs = lib.ptr(m.adam_steps), lib.ptr(self.lrs)
        a.clip_param, a.entropy_coef, a.value_loss_coef = cfg.clip_param, cfg.entropy_coef, cfg.value_loss_coef
        a.huber_delta, a.max_grad_norm = cfg.huber_delta, cfg.max_grad_norm
        g = op.param_groups[0]
        a.adam_beta1, a.adam_beta2, a.adam_eps, a.weight_decay = g["betas"][0], g["betas"][1], g["eps"], g["weight_decay"]
        a.vn_beta = 0.99999 if vn is None else vn.beta
        a.partials, a.folded, a.grads, a.train_info = (lib.ptr(self.partials), lib.ptr(self.folded),
                                                        lib.ptr(self.grads), lib.ptr(self.train_info))
        return a

    def _share_update(self, buf, batch_rows, indices, row_begin, mb_stats):
        """One minibatch update of the shared policy-value network (ppo.py:46-176 with `_use_share_model`)."""
        L, s = self._lib, lib.current_stream()
        need = int(L.orl_share_workspace_floats(int(batch_rows), self.d, self.n))
        if self.share_ws is None or self.share_ws.numel() < need:
            self.share_ws = torch.empty(need, dtype=torch.float32, device=self.device)
        a = self._args(buf, batch_rows, indices, row_begin)
        a.mb_stats = lib.ptr(mb_stats)
        a.partials, a.grads, a.folded = lib.ptr(self.share_ws), lib.ptr(self.share_grads), lib.ptr(self.share_loss)
        lib.check(L.orl_share_fwdbwd(a, s), "orl_share_fwdbwd")
        parallel.allreduce_sum_(self.share_bucket)   # gradients + loss sums (no-op on one GPU)
        lib.check(L.orl_share_apply(a, s), "orl_share_apply")
        self.gpu_launches += 5

    def ppo_update(self, buf, batch_rows, indices=None, row_begin=0, mb_stats=None):
        """One minibatch update (ppo.py:46-176) — asynchronous."""
        L, s = self._lib, lib.current_stream()
        if mb_stats is None:
            lib.check(L.orl_minibatch_stats(lib.ptr(indices), int(batch_rows), lib.ptr(buf.returns),
                                            lib.ptr(buf.active_masks), lib.ptr(self.mb_stats), s), "orl_minibatch_stats")
            mb_stats = self.mb_stats
            self.gpu_launches += 1
            parallel.allreduce_sum_(mb_stats)
        if self.share:
            return self._share_update(buf, batch_rows, indices, row_begin, mb_stats)
        a = self._args(buf, batch_rows, indices, row_begin)
        a.mb_stats = lib.ptr(mb_stats)
        lib.check(L.orl_ppo_fwdbwd(a, s), "orl_ppo_fwdbwd")
        if self.peer is not None:
            # the single gradient-bucket exchange of the update, inside the optimiser kernel (peer loads over NVLink)
            lib.check(L.orl_ppo_reduce_peer(a, self.peer.args, s), "orl_ppo_reduce_peer")
            lib.check(L.orl_ppo_apply_peer(a, self.peer.args, s), "orl_ppo_apply_peer")
            self.gpu_launches += 3
            return
        lib.check(L.orl_ppo_reduce(a, s), "orl_ppo_reduce")
        summed = parallel.allreduce_sum_into(self.folded)  # the single gradient-bucket all-reduce of the update
        a.folded = lib.ptr(summed)
        lib.check(L.orl_ppo_apply(a, s), "orl_ppo_apply")
        self.gpu_launches += 3

    def _rnn_args(self, buf, chunk_ids, mb_stats):
        m = self.algo_module
        pol, cri = m.models["policy"], m.models["critic"]
        op, oc = m.optimizers["policy"], m.optimizers["critic"]
        cfg = self.cfg
        a = lib.OrlRnnArgs()
        a.n_envs, a.n_agents, a.episode_length = buf.n_rollout_threads, buf.num_agents, buf.episode_length
        a.obs_dim, a.critic_obs_dim, a.n_actions, a.activation_id = self.d, self.dc, self.n, pol.activation_id
        a.chunk_length, a.flags = self.chunk_length, self.flags
        a.n_chunks, a.chunk_ids = int(chunk_ids.numel()), lib.ptr(chunk_ids)
        a.policy_params, a.critic_params = lib.ptr(pol.flat_params), lib.ptr(cri.flat_params)
        a.policy_obs, a.critic_obs = lib.ptr(buf.policy_obs), lib.ptr(buf.critic_obs)
        a.rnn_states, a.rnn_states_critic = lib.ptr(buf.rnn_states), lib.ptr(buf.rnn_states_critic)
        a.actions, a.action_log_probs = lib.ptr(buf.actions), lib.ptr(buf.action_log_probs)
        a.masks, a.active_masks = lib.ptr(buf.masks), lib.ptr(buf.active_masks)
        a.value_preds, a.returns, a.advantages = lib.ptr(buf.value_preds), lib.ptr(buf.returns), lib.ptr(buf.advantages)
        a.gae_stats, a.mb_stats = lib.ptr(buf.gae_stats), lib.ptr(mb_stats)
        vn = cri.value_normalizer
        a.vn_state = None if vn is None else lib.ptr(vn.state)
        a.tape, a.grads, a.grads_stride, a.loss_acc = lib.ptr(self.tape), lib.ptr(self.rnn_grads), self.rnn_stride, lib.ptr(self.loss_acc)
        a.policy_adam_m, a.policy_adam_v = lib.ptr(op.exp_avg), lib.ptr(op.exp_avg_sq)
        a.critic_adam_m, a.critic_adam_v = lib.ptr(oc.exp_avg), lib.ptr(oc.exp_avg_sq)
        a.adam_steps, a.lrs = lib.ptr(m.adam_steps), lib.ptr(self.lrs)
        a.clip_param, a.entropy_coef, a.value_loss_coef = cfg.clip_param, cfg.entropy_coef, cfg.value_loss_coef
        a.huber_delta, a.max_grad_norm = cfg.huber_delta, cfg.max_grad_norm
        g = op.param_groups[0]
        a.adam_beta1, a.adam_beta2, a.adam_eps, a.weight_decay = g["betas"][0], g["betas"][1], g["eps"], g["weight_decay"]
        a.dual_clip_coeff = float(getattr(cfg, "dual_clip_coeff", 3.0))
        a.vn_beta = 0.99999 if vn is None else vn.beta
        a.train_info = lib.ptr(self.train_info)
        rows = int(chunk_ids.numel()) * self.chunk_length
        a.norm_rows = rows * self.world_size if self.world_size > 1 else 0
        return a

    def joint_minibatch_stats(self, buf, chunk_ids, chunk_length):
        """JRPO minibatch moments {sum ret_0, sum ret_0^2, sum active_0, sum active_all} of the given v3 chunks into
        self.mb_stats (this rank's rows only).  The all-agent pass writes slots 1..3 first, then the agent-0 pass
        overwrites slots 0..2, so slot 3 keeps the all-agent active sum."""
        s, T, N, A = lib.current_stream(), buf.episode_length, buf.n_rollout_threads, buf.num_agents
        for agent0, out in ((False, self.mb_stats[1:]), (True, self.mb_stats)):
            bi = chunk_row_indices_v3(chunk_ids, chunk_length, T, N, A, agent0_only=agent0)
            lib.check(self._lib.orl_minibatch_stats(lib.ptr(bi), int(bi.numel()), lib.ptr(buf.returns),
                                                    lib.ptr(buf.active_masks), lib.ptr(out), s), "orl_minibatch_stats")
        self.gpu_launches += 2
        return self.mb_stats

    def _train_recurrent(self, buf):
        """train_ppo with ReplayData.recurrent_generator (replay_data.py:1062-1258): per epoch one permutation of
        the data chunks (L consecutive steps of the agent-major / time-minor flattening f = (n*A + a)*T + t);
        a minibatch is a slice of chunk ids, gathered inside the kernels.

        With the joint-action loss (recurrent_generator_v3, replay_data.py:425-551) the chunks run over the env-major /
        time-minor flattening g = n*T + t instead, every chunk step carrying all A agents; the minibatch moments are
        agent 0's returns / active masks plus the all-agent active sum (4 doubles)."""
        cfg = self.cfg
        T, A = buf.episode_length, buf.num_agents
        B = buf.n_rollout_threads * A
        total, L = T * B, (T if self.naive else cfg.data_chunk_length)
        flat = T * buf.n_rollout_threads if self.joint else total   # flattened samples that are cut into chunks
        if flat < L:
            raise AssertionError(f"PPO requires the number of processes ({buf.n_rollout_threads}) * episode length ({T}) "
                                 f"{'' if self.joint else '* agents '}to be greater than or equal to the data chunk length ({L}).")
        data_chunks = flat // L
        mbc = data_chunks // self.num_mini_batch
        rows = mbc * L
        tape_rows = rows * A if self.joint else rows   # the JRPO policy tape has one row per agent and chunk step
        need = int(self._lib.orl_rnn_workspace_floats(tape_rows, self.rnn_stride))   # tape rows + reduction partials
        if self.tape is None or self.tape.numel() < need:
            self.tape = torch.empty(need, dtype=torch.float32, device=self.device)
        whole = self.num_mini_batch == 1 and rows == flat
        s, Lb = lib.current_stream(), self._lib
        for epoch in range(self.ppo_epoch):
            if cfg.parity_mode:
                perm = torch.randperm(data_chunks).to(self.device, non_blocking=True)   # global CPU generator
                self.h2d_bytes += data_chunks * 8
            else:
                perm = torch.randperm(data_chunks, device=self.device)
            for i in range(self.num_mini_batch):
                ids = perm[i * mbc:(i + 1) * mbc].contiguous()
                if whole and not self.joint:
                    mb_stats = buf.gae_stats[5:8]
                elif whole and epoch > 0:
                    mb_stats = self.mb_stats   # JRPO, one minibatch of every chunk: the moments of epoch 0 still hold
                elif self.joint:
                    mb_stats = self.joint_minibatch_stats(buf, ids, L)
                    parallel.allreduce_sum_(mb_stats)
                else:
                    bi = chunk_row_indices(ids, L, T, B)
                    lib.check(Lb.orl_minibatch_stats(lib.ptr(bi), int(rows), lib.ptr(buf.returns), lib.ptr(buf.active_masks),
                                                     lib.ptr(self.mb_stats), s), "orl_minibatch_stats")
                    mb_stats = self.mb_stats
                    self.gpu_launches += 1
                    parallel.allreduce_sum_(mb_stats)
                a = self._rnn_args(buf, ids, mb_stats)
                lib.check(Lb.orl_rnn_fwdbwd(a, s), "orl_rnn_fwdbwd")
                parallel.allreduce_sum_(self.rnn_bucket)   # gradients of both nets + loss sums (no-op on one GPU)
                lib.check(Lb.orl_rnn_apply(a, s), "orl_rnn_apply")
                self.gpu_launches += 9   # 2 x (chunk, tape gemm, tape colsum, partial sum) + apply

    def train(self, buffer, turn_on=True):
        """train_ppo (ppo.py:383-458).  `buffer` is the device ReplayData whose returns/advantages
        were produced by `compute_returns` (orl_gae).  Returns the averaged metrics (one D2H read)."""
        if not isinstance(buffer, ReplayData):
            # a HOST buffer (the reference's numpy ReplayData): upload it once, then the device path
            buffer = ReplayData.from_host(buffer, self.cfg, self.algo_module.get_critic_value_normalizer(), device=self.device)
            self.h2d_bytes += buffer.h2d_bytes
        self.train_async(buffer)
        return self.read_train_info()

    def read_train_info(self):
        num_updates = self.ppo_epoch * self.num_mini_batch
        info = (self.train_info / num_updates).cpu().numpy()
        self.d2h_bytes += info.nbytes
        if self.peer is not None and not (info == info).all():
            self.peer.check()
        keys = ["value_loss", "critic_grad_norm", "policy_loss", "dist_entropy", "actor_grad_norm", "ratio"]
        return {k: float(v) for k, v in zip(keys, info)}

    def sync_lrs(self):
        """Learning rates live in a device buffer (the kernels read them there, so a captured graph can be replayed while
        a schedule changes them): one 8-byte H2D copy, only when the host values changed."""
        m = self.algo_module
        lrs = (m.optimizers["policy"].param_groups[0]["lr"], m.optimizers["critic"].param_groups[0]["lr"])
        if lrs != self._lrs_host:
            self.lrs.copy_(torch.tensor(lrs, dtype=torch.float32), non_blocking=True)
            self._lrs_host = lrs
            self.h2d_bytes += 8

    def train_async(self, buffer):
        """All launches of one training phase, no host read-back."""
        buf = buffer
        if not torch.cuda.is_current_stream_capturing():
            self.sync_lrs()
        self.train_info.zero_()
        if not getattr(buf, "returns_ready", True):
            # train() on a buffer whose returns were never computed (the reference's algorithm tests call it on a fresh
            # buffer, tests/test_algorithm/test_ppo_algorithm.py:76-82): the reference derives the advantages inside
            # train_ppo from whatever the buffer holds; here that is the GAE launch with the bootstrap value of slot T
            buf.compute_returns(None, self.algo_module.get_critic_value_normalizer())
            self.gpu_launches += 1
        if not getattr(buf, "stats_global", False):
            # global advantage / return moments (ppo.py:402-409 semantics); once per compute_returns — a second train() on
            # the same buffer must not sum the already-global moments again
            if self.peer is not None and buf.gae_stats.numel() <= 16:
                lib.check(self._lib.orl_peer_sum_f64(self.peer.args, self.stride, lib.ptr(buf.gae_stats), buf.gae_stats.numel(),
                                                     lib.current_stream()), "orl_peer_sum_f64")
                self.gpu_launches += 1
            else:
                parallel.allreduce_sum_(buf.gae_stats)
            buf.stats_global = True
        if self.recurrent:
            return self._train_recurrent(buf)
        total = buf.episode_length * buf.n_rollout_threads * buf.num_agents
        mb = total // self.num_mini_batch
        whole = self.num_mini_batch == 1
        for _ in range(self.ppo_epoch):
            if self.cfg.parity_mode:
                perm = torch.randperm(total).to(self.device, non_blocking=True)  # global CPU generator, like the reference
                self.h2d_bytes += total * 8
            elif whole:
                perm = None
            else:
                perm = torch.randperm(total, device=self.device)
            for i in range(self.num_mini_batch):
                if whole:
                    # {sum ret, sum ret^2, sum active} over the whole buffer == gae_stats[5:8]
                    self.ppo_update(buf, mb, perm, 0, mb_stats=buf.gae_stats[5:8])
                else:
                    self.ppo_update(buf, mb, perm[i * mb:(i + 1) * mb])
