"""Device-resident rollout storage with the attribute names and shapes of the reference's
`ReplayData` (openrl/buffers/replay_data.py:40-184): float32 torch CUDA tensors

    policy_obs, critic_obs (T+1,N,A,d)   value_preds, returns, masks, bad_masks, active_masks (T+1,N,A,1)
    action_masks (T+1,N,A,n) [Discrete]  actions, action_log_probs, rewards (T,N,A,1)

The env / policy kernels write slots in place (no insert copies); `compute_returns` is the CUDA
GAE scan; minibatch gathers happen inside the PPO kernel.  HBM layout: element (t,n,a,k) at
((t*N+n)*A+a)*K+k, i.e. B = N*A contiguous columns per time slot so that time scans are coalesced.
Unlike the reference, rnn_states* are only allocated for recurrent policies (they are 88 % of the
reference's 308 MB at 4096 envs, SURVEY.md §8a).
"""
import torch

from .. import lib


def chunk_row_indices(chunk_ids, chunk_length, episode_length, rows):
    """Buffer row index t*B + row of every step of the given data chunks, chunk-major / step-minor.

    `recurrent_generator` (replay_data.py:1062-1258) flattens (T, N, A, ...) agent-major / time-minor
    (`_cast`, buffers/utils/util.py:96-97): sample f = (n*A + a)*T + t; chunk c holds f in [c*L, c*L + L) and does
    not stop at trajectory boundaries.  The device buffer keeps the (T, B) layout, so sample f is row
    (f % T)*B + f // T."""
    import torch

    lane = torch.arange(chunk_length, device=chunk_ids.device)
    f = (chunk_ids[:, None] * chunk_length + lane[None, :]).reshape(-1)
    return ((f % episode_length) * rows + f // episode_length).contiguous()


def chunk_row_indices_v3(chunk_ids, chunk_length, episode_length, n_envs, n_agents, agent0_only=False):
    """Buffer row indices of the data chunks of `recurrent_generator_v3` (replay_data.py:425-551, the joint-action
    loss): (T, N, A, ...) is flattened env-major / time-minor (`_cast_v3`, buffers/utils/util.py:99-101), sample
    g = n*T + t carrying all A agents; chunk c holds g in [c*L, c*L + L).  Step g of agent a is buffer row
    (g % T)*N*A + (g // T)*A + a.  Ordered (chunk, step, agent); agent0_only keeps agent 0's rows (the critic's
    `to_single_np`, ppo.py:222-224)."""
    lane = torch.arange(chunk_length, device=chunk_ids.device)
    g = (chunk_ids[:, None] * chunk_length + lane[None, :]).reshape(-1, 1)
    base = (g % episode_length) * (n_envs * n_agents) + (g // episode_length) * n_agents
    agents = torch.arange(1 if agent0_only else n_agents, device=chunk_ids.device)
    return (base + agents[None, :]).reshape(-1).contiguous()


class ReplayData:
    def __init__(self, cfg, num_agents, obs_space, act_space, data_client=None, episode_length=None, device="cuda:0"):
        T = cfg.episode_length if episode_length is None else episode_length
        N, A = cfg.n_rollout_threads, num_agents
        self.episode_length, self.n_rollout_threads, self.num_agents = T, N, A
        self.device = torch.device(device)
        self.gamma, self.gae_lambda = cfg.gamma, cfg.gae_lambda
        self._use_gae = cfg.use_gae
        self._use_popart = cfg.use_popart
        self._use_valuenorm = cfg.use_valuenorm
        self._use_proper_time_limits = cfg.use_proper_time_limits
        if obs_space.__class__.__name__ == "Dict":
            d_p, d_c = obs_space["policy"].shape[0], obs_space["critic"].shape[0]
        else:
            d_p = d_c = obs_space.shape[0]
        self.obs_dim, self.critic_obs_dim = d_p, d_c
        self.continuous = act_space.__class__.__name__ == "Box"
        n = act_space.shape[0] if self.continuous else act_space.n
        self.n_actions = n
        act_w = n if self.continuous else 1   # per-dimension actions / log-probs for Box (distributions.py:35-37)
        f = lambda *s: torch.zeros(*s, dtype=torch.float32, device=self.device)  # noqa: E731
        self.policy_obs = f(T + 1, N, A, d_p)
        # single-observation envs share one tensor (the reference stores two equal copies)
        self.critic_obs = self.policy_obs if d_c == d_p and obs_space.__class__.__name__ != "Dict" else f(T + 1, N, A, d_c)
        self.value_preds = f(T + 1, N, A, 1)
        self.returns = f(T + 1, N, A, 1)
        self.masks = torch.ones(T + 1, N, A, 1, dtype=torch.float32, device=self.device)
        self.bad_masks = torch.ones_like(self.masks)
        self.active_masks = torch.ones_like(self.masks)
        self.action_masks = torch.ones(T + 1, N, A, n, dtype=torch.float32, device=self.device)
        self.action_masks_trivial = True  # all ones: kernels are given NULL
        self.actions = f(T, N, A, act_w)
        self.action_log_probs = f(T, N, A, act_w)
        self.rewards = f(T, N, A, 1)
        self.advantages = f(T, N, A, 1)  # raw returns - V, written by the GAE kernel (ppo.py:384-399)
        self.gae_stats = torch.zeros(8, dtype=torch.float64, device=self.device)
        # hidden states, one per (slot, row): replay_data.py:96-111.  (T+1, N, A, recurrent_N, H)
        self.recurrent = bool(cfg.use_recurrent_policy or getattr(cfg, "use_naive_recurrent_policy", False))
        if self.recurrent:
            self.rnn_states = f(T + 1, N, A, cfg.recurrent_N, cfg.hidden_size)
            self.rnn_states_critic = f(T + 1, N, A, cfg.recurrent_N, cfg.hidden_size)
        else:
            self.rnn_states = self.rnn_states_critic = None
        self.step = 0
        self.returns_ready = False   # set by compute_returns, cleared by after_update (see PPOAlgorithm.train_async)
        self._lib = lib.load()

    @classmethod
    def from_host(cls, host, cfg, value_normalizer=None, device="cuda:0"):
        """Upload a HOST rollout buffer — the reference's numpy `ReplayData` or any object with its attribute names
        (replay_data.py:40-184) — into a device ReplayData: the algorithm-level seam
        `PPOAlgorithm(cfg, module).train(buffer.data)` (tests/test_algorithm/test_ppo_algorithm.py:76-82).
        `returns` are taken as the host buffer holds them; the advantages and their moments are rebuilt on the
        device exactly as train_ppo does (ppo.py:384-409: returns[:-1] - denormalize(value_preds[:-1]))."""
        import numpy as np

        from .. import spaces

        def arr(name):
            v = getattr(host, name)
            if isinstance(v, dict) or hasattr(v, "keys"):       # Dict observations: ObsData of per-key arrays
                v = v["policy" if name == "policy_obs" else "critic"]
            return np.ascontiguousarray(np.asarray(v, dtype=np.float32))

        pobs, cobs = arr("policy_obs"), arr("critic_obs")
        T, N, A = pobs.shape[0] - 1, pobs.shape[1], pobs.shape[2]
        acts = arr("actions")
        am = getattr(host, "action_masks", None)
        if am is not None:
            act_space = spaces.Discrete(int(np.asarray(am).shape[-1]))
        else:
            act_space = spaces.Box(-np.inf, np.inf, (acts.shape[-1],), np.float32)
        same = pobs.shape == cobs.shape and np.array_equal(pobs, cobs)
        box = lambda d: spaces.Box(-np.inf, np.inf, (d,), np.float32)   # noqa: E731
        obs_space = box(pobs.shape[-1]) if same else spaces.Dict({"policy": box(pobs.shape[-1]), "critic": box(cobs.shape[-1])})
        import copy

        c2 = copy.copy(cfg)
        c2.n_rollout_threads = N
        self = cls(c2, A, obs_space, act_space, episode_length=T, device=device)
        staged = 0
        for name in ("value_preds", "returns", "masks", "bad_masks", "active_masks", "actions", "action_log_probs", "rewards"):
            h = torch.from_numpy(arr(name))
            getattr(self, name).copy_(h.view_as(getattr(self, name)), non_blocking=False)
            staged += h.numel() * 4
        self.policy_obs.copy_(torch.from_numpy(pobs).view_as(self.policy_obs))
        if self.critic_obs is not self.policy_obs:
            self.critic_obs.copy_(torch.from_numpy(cobs).view_as(self.critic_obs))
        staged += pobs.size * 4 + (0 if same else cobs.size * 4)
        if am is not None:
            amh = torch.from_numpy(np.ascontiguousarray(np.asarray(am, dtype=np.float32)))
            self.action_masks.copy_(amh.view_as(self.action_masks))
            self.action_masks_trivial = bool((amh == 1).all())
            staged += amh.numel() * 4
        if self.recurrent:
            for name in ("rnn_states", "rnn_states_critic"):
                getattr(self, name).copy_(torch.from_numpy(arr(name)).view_as(getattr(self, name)))
        self.h2d_bytes = staged
        self.rebuild_advantages(value_normalizer)
        return self

    def rebuild_advantages(self, value_normalizer=None):
        """advantages = returns[:-1] - denormalize(value_preds[:-1]) and the moment vector `gae_stats` that
        orl_gae would have produced (ppo.py:384-409); used when returns come from outside (host buffers)."""
        vp = self.value_preds[:-1]
        if (self._use_popart or self._use_valuenorm) and value_normalizer is not None:
            m, var = value_normalizer.running_mean_var()
            vp = vp * torch.sqrt(var) + m
        self.advantages.copy_(self.returns[:-1] - vp)
        adv = self.advantages.double().view(-1)
        act = (self.active_masks[:-1].view(-1) != 0).double()
        ret = self.returns[:-1].double().view(-1)
        self.gae_stats.copy_(torch.stack([adv.sum(), (adv * adv).sum(), torch.tensor(float(adv.numel()), dtype=torch.float64, device=self.device),
                                          (adv * act).sum(), (adv * adv * act).sum(), ret.sum(), (ret * ret).sum(),
                                          self.active_masks[:-1].double().sum()]))
        self.returns_ready = True
        self.stats_global = False   # gae_stats now hold this rank's moments only (PPOAlgorithm.train_async all-reduces them once)

    def init_buffer(self, raw_obs, action_masks=None):
        """replay_data.py:286-298 — slot 0 <- first observation (host array or device tensor)."""
        obs = torch.as_tensor(raw_obs, dtype=torch.float32).to(self.device)
        self.policy_obs[0].copy_(obs.view_as(self.policy_obs[0]))

    def after_update(self):
        """replay_data.py:300-318 — slot T becomes slot 0 of the next rollout."""
        self.returns_ready = False
        self.policy_obs[0].copy_(self.policy_obs[-1])
        if self.critic_obs is not self.policy_obs:
            self.critic_obs[0].copy_(self.critic_obs[-1])
        self.masks[0].copy_(self.masks[-1])
        self.bad_masks[0].copy_(self.bad_masks[-1])
        self.active_masks[0].copy_(self.active_masks[-1])
        if not self.action_masks_trivial:
            self.action_masks[0].copy_(self.action_masks[-1])
        if self.recurrent:
            self.rnn_states[0].copy_(self.rnn_states[-1])
            self.rnn_states_critic[0].copy_(self.rnn_states_critic[-1])

    def compute_returns(self, next_value, value_normalizer=None):
        """replay_data.py:320-423 on the device (orl_gae), fused with the advantage build.

        next_value: (N,A,1) device tensor, or None when value_preds[-1] already holds the
        bootstrap value (written there by orl_critic_values)."""
        T, B = self.episode_length, self.n_rollout_threads * self.num_agents
        flags = (lib.GAE_USE_GAE if self._use_gae else 0) | (lib.GAE_PROPER_TIME_LIMITS if self._use_proper_time_limits else 0)
        vn = None
        if (self._use_popart or self._use_valuenorm) and value_normalizer is not None:
            flags |= lib.GAE_DENORM
            vn = value_normalizer.state
        nv = self.value_preds[-1] if next_value is None else torch.as_tensor(next_value, dtype=torch.float32).to(self.device).contiguous()
        lib.check(self._lib.orl_gae(lib.ptr(self.rewards), lib.ptr(self.value_preds), lib.ptr(self.masks),
                                    lib.ptr(self.bad_masks), lib.ptr(self.active_masks), lib.ptr(nv), lib.ptr(vn),
                                    lib.ptr(self.returns), lib.ptr(self.advantages), lib.ptr(self.gae_stats), T, B,
                                    float(self.gamma), float(self.gae_lambda), flags, lib.current_stream()), "orl_gae")
        self.returns_ready = True
        self.stats_global = False   # gae_stats now hold this rank's moments only (PPOAlgorithm.train_async all-reduces them once)
