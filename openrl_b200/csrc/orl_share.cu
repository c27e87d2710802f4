// cfg.use_share_model: ONE policy-value network (reference: PolicyValueNetwork, policy_value_network.py:33-174) with one
// optimiser — rollout, value pass and the PPO update (ppo.py:46-176 with `_use_share_model`: both losses back-propagate
// into the same parameters, both clip_grad_norm_ calls see all of them, one Adam step).
//
// Correctness-first implementation (this option is not on the benchmarked configs): one thread per row runs the
// sequential core of orl_deep_core.h (verified on the CPU against torch autograd of the oracle, tests/test_deep_core_cpu.py);
// the update writes a per-row tape and the parameter gradients are deterministic tape reductions dW = sum_rows P^T Q.
#include <algorithm>

#include "orl_deep_core.h"
#include "orl_envstep.cuh"
#include "orl_loss.cuh"

namespace {
using namespace orl;
namespace dc = orl_deep;

constexpr int S_NT = 128;

__device__ __forceinline__ void load_obs_row(const float* __restrict__ obs, size_t row, int d, float* x) {
    for (int k = 0; k < d; ++k) x[k] = obs[row * d + k];
}

// ---- rollout (single-agent device envs, or ENV_NONE = act only): one thread per env for all steps ----
template <int ENV>
__global__ void __launch_bounds__(S_NT) share_rollout_kernel(const OrlRolloutArgs a) {
    const int N = a.n_envs, B = N * a.n_agents, d = a.obs_dim, n = a.n_actions;
    const int e = blockIdx.x * S_NT + threadIdx.x;
    if (e >= B) return;
    const dc::Offsets o = dc::deep_offsets(d, n);
    const uint64_t rng_base = a.rng_step_base + (a.rng_counter ? *a.rng_counter : 0ull);
    float x[dc::MAXD];
    load_obs_row(a.policy_obs, (size_t)a.t_begin * B + e, d, x);
    for (int t = a.t_begin; t < a.t_end; ++t) {
        float logit[MAX_OUT];
#pragma unroll
        for (int j = 0; j < MAX_OUT; ++j) logit[j] = 0.f;
        dc::deep_forward(a.policy_params, o, a.activation_id, x, nullptr, logit, nullptr, nullptr);
        const size_t grow = (size_t)t * B + e;
        if (a.action_masks) {
#pragma unroll
            for (int j = 0; j < MAX_OUT; ++j) if (j < n && a.action_masks[grow * n + j] == 0.f) logit[j] = -6e4f;
        }
        float nl[MAX_OUT], pr[MAX_OUT];
        log_softmax_n(logit, n, nl, pr);
        int act;
        if (a.deterministic) {
            act = 0;
#pragma unroll
            for (int j = 1; j < MAX_OUT; ++j) if (j < n && pr[j] > pr[act]) act = j;
        } else {
            float q[MAX_OUT];
            if (a.exp_noise) {
#pragma unroll
                for (int j = 0; j < MAX_OUT; ++j) q[j] = (j < n) ? a.exp_noise[grow * n + j] : 1.f;
            } else {
                const uint64_t step = rng_base + (uint64_t)t;
                const uint2 key = make_uint2((uint32_t)a.rng_seed, (uint32_t)(a.rng_seed >> 32));
                const uint4 r0 = philox4x32_10(make_uint4((uint32_t)step, (uint32_t)(step >> 32), (uint32_t)(e + a.rng_row_offset), 0u), key);
                const uint4 r1 = philox4x32_10(make_uint4((uint32_t)step, (uint32_t)(step >> 32), (uint32_t)(e + a.rng_row_offset), 1u), key);
                const uint32_t rr[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
#pragma unroll
                for (int j = 0; j < MAX_OUT; ++j) q[j] = -logf(u32_to_unit_open(rr[j]));
            }
            act = sample_categorical(pr, n, q);
        }
        float lp = nl[0];
#pragma unroll
        for (int j = 1; j < MAX_OUT; ++j) if (j == act) lp = nl[j];
        a.actions[grow] = (float)act;
        a.action_log_probs[grow] = lp;
        if (ENV != ORL_ENV_NONE) {
            if constexpr (ENV == ORL_ENV_CARTPOLE || ENV == ORL_ENV_GRIDWORLD) {
                EnvPtrs E{a.env_f64, a.env_u64, a.env_i32, a.env_table, a.env_table_len, a.rng_seed,
                          a.ep_return, a.ep_length, a.episode_stats, a.rng_row_offset};
                float ob[4], fin[4], reward; bool done;
                env_step_single(E, ENV, e, N, act, ob, reward, done, fin);
                const size_t o1 = (size_t)(t + 1) * B + e;
#pragma unroll
                for (int k = 0; k < 4; ++k) { x[k] = ob[k]; a.policy_obs[o1 * 4 + k] = ob[k]; }
                a.rewards[grow] = reward;
                a.masks[o1] = done ? 0.f : 1.f;
                a.active_masks[o1] = 1.f;
            }
        }
    }
}

__global__ void share_bump_counter_kernel(uint64_t* c, uint64_t by) { *c += by; }

__global__ void __launch_bounds__(S_NT) share_values_kernel(const float* __restrict__ params, int d, int n, int activation_id,
                                                            const float* __restrict__ obs, float* __restrict__ values, long long rows) {
    const long long r = (long long)blockIdx.x * S_NT + threadIdx.x;
    if (r >= rows) return;
    const dc::Offsets o = dc::deep_offsets(d, n);
    float x[dc::MAXD];
    load_obs_row(obs, (size_t)r, d, x);
    float v;
    dc::deep_forward(params, o, activation_id, x, &v, nullptr, nullptr, nullptr);
    values[r] = v;
}

// ---- update: forward + both losses + backward of one minibatch row per thread -> tape row; loss sums -> loss_acc ----
__global__ void __launch_bounds__(S_NT) share_fwdbwd_kernel(const OrlPpoArgs a, float* __restrict__ tape, float* __restrict__ loss_acc) {
    const long long r = (long long)blockIdx.x * S_NT + threadIdx.x;
    const int d = a.obs_dim, n = a.n_actions;
    const dc::Offsets o = dc::deep_offsets(d, n);
    float l_pol = 0.f, l_ent = 0.f, l_ratio = 0.f, l_val = 0.f;
    if (r < a.batch_rows) {
        const long long gi = a.indices ? a.indices[r] : a.row_begin + r;
        const bool pol_masks = a.flags & ORL_PPO_POLICY_ACTIVE_MASKS, val_masks = a.flags & ORL_PPO_VALUE_ACTIVE_MASKS;
        const double rows_d = (double)(a.norm_rows > 0 ? a.norm_rows : a.batch_rows);
        const float inv_rows = (float)(1.0 / rows_d), inv_act = (float)(1.0 / a.mb_stats[2]);
        const AdvNorm advn = make_adv_norm(a.gae_stats, a.flags & ORL_PPO_ADV_NORMALIZE);
        float vn_mean = 0.f, vn_std = 1.f;
        if (a.flags & ORL_PPO_VALUENORM) {
            float st[3];
            vn_updated(a.vn_state, a.mb_stats, rows_d, a.vn_beta, st);
            const VnScalars s = vn_mean_std(st);
            vn_mean = s.mean; vn_std = s.std;
        }
        float x[dc::MAXD];
        load_obs_row(a.policy_obs, (size_t)gi, d, x);
        dc::Save sv;
        float value, logit[MAX_OUT];
#pragma unroll
        for (int j = 0; j < MAX_OUT; ++j) logit[j] = 0.f;
        float* tp = tape + (size_t)r * dc::TAPE;
        dc::deep_forward(a.policy_params, o, a.activation_id, x, &value, logit, &sv, tp);
        const float active = a.active_masks[gi];
        // policy loss (ppo.py:300-319) + entropy (act.py:160-168)
        unsigned masked = 0;
        if (a.action_masks) {
#pragma unroll
            for (int j = 0; j < MAX_OUT; ++j) if (j < n && a.action_masks[gi * n + j] == 0.f) { logit[j] = -6e4f; masked |= 1u << j; }
        }
        float nl[MAX_OUT], pr[MAX_OUT];
        log_softmax_n(logit, n, nl, pr);
        const int act = (int)a.actions[gi];
        float lp = nl[0];
#pragma unroll
        for (int j = 1; j < MAX_OUT; ++j) if (j == act) lp = nl[j];
        const float adv = apply_adv_norm(advn, a.advantages[gi]);
        const PgTerm pg = pg_term(lp, a.old_log_probs[gi], adv, a.clip_param, a.flags, a.dual_clip_coeff);
        const float wrow = pol_masks ? active * inv_act : inv_rows;
        float ent = 0.f;
#pragma unroll
        for (int j = 0; j < MAX_OUT; ++j) if (j < n) ent -= pr[j] * nl[j];
        l_pol = pg.loss * wrow; l_ent = ent * wrow; l_ratio = pg.ratio;
        const float dlp = pg.dlogp * wrow, went = a.entropy_coef * wrow;
        float dl[MAX_OUT];
#pragma unroll
        for (int j = 0; j < MAX_OUT; ++j) {
            dl[j] = 0.f;
            if (j < n && !((masked >> j) & 1u)) dl[j] = dlp * ((j == act ? 1.f : 0.f) - pr[j]) + went * pr[j] * (nl[j] + ent);
        }
        // value loss (ppo.py:178-220)
        const float ret = a.returns[gi];
        const float target = (a.flags & ORL_PPO_VALUENORM) ? (ret - vn_mean) / vn_std : ret;
        const ValueTerm vt = value_term(value, a.value_preds[gi], target, a.clip_param, a.huber_delta, a.flags);
        const float wv = val_masks ? active * inv_act : inv_rows;
        l_val = vt.loss * wv;
        dc::deep_backward(a.policy_params, o, a.activation_id, sv, a.value_loss_coef * wv * vt.dv, dl, tp);
    }
    // block sums -> one atomicAdd per block and slot (order across blocks is not fixed: last-ulp noise on the logged sums only)
    __shared__ float red[4][S_NT / 32];
    float v[4] = {l_pol, l_ent, l_ratio, l_val};
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < 4; ++k) { const float s = warp_sum(v[k]); if (lane == 0) red[k][warp] = s; }
    __syncthreads();
    if (threadIdx.x < 4) {
        float s = 0.f;
        for (int w = 0; w < S_NT / 32; ++w) s += red[threadIdx.x][w];
        atomicAdd(loss_acc + threadIdx.x, s);
    }
}

// ---- tape reductions: out[m*N + k] = sum_rows tape[r][p_off + m] * tape[r][q_off + k]  (q_off < 0: column sum, N = 1) ----
struct SJob { int p_off, M, q_off, N, out_off; };
constexpr int S_MAX_JOBS = 24, SR_ROWS = 512, SR_SUB = 32;
struct SJobs { SJob job[S_MAX_JOBS]; int n; };

__global__ void __launch_bounds__(256) share_tape_reduce_kernel(const float* __restrict__ tape, long long rows, SJobs jobs,
                                                                float* __restrict__ partials, int stride) {
    __shared__ float Ps[SR_SUB][64 + 1], Qs[SR_SUB][64 + 1];
    const SJob jb = jobs.job[blockIdx.y];
    const long long r_begin = (long long)blockIdx.x * SR_ROWS;
    const int rows_here = (int)min((long long)SR_ROWS, rows - r_begin);
    const int tid = threadIdx.x, tk = tid & 15, tm = tid >> 4;   // outputs m = tm + 16 i (i < 4), k = 4 tk + c (c < 4)
    float acc[4][4] = {};
    for (int s0 = 0; s0 < rows_here; s0 += SR_SUB) {
        const int sub = min(SR_SUB, rows_here - s0);
        for (int i = tid; i < SR_SUB * 64; i += 256) {
            const int r = i >> 6, c = i & 63;
            const float* row = tape + (size_t)(r_begin + s0 + (r < sub ? r : 0)) * dc::TAPE;
            Ps[r][c] = (r < sub && c < jb.M) ? row[jb.p_off + c] : 0.f;
            Qs[r][c] = (r < sub && c < jb.N) ? (jb.q_off >= 0 ? row[jb.q_off + c] : 1.f) : 0.f;
        }
        __syncthreads();
        for (int r = 0; r < SR_SUB; ++r) {
            float q[4], p[4];
#pragma unroll
            for (int c = 0; c < 4; ++c) q[c] = Qs[r][4 * tk + c];
#pragma unroll
            for (int i = 0; i < 4; ++i) p[i] = Ps[r][tm + 16 * i];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int c = 0; c < 4; ++c) acc[i][c] = fmaf(p[i], q[c], acc[i][c]);
        }
        __syncthreads();
    }
    float* part = partials + (size_t)blockIdx.x * stride + jb.out_off;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int m = tm + 16 * i;
        if (m < jb.M) {
#pragma unroll
            for (int c = 0; c < 4; ++c) { const int k = 4 * tk + c; if (k < jb.N) part[m * jb.N + k] = acc[i][c]; }
        }
    }
}

__global__ void share_partial_sum_kernel(const float* __restrict__ partials, int row_blocks, int stride, int total, float* __restrict__ grads) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    float s = 0.f;
    for (int rb = 0; rb < row_blocks; ++rb) s += partials[(size_t)rb * stride + i];   // fixed order: deterministic
    grads[i] = s;
}

SJobs make_share_jobs(int d, int n) {
    const dc::Offsets o = dc::deep_offsets(d, n);
    SJobs t; int g = 0;
    auto gemm = [&](int p, int M, int q, int N, int out) { t.job[g++] = SJob{p, M, q, N, out}; };
    auto col = [&](int p, int M, int out) { t.job[g++] = SJob{p, M, -1, 1, out}; };
    gemm(dc::TP_DZ1, dc::H, dc::TQ_X, d, o.w1);       col(dc::TP_DZ1, dc::H, o.b1);  col(dc::TS_DY1N1, dc::H, o.g1); col(dc::TS_DY1, dc::H, o.be1);
    gemm(dc::TP_DZ3, dc::H, dc::TQ_Y1, dc::H, o.w3);  col(dc::TP_DZ3, dc::H, o.b3);  col(dc::TS_DY3N3, dc::H, o.g3); col(dc::TS_DY3, dc::H, o.be3);
    gemm(dc::TP_DZ5, dc::H, dc::TQ_Y3, dc::H, o.w5);  col(dc::TP_DZ5, dc::H, o.b5);  col(dc::TS_DY5N5, dc::H, o.g5); col(dc::TS_DY5, dc::H, o.be5);
    gemm(dc::TP_DZ7, dc::H, dc::TQ_Y5, dc::H, o.w7);  col(dc::TP_DZ7, dc::H, o.b7);  col(dc::TS_DY7N7, dc::H, o.g7); col(dc::TS_DY7, dc::H, o.be7);
    gemm(dc::TP_DV, 1, dc::TQ_Y7, dc::H, o.wv);       col(dc::TP_DV, 1, o.bv);
    gemm(dc::TP_DLOG, n, dc::TQ_Y7, dc::H, o.wa);     col(dc::TP_DLOG, n, o.ba);
    t.n = g;
    return t;
}

// ---- optimiser: ppo.py:120-158 with a shared model — clip_grad_norm_(all) twice, one Adam step (lr = lrs[0]) ----
__global__ void __launch_bounds__(1024) share_apply_kernel(const OrlPpoArgs a, const float* __restrict__ loss_acc) {
    const int total = dc::deep_offsets(a.obs_dim, a.n_actions).total;
    float* params = a.policy_params;
    float* am = a.policy_adam_m;
    float* av = a.policy_adam_v;
    const float* grads = a.grads;
    __shared__ float red[32];
    __shared__ float s_norm;
    const int tid = threadIdx.x;
    float sq = 0.f;
    for (int i = tid; i < total; i += blockDim.x) { const float g = grads[i]; sq = fmaf(g, g, sq); }
    {
        const float s = warp_sum(sq);
        if ((tid & 31) == 0) red[tid >> 5] = s;
        __syncthreads();
        if (tid < 32) {
            float v = (tid < (int)(blockDim.x >> 5)) ? red[tid] : 0.f;
            v = warp_sum(v);
            if (tid == 0) s_norm = sqrtf(v);
        }
        __syncthreads();
    }
    const float norm1 = s_norm;                       // actor_grad_norm: norm before the first clip
    float c1 = 1.f, norm2 = norm1, c2 = 1.f;
    if (a.flags & ORL_PPO_MAX_GRAD_NORM) {
        c1 = fminf(a.max_grad_norm / (norm1 + 1e-6f), 1.0f);
        norm2 = norm1 * c1;                           // critic_grad_norm: what the second clip_grad_norm_ measures
        c2 = fminf(a.max_grad_norm / (norm2 + 1e-6f), 1.0f);
    }
    const float clip = c1 * c2;
    const int step = a.adam_steps[0] + 1;
    const double bc1 = 1.0 - pow((double)a.adam_beta1, (double)step);
    const double bc2 = 1.0 - pow((double)a.adam_beta2, (double)step);
    const float step_size = (float)((double)a.lrs[0] / bc1);
    const float bc2_sqrt = (float)sqrt(bc2);
    for (int i = tid; i < total; i += blockDim.x) {
        float g = grads[i] * clip;
        const float pv = params[i];
        if (a.weight_decay != 0.f) g = fmaf(a.weight_decay, pv, g);
        const float m = am[i] + (g - am[i]) * (1.f - a.adam_beta1);
        const float v = fmaf(av[i], a.adam_beta2, (g * g) * (1.f - a.adam_beta2));
        am[i] = m; av[i] = v;
        params[i] = pv - step_size * (m / (sqrtf(v) / bc2_sqrt + a.adam_eps));
    }
    if (tid == 0) {
        a.adam_steps[0] = step;
        const double rows_d = (double)(a.norm_rows > 0 ? a.norm_rows : a.batch_rows);
        a.train_info[0] += loss_acc[3];
        a.train_info[1] += norm2;
        a.train_info[2] += loss_acc[0];
        a.train_info[3] += loss_acc[1];
        a.train_info[4] += norm1;
        a.train_info[5] += loss_acc[2] / (float)rows_d;
        if (a.flags & ORL_PPO_VALUENORM) {
            float st[3];
            vn_updated(a.vn_state, a.mb_stats, rows_d, a.vn_beta, st);
            a.vn_state[0] = st[0]; a.vn_state[1] = st[1]; a.vn_state[2] = st[2];
        }
    }
}

}  // namespace

extern "C" {

int orl_share_param_count(int obs_dim, int n_actions) { return dc::deep_offsets(obs_dim, n_actions).total; }
int orl_share_tape_width(void) { return dc::TAPE; }
/* floats of the update workspace for a minibatch of `rows` rows: tape rows, then reduction partials */
long long orl_share_workspace_floats(long long rows, int obs_dim, int n_actions) {
    const long long rb = (rows + SR_ROWS - 1) / SR_ROWS;
    return rows * dc::TAPE + rb * (long long)((dc::deep_offsets(obs_dim, n_actions).total + 3) & ~3);
}

int orl_share_rollout(const OrlRolloutArgs* ap, void* stream) {
    ORL_CHECK_ARG(ap, "args");
    const OrlRolloutArgs& a = *ap;
    ORL_CHECK_ARG(a.n_envs > 0 && a.obs_dim > 0 && a.obs_dim <= dc::MAXD && a.n_actions > 0 && a.n_actions <= MAX_OUT, "shapes");
    ORL_CHECK_ARG(a.t_begin >= 0 && a.t_begin < a.t_end, "step range");
    ORL_CHECK_ARG(a.policy_params && a.policy_obs && a.actions && a.action_log_probs, "null buffer");
    ORL_CHECK_ARG(a.head_kind == ORL_HEAD_CATEGORICAL, "the shared-model kernels are built for Discrete action spaces");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const int B = a.n_envs * a.n_agents;
    const int grid = (B + S_NT - 1) / S_NT;
    if (a.env_kind == ORL_ENV_NONE) {
        ORL_CHECK_ARG(a.t_end == a.t_begin + 1, "ORL_ENV_NONE acts for one step per call");
        share_rollout_kernel<ORL_ENV_NONE><<<grid, S_NT, 0, st>>>(a);
    } else if (a.env_kind == ORL_ENV_CARTPOLE) {
        ORL_CHECK_ARG(a.n_agents == 1 && a.obs_dim == 4 && a.n_actions == 2 && a.env_f64 && a.env_u64 && a.env_i32, "CartPole shapes / state");
        share_rollout_kernel<ORL_ENV_CARTPOLE><<<grid, S_NT, 0, st>>>(a);
    } else if (a.env_kind == ORL_ENV_GRIDWORLD) {
        ORL_CHECK_ARG(a.n_agents == 1 && a.obs_dim == 4 && a.n_actions == 5 && a.env_i32, "GridWorld shapes / state");
        share_rollout_kernel<ORL_ENV_GRIDWORLD><<<grid, S_NT, 0, st>>>(a);
    } else {
        orl::set_last_error("orl_share_rollout: env_kind %d is not built for the shared model (single-agent device envs and ORL_ENV_NONE are)", a.env_kind);
        return ORL_ERR_UNSUPPORTED;
    }
    ORL_LAUNCH_CHECK("share_rollout_kernel");
    if (a.rng_counter) {
        share_bump_counter_kernel<<<1, 1, 0, st>>>(a.rng_counter, (uint64_t)(a.t_end - a.t_begin));
        ORL_LAUNCH_CHECK("share_bump_counter_kernel");
    }
    return 0;
}

int orl_share_values(const float* params, int obs_dim, int n_actions, int activation_id, const float* obs, float* values, long long rows,
                     void* stream) {
    ORL_CHECK_ARG(params && obs && values && rows > 0, "null buffer / rows");
    ORL_CHECK_ARG(obs_dim > 0 && obs_dim <= dc::MAXD && n_actions > 0 && n_actions <= MAX_OUT, "shapes");
    share_values_kernel<<<(unsigned)((rows + S_NT - 1) / S_NT), S_NT, 0, reinterpret_cast<cudaStream_t>(stream)>>>(params, obs_dim, n_actions,
                                                                                                               activation_id, obs, values, rows);
    ORL_LAUNCH_CHECK("share_values_kernel");
    return 0;
}

/* forward + losses + backward + deterministic gradient reduction: args->policy_* = the shared model, args->partials =
 * workspace (orl_share_workspace_floats), args->grads = true gradients (out), args->folded[0..3] = loss sums (out) */
int orl_share_fwdbwd(const OrlPpoArgs* ap, void* stream) {
    ORL_CHECK_ARG(ap, "args");
    const OrlPpoArgs& a = *ap;
    ORL_CHECK_ARG(a.obs_dim > 0 && a.obs_dim <= dc::MAXD && a.n_actions > 0 && a.n_actions <= MAX_OUT && a.batch_rows > 0, "shapes");
    ORL_CHECK_ARG(a.policy_params && a.partials && a.folded && a.grads && a.policy_obs && a.actions && a.old_log_probs && a.advantages &&
                      a.value_preds && a.returns && a.active_masks && a.gae_stats && a.mb_stats, "null buffer");
    ORL_CHECK_ARG(a.head_kind == ORL_HEAD_CATEGORICAL, "the shared-model kernels are built for Discrete action spaces");
    if (a.flags & ORL_PPO_JOINT_ACTION) {
        orl::set_last_error("orl_share_fwdbwd: ORL_PPO_JOINT_ACTION needs chunked recurrence (orl_rnn_fwdbwd)");
        return ORL_ERR_UNSUPPORTED;
    }
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    float* tape = a.partials;
    const long long rows = a.batch_rows;
    const int rb = (int)((rows + SR_ROWS - 1) / SR_ROWS);
    const int total = dc::deep_offsets(a.obs_dim, a.n_actions).total, stride = (total + 3) & ~3;
    float* partials = tape + (size_t)rows * dc::TAPE;
    int e = orl::check_cuda(cudaMemsetAsync(a.folded, 0, 8 * sizeof(float), st), "memset loss sums");
    if (e) return e;
    share_fwdbwd_kernel<<<(unsigned)((rows + S_NT - 1) / S_NT), S_NT, 0, st>>>(a, tape, a.folded);
    ORL_LAUNCH_CHECK("share_fwdbwd_kernel");
    const SJobs jobs = make_share_jobs(a.obs_dim, a.n_actions);
    share_tape_reduce_kernel<<<dim3(rb, jobs.n), 256, 0, st>>>(tape, rows, jobs, partials, stride);
    ORL_LAUNCH_CHECK("share_tape_reduce_kernel");
    share_partial_sum_kernel<<<(total + 255) / 256, 256, 0, st>>>(partials, rb, stride, total, a.grads);
    ORL_LAUNCH_CHECK("share_partial_sum_kernel");
    return 0;
}

int orl_share_apply(const OrlPpoArgs* ap, void* stream) {
    ORL_CHECK_ARG(ap, "args");
    const OrlPpoArgs& a = *ap;
    ORL_CHECK_ARG(a.policy_params && a.policy_adam_m && a.policy_adam_v && a.adam_steps && a.lrs && a.grads && a.folded && a.train_info && a.mb_stats,
                  "null buffer");
    share_apply_kernel<<<1, 1024, 0, reinterpret_cast<cudaStream_t>(stream)>>>(a, a.folded);
    ORL_LAUNCH_CHECK("share_apply_kernel");
    return 0;
}

}  // extern "C"
