// Recurrent (GRU) policy / value networks: rollout, critic pass, chunked-BPTT update, optimizer.
//
// Replaces, for cfg.use_recurrent_policy:
//   RNNLayer.forward                      openrl/modules/networks/utils/rnn.py:39-99
//   OnPolicyDriver.act / add2buffer       openrl/drivers/onpolicy_driver.py:80-152,236-279 (rnn-state carry,
//                                         zeroing on dones_env)
//   ReplayData.recurrent_generator        openrl/buffers/replay_data.py:1062-1258 (chunks of L over f=(n*A+a)*T+t)
//   ReplayData.recurrent_generator_v3     openrl/buffers/replay_data.py:425-551 (JRPO: chunks of L over g=n*T+t, all agents
//                                         of a step together; joint-action loss ppo.py:254-321)
//   PPOAlgorithm.ppo_update (BPTT part)   openrl/algorithms/ppo.py:46-458
//
// Design (DESIGN.md "recurrent path"): ONE WARP per env (rollout), per row (critic) or per chunk (update) running
// the warp-cooperative step of orl_rnn_warp.cuh — 64-vectors as two registers per lane, the net's weights staged
// once per persistent CTA in 136 KB of shared memory, mat-vecs by shuffle broadcast (shared-memory-bandwidth
// bound: one LDS per FMA).  The update writes a per-row-step tape (forward activations, local gradients);
// parameter gradients are reductions of the tape, dW = sum_rows P^T Q, by a staged-GEMM kernel with float atomics
// into the true-layout gradient buffer.  The sequential restatement of the same step (orl_rnn_core.h, pinned to
// the torch oracle on the CPU) serves PPOModule.act and is the element-wise checker of the warp path
// (tests/debug_gru.py).
#include <algorithm>

#include "orl_envstep.cuh"
#include "orl_loss.cuh"
#include "orl_rnn_core.h"
#include "orl_rnn_warp.cuh"

namespace {
using namespace orl;
namespace rc = orl_rnn;
namespace rw = orl_rnnw;

static_assert(rc::MAXN == MAX_OUT, "head width limits must agree");
constexpr int LMAX = 32;     // data_chunk_length limit accepted by the host API (the chunk kernels loop over l; the tape is n_chunks * L rows)
constexpr int RNN_NT = 64;   // threads per CTA of the sequential kernels

__device__ __forceinline__ int pick_action(const OrlRnnArgs& a, const float (&pr)[MAX_OUT], int n, size_t grow, int row,
                                           int t, uint64_t rng_base) {
    if (a.deterministic) {
        int act = 0;
#pragma unroll
        for (int j = 1; j < MAX_OUT; ++j) if (j < n && pr[j] > pr[act]) act = j;
        return act;
    }
    float q[MAX_OUT];
    if (a.exp_noise) {
#pragma unroll
        for (int j = 0; j < MAX_OUT; ++j) q[j] = (j < n) ? a.exp_noise[grow * n + j] : 1.f;
    } else {
        const uint64_t step = rng_base + (uint64_t)t;
        const uint2 key = make_uint2((uint32_t)a.rng_seed, (uint32_t)(a.rng_seed >> 32));
        const uint4 r0 = philox4x32_10(make_uint4((uint32_t)step, (uint32_t)(step >> 32), (uint32_t)row, 0u), key);
        const uint4 r1 = philox4x32_10(make_uint4((uint32_t)step, (uint32_t)(step >> 32), (uint32_t)row, 1u), key);
        const uint32_t rr[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
#pragma unroll
        for (int j = 0; j < MAX_OUT; ++j) q[j] = -logf(u32_to_unit_open(rr[j]));
    }
    return sample_categorical(pr, n, q);
}

// ---- act only (PPOModule.act / PPONet.act): one thread per row runs the sequential core; the caller owns env.step ----
__global__ void __launch_bounds__(RNN_NT) rnn_act_kernel(const OrlRnnArgs a) {
    const int B = a.n_envs, n = a.n_actions, d = a.obs_dim;
    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= B) return;
    const rc::Offsets o = rc::rnn_offsets(d, n);
    const uint64_t rng_base = a.rng_step_base + (a.rng_counter ? *a.rng_counter : 0ull);
    for (int t = a.t_begin; t < a.t_end; ++t) {
        const size_t grow = (size_t)t * B + row;
        float x[rc::MAXD], h[rc::H], hn[rc::H], logit[MAX_OUT];
        for (int k = 0; k < rc::MAXD; ++k) x[k] = k < d ? a.policy_obs[grow * d + k] : 0.f;
        for (int j = 0; j < rc::H; ++j) h[j] = a.rnn_states[grow * rc::H + j];
        rc::rnn_step_forward(a.policy_params, o, a.activation_id, x, h, a.masks[grow], hn, logit, nullptr, nullptr);
        for (int j = 0; j < rc::H; ++j) a.rnn_states[((size_t)(t + 1) * B + row) * rc::H + j] = hn[j];
#pragma unroll
        for (int j = 0; j < MAX_OUT; ++j) if (j >= n) logit[j] = 0.f;
        float nl[MAX_OUT], pr[MAX_OUT];
        log_softmax_n(logit, n, nl, pr);
        const int act = pick_action(a, pr, n, grow, row, t, rng_base);
        float lp = nl[0];
#pragma unroll
        for (int j = 1; j < MAX_OUT; ++j) if (j == act) lp = nl[j];
        a.actions[grow] = (float)act;
        a.action_log_probs[grow] = lp;
    }
}

__global__ void rnn_bump_counter_kernel(uint64_t* c, uint64_t by) { *c += by; }

constexpr int W_NT = 512, W_WPC = W_NT / 32;   // one persistent CTA per SM, 16 warps, weights of one net in smem

// ---- rollout: one warp per env advances its A agent rows together; env.step on lane 0 ----
template <int ENV>
__global__ void __launch_bounds__(W_NT, 1) rnn_rollout_warp_kernel(const OrlRnnArgs a) {
    extern __shared__ __align__(16) float smem[];
    constexpr int A = ENV == ORL_ENV_MPE_SPREAD ? 3 : 1;
    constexpr int D = ENV == ORL_ENV_MPE_SPREAD ? 18 : 4;
    const int N = a.n_envs, B = N * A, n = a.n_actions;
    const rc::Offsets o = rc::rnn_offsets(D, n);
    const rw::SmemNet W = rw::load_net(smem, a.policy_params, o, threadIdx.x, W_NT);
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float* scr = smem + rw::smem_net_floats() + warp * A * rw::SCR;
    EnvPtrs E{a.env_f64, a.env_u64, a.env_i32, a.env_table, a.env_table_len, a.rng_seed, a.ep_return, a.ep_length, a.episode_stats};
    const uint64_t rng_base = a.rng_step_base + (a.rng_counter ? *a.rng_counter : 0ull);
    float* const no_tape[A] = {};
    for (int e = blockIdx.x * W_WPC + warp; e < N; e += gridDim.x * W_WPC) {
        for (int t = a.t_begin; t < a.t_end; ++t) {
            rw::V2 x[A], h[A], hn[A];
            float mk[A], logit[A][MAX_OUT];
            int acts[A];
#pragma unroll
            for (int ag = 0; ag < A; ++ag) {
                const size_t grow = (size_t)t * B + e * A + ag;
                const float* ob = a.policy_obs + grow * D;
                x[ag] = rw::V2{lane < D ? ob[lane] : 0.f, lane + 32 < D ? ob[lane + 32] : 0.f};
                h[ag] = rw::ldv(a.rnn_states + grow * rc::H, lane);
                mk[ag] = a.masks[grow];
            }
            rw::step_forward<A>(W, scr, D, n, a.activation_id, x, h, mk, hn, logit, no_tape, lane);
#pragma unroll
            for (int ag = 0; ag < A; ++ag) {
                const int row = e * A + ag;
                const size_t grow = (size_t)t * B + row;
                float nl[MAX_OUT], pr[MAX_OUT];
                log_softmax_n(logit[ag], n, nl, pr);                 // identical on every lane
                const int act = pick_action(a, pr, n, grow, row, t, rng_base);
                float lp = nl[0];
#pragma unroll
                for (int j = 1; j < MAX_OUT; ++j) if (j == act) lp = nl[j];
                if (lane == 0) { a.actions[grow] = (float)act; a.action_log_probs[grow] = lp; }
                acts[ag] = act;
            }
            int done_i = 0;
            if (lane == 0) {
                bool done = false; float reward = 0.f;
                if constexpr (ENV == ORL_ENV_MPE_SPREAD) {
                    float ob[3][18];
                    const int acts3[3] = {acts[0], acts[A > 1 ? 1 : 0], acts[A > 2 ? 2 : 0]};
                    env_step_mpe(E, e, N, acts3, ob, reward, done);
                    const size_t r1 = (size_t)(t + 1) * B + (size_t)e * 3;
                    for (int ag = 0; ag < 3; ++ag)
                        for (int k = 0; k < 18; ++k) {
                            a.policy_obs[(r1 + ag) * 18 + k] = ob[ag][k];
                            for (int dst = 0; dst < 3; ++dst) a.critic_obs[(r1 + dst) * 54 + ag * 18 + k] = ob[ag][k];
                        }
                } else {
                    float ob[4], fin[4];
                    env_step_single(E, ENV, e, N, acts[0], ob, reward, done, fin);
                    const size_t o1 = (size_t)(t + 1) * B + e;
                    for (int k = 0; k < 4; ++k) {
                        a.policy_obs[o1 * 4 + k] = ob[k];
                        if (a.critic_obs != a.policy_obs) a.critic_obs[o1 * 4 + k] = ob[k];
                    }
                }
                for (int ag = 0; ag < A; ++ag) {
                    const size_t r1 = (size_t)(t + 1) * B + (size_t)e * A + ag;
                    a.rewards[(size_t)t * B + (size_t)e * A + ag] = reward;
                    a.masks[r1] = done ? 0.f : 1.f;
                    a.active_masks[r1] = 1.f;
                }
                done_i = done ? 1 : 0;
            }
            done_i = __shfl_sync(0xffffffffu, done_i, 0);
#pragma unroll
            for (int ag = 0; ag < A; ++ag) {   // rnn_states[dones_env] = 0 (onpolicy_driver.py:262-269)
                const size_t r1 = (size_t)(t + 1) * B + (size_t)e * A + ag;
                rw::stv(a.rnn_states + r1 * rc::H, lane, done_i ? rw::V2{0.f, 0.f} : hn[ag]);
            }
            __syncwarp();   // lane 0's observation / mask writes are read by the whole warp in the next step
        }
    }
}

// ---- recurrent critic over all T+1 slots: one warp per row ----
__global__ void __launch_bounds__(W_NT, 1) rnn_critic_warp_kernel(const OrlRnnArgs a) {
    extern __shared__ __align__(16) float smem[];
    const int B = a.n_envs * a.n_agents, T = a.episode_length, dc = a.critic_obs_dim;
    const rc::Offsets o = rc::rnn_offsets(dc, 1);
    const rw::SmemNet W = rw::load_net(smem, a.critic_params, o, threadIdx.x, W_NT);
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float* scr = smem + rw::smem_net_floats() + warp * rw::SCR;
    float* const no_tape[1] = {nullptr};
    for (int row = blockIdx.x * W_WPC + warp; row < B; row += gridDim.x * W_WPC) {
        rw::V2 h[1] = {rw::ldv(a.rnn_states_critic + (size_t)row * rc::H, lane)};
        for (int t = 0; t <= T; ++t) {
            const size_t grow = (size_t)t * B + row;
            const float* ob = a.critic_obs + grow * dc;
            const rw::V2 x[1] = {rw::V2{lane < dc ? ob[lane] : 0.f, lane + 32 < dc ? ob[lane + 32] : 0.f}};
            const float mk[1] = {a.masks[grow]};
            rw::V2 hn[1]; float out[1][MAX_OUT];
            rw::step_forward<1>(W, scr, dc, 1, a.activation_id, x, h, mk, hn, out, no_tape, lane);
            if (lane == 0) a.value_preds[grow] = out[0][0];
            if (t < T) {
                const float keep = a.masks[grow + B] == 0.f ? 0.f : 1.f;   // rnn_states_critic[dones_env] = 0
                h[0] = rw::V2{hn[0].a * keep, hn[0].b * keep};
                rw::stv(a.rnn_states_critic + (grow + B) * rc::H, lane, h[0]);
            }
        }
    }
}

// ---- update: one warp per C_R chunks; L forward steps (tape), per-step loss, L backward steps ----
// JOINT (ORL_PPO_JOINT_ACTION, chunks over g = n*T + t): the policy warp owns ONE chunk and its C_R = A agent rows
// (tape row (cpos*L + l)*A + a) and takes the joint-action loss once per step; the critic warp runs agent 0's row
// n*A of each of its C_R chunks.
template <bool POLICY, int C_R, int C_NT, bool JOINT = false>
__global__ void __launch_bounds__(C_NT, 1) rnn_chunk_warp_kernel(const OrlRnnArgs a) {
    constexpr int C_WPC = C_NT / 32;
    constexpr bool JPOL = JOINT && POLICY;   // the warp's rows are the agents of one chunk
    extern __shared__ __align__(16) float smem[];
    const int B = a.n_envs * a.n_agents, T = a.episode_length, L = a.chunk_length;
    const int rstride = JOINT ? a.n_agents : 1;   // buffer row of flattened sample f (agent r): (f / T) * rstride + r
    const int d = POLICY ? a.obs_dim : a.critic_obs_dim, n = POLICY ? a.n_actions : 1;
    const float* obs = POLICY ? a.policy_obs : a.critic_obs;
    const float* states = POLICY ? a.rnn_states : a.rnn_states_critic;
    const rc::Offsets o = rc::rnn_offsets(d, n);
    const rw::SmemNet W = rw::load_net(smem, POLICY ? a.policy_params : a.critic_params, o, threadIdx.x, C_NT);
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float* scr = smem + rw::smem_net_floats() + warp * C_R * rw::SCR;
    float loss0 = 0.f, loss1 = 0.f, loss2 = 0.f;   // identical on every lane; lane 0's copy is reduced

    const double rows_d = a.norm_rows > 0 ? (double)a.norm_rows : (double)a.n_chunks * L;   // JOINT: chunk steps
    const float inv_rows = (float)(1.0 / rows_d);
    const float inv_act = (float)(1.0 / a.mb_stats[2]);   // JOINT: agent 0's active sum
    // JRPO entropy: mean over all agent rows, or weighted by every agent's active mask (act.py:114-118)
    const float inv_ent_rows = JPOL ? (float)(1.0 / (rows_d * C_R)) : inv_rows;
    const float inv_ent_act = JPOL ? (float)(1.0 / a.mb_stats[3]) : inv_act;
    const bool pol_masks = a.flags & ORL_PPO_POLICY_ACTIVE_MASKS, val_masks = a.flags & ORL_PPO_VALUE_ACTIVE_MASKS;
    AdvNorm advn;
    float vn_mean = 0.f, vn_std = 1.f;
    if (POLICY) advn = make_adv_norm(a.gae_stats, a.flags & ORL_PPO_ADV_NORMALIZE);
    else if (a.flags & ORL_PPO_VALUENORM) {
        float st[3];
        vn_updated(a.vn_state, a.mb_stats, rows_d, a.vn_beta, st);
        const VnScalars s = vn_mean_std(st);
        vn_mean = s.mean; vn_std = s.std;
    }

    const long long n_groups = JPOL ? a.n_chunks : (a.n_chunks + C_R - 1) / C_R;
    for (long long grp = (long long)blockIdx.x * C_WPC + warp; grp < n_groups; grp += (long long)gridDim.x * C_WPC) {
        long long cpos[C_R], f0[C_R];
        int agent[C_R];
        bool valid[C_R];
        rw::V2 h[C_R];
#pragma unroll
        for (int r = 0; r < C_R; ++r) {
            if (JPOL) {
                valid[r] = true; cpos[r] = grp; agent[r] = r;
            } else {
                valid[r] = grp * C_R + r < a.n_chunks;
                cpos[r] = valid[r] ? grp * C_R + r : grp * C_R;   // a tail slot recomputes chunk 0 of the group (same values, same addresses)
                agent[r] = 0;
            }
            f0[r] = a.chunk_ids[cpos[r]] * (long long)L;
            h[r] = rw::ldv(states + ((size_t)(f0[r] % T) * B + (size_t)(f0[r] / T) * rstride + agent[r]) * rc::H, lane);
        }
        for (int l = 0; l < L; ++l) {
            rw::V2 x[C_R], h2[C_R];
            float mk[C_R], out[C_R][MAX_OUT];
            float* tape[C_R];
            size_t bi[C_R];
#pragma unroll
            for (int r = 0; r < C_R; ++r) {
                const long long f = f0[r] + l, row = (f / T) * rstride + agent[r], t = f % T;
                bi[r] = (size_t)t * B + row;
                const float* ob = obs + bi[r] * d;
                x[r] = rw::V2{lane < d ? ob[lane] : 0.f, lane + 32 < d ? ob[lane + 32] : 0.f};
                mk[r] = a.masks[bi[r]];
                tape[r] = a.tape + (JPOL ? ((size_t)cpos[r] * L + l) * C_R + r : (size_t)cpos[r] * L + l) * rw::TAPE_W;
            }
            rw::step_forward<C_R>(W, scr, d, n, a.activation_id, x, h, mk, h2, out, tape, lane);
            if constexpr (JPOL) {
                // joint log-prob of the step: register sum over the warp's agent rows, in agent order (ppo.py:284-300)
                float joint = 0.f, old_joint = 0.f;
#pragma unroll
                for (int r = 0; r < C_R; ++r) {
                    h[r] = h2[r];
                    float nl[MAX_OUT], pr[MAX_OUT];
                    log_softmax_n(out[r], n, nl, pr);
                    const int act = (int)a.actions[bi[r]];
                    float lp = nl[0];
#pragma unroll
                    for (int j = 1; j < MAX_OUT; ++j) if (j == act) lp = nl[j];
                    joint += lp;
                    old_joint += a.action_log_probs[bi[r]];
                }
                const float adv = apply_adv_norm(advn, a.advantages[bi[0]]);
                const PgTerm pg = pg_term(joint, old_joint, adv, a.clip_param, a.flags, a.dual_clip_coeff);
                const float wrow = pol_masks ? a.active_masks[bi[0]] * inv_act : inv_rows;
                loss0 += pg.loss * wrow; loss2 += pg.ratio;
                const float dlp = pg.dlogp * wrow;   // every agent row of the step receives the same dL/dlogp_joint
#pragma unroll
                for (int r = 0; r < C_R; ++r) {
                    float nl[MAX_OUT], pr[MAX_OUT], dl[MAX_OUT];
                    log_softmax_n(out[r], n, nl, pr);
                    const int act = (int)a.actions[bi[r]];
                    const float went = pol_masks ? a.active_masks[bi[r]] * inv_ent_act : inv_ent_rows;
                    float ent = 0.f;
#pragma unroll
                    for (int j = 0; j < MAX_OUT; ++j) if (j < n) ent -= pr[j] * nl[j];
                    loss1 += ent * went;
                    const float wec = a.entropy_coef * went;
#pragma unroll
                    for (int j = 0; j < MAX_OUT; ++j)
                        dl[j] = j < n ? dlp * ((j == act ? 1.f : 0.f) - pr[j]) + wec * pr[j] * (nl[j] + ent) : 0.f;
                    float mine = 0.f;   // lane m < 8 stores dL/dout[m]
#pragma unroll
                    for (int j = 0; j < MAX_OUT; ++j) if (lane == j) mine = dl[j];
                    if (lane < MAX_OUT) tape[r][rc::TP_DLOG + lane] = mine;
                }
            } else {
#pragma unroll
                for (int r = 0; r < C_R; ++r) {
                    h[r] = h2[r];
                    float dl[MAX_OUT];
#pragma unroll
                    for (int j = 0; j < MAX_OUT; ++j) dl[j] = 0.f;
                    const float active = a.active_masks[bi[r]];
                    const float keep = valid[r] ? 1.f : 0.f;
                    if (POLICY) {
                        float nl[MAX_OUT], pr[MAX_OUT];
                        log_softmax_n(out[r], n, nl, pr);
                        const int act = (int)a.actions[bi[r]];
                        float lp = nl[0];
#pragma unroll
                        for (int j = 1; j < MAX_OUT; ++j) if (j == act) lp = nl[j];
                        const float adv = apply_adv_norm(advn, a.advantages[bi[r]]);
                        const PgTerm pg = pg_term(lp, a.action_log_probs[bi[r]], adv, a.clip_param, a.flags, a.dual_clip_coeff);
                        const float wrow = pol_masks ? active * inv_act : inv_rows;
                        float ent = 0.f;
#pragma unroll
                        for (int j = 0; j < MAX_OUT; ++j) if (j < n) ent -= pr[j] * nl[j];
                        loss0 += keep * pg.loss * wrow; loss1 += keep * ent * wrow; loss2 += keep * pg.ratio;
                        const float dlp = pg.dlogp * wrow, went = a.entropy_coef * wrow;
#pragma unroll
                        for (int j = 0; j < MAX_OUT; ++j)
                            if (j < n) dl[j] = dlp * ((j == act ? 1.f : 0.f) - pr[j]) + went * pr[j] * (nl[j] + ent);
                    } else {
                        const float ret = a.returns[bi[r]];
                        const float target = (a.flags & ORL_PPO_VALUENORM) ? (ret - vn_mean) / vn_std : ret;
                        const ValueTerm vt = value_term(out[r][0], a.value_preds[bi[r]], target, a.clip_param, a.huber_delta, a.flags);
                        const float wrow = val_masks ? active * inv_act : inv_rows;
                        loss0 += keep * vt.loss * wrow;
                        dl[0] = a.value_loss_coef * wrow * vt.dv;
                    }
                    float mine = 0.f;   // lane m < 8 stores dL/dout[m]
#pragma unroll
                    for (int j = 0; j < MAX_OUT; ++j) if (lane == j) mine = dl[j];
                    if (lane < MAX_OUT) tape[r][rc::TP_DLOG + lane] = mine;
                }
            }
        }
        __syncwarp();   // tape scalars (lane 0) and dL/dout (lanes < 8) are read by every lane below
        rw::V2 dh[C_R];
#pragma unroll
        for (int r = 0; r < C_R; ++r) dh[r] = rw::V2{0.f, 0.f};
        for (int l = L - 1; l >= 0; --l) {
            float* tape[C_R];
#pragma unroll
            for (int r = 0; r < C_R; ++r)
                tape[r] = a.tape + (JPOL ? ((size_t)cpos[r] * L + l) * C_R + r : (size_t)cpos[r] * L + l) * rw::TAPE_W;
            rw::step_backward<C_R>(W, scr, n, a.activation_id, tape, dh, lane);
        }
    }
    __shared__ float red[3][C_WPC];
    if (lane == 0) { red[0][warp] = loss0; red[1][warp] = loss1; red[2][warp] = loss2; }
    __syncthreads();
    if (threadIdx.x < 3) {
        float s = 0.f;
        for (int w = 0; w < C_WPC; ++w) s += red[threadIdx.x][w];
        if (POLICY) atomicAdd(a.loss_acc + threadIdx.x, s);
        else if (threadIdx.x == 0) atomicAdd(a.loss_acc + 3, s);
    }
}

// ---- tape reductions (deterministic, two stages) ----
// Stage 1: every CTA owns TR_ROWS tape rows and one job and writes its partial result to partials[row_block][...]:
//   gemm job   part[out_off + m*N + k] = sum_rows tape[r][p_off+m] * tape[r][q_off+k]     (register-tiled, 12x4 per thread)
//   column job part[out_off + m]       = sum_rows tape[r][p_off+m]
// Stage 2: grads[i] = sum over row blocks of partials[rb][i], fixed order.
struct TapeJob { int p_off, M, q_off, N, out_off; };
constexpr int MAX_GEMM_JOBS = 5, MAX_COL_JOBS = 11;
struct TapeJobs { TapeJob gemm[MAX_GEMM_JOBS]; TapeJob col[MAX_COL_JOBS]; int n_gemm, n_col; };
constexpr int TR_NT = 256, TR_ROWS = 1024, TR_SUB = 32, TR_MI = rc::G3 / 16;   // 16 x 16 threads; thread tile (M/16) x 4

__device__ __forceinline__ void cp_async16(float* smem_dst, const float* gmem_src, bool valid) {
    const unsigned dst = (unsigned)__cvta_generic_to_shared(smem_dst);
    const int src_size = valid ? 16 : 0;   // 0: the 16 bytes are zero-filled
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(dst), "l"(gmem_src), "r"(src_size));
}
constexpr size_t TR_SMEM = 2 * (size_t)TR_SUB * (rc::G3 + rc::H) * sizeof(float);   // two stages of P and Q tiles

__global__ void __launch_bounds__(TR_NT) tape_gemm_kernel(const float* __restrict__ tape, long long rows, TapeJobs jobs,
                                                          float* __restrict__ partials, int stride) {
    extern __shared__ __align__(16) float tsm[];
    const TapeJob jb = jobs.gemm[blockIdx.y];
    const long long r_begin = (long long)blockIdx.x * TR_ROWS;
    const int rows_here = (int)min((long long)TR_ROWS, rows - r_begin);
    auto Ps = [&](int buf) { return tsm + buf * (TR_SUB * rc::G3); };
    auto Qs = [&](int buf) { return tsm + 2 * TR_SUB * rc::G3 + buf * (TR_SUB * rc::H); };
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int MI = (jb.M + 15) >> 4, Mq = MI * 4;   // P columns are read in whole float4 up to 16*MI (fields are zero / foreign beyond M: discarded)
    // stage loader: rows beyond the block's tail are zero-filled
    auto load_stage = [&](int buf, int s0) {
        const int sub = min(TR_SUB, rows_here - s0);
        const float* base = tape + (size_t)(r_begin + s0) * rw::TAPE_W;
        for (int i = tid; i < TR_SUB * Mq; i += TR_NT) {
            const int r = i / Mq, c = i % Mq;
            cp_async16(Ps(buf) + r * rc::G3 + 4 * c, base + (size_t)(r < sub ? r : 0) * rw::TAPE_W + jb.p_off + 4 * c, r < sub);
        }
        for (int i = tid; i < TR_SUB * (rc::H / 4); i += TR_NT) {
            const int r = i >> 4, c = i & 15;
            cp_async16(Qs(buf) + r * rc::H + 4 * c, base + (size_t)(r < sub ? r : 0) * rw::TAPE_W + jb.q_off + 4 * c, r < sub);
        }
        asm volatile("cp.async.commit_group;\n" ::);
    };
    float acc[TR_MI][4];
#pragma unroll
    for (int i = 0; i < TR_MI; ++i) { acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.f; }
    const int n_sub = (rows_here + TR_SUB - 1) / TR_SUB;
    load_stage(0, 0);
    for (int s = 0; s < n_sub; ++s) {
        const int buf = s & 1;
        if (s + 1 < n_sub) { load_stage(buf ^ 1, (s + 1) * TR_SUB); asm volatile("cp.async.wait_group 1;\n" ::); }
        else asm volatile("cp.async.wait_group 0;\n" ::);
        __syncthreads();
        const float* P = Ps(buf);
        const float* Q = Qs(buf);
#pragma unroll 4
        for (int r = 0; r < TR_SUB; ++r) {
            const float4 q = *reinterpret_cast<const float4*>(Q + r * rc::H + 4 * tx);
#pragma unroll
            for (int i = 0; i < TR_MI; ++i) {
                if (i < MI) {
                    const float p = P[r * rc::G3 + ty + 16 * i];
                    acc[i][0] = fmaf(p, q.x, acc[i][0]); acc[i][1] = fmaf(p, q.y, acc[i][1]);
                    acc[i][2] = fmaf(p, q.z, acc[i][2]); acc[i][3] = fmaf(p, q.w, acc[i][3]);
                }
            }
        }
        __syncthreads();   // the stage just read is refilled by the next iteration's load
    }
    float* part = partials + (size_t)blockIdx.x * stride + jb.out_off;
#pragma unroll
    for (int i = 0; i < TR_MI; ++i) {
        const int m = ty + 16 * i;
        if (i < MI && m < jb.M) {
#pragma unroll
            for (int c = 0; c < 4; ++c) { const int k = 4 * tx + c; if (k < jb.N) part[m * jb.N + k] = acc[i][c]; }
        }
    }
}

__global__ void __launch_bounds__(rc::G3) tape_colsum_kernel(const float* __restrict__ tape, long long rows, TapeJobs jobs,
                                                             float* __restrict__ partials, int stride) {
    const TapeJob jb = jobs.col[blockIdx.y];
    const long long r_begin = (long long)blockIdx.x * TR_ROWS;
    const int rows_here = (int)min((long long)TR_ROWS, rows - r_begin);
    const int m = threadIdx.x;
    if (m >= jb.M) return;
    const float* p = tape + (size_t)r_begin * rw::TAPE_W + jb.p_off + m;
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
    int r = 0;
    for (; r + 4 <= rows_here; r += 4) {
        s0 += p[(size_t)r * rw::TAPE_W]; s1 += p[(size_t)(r + 1) * rw::TAPE_W];
        s2 += p[(size_t)(r + 2) * rw::TAPE_W]; s3 += p[(size_t)(r + 3) * rw::TAPE_W];
    }
    for (; r < rows_here; ++r) s0 += p[(size_t)r * rw::TAPE_W];
    partials[(size_t)blockIdx.x * stride + jb.out_off + m] = (s0 + s1) + (s2 + s3);
}

__global__ void tape_partial_sum_kernel(const float* __restrict__ partials, int row_blocks, int stride, int total,
                                        float* __restrict__ grads) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    float s = 0.f;
    for (int rb = 0; rb < row_blocks; ++rb) s += partials[(size_t)rb * stride + i];
    grads[i] = s;
}

TapeJobs make_jobs(int d, int n) {
    const rc::Offsets o = rc::rnn_offsets(d, n);
    TapeJobs t; int g = 0, c = 0;
    auto gemm = [&](int p, int M, int q, int N, int out) { t.gemm[g++] = TapeJob{p, M, q, N, out}; };
    auto col = [&](int p, int M, int out) { t.col[c++] = TapeJob{p, M, -1, 1, out}; };
    gemm(rc::TP_DZ1, rc::H, rc::TQ_X, d, o.w1);     col(rc::TP_DZ1, rc::H, o.b1);
    col(rc::TS_DY1N1, rc::H, o.g1);                  col(rc::TS_DY1, rc::H, o.be1);
    gemm(rc::TP_DZ3, rc::H, rc::TQ_Y1, rc::H, o.w3); col(rc::TP_DZ3, rc::H, o.b3);
    col(rc::TS_DY3N3, rc::H, o.g3);                  col(rc::TS_DY3, rc::H, o.be3);
    gemm(rc::TP_DGI, rc::G3, rc::TQ_Y3, rc::H, o.wih); gemm(rc::TP_DGH, rc::G3, rc::TQ_HM, rc::H, o.whh);
    col(rc::TP_DGI, rc::G3, o.bih);                  col(rc::TP_DGH, rc::G3, o.bhh);
    col(rc::TS_DONO, rc::H, o.gr);                   col(rc::TS_DO, rc::H, o.ber);
    gemm(rc::TP_DLOG, n, rc::TQ_O, rc::H, o.wh);     col(rc::TP_DLOG, n, o.bh);
    t.n_gemm = g; t.n_col = c;
    return t;
}

// workspace = tape (rows x TAPE_W) followed by the reduction partials (row blocks x grads_stride)
long long ws_tape_floats(long long rows) { return rows * rw::TAPE_W; }
int ws_row_blocks(long long rows) { return (int)((rows + TR_ROWS - 1) / TR_ROWS); }

// ---- optimizer: per-net global-norm clip + Adam on the true-layout gradients (one CTA per net) ----
__global__ void __launch_bounds__(1024) rnn_apply_kernel(const OrlRnnArgs a) {
    const int net = blockIdx.x;
    const int total = net == 0 ? rc::rnn_offsets(a.obs_dim, a.n_actions).total : rc::rnn_offsets(a.critic_obs_dim, 1).total;
    float* params = net == 0 ? a.policy_params : a.critic_params;
    float* am = net == 0 ? a.policy_adam_m : a.critic_adam_m;
    float* av = net == 0 ? a.policy_adam_v : a.critic_adam_v;
    const float* grads = a.grads + (size_t)net * a.grads_stride;
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
    const float norm = s_norm;
    float clip = 1.f;
    if (a.flags & ORL_PPO_MAX_GRAD_NORM) clip = fminf(a.max_grad_norm / (norm + 1e-6f), 1.0f);
    const int step = a.adam_steps[net] + 1;
    const double bc1 = 1.0 - pow((double)a.adam_beta1, (double)step);
    const double bc2 = 1.0 - pow((double)a.adam_beta2, (double)step);
    const float step_size = (float)((double)a.lrs[net] / bc1);
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
        a.adam_steps[net] = step;
        if (net == 0) {
            a.train_info[2] += a.loss_acc[0];
            a.train_info[3] += a.loss_acc[1];
            a.train_info[4] += norm;
            a.train_info[5] += a.loss_acc[2] / (float)(a.norm_rows > 0 ? (double)a.norm_rows : (double)a.n_chunks * a.chunk_length);
        } else {
            a.train_info[0] += a.loss_acc[3];
            a.train_info[1] += norm;
            if (a.flags & ORL_PPO_VALUENORM) {
                float st[3];
                vn_updated(a.vn_state, a.mb_stats, a.norm_rows > 0 ? (double)a.norm_rows : (double)a.n_chunks * a.chunk_length, a.vn_beta, st);
                a.vn_state[0] = st[0]; a.vn_state[1] = st[1]; a.vn_state[2] = st[2];
            }
        }
    }
}

constexpr size_t w_smem(int rows_per_warp) {   // weights of one net + the per-warp mat-vec scratch
    return (size_t)(rw::smem_net_floats() + rw::smem_scratch_floats(W_WPC, rows_per_warp)) * sizeof(float);
}
template <typename K>
int warp_kernel_prepare(K kernel, size_t smem, const char* what) {
    return orl::check_cuda(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), what);
}
int warp_grid(long long units) {   // persistent CTAs: one per SM, never more than the work needs
    const long long need = (units + W_WPC - 1) / W_WPC;
    return (int)std::max(1LL, std::min<long long>(need, orl::sm_count()));
}

constexpr int JOINT_MAX_AGENTS = 4;   // JRPO policy warps hold one chunk's A agent rows (C_R = A)
static_assert(w_smem(JOINT_MAX_AGENTS) <= 227 * 1024, "JRPO policy weights + scratch must fit one CTA per SM");

// one persistent warp kernel launch over `units` warp work items (chunk groups)
template <bool POLICY, int C_R, bool JOINT>
int launch_chunk(const OrlRnnArgs& a, long long units, cudaStream_t st) {
    auto k = rnn_chunk_warp_kernel<POLICY, C_R, W_NT, JOINT>;
    if (int e = warp_kernel_prepare(k, w_smem(C_R), POLICY ? "smem attr (rnn chunk policy)" : "smem attr (rnn chunk critic)")) return e;
    k<<<warp_grid(units), W_NT, w_smem(C_R), st>>>(a);
    return 0;
}
template <int A>
int launch_joint_policy(const OrlRnnArgs& a, cudaStream_t st) { return launch_chunk<true, A, true>(a, a.n_chunks, st); }

int check_common(const OrlRnnArgs& a) {
    ORL_CHECK_ARG(a.n_envs > 0 && a.n_agents > 0 && a.episode_length > 0, "n_envs / n_agents / episode_length");
    ORL_CHECK_ARG(a.obs_dim > 0 && a.obs_dim <= rc::MAXD && a.critic_obs_dim > 0 && a.critic_obs_dim <= rc::MAXD, "obs dims (<= 64)");
    ORL_CHECK_ARG(a.n_actions > 0 && a.n_actions <= MAX_OUT, "n_actions (<= 8)");
    ORL_CHECK_ARG(a.activation_id >= 0 && a.activation_id <= 3, "activation_id");
    return 0;
}

}  // namespace

extern "C" {

int orl_rnn_param_count(int obs_dim, int n_out) { return rc::rnn_offsets(obs_dim, n_out).total; }
int orl_rnn_tape_width(void) { return rw::TAPE_W; }
long long orl_rnn_workspace_floats(long long rows, int grads_stride) {
    return ws_tape_floats(rows) + (long long)ws_row_blocks(rows) * grads_stride;
}

int orl_rnn_rollout(const OrlRnnArgs* ap, void* stream) {
    ORL_CHECK_ARG(ap, "args");
    const OrlRnnArgs& a = *ap;
    if (int e = check_common(a)) return e;
    ORL_CHECK_ARG(a.policy_params && a.policy_obs && a.rnn_states && a.actions && a.action_log_probs && a.masks, "null rollout buffer");
    ORL_CHECK_ARG(a.t_begin >= 0 && a.t_end <= a.episode_length && a.t_begin <= a.t_end, "t range");
    cudaStream_t st = (cudaStream_t)stream;
    const int grid = (a.n_envs + RNN_NT - 1) / RNN_NT;
    if (a.env_kind == ORL_ENV_NONE) {   // policy step(s) only: rows = n_envs, slot t -> actions[t], rnn_states[t+1]
        ORL_CHECK_ARG(a.n_agents == 1, "ENV_NONE rows are passed as n_envs with n_agents == 1");
        if (a.t_end > a.t_begin) rnn_act_kernel<<<grid, RNN_NT, 0, st>>>(a);
        if (a.rng_counter) rnn_bump_counter_kernel<<<1, 1, 0, st>>>(a.rng_counter, (uint64_t)(a.t_end - a.t_begin));
        return orl::check_cuda(cudaGetLastError(), "rnn_act_kernel launch");
    }
    ORL_CHECK_ARG(a.critic_obs && a.rewards && a.active_masks, "null rollout buffer");
    ORL_CHECK_ARG(a.env_kind == ORL_ENV_MPE_SPREAD || a.env_kind == ORL_ENV_CARTPOLE || a.env_kind == ORL_ENV_GRIDWORLD,
                  "unknown env kind");
    ORL_CHECK_ARG(a.ep_return && a.ep_length && a.episode_stats, "episode statistics buffers");
    if (a.env_kind == ORL_ENV_MPE_SPREAD) {
        ORL_CHECK_ARG(a.n_agents == 3 && a.obs_dim == 18 && a.critic_obs_dim == 54 && a.env_f64 && a.env_u64 && a.env_i32,
                      "simple_spread shapes / state");
    } else {
        ORL_CHECK_ARG(a.n_agents == 1 && a.obs_dim == 4, "single-agent env shapes");
    }
    if (a.t_end > a.t_begin) {
        const int wg = warp_grid(a.n_envs);
        int e = 0;
        switch (a.env_kind) {
            case ORL_ENV_MPE_SPREAD:
                if ((e = warp_kernel_prepare(rnn_rollout_warp_kernel<ORL_ENV_MPE_SPREAD>, w_smem(3), "smem attr (rnn rollout)"))) return e;
                rnn_rollout_warp_kernel<ORL_ENV_MPE_SPREAD><<<wg, W_NT, w_smem(3), st>>>(a); break;
            case ORL_ENV_CARTPOLE:
                if ((e = warp_kernel_prepare(rnn_rollout_warp_kernel<ORL_ENV_CARTPOLE>, w_smem(1), "smem attr (rnn rollout)"))) return e;
                rnn_rollout_warp_kernel<ORL_ENV_CARTPOLE><<<wg, W_NT, w_smem(1), st>>>(a); break;
            default:
                if ((e = warp_kernel_prepare(rnn_rollout_warp_kernel<ORL_ENV_GRIDWORLD>, w_smem(1), "smem attr (rnn rollout)"))) return e;
                rnn_rollout_warp_kernel<ORL_ENV_GRIDWORLD><<<wg, W_NT, w_smem(1), st>>>(a); break;
        }
    }
    if (a.rng_counter) rnn_bump_counter_kernel<<<1, 1, 0, st>>>(a.rng_counter, (uint64_t)(a.t_end - a.t_begin));
    return orl::check_cuda(cudaGetLastError(), "rnn_rollout_warp_kernel launch");
}

int orl_rnn_critic(const OrlRnnArgs* ap, void* stream) {
    ORL_CHECK_ARG(ap, "args");
    const OrlRnnArgs& a = *ap;
    if (int e = check_common(a)) return e;
    ORL_CHECK_ARG(a.critic_params && a.critic_obs && a.rnn_states_critic && a.masks && a.value_preds, "null critic buffer");
    const int B = a.n_envs * a.n_agents;
    if (int e = warp_kernel_prepare(rnn_critic_warp_kernel, w_smem(1), "smem attr (rnn critic)")) return e;
    rnn_critic_warp_kernel<<<warp_grid(B), W_NT, w_smem(1), (cudaStream_t)stream>>>(a);
    return orl::check_cuda(cudaGetLastError(), "rnn_critic_warp_kernel launch");
}

int orl_rnn_fwdbwd(const OrlRnnArgs* ap, void* stream) {
    ORL_CHECK_ARG(ap, "args");
    const OrlRnnArgs& a = *ap;
    if (int e = check_common(a)) return e;
    ORL_CHECK_ARG(a.chunk_length >= 1 && a.chunk_length <= LMAX, "chunk_length (data_chunk_length) must be in [1, 32]");
    ORL_CHECK_ARG(a.n_chunks > 0 && a.chunk_ids, "chunks");
    ORL_CHECK_ARG(a.policy_params && a.critic_params && a.policy_obs && a.critic_obs && a.rnn_states && a.rnn_states_critic &&
                      a.actions && a.action_log_probs && a.masks && a.active_masks && a.value_preds && a.returns && a.advantages,
                  "null update buffer");
    ORL_CHECK_ARG(a.gae_stats && a.mb_stats && a.tape && a.grads && a.loss_acc, "stats / workspace");
    ORL_CHECK_ARG(a.grads_stride >= rc::rnn_offsets(a.obs_dim, a.n_actions).total &&
                      a.grads_stride >= rc::rnn_offsets(a.critic_obs_dim, 1).total, "grads_stride");
    if (a.flags & ORL_PPO_VALUENORM) { ORL_CHECK_ARG(a.vn_state, "vn_state"); }
    const bool joint = a.flags & ORL_PPO_JOINT_ACTION;
    if (joint && a.n_agents > JOINT_MAX_AGENTS) {
        orl::set_last_error("orl_rnn_fwdbwd: ORL_PPO_JOINT_ACTION is built for n_agents <= %d (got %d)", JOINT_MAX_AGENTS, a.n_agents);
        return ORL_ERR_UNSUPPORTED;
    }
    cudaStream_t st = (cudaStream_t)stream;
    int e = orl::check_cuda(cudaMemsetAsync(a.loss_acc, 0, 8 * sizeof(float), st), "memset loss_acc");
    if (e) return e;
    // tape rows per net: n_chunks*L chunk steps, times A policy rows per step with the joint-action loss
    const long long steps = a.n_chunks * a.chunk_length;
    const long long net_rows[2] = {joint ? steps * a.n_agents : steps, steps};
    float* partials = a.tape + ws_tape_floats(net_rows[0]);
    // two chunks per warp: every weight read from shared memory feeds two rows (four per warp with 8 warps / CTA
    // measured 12 % slower on B200: profiles/r1_gru_perf.md).  JRPO policy: one chunk per warp, its A agent rows.
    constexpr int C_R = 2;
    if ((e = orl::check_cuda(cudaFuncSetAttribute(tape_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TR_SMEM),
                             "smem attr (tape gemm)"))) return e;
    for (int net = 0; net < 2; ++net) {
        const int d = net == 0 ? a.obs_dim : a.critic_obs_dim, n = net == 0 ? a.n_actions : 1;
        if (net == 0 && joint) {
            switch (a.n_agents) {
                case 1: e = launch_joint_policy<1>(a, st); break;
                case 2: e = launch_joint_policy<2>(a, st); break;
                case 3: e = launch_joint_policy<3>(a, st); break;
                default: e = launch_joint_policy<4>(a, st); break;
            }
        } else if (net == 0) {
            e = launch_chunk<true, C_R, false>(a, (a.n_chunks + C_R - 1) / C_R, st);
        } else {
            e = joint ? launch_chunk<false, C_R, true>(a, (a.n_chunks + C_R - 1) / C_R, st)
                      : launch_chunk<false, C_R, false>(a, (a.n_chunks + C_R - 1) / C_R, st);
        }
        if (e) return e;
        const long long rows = net_rows[net];
        const int rb = ws_row_blocks(rows);
        const TapeJobs jobs = make_jobs(d, n);
        tape_gemm_kernel<<<dim3(rb, jobs.n_gemm), TR_NT, TR_SMEM, st>>>(a.tape, rows, jobs, partials, a.grads_stride);
        tape_colsum_kernel<<<dim3(rb, jobs.n_col), rc::G3, 0, st>>>(a.tape, rows, jobs, partials, a.grads_stride);
        const int total = rc::rnn_offsets(d, n).total;
        tape_partial_sum_kernel<<<(total + 255) / 256, 256, 0, st>>>(partials, rb, a.grads_stride, total,
                                                                     a.grads + (size_t)net * a.grads_stride);
    }
    return orl::check_cuda(cudaGetLastError(), "rnn update launches");
}

int orl_rnn_apply(const OrlRnnArgs* ap, void* stream) {
    ORL_CHECK_ARG(ap, "args");
    const OrlRnnArgs& a = *ap;
    if (int e = check_common(a)) return e;
    ORL_CHECK_ARG(a.policy_params && a.critic_params && a.grads && a.loss_acc && a.policy_adam_m && a.policy_adam_v &&
                      a.critic_adam_m && a.critic_adam_v && a.adam_steps && a.lrs && a.train_info && a.mb_stats, "null optimizer buffer");
    ORL_CHECK_ARG(a.n_chunks > 0 && a.chunk_length >= 1, "chunks");
    if (a.flags & ORL_PPO_VALUENORM) { ORL_CHECK_ARG(a.vn_state, "vn_state"); }
    rnn_apply_kernel<<<2, 1024, 0, (cudaStream_t)stream>>>(a);
    return orl::check_cuda(cudaGetLastError(), "rnn_apply_kernel launch");
}

}  // extern "C"
