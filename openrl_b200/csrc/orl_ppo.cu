// PPO minibatch update: fused gather + forward + loss + backward (orl_ppo_fwdbwd), deterministic
// partial reduction (orl_ppo_reduce) and unfold + clip + Adam (orl_ppo_apply).
// Reference semantics: openrl/algorithms/ppo.py:46-361 (see include/openrl_b200.h).
//
// orl_ppo_fwdbwd: persistent CTAs of 256 threads; CTAs [0, G) run the policy net, [G, 2G) the
// critic net (the two losses are independent once the minibatch moments are known).  A CTA walks
// tiles of 128 minibatch rows; per tile it runs, entirely in shared memory / registers,
//   trunk forward (2 tile GEMMs + LayerNorms)  -> head + loss + dLoss/dhead (2 lanes per row)
//   -> dn3 = dL.Whf, LN3 backward -> G3 += dZ3^T n1 ; dn1 = dZ3.W3f, LN1 + activation backward
//   -> G1 += dZ1^T X
// with the weight-gradient blocks (4x4 per thread) accumulated in registers across all tiles of
// the CTA and written once at the end.  fp32 FFMA throughout (1e-4 loss-parity bar; see DESIGN.md).
// Arithmetic per row (d=4, n=2, both nets): ~53 kFLOP; bytes per row: ~60 B  => fp32-pipe bound.
#include <algorithm>

#include "orl_loss.cuh"

namespace {
using namespace orl;

constexpr int P_M = 128;   // rows per tile
constexpr int P_NT = 256;  // threads per CTA
constexpr int P_TY = P_NT / 16, P_RPT = P_M / P_TY;
constexpr int DLW = 8;     // leading dimension of the dL/dhead tile
constexpr int N_LOSS = 8;  // loss-sum slots at the tail of a partial row

__host__ __device__ inline int ppo_stride(int obs_dim, int critic_obs_dim, int n_actions) {
    const int a = orl::fold_offsets(obs_dim, n_actions).total, b = orl::fold_offsets(critic_obs_dim, 1).total;
    return ((a > b ? a : b) + N_LOSS + 3) & ~3;
}

__host__ __device__ inline int ppo_grads_stride(int obs_dim, int critic_obs_dim, int n_actions) {
    const int a = orl::net_offsets(obs_dim, n_actions, 1).total, b = orl::net_offsets(critic_obs_dim, 1).total;
    return ((a > b ? a : b) + 3) & ~3;
}

struct WgMap { int jb, kb, mg, MG; bool active; };
__device__ __forceinline__ WgMap wg_map(int JB, int KB) {
    WgMap m;
    const int nb = JB * KB;
    m.MG = P_NT / nb;
    const int tid = threadIdx.x;
    m.active = tid < nb * m.MG;
    const int b = tid % nb;
    m.mg = tid / nb;
    m.jb = b / KB;
    m.kb = b % KB;
    return m;
}
// g[a][b] += sum_{m = mg, mg+MG, ...} P[m][4jb+a] * Q[m][4kb+b];  db[a] += P[m][4jb+a] when kb == 0
__device__ __forceinline__ void wgrad_acc(const float* __restrict__ P, int ldp, const float* __restrict__ Q, int ldq,
                                          const WgMap& mp, float (&g)[4][4], float (&db)[4]) {
    if (!mp.active) return;
    const float* pp = P + 4 * mp.jb;
    const float* qq = Q + 4 * mp.kb;
    const bool bias = mp.kb == 0;
#pragma unroll 4
    for (int m = mp.mg; m < P_M; m += mp.MG) {
        const float4 p = *reinterpret_cast<const float4*>(pp + m * ldp);
        const float4 q = *reinterpret_cast<const float4*>(qq + m * ldq);
        g[0][0] = fmaf(p.x, q.x, g[0][0]); g[0][1] = fmaf(p.x, q.y, g[0][1]); g[0][2] = fmaf(p.x, q.z, g[0][2]); g[0][3] = fmaf(p.x, q.w, g[0][3]);
        g[1][0] = fmaf(p.y, q.x, g[1][0]); g[1][1] = fmaf(p.y, q.y, g[1][1]); g[1][2] = fmaf(p.y, q.z, g[1][2]); g[1][3] = fmaf(p.y, q.w, g[1][3]);
        g[2][0] = fmaf(p.z, q.x, g[2][0]); g[2][1] = fmaf(p.z, q.y, g[2][1]); g[2][2] = fmaf(p.z, q.z, g[2][2]); g[2][3] = fmaf(p.z, q.w, g[2][3]);
        g[3][0] = fmaf(p.w, q.x, g[3][0]); g[3][1] = fmaf(p.w, q.y, g[3][1]); g[3][2] = fmaf(p.w, q.z, g[3][2]); g[3][3] = fmaf(p.w, q.w, g[3][3]);
        if (bias) { db[0] += p.x; db[1] += p.y; db[2] += p.z; db[3] += p.w; }
    }
}

// Reduce a thread-block-distributed gradient (4x4 blocks, MG row groups) through shared scratch and
// write rows < jdim, cols < kdim to global out[j*kdim + k]; bias sums to out_b[j].
__device__ __forceinline__ void wgrad_flush(float* __restrict__ scratch, const WgMap& mp, int JB, int KB,
                                            const float (&g)[4][4], const float (&db)[4], int jdim, int kdim,
                                            float* __restrict__ out, float* __restrict__ out_b) {
    const int W = 4 * KB, R = 4 * JB;
    __syncthreads();
    if (mp.active) {
        float* s = scratch + (size_t)mp.mg * (R * W + R);
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int b = 0; b < 4; ++b) s[(4 * mp.jb + a) * W + 4 * mp.kb + b] = g[a][b];
        if (mp.kb == 0) {
#pragma unroll
            for (int a = 0; a < 4; ++a) s[R * W + 4 * mp.jb + a] = db[a];
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < R * W + R; i += P_NT) {
        float v = 0.f;
        for (int g2 = 0; g2 < mp.MG; ++g2) v += scratch[(size_t)g2 * (R * W + R) + i];
        if (i < R * W) {
            const int j = i / W, k = i % W;
            if (j < jdim && k < kdim) out[j * kdim + k] = v;
        } else {
            const int j = i - R * W;
            if (j < jdim) out_b[j] = v;
        }
    }
}


template <bool POLICY>
__device__ __forceinline__ void ppo_net_pass(const OrlPpoArgs& a, float* smem, int cta, int G) {
    const int d = POLICY ? a.obs_dim : a.critic_obs_dim;
    const int n = POLICY ? a.n_actions : 1;
    const float* params = POLICY ? a.policy_params : a.critic_params;
    const float* obs = POLICY ? a.policy_obs : a.critic_obs;
    const int dp = pad4(d), ldx = dp + 4;
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;

    float* p = smem;
    SmemWeights w = carve_weights(p, d, true);
    float* Xs = p;  p += P_M * ldx;
    float* N1s = p; p += P_M * LDA;
    float* N3s = p; p += P_M * LDA;
    float* DZs = p; p += P_M * LDA;
    float* DLs = p; p += P_M * DLW;
    float* row_a = p; p += P_M;   // policy: action      | critic: value_pred
    float* row_b = p; p += P_M;   // policy: old logp    | critic: return
    float* row_c = p; p += P_M;   // policy: raw adv
    float* row_act = p; p += P_M; // active mask
    float* red = p; p += 32;
    long long* row_idx = reinterpret_cast<long long*>(p); p += 2 * P_M;

    load_weights_folded<P_NT>(w, params, d, n, true);

    const bool pol_masks = a.flags & ORL_PPO_POLICY_ACTIVE_MASKS, val_masks = a.flags & ORL_PPO_VALUE_ACTIVE_MASKS;
    const double rows_d = (double)(a.norm_rows > 0 ? a.norm_rows : a.batch_rows);
    const float inv_rows = (float)(1.0 / rows_d);
    const float inv_act = (float)(1.0 / a.mb_stats[2]);
    AdvNorm advn;
    float vn_mean = 0.f, vn_std = 1.f;
    if (POLICY) {
        advn = make_adv_norm(a.gae_stats, a.flags & ORL_PPO_ADV_NORMALIZE);
    } else if (a.flags & ORL_PPO_VALUENORM) {
        float st[3];
        vn_updated(a.vn_state, a.mb_stats, rows_d, a.vn_beta, st);
        const VnScalars s = vn_mean_std(st);
        vn_mean = s.mean; vn_std = s.std;
    }

    const WgMap map3 = wg_map(16, 16);
    const WgMap map1 = wg_map(16, dp / 4);
    const int JBH = n > 4 ? 2 : 1;
    const WgMap maph = wg_map(JBH, 16);
    float g3[4][4] = {}, g1[4][4] = {}, gh[4][4] = {}, db3[4] = {}, db1[4] = {}, dbh[4] = {};
    const bool gaussian = POLICY && a.head_kind == ORL_HEAD_GAUSSIAN;
    float dls_acc[MAX_OUT] = {};   // dL/dlogstd partial sums of this thread's rows (Gaussian head)
    float loss0 = 0.f, loss1 = 0.f, loss2 = 0.f;  // policy: policy_loss, entropy, ratio | critic: value_loss

    const long long n_tiles = (a.batch_rows + P_M - 1) / P_M;
    for (long long tile = cta; tile < n_tiles; tile += G) {
        const long long r0 = tile * P_M;
        const int rows_here = (int)min((long long)P_M, a.batch_rows - r0);
        // ---- gather (replay_data.py:616-646) ----
        if (tid < P_M) {
            long long gi = -1;
            if (tid < rows_here) gi = a.indices ? a.indices[r0 + tid] : a.row_begin + r0 + tid;
            row_idx[tid] = gi;
            if (gi >= 0) {
                if (POLICY) { row_a[tid] = a.actions[gi]; row_b[tid] = a.old_log_probs[gi]; row_c[tid] = a.advantages[gi]; }
                else { row_a[tid] = a.value_preds[gi]; row_b[tid] = a.returns[gi]; }
                row_act[tid] = a.active_masks[gi];
            }
        }
        __syncthreads();
        for (int i = tid; i < P_M * ldx; i += P_NT) {
            const int r = i / ldx, k = i % ldx;
            const long long gi = row_idx[r];
            Xs[i] = (gi >= 0 && k < d) ? obs[gi * d + k] : 0.f;
        }
        __syncthreads();

        // ---- forward ----
        float mu1[P_RPT], rstd1[P_RPT], rstd3[P_RPT];
        unsigned posmask;
        trunk_forward<P_M, P_NT, true>(w, Xs, ldx, d, a.activation_id, N1s, N3s, mu1, rstd1, rstd3, posmask);
        __syncthreads();
        float out[MAX_OUT];
        head_dots<P_M, P_NT>(w, N3s, n, out);
        {
            constexpr int PPR = P_NT / P_M;
            const int row = tid / PPR;
            if (tid % PPR == 0) {
                float dl[DLW];
#pragma unroll
                for (int j = 0; j < DLW; ++j) dl[j] = 0.f;
                if (row < rows_here) {
                    const float active = row_act[row];
                    if (POLICY && gaussian) {
                        // DiagGaussian head (act.py:150-158, distributions.py:34-47): per-dimension ratios,
                        // surrogate summed over the action dimension (ppo.py:307-319)
                        const long long gi = row_idx[row];
                        const float* logstd = params + net_offsets(d, n, 1).ls;
                        const float adv = apply_adv_norm(advn, row_c[row]);
                        const float wrow = pol_masks ? active * inv_act : inv_rows;
                        const float went_row = pol_masks ? active * inv_act : inv_rows / (float)n;
#pragma unroll
                        for (int j = 0; j < MAX_OUT; ++j) {
                            if (j < n) {
                                const float mean = out[j], ls = logstd[j], std = expf(ls), var = std * std;
                                const float act = a.actions[gi * n + j], diff = act - mean;
                                const float lp = -(diff * diff) / (2.0f * var) - ls - 0.9189385332046727f;
                                const PgTerm pg = pg_term(lp, a.old_log_probs[gi * n + j], adv, a.clip_param, a.flags, a.dual_clip_coeff);
                                loss0 += pg.loss * wrow;
                                loss1 += (1.4189385332046727f + ls) * went_row;   // 0.5 + 0.5 log(2 pi) + log(std)
                                loss2 += pg.ratio / (float)n;
                                const float dlp = pg.dlogp * wrow;
                                dl[j] = dlp * diff / var;                                               // dL/dmean
                                dls_acc[j] += dlp * (diff * diff / var - 1.0f) - a.entropy_coef * went_row;   // dL/dlogstd
                            }
                        }
                    } else if (POLICY) {
                        const long long gi = row_idx[row];
                        unsigned masked = 0;
                        if (a.action_masks) {
#pragma unroll
                            for (int j = 0; j < MAX_OUT; ++j)
                                if (j < n && a.action_masks[gi * n + j] == 0.f) { out[j] = -6e4f; masked |= 1u << j; }
                        }
                        float nl[MAX_OUT], pr[MAX_OUT];
                        log_softmax_n(out, n, nl, pr);
                        const int act = (int)row_a[row];
                        float lp = nl[0];
#pragma unroll
                        for (int j = 1; j < MAX_OUT; ++j) if (j == act) lp = nl[j];
                        const float adv = apply_adv_norm(advn, row_c[row]);
                        const PgTerm pg = pg_term(lp, row_b[row], adv, a.clip_param, a.flags, a.dual_clip_coeff);
                        const float wrow = pol_masks ? active * inv_act : inv_rows;
                        float ent = 0.f;
#pragma unroll
                        for (int j = 0; j < MAX_OUT; ++j) if (j < n) ent -= pr[j] * nl[j];
                        loss0 += pg.loss * wrow;
                        loss1 += ent * wrow;
                        loss2 += pg.ratio;
                        const float dlp = pg.dlogp * wrow;
                        const float went = a.entropy_coef * wrow;
#pragma unroll
                        for (int j = 0; j < MAX_OUT; ++j) {
                            if (j < n && !((masked >> j) & 1u)) {
                                const float onehot = (j == act) ? 1.f : 0.f;
                                dl[j] = dlp * (onehot - pr[j]) + went * pr[j] * (nl[j] + ent);
                            }
                        }
                    } else {
                        const float v = out[0], vp = row_a[row], ret = row_b[row];
                        const float target = (a.flags & ORL_PPO_VALUENORM) ? (ret - vn_mean) / vn_std : ret;
                        const float diff = v - vp;
                        const float clipped = vp + fminf(fmaxf(diff, -a.clip_param), a.clip_param);
                        const float e_c = target - clipped, e_o = target - v;
                        const bool hub = a.flags & ORL_PPO_HUBER;
                        const float l_c = hub ? huber(e_c, a.huber_delta) : 0.5f * e_c * e_c;
                        const float l_o = hub ? huber(e_o, a.huber_delta) : 0.5f * e_o * e_o;
                        const float gc = hub ? huber_grad(e_c, a.huber_delta) : e_c;
                        const float go = hub ? huber_grad(e_o, a.huber_delta) : e_o;
                        float l = l_o, dv = -go;
                        if (a.flags & ORL_PPO_CLIP_VALUE) {
                            const bool inrange = diff >= -a.clip_param && diff <= a.clip_param;
                            const float dc = inrange ? -gc : 0.f;
                            if (l_o > l_c) { l = l_o; dv = -go; }
                            else if (l_c > l_o) { l = l_c; dv = dc; }
                            else { l = l_o; dv = 0.5f * (-go) + 0.5f * dc; }
                        }
                        const float wrow = val_masks ? active * inv_act : inv_rows;
                        loss0 += l * wrow;
                        dl[0] = a.value_loss_coef * wrow * dv;
                    }
                }
                *reinterpret_cast<float4*>(DLs + row * DLW) = make_float4(dl[0], dl[1], dl[2], dl[3]);
                *reinterpret_cast<float4*>(DLs + row * DLW + 4) = make_float4(dl[4], dl[5], dl[6], dl[7]);
            }
        }
        __syncthreads();

        // ---- backward: head -> LN3 ----
        float acc[P_RPT][4];
#pragma unroll
        for (int i = 0; i < P_RPT; ++i) { acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.f; }
        for (int j = 0; j < n; ++j) {
            const float4 wv = *reinterpret_cast<const float4*>(w.whf + j * H + 4 * tx);
#pragma unroll
            for (int i = 0; i < P_RPT; ++i) {
                const float dlv = DLs[(ty + P_TY * i) * DLW + j];
                acc[i][0] = fmaf(dlv, wv.x, acc[i][0]); acc[i][1] = fmaf(dlv, wv.y, acc[i][1]);
                acc[i][2] = fmaf(dlv, wv.z, acc[i][2]); acc[i][3] = fmaf(dlv, wv.w, acc[i][3]);
            }
        }
        {
            float nrm[P_RPT][4];
            load_tile<P_RPT, P_TY>(N3s, nrm, tx, ty);
            layernorm_bwd_rows<P_RPT>(acc, nrm, rstd3);
        }
        store_tile<P_RPT, P_TY>(DZs, acc, tx, ty);   // dZ3
        wgrad_acc(DLs, DLW, N3s, LDA, maph, gh, dbh);  // GH += dL^T n3
        __syncthreads();

        // ---- fc3 backward ----
        wgrad_acc(DZs, LDA, N1s, LDA, map3, g3, db3);  // G3 += dZ3^T n1
#pragma unroll
        for (int i = 0; i < P_RPT; ++i) { acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.f; }
        gemm_tile<P_RPT, P_TY>(DZs, LDA, w.w3n, H, acc, tx, ty);  // dn1 = dZ3 . W3f
        {
            float nrm[P_RPT][4];
            load_tile<P_RPT, P_TY>(N1s, nrm, tx, ty);
            layernorm_bwd_rows<P_RPT>(acc, nrm, rstd1);
#pragma unroll
            for (int i = 0; i < P_RPT; ++i) {
                const float stdv = 1.0f / rstd1[i];
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const float aval = fmaf(nrm[i][c], stdv, mu1[i]);
                    acc[i][c] *= act_bwd(aval, (posmask >> (i * 4 + c)) & 1u, a.activation_id);
                }
            }
        }
        __syncthreads();                               // all reads of dZ3 done
        store_tile<P_RPT, P_TY>(DZs, acc, tx, ty);     // dZ1
        __syncthreads();
        wgrad_acc(DZs, LDA, Xs, ldx, map1, g1, db1);   // G1 += dZ1^T X
        __syncthreads();
    }

    // ---- flush this CTA's partial folded gradients + loss sums ----
    const int stride = ppo_stride(a.obs_dim, a.critic_obs_dim, a.n_actions);
    float* part = a.partials + (size_t)((POLICY ? 0 : G) + cta) * stride;
    const FoldOffsets fo = fold_offsets(d, n);
    float* scratch = N1s;  // >= 16*(64*4+64) floats needed at most; N1s..DZs is 3*128*68 floats
    wgrad_flush(scratch, map1, 16, dp / 4, g1, db1, H, d, part + fo.g1, part + fo.db1);
    wgrad_flush(scratch, map3, 16, 16, g3, db3, H, H, part + fo.g3, part + fo.db3);
    wgrad_flush(scratch, maph, JBH, 16, gh, dbh, n, H, part + fo.gh, part + fo.dbh);
    __syncthreads();
    if (POLICY) {   // dL/dlogstd: block reduction of the per-thread partial sums (zero for categorical heads)
        const int lane = tid & 31, warp = tid >> 5;
#pragma unroll
        for (int j = 0; j < MAX_OUT; ++j) {
            const float sv = warp_sum(dls_acc[j]);
            if (lane == 0) scratch[j * 8 + warp] = sv;
        }
        __syncthreads();
        if (tid < n) {
            float sv = 0.f;
            for (int wv = 0; wv < P_NT / 32; ++wv) sv += scratch[tid * 8 + wv];
            part[fo.dls + tid] = sv;
        }
        __syncthreads();
    } else if (tid < n) {
        part[fo.dls + tid] = 0.f;
    }
    {
        float v[3] = {loss0, loss1, loss2};
        const int lane = tid & 31, warp = tid >> 5;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const float s = warp_sum(v[k]);
            if (lane == 0) red[k * 8 + warp] = s;
        }
        __syncthreads();
        if (tid < N_LOSS) {
            float s = 0.f;
            if (tid < 3) for (int wv = 0; wv < P_NT / 32; ++wv) s += red[tid * 8 + wv];
            part[stride - N_LOSS + tid] = s;
        }
    }
}

__global__ void __launch_bounds__(P_NT, 1) ppo_fwdbwd_kernel(const OrlPpoArgs a) {
    extern __shared__ __align__(16) float smem[];
    const int G = a.grid_per_net;
    if ((int)blockIdx.x < G) ppo_net_pass<true>(a, smem, blockIdx.x, G);
    else ppo_net_pass<false>(a, smem, blockIdx.x - G, G);
}

// Sum over the G partial rows of one net for 32 consecutive bucket elements per CTA (8 warps): warp w adds rows
// w, w+8, ... (coalesced 128-byte loads, 8 independent loads in flight per thread), the 8 partial sums are combined in
// warp order -> a fixed summation order (deterministic), ~2 us instead of ~12 us for the G = 148 sequential loads per thread.
constexpr int RED_W = 8, RED_NT = 32 * RED_W;
__device__ __forceinline__ float reduce_partials(const float* __restrict__ partials, int net, int G, int stride, int el,
                                                 float (*part)[32]) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    float s0 = 0.f, s1 = 0.f;
    if (el < stride) {
        const float* p = partials + (size_t)net * G * stride + el;
        int g = w;
#pragma unroll 4
        for (; g + RED_W < G; g += 2 * RED_W) { s0 += p[(size_t)g * stride]; s1 += p[(size_t)(g + RED_W) * stride]; }
        if (g < G) s0 += p[(size_t)g * stride];
    }
    part[w][lane] = s0 + s1;
    __syncthreads();
    float t = 0.f;
    if (w == 0) {
#pragma unroll
        for (int k = 0; k < RED_W; ++k) t += part[k][lane];
    }
    return t;   // valid in warp 0
}

// folded[net][i] = sum over the G partial rows of that net
__global__ void __launch_bounds__(RED_NT) ppo_reduce_kernel(const float* __restrict__ partials, float* __restrict__ folded, int G, int stride) {
    __shared__ float part[RED_W][32];
    const int net = blockIdx.y, el = blockIdx.x * 32 + (threadIdx.x & 31);
    const float s = reduce_partials(partials, net, G, stride, el, part);
    if (threadIdx.x < 32 && el < stride) folded[(size_t)net * stride + el] = s;
}

// ---- gradient-bucket exchange over NVLink peer memory, fused into the reduce and optimiser kernels -------------------
// Every rank owns a symmetric allocation mapped into all peers: floats [parity 2][source rank W][net 2][stride], then
// uint32 arrival flags [3][ORL_PEER_MAX_WORLD], then doubles [parity 2][ORL_PEER_SMALL_MAX] (orl_peer_sum_f64).
// Update number e of a net (1-based) uses half (e-1)&1.  PUSH: ppo_reduce_peer_kernel (76 CTAs) stores this rank's
// bucket straight into slot [half][my rank] of EVERY rank's allocation - posted NVLink writes, no round trip.  The apply
// CTA of that net then (a) publishes "my bucket for update e has been written everywhere" into every peer's flag word
// [net][my rank] (fence.sys + st.release.sys; the pushes are ordered before it by the kernel boundary), (b) waits until
// all W flag words of its own copy show >= e (ld.acquire.sys), (c) sums the W slots of its OWN copy in rank order - local
// reads, the same order on every rank, so all ranks hold bit-identical sums - and continues as the single-GPU optimiser.
// Two halves suffice: a rank pushes into half h again in update e+2, after its apply of e+1 saw every peer's flag e+1,
// and a peer raises flag e+1 only after its apply of e (the last reader of its half h) has retired.
__global__ void __launch_bounds__(RED_NT) ppo_reduce_peer_kernel(const float* __restrict__ partials, const OrlPeerArgs pa, int G, int stride) {
    __shared__ float part[RED_W][32];
    const int net = blockIdx.y, el = blockIdx.x * 32 + (threadIdx.x & 31);
    const float s = reduce_partials(partials, net, G, stride, el, part);
    if (threadIdx.x < 32 && el < stride) {
        const size_t off = ((size_t)(pa.epochs[net] & 1u) * pa.world + pa.rank) * 2u * stride + (size_t)net * stride + el;
        for (int q = 0; q < pa.world; ++q) reinterpret_cast<float*>(pa.peer_buffers[q])[off] = s;
    }
}

__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ float4 ld_peer4(const float* p) {
    float4 v;
    asm volatile("ld.relaxed.sys.global.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ uint64_t global_ns() {
    uint64_t t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}

__host__ __device__ __forceinline__ size_t peer_flag_word(int world, int stride) { return (size_t)4 * world * stride; }

// signal every peer's flag word [slot][my rank] with `e`, then wait until all W words of my own copy show >= e
__device__ __forceinline__ void peer_handshake(const OrlPeerArgs& pa, int slot, uint32_t e, size_t flag_word) {
    const int tid = threadIdx.x, W = pa.world;
    if (tid < W) {
        __threadfence_system();
        uint32_t* remote = reinterpret_cast<uint32_t*>(pa.peer_buffers[tid]) + flag_word + slot * ORL_PEER_MAX_WORLD + pa.rank;
        st_release_sys(remote, e);
        const uint32_t* mine = reinterpret_cast<const uint32_t*>(pa.peer_buffers[pa.rank]) + flag_word + slot * ORL_PEER_MAX_WORLD + tid;
        const uint64_t t0 = global_ns();
        unsigned spins = 0;
        while ((int32_t)(ld_acquire_sys(mine) - e) < 0) {
            if ((++spins & 1023u) == 0 && global_ns() - t0 > (uint64_t)pa.timeout_ms * 1000000ull) {
                atomicExch(pa.error_flag, 1 + tid);   // peer `tid` never arrived: the host raises on the next read-back
                break;
            }
        }
        __threadfence_system();
    }
    __syncthreads();
}

__device__ const float* peer_gather(const OrlPeerArgs& pa, int net, int stride) {
    const int tid = threadIdx.x, W = pa.world;
    const uint32_t e = pa.epochs[net] + 1u;
    peer_handshake(pa, net, e, peer_flag_word(W, stride));
    // the W slots of this rank's own copy (written by the peers; L1 is bypassed: ld.relaxed.sys)
    const float* base = pa.local_buffer + (size_t)((e - 1u) & 1u) * W * 2u * stride + (size_t)net * stride;
    float* out = pa.summed + (size_t)net * stride;
    for (int i = tid * 4; i < stride; i += blockDim.x * 4) {
        float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int q0 = 0; q0 < W; q0 += 8) {
            float4 v[8];
#pragma unroll
            for (int q = 0; q < 8; ++q)
                if (q0 + q < W) v[q] = ld_peer4(base + (size_t)(q0 + q) * 2u * stride + i);
#pragma unroll
            for (int q = 0; q < 8; ++q)
                if (q0 + q < W) { s.x += v[q].x; s.y += v[q].y; s.z += v[q].z; s.w += v[q].w; }
        }
        *reinterpret_cast<float4*>(out + i) = s;
    }
    __syncthreads();
    return out;
}

// SUM of n <= ORL_PEER_SMALL_MAX doubles over all ranks, in place (the once-per-iteration rollout moments): one CTA
__global__ void __launch_bounds__(64) peer_sum_f64_kernel(const OrlPeerArgs pa, double* __restrict__ data, int n, int stride) {
    const int tid = threadIdx.x, W = pa.world;
    const uint32_t e = pa.epochs[2] + 1u;
    const size_t flag_word = peer_flag_word(W, stride);
    const size_t small_byte = flag_word * 4 + (size_t)3 * ORL_PEER_MAX_WORLD * 4 + (size_t)((e - 1u) & 1u) * ORL_PEER_SMALL_MAX * 8;
    double* mine = reinterpret_cast<double*>(reinterpret_cast<char*>(pa.peer_buffers[pa.rank]) + small_byte);
    if (tid < n) mine[tid] = data[tid];
    __syncthreads();
    peer_handshake(pa, 2, e, flag_word);
    if (tid < n) {
        double s = 0.0;
        for (int q = 0; q < W; ++q) {
            double v;
            asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(v)
                         : "l"(reinterpret_cast<const double*>(reinterpret_cast<const char*>(pa.peer_buffers[q]) + small_byte) + tid) : "memory");
            s += v;
        }
        data[tid] = s;
    }
    if (tid == 0) pa.epochs[2] = e;
}

template <bool PEER>
__global__ void __launch_bounds__(1024) ppo_apply_kernel(const OrlPpoArgs a, const OrlPeerArgs pa) {
    const int net = blockIdx.x;  // 0 policy, 1 critic
    const int d = net == 0 ? a.obs_dim : a.critic_obs_dim;
    const int n = net == 0 ? a.n_actions : 1;
    const int stride = ppo_stride(a.obs_dim, a.critic_obs_dim, a.n_actions);
    const NetOffsets po = net_offsets(d, n, net == 0 && a.head_kind == ORL_HEAD_GAUSSIAN);
    const FoldOffsets fo = fold_offsets(d, n);
    float* params = net == 0 ? a.policy_params : a.critic_params;
    float* am = net == 0 ? a.policy_adam_m : a.critic_adam_m;
    float* av = net == 0 ? a.policy_adam_v : a.critic_adam_v;
    float* grads = a.grads + (size_t)net * ppo_grads_stride(a.obs_dim, a.critic_obs_dim, a.n_actions);
    __shared__ float red[32];
    __shared__ float s_norm;
    const int tid = threadIdx.x;
    const float* f = PEER ? peer_gather(pa, net, stride) : a.folded + (size_t)net * stride;

    float sq = 0.f;
    for (int i = tid; i < po.total; i += blockDim.x) {
        float g;
        if (i < po.b1) g = f[fo.g1 + (i - po.w1)];
        else if (i < po.g1) g = f[fo.db1 + (i - po.b1)];
        else if (i < po.be1) {  // dg1[k] = sum_j W3[j][k] * G3[j][k]
            const int k = i - po.g1; float s = 0.f;
            for (int j = 0; j < H; ++j) s = fmaf(params[po.w3 + j * H + k], f[fo.g3 + j * H + k], s);
            g = s;
        } else if (i < po.w3) {  // dbe1[k] = sum_j W3[j][k] * db3[j]
            const int k = i - po.be1; float s = 0.f;
            for (int j = 0; j < H; ++j) s = fmaf(params[po.w3 + j * H + k], f[fo.db3 + j], s);
            g = s;
        } else if (i < po.b3) {  // dW3[j][k] = G3[j][k]*g1[k] + db3[j]*be1[k]
            const int j = (i - po.w3) / H, k = (i - po.w3) % H;
            g = fmaf(f[fo.g3 + j * H + k], params[po.g1 + k], f[fo.db3 + j] * params[po.be1 + k]);
        } else if (i < po.g3) g = f[fo.db3 + (i - po.b3)];
        else if (i < po.be3) {
            const int k = i - po.g3; float s = 0.f;
            for (int j = 0; j < n; ++j) s = fmaf(params[po.wh + j * H + k], f[fo.gh + j * H + k], s);
            g = s;
        } else if (i < po.wh) {
            const int k = i - po.be3; float s = 0.f;
            for (int j = 0; j < n; ++j) s = fmaf(params[po.wh + j * H + k], f[fo.dbh + j], s);
            g = s;
        } else if (i < po.bh) {
            const int j = (i - po.wh) / H, k = (i - po.wh) % H;
            g = fmaf(f[fo.gh + j * H + k], params[po.g3 + k], f[fo.dbh + j] * params[po.be3 + k]);
        } else if (i < po.ls) g = f[fo.dbh + (i - po.bh)];
        else g = f[fo.dls + (i - po.ls)];
        grads[i] = g;
        sq = fmaf(g, g, sq);
    }
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
    __shared__ float s_adam[2];
    if (tid == (int)blockDim.x - 1) {   // the two double-precision pow() once per CTA (f64 is slow here), not once per thread
        const double bc1 = 1.0 - pow((double)a.adam_beta1, (double)step);
        const double bc2 = 1.0 - pow((double)a.adam_beta2, (double)step);
        s_adam[0] = (float)((double)a.lrs[net] / bc1);
        s_adam[1] = (float)sqrt(bc2);
    }
    __syncthreads();  // every thread has read the parameters it needs for unfolding; the step constants are in place
    const float step_size = s_adam[0], bc2_sqrt = s_adam[1];
    for (int i = tid; i < po.total; i += blockDim.x) {
        float g = grads[i] * clip;
        float pv = params[i];
        if (a.weight_decay != 0.f) g = fmaf(a.weight_decay, pv, g);
        const float m = am[i] + (g - am[i]) * (1.f - a.adam_beta1);          // exp_avg.lerp_(grad, 1-beta1)
        const float v = fmaf(av[i], a.adam_beta2, (g * g) * (1.f - a.adam_beta2));  // mul_(beta2).addcmul_(g,g,1-beta2)
        am[i] = m; av[i] = v;
        const float denom = sqrtf(v) / bc2_sqrt + a.adam_eps;
        params[i] = pv - step_size * (m / denom);
    }
    if (tid == 0) {
        a.adam_steps[net] = step;
        if (PEER) {
            pa.epochs[net] += 1u;
            // a peer timed out: poison the logged scalars so that the host's one read-back sees it (it then reads error_flag)
            if (*reinterpret_cast<volatile int32_t*>(pa.error_flag) != 0) a.train_info[net == 0 ? 2 : 0] = __int_as_float(0x7fc00000);
        }
        const float* ls = f + stride - N_LOSS;
        if (net == 0) {
            a.train_info[2] += ls[0];
            a.train_info[3] += ls[1];
            a.train_info[4] += norm;
            a.train_info[5] += ls[2] / (float)(a.norm_rows > 0 ? a.norm_rows : a.batch_rows);
        } else {
            a.train_info[0] += ls[0];
            a.train_info[1] += norm;
            if (a.flags & ORL_PPO_VALUENORM) {
                float st[3];
                vn_updated(a.vn_state, a.mb_stats, (double)(a.norm_rows > 0 ? a.norm_rows : a.batch_rows), a.vn_beta, st);
                a.vn_state[0] = st[0]; a.vn_state[1] = st[1]; a.vn_state[2] = st[2];
            }
        }
    }
}

__global__ void minibatch_stats_kernel(const int64_t* __restrict__ idx, int64_t rows, const float* __restrict__ returns,
                                       const float* __restrict__ active, double* __restrict__ out) {
    double s0 = 0, s1 = 0, s2 = 0;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < rows; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t g = idx[i];
        const double r = returns[g];
        s0 += r; s1 += r * r; s2 += active[g];
    }
    __shared__ double red[3][8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    s0 = warp_sum(s0); s1 = warp_sum(s1); s2 = warp_sum(s2);
    if (lane == 0) { red[0][warp] = s0; red[1][warp] = s1; red[2][warp] = s2; }
    __syncthreads();
    if (threadIdx.x < 3) {
        double t = 0;
        for (int wv = 0; wv < (int)(blockDim.x >> 5); ++wv) t += red[threadIdx.x][wv];
        atomicAdd(out + threadIdx.x, t);
    }
}

size_t fwdbwd_smem_bytes(int d, int dc) {
    const int dm = std::max(d, dc);
    const int ldx = orl::pad4(dm) + 4;
    const size_t floats = orl::smem_weights_floats(dm, true) + (size_t)P_M * ldx + 3 * (size_t)P_M * orl::LDA +
                          (size_t)P_M * DLW + 4 * P_M + 32 + 4 * P_M /* row_idx as 2 floats each */ + 16;
    return floats * sizeof(float);
}

int check_ppo_args(const OrlPpoArgs& a) {
    ORL_CHECK_ARG(a.obs_dim > 0 && a.obs_dim <= 64 && a.critic_obs_dim > 0 && a.critic_obs_dim <= 64, "obs dims must be in 1..64");
    ORL_CHECK_ARG(a.n_actions > 0 && a.n_actions <= orl::MAX_OUT, "n_actions must be in 1..8");
    ORL_CHECK_ARG(a.activation_id >= 0 && a.activation_id <= 3, "activation_id");
    ORL_CHECK_ARG(a.grid_per_net > 0, "grid_per_net");
    ORL_CHECK_ARG(a.batch_rows > 0, "batch_rows");
    ORL_CHECK_ARG(a.policy_params && a.critic_params && a.partials && a.folded && a.grads && a.train_info, "null buffer");
    return 0;
}

}  // namespace

namespace orl {
int ppo_stride_host(int obs_dim, int critic_obs_dim, int n_actions) { return ppo_stride(obs_dim, critic_obs_dim, n_actions); }
int launch_ppo_fwdbwd_tc(const OrlPpoArgs& a, cudaStream_t st);
}  // namespace orl

extern "C" int orl_ppo_stride(int obs_dim, int critic_obs_dim, int n_actions) {
    return ppo_stride(obs_dim, critic_obs_dim, n_actions);
}

extern "C" int orl_ppo_grads_stride(int obs_dim, int critic_obs_dim, int n_actions) {
    return ppo_grads_stride(obs_dim, critic_obs_dim, n_actions);
}

extern "C" int orl_net_param_count(int obs_dim, int n_out) { return orl::net_offsets(obs_dim, n_out).total; }

extern "C" int orl_ppo_fwdbwd(const OrlPpoArgs* args, void* stream) {
    ORL_CHECK_ARG(args, "args");
    const OrlPpoArgs& a = *args;
    if (int e = check_ppo_args(a)) return e;
    if (a.flags & ORL_PPO_JOINT_ACTION) {
        orl::set_last_error("orl_ppo_fwdbwd: ORL_PPO_JOINT_ACTION needs chunked recurrence (orl_rnn_fwdbwd)");
        return ORL_ERR_UNSUPPORTED;
    }
    ORL_CHECK_ARG(a.policy_obs && a.critic_obs && a.actions && a.old_log_probs && a.advantages && a.value_preds &&
                      a.returns && a.active_masks && a.gae_stats && a.mb_stats, "null rollout buffer");
    ORL_CHECK_ARG(!(a.flags & ORL_PPO_VALUENORM) || a.vn_state, "vn_state required with VALUENORM");
    ORL_CHECK_ARG(a.indices || (a.row_begin >= 0 && a.row_begin + a.batch_rows <= a.total_rows), "row range");
    ORL_CHECK_ARG(a.head_kind == ORL_HEAD_CATEGORICAL || a.head_kind == ORL_HEAD_GAUSSIAN, "head_kind");
    if (a.flags & ORL_PPO_TF32) {
        if (a.head_kind != ORL_HEAD_CATEGORICAL) {
            orl::set_last_error("orl_ppo_fwdbwd: ORL_PPO_TENSORCORE supports categorical heads only");
            return ORL_ERR_UNSUPPORTED;
        }
        return orl::launch_ppo_fwdbwd_tc(a, reinterpret_cast<cudaStream_t>(stream));
    }
    const size_t smem = fwdbwd_smem_bytes(a.obs_dim, a.critic_obs_dim);
    static bool attr_set = false;
    if (!attr_set) {
        int e = orl::check_cuda(cudaFuncSetAttribute(ppo_fwdbwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024),
                                "cudaFuncSetAttribute(ppo_fwdbwd)");
        if (e) return e;
        attr_set = true;
    }
    ppo_fwdbwd_kernel<<<2 * a.grid_per_net, P_NT, smem, reinterpret_cast<cudaStream_t>(stream)>>>(a);
    ORL_LAUNCH_CHECK("ppo_fwdbwd_kernel");
    return 0;
}

extern "C" int orl_ppo_reduce(const OrlPpoArgs* args, void* stream) {
    ORL_CHECK_ARG(args, "args");
    const OrlPpoArgs& a = *args;
    if (int e = check_ppo_args(a)) return e;
    const int stride = orl_ppo_stride(a.obs_dim, a.critic_obs_dim, a.n_actions);
    dim3 grid((stride + 31) / 32, 2);
    ppo_reduce_kernel<<<grid, RED_NT, 0, reinterpret_cast<cudaStream_t>(stream)>>>(a.partials, a.folded, a.grid_per_net, stride);
    ORL_LAUNCH_CHECK("ppo_reduce_kernel");
    return 0;
}

static int check_peer_args(const OrlPeerArgs& pa) {
    ORL_CHECK_ARG(pa.world >= 2 && pa.world <= ORL_PEER_MAX_WORLD && pa.rank >= 0 && pa.rank < pa.world, "peer world / rank");
    ORL_CHECK_ARG(pa.peer_buffers && pa.local_buffer && pa.epochs && pa.error_flag && pa.summed, "null peer buffer");
    ORL_CHECK_ARG(pa.timeout_ms > 0, "timeout_ms");
    return 0;
}

extern "C" long long orl_ppo_peer_bucket_bytes(int obs_dim, int critic_obs_dim, int n_actions, int world) {
    const int stride = orl_ppo_stride(obs_dim, critic_obs_dim, n_actions);
    return (long long)peer_flag_word(world, stride) * sizeof(float) + (long long)3 * ORL_PEER_MAX_WORLD * sizeof(uint32_t) +
           (long long)2 * ORL_PEER_SMALL_MAX * sizeof(double);
}

extern "C" int orl_peer_sum_f64(const OrlPeerArgs* peer, int stride, double* data, int n, void* stream) {
    ORL_CHECK_ARG(peer && data && stride > 0 && stride % 4 == 0, "args");
    if (int e = check_peer_args(*peer)) return e;
    ORL_CHECK_ARG(n > 0 && n <= ORL_PEER_SMALL_MAX, "n must be in 1..ORL_PEER_SMALL_MAX");
    peer_sum_f64_kernel<<<1, 64, 0, reinterpret_cast<cudaStream_t>(stream)>>>(*peer, data, n, stride);
    ORL_LAUNCH_CHECK("peer_sum_f64_kernel");
    return 0;
}

extern "C" int orl_ppo_reduce_peer(const OrlPpoArgs* args, const OrlPeerArgs* peer, void* stream) {
    ORL_CHECK_ARG(args && peer, "args");
    const OrlPpoArgs& a = *args;
    if (int e = check_ppo_args(a)) return e;
    if (int e = check_peer_args(*peer)) return e;
    const int stride = orl_ppo_stride(a.obs_dim, a.critic_obs_dim, a.n_actions);
    dim3 grid((stride + 31) / 32, 2);
    ppo_reduce_peer_kernel<<<grid, RED_NT, 0, reinterpret_cast<cudaStream_t>(stream)>>>(a.partials, *peer, a.grid_per_net, stride);
    ORL_LAUNCH_CHECK("ppo_reduce_kernel(peer)");
    return 0;
}

extern "C" int orl_ppo_apply_peer(const OrlPpoArgs* args, const OrlPeerArgs* peer, void* stream) {
    ORL_CHECK_ARG(args && peer, "args");
    const OrlPpoArgs& a = *args;
    if (int e = check_ppo_args(a)) return e;
    if (int e = check_peer_args(*peer)) return e;
    ORL_CHECK_ARG(a.policy_adam_m && a.policy_adam_v && a.critic_adam_m && a.critic_adam_v && a.adam_steps && a.lrs,
                  "null optimiser state");
    ORL_CHECK_ARG(a.mb_stats, "mb_stats");
    ppo_apply_kernel<true><<<2, 1024, 0, reinterpret_cast<cudaStream_t>(stream)>>>(a, *peer);
    ORL_LAUNCH_CHECK("ppo_apply_kernel(peer)");
    return 0;
}

extern "C" int orl_ppo_apply(const OrlPpoArgs* args, void* stream) {
    ORL_CHECK_ARG(args, "args");
    const OrlPpoArgs& a = *args;
    if (int e = check_ppo_args(a)) return e;
    ORL_CHECK_ARG(a.policy_adam_m && a.policy_adam_v && a.critic_adam_m && a.critic_adam_v && a.adam_steps && a.lrs,
                  "null optimiser state");
    ORL_CHECK_ARG(a.mb_stats, "mb_stats");
    ppo_apply_kernel<false><<<2, 1024, 0, reinterpret_cast<cudaStream_t>(stream)>>>(a, OrlPeerArgs{});
    ORL_LAUNCH_CHECK("ppo_apply_kernel");
    return 0;
}

extern "C" int orl_minibatch_stats(const int64_t* indices, int64_t batch_rows, const float* returns,
                                   const float* active_masks, double* mb_stats_out, void* stream) {
    ORL_CHECK_ARG(indices && returns && active_masks && mb_stats_out && batch_rows > 0, "null buffer / rows");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    int e = orl::check_cuda(cudaMemsetAsync(mb_stats_out, 0, 3 * sizeof(double), st), "memset mb_stats");
    if (e) return e;
    const int grid = (int)std::min<int64_t>((batch_rows + 255) / 256, 4LL * orl::sm_count());
    minibatch_stats_kernel<<<grid, 256, 0, st>>>(indices, batch_rows, returns, active_masks, mb_stats_out);
    ORL_LAUNCH_CHECK("minibatch_stats_kernel");
    return 0;
}
