// kin_ppo.cu -- K3: the PPO agent update (strict-fp32 variant) and the small kernels around it.
//
//   kin_policy_act      stochastic policy step for rollout collection (actor + critic forward, Gaussian sample, log-prob)
//   kin_ppo_bootstrap   TimeLimit bootstrap  r += gamma * V(terminal_obs)  for truncated episodes
//   kin_ppo_gae         generalised advantage estimation, one thread per env scanning T steps backwards
//   kin_ppo_grad        one minibatch: fused actor+critic forward, clipped-surrogate / value / entropy loss, backward
//                       and weight-gradient accumulation; persistent CTAs, 64-sample tiles, all operands in shared
//                       memory, weight gradients accumulated in registers across tiles, deterministic two-stage
//                       reduction over CTAs (no atomics on the gradient)
//   kin_ppo_adam        global-norm clip + Adam on the flat parameter buffer
//
// Third-party arithmetic restated here: stable-baselines3 2.8.0 (ppo.py train(), on_policy_algorithm.py
// collect_rollouts(), buffers.py compute_returns_and_advantage(), distributions.py DiagGaussianDistribution) -- the
// reference only calls it (kinematic_phase1/train_workspace_expansion.py:189-232).  tests/test_gpu_ppo.py checks every
// kernel against a PyTorch autograd restatement of the same formulas.
//
// This is the FP32-pipe variant (the strict-parity path north_star asks to keep); the GEMM-shaped parts are classic
// register-tiled shared-memory SGEMMs.  The tcgen05 variant of the update is the next step (DESIGN.md).
#include <cuda_bf16.h>

#include "kin_internal.h"
#include "kin_mlp.cuh"
#include "kin_ppo_layout.cuh"
#include "kin_ppo_math.cuh"
#include "kin_state.cuh"

namespace kin {

constexpr int PPO_THREADS = 256;
constexpr int TS = KIN_PPO_TILE;      // 64 samples per tile
constexpr int HS = 132;               // row stride of the [TS][128] activation tiles (16-byte aligned rows)

// ---------------------------------------------------------------------------------------------------------
// rollout-side kernels
// ---------------------------------------------------------------------------------------------------------
struct ActW {
    const float *w0, *b0, *w1, *b1, *wo, *bo;
};

template <int IN>
__global__ void __launch_bounds__(128)
kin_policy_act_kernel(ActW pi, ActW vf, const float* __restrict__ log_std, const float* __restrict__ obs, float* __restrict__ action,
                      float* __restrict__ logp, float* __restrict__ value, int n, uint64_t seed, uint32_t step, int deterministic) {
    extern __shared__ __align__(16) float smem[];
    float* sw = smem;
    float* scratch = smem + MlpSmem<IN>::FLOATS + threadIdx.x;
    const int tid = threadIdx.x;
    const int i = blockIdx.x * 128 + tid;
    const int ic = min(i, n - 1);
    float x[IN];
    const float4* src = reinterpret_cast<const float4*>(obs + (size_t)ic * IN);
#pragma unroll
    for (int k = 0; k < IN / 4; ++k) {
        float4 v = __ldg(src + k);
        x[4 * k] = v.x; x[4 * k + 1] = v.y; x[4 * k + 2] = v.z; x[4 * k + 3] = v.w;
    }
    mlp_load_smem<IN>(sw, pi.w0, pi.b0, pi.w1, pi.b1, pi.wo, pi.bo, ACT, tid, 128);
    __syncthreads();
    float mean[ACT];
    mlp_forward<IN, ACT, 128>(sw, x, mean, scratch);
    if (i < n) {
        Philox rng(seed, (unsigned)i, step);
        float lp = 0.0f;
        float eps[8];
#pragma unroll
        for (int k = 0; k < 8; k += 2) eps[k] = gauss_pair(rng, &eps[k + 1]);
#pragma unroll
        for (int k = 0; k < ACT; ++k) {
            const float ls = __ldg(log_std + k);
            const float e = deterministic ? 0.0f : eps[k];
            action[(size_t)i * ACT + k] = fmaf(expf(ls), e, mean[k]);
            lp += gauss_logp_term(e, ls);   // (a - mean) / sigma == eps
        }
        logp[i] = lp;
    }
    if (value) {
        __syncthreads();
        mlp_load_smem<IN>(sw, vf.w0, vf.b0, vf.w1, vf.b1, vf.wo, vf.bo, 1, tid, 128);
        __syncthreads();
        float v[1];
        mlp_forward<IN, 1, 128>(sw, x, v, scratch);
        if (i < n) value[i] = v[0];
    }
}

template <int IN>
__global__ void __launch_bounds__(128)
kin_ppo_bootstrap_kernel(ActW vf, const float* __restrict__ terminal_obs, const uint8_t* __restrict__ done, float* __restrict__ reward,
                         float gamma, int n) {
    extern __shared__ __align__(16) float smem[];
    const int tid = threadIdx.x;
    const int i = blockIdx.x * 128 + tid;
    const bool trunc = i < n && (done[i] & KIN_DONE_TRUNCATED) && !(done[i] & KIN_DONE_TERMINATED);
    if (!__syncthreads_or(trunc)) return;   // block-uniform early exit: most steps truncate nothing
    float* sw = smem;
    float* scratch = smem + MlpSmem<IN>::FLOATS + tid;
    const int ic = min(i, n - 1);
    float x[IN];
    const float4* src = reinterpret_cast<const float4*>(terminal_obs + (size_t)ic * IN);
#pragma unroll
    for (int k = 0; k < IN / 4; ++k) {
        float4 v = __ldg(src + k);
        x[4 * k] = v.x; x[4 * k + 1] = v.y; x[4 * k + 2] = v.z; x[4 * k + 3] = v.w;
    }
    mlp_load_smem<IN>(sw, vf.w0, vf.b0, vf.w1, vf.b1, vf.wo, vf.bo, 1, tid, 128);
    __syncthreads();
    float v[1];
    mlp_forward<IN, 1, 128>(sw, x, v, scratch);
    if (trunc) reward[i] = fmaf(gamma, v[0], reward[i]);
}

// POP (the kin_pop_* population launches, kin_b200.h): the kernels below take their per-run pointers and hyper-parameters from member
// blockIdx.y's KinPopMember descriptor, whose table arrives in the first pointer argument; the body is the standalone kernel's.

// buffers.py compute_returns_and_advantage: one thread per env, backwards over T; [T][n] arrays are coalesced over envs
template <bool POP = false>
__global__ void __launch_bounds__(256)
kin_ppo_gae_kernel(const float* __restrict__ reward, const float* __restrict__ value, const uint8_t* __restrict__ episode_start,
                   const float* __restrict__ last_value, const uint8_t* __restrict__ last_done, float gamma, float lam, int T, int n,
                   float* __restrict__ adv, float* __restrict__ ret) {
    if constexpr (POP) {
        const KinPopMember& M = reinterpret_cast<const KinPopMember*>(reward)[blockIdx.y];
        reward = M.reward;
        value = M.value;
        episode_start = M.episode_start;
        last_value = M.last_value;
        last_done = M.done + (size_t)(T - 1) * n;
        gamma = M.hyper.gamma;
        lam = M.hyper.gae_lambda;
        adv = M.advantage;
        ret = M.returns;
    }
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    float next_value = last_value[e];
    float next_non_terminal = (last_done[e] & (KIN_DONE_TERMINATED | KIN_DONE_TRUNCATED)) ? 0.0f : 1.0f;
    float last_gae = 0.0f;
    for (int t = T - 1; t >= 0; --t) {
        const size_t idx = (size_t)t * n + e;
        const float v = value[idx];
        const float delta = fmaf(gamma * next_value, next_non_terminal, reward[idx]) - v;
        last_gae = fmaf(gamma * lam * next_non_terminal, last_gae, delta);
        adv[idx] = last_gae;
        ret[idx] = last_gae + v;
        next_value = v;
        next_non_terminal = episode_start[idx] ? 0.0f : 1.0f;
    }
}

// (sum adv, sum adv^2) per 64-sample tile, in double
template <bool POP = false>
__global__ void __launch_bounds__(64)
kin_ppo_tile_sums_kernel(const float* __restrict__ adv, double* __restrict__ tile_sums) {
    if constexpr (POP) {
        const KinPopMember& M = reinterpret_cast<const KinPopMember*>(adv)[blockIdx.y];
        adv = M.advantage;
        tile_sums = M.tile_sums;
    }
    const int tile = blockIdx.x;
    const double a = (double)adv[(size_t)tile * TS + threadIdx.x];
    double s1 = a, s2 = a * a;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        s1 += __shfl_xor_sync(0xffffffffu, s1, off);
        s2 += __shfl_xor_sync(0xffffffffu, s2, off);
    }
    __shared__ double sh[4];
    if ((threadIdx.x & 31) == 0) { sh[(threadIdx.x >> 5) * 2] = s1; sh[(threadIdx.x >> 5) * 2 + 1] = s2; }
    __syncthreads();
    if (threadIdx.x == 0) { tile_sums[2 * tile] = sh[0] + sh[2]; tile_sums[2 * tile + 1] = sh[1] + sh[3]; }
}

// ---------------------------------------------------------------------------------------------------------
// the minibatch gradient
// ---------------------------------------------------------------------------------------------------------
template <int IN>
struct GradSmem {
    static constexpr int XS = IN + 1;                 // X row stride
    static constexpr int W0T = 0;                     // [IN][128]
    static constexpr int B0 = W0T + IN * 128;         // [128]
    static constexpr int W1 = B0 + 128;               // [2][64][64]  (u, i)
    static constexpr int W1T = W1 + 2 * 4096;         // [2][64][64]  (i, u)
    static constexpr int B1 = W1T + 2 * 4096;         // [128]
    static constexpr int WOA = B1 + 128;              // [7][64]
    static constexpr int WOC = WOA + 448;             // [64]
    static constexpr int BO = WOC + 64;               // [8]
    static constexpr int LS = BO + 8;                 // log_std [8]
    static constexpr int X = LS + 8;                  // [TS][XS]
    static constexpr int H1 = X + TS * XS + ((4 - (TS * XS) % 4) % 4);   // [TS][HS]
    static constexpr int H2 = H1 + TS * HS;
    static constexpr int G = H2 + TS * HS;
    static constexpr int OUT8 = G + TS * HS;          // [TS][8]
    static constexpr int SCAL = OUT8 + TS * 8;        // [0] adv mean, [1] 1/(std+eps), then RED
    static constexpr int RED = SCAL + 8;              // [2][12] per loss warp: the 5 statistics, the 7 d log_std, summed over its tiles
    static constexpr int FLOATS = SCAL + 32;
    static_assert(RED + 2 * 12 <= FLOATS, "the loss warps' rows fit the scalar block");
};

template <int IN>
__global__ void __launch_bounds__(PPO_THREADS, 1)
kin_ppo_grad_kernel(const float* __restrict__ params, KinPpoHyper hp, const float* __restrict__ obs, const float* __restrict__ action,
                    const float* __restrict__ old_logp, const float* __restrict__ advantage, const float* __restrict__ returns,
                    const double* __restrict__ tile_sums, const int* __restrict__ tile_ids, int n_tiles, float inv_global_batch,
                    float* __restrict__ partials, const float* __restrict__ adv_stats) {
    using L = GradSmem<IN>;
    extern __shared__ __align__(16) float sm[];
    const PpoOffsets O = ppo_offsets(IN);
    const int tid = threadIdx.x;
    const int P = O.total;

    // ---- stage the weights (both nets) -----------------------------------------------------------------
    for (int i = tid; i < 64 * IN; i += PPO_THREADS) {
        const int u = i / IN, k = i - u * IN;
        sm[L::W0T + k * 128 + u] = __ldg(params + O.pi_w0 + i);
        sm[L::W0T + k * 128 + 64 + u] = __ldg(params + O.vf_w0 + i);
    }
    for (int i = tid; i < 4096; i += PPO_THREADS) {
        const int u = i >> 6, k = i & 63;
        const float wa = __ldg(params + O.pi_w1 + i), wc = __ldg(params + O.vf_w1 + i);
        sm[L::W1 + i] = wa;
        sm[L::W1 + 4096 + i] = wc;
        sm[L::W1T + k * 64 + u] = wa;
        sm[L::W1T + 4096 + k * 64 + u] = wc;
    }
    if (tid < 64) {
        sm[L::B0 + tid] = __ldg(params + O.pi_b0 + tid);
        sm[L::B0 + 64 + tid] = __ldg(params + O.vf_b0 + tid);
        sm[L::B1 + tid] = __ldg(params + O.pi_b1 + tid);
        sm[L::B1 + 64 + tid] = __ldg(params + O.vf_b1 + tid);
        sm[L::WOC + tid] = __ldg(params + O.val_w + tid);
    }
    for (int i = tid; i < 448; i += PPO_THREADS) sm[L::WOA + i] = __ldg(params + O.act_w + i);
    if (tid < 8) {
        sm[L::BO + tid] = tid < 7 ? __ldg(params + O.act_b + tid) : __ldg(params + O.val_b);
        sm[L::LS + tid] = tid < 7 ? __ldg(params + O.log_std + tid) : 0.0f;
    }
    if (tid < 32) sm[L::SCAL + tid] = 0.0f;
    // advantage statistics of this minibatch (torch: mean, unbiased std): precomputed (kin_ppo_adv_stats) or from the per-tile sums
    if (adv_stats) {
        if (tid == 0) { sm[L::SCAL + 0] = adv_stats[0]; sm[L::SCAL + 1] = adv_stats[1]; }
    } else if (tid < 32) {
        const double2 s = warp_tile_sums(tile_sums, tile_ids, n_tiles, tid, 32);
        if (tid == 0) adv_normaliser(s.x, s.y, (double)n_tiles * TS, hp.normalize_advantage, &sm[L::SCAL]);
    }
    __syncthreads();

    // ---- register accumulators (live across all tiles of this CTA) --------------------------------------
    const int ty = tid >> 4, tx = tid & 15;              // 16 x 16 thread grid for the [64 x 128] tiles: 4 samples x 8 units
    const int net_col = tx >= 8 ? 64 : 0;                // activation column offset of this thread's net
    const int net_id = tx >= 8 ? 1 : 0;
    const int ucol = (tx & 7) * 8;
    const int w1_net = tid >> 7, w1_t = tid & 127;       // dW1: 128 threads per net, 4(u) x 8(i) block
    const int w1_u0 = (w1_t >> 3) * 4, w1_i0 = (w1_t & 7) * 8;
    constexpr int KB = IN / 8;                           // dW0: 4(u) x KB(k) block
    const int w0_u0 = (tid & 31) * 4, w0_k0 = (tid >> 5) * KB;
    float acc_w1[4][8], acc_w0[KB][4], acc_wo[2] = {0.0f, 0.0f}, acc_b1 = 0.0f, acc_b0 = 0.0f, acc_bo = 0.0f;
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 8; ++b) acc_w1[a][b] = 0.0f;
#pragma unroll
    for (int a = 0; a < KB; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) acc_w0[a][b] = 0.0f;

    for (int j = blockIdx.x; j < n_tiles; j += gridDim.x) {
        const size_t base = (size_t)tile_ids[j] * TS;
        // ---- load the observation tile (coalesced) -----------------------------------------------------
        for (int i = tid; i < TS * IN; i += PPO_THREADS) {
            const int s = i / IN, k = i - s * IN;
            sm[L::X + s * L::XS + k] = __ldg(obs + base * IN + i);
        }
        __syncthreads();
        // ---- layer 1: H1 = tanh(X W0^T + b0), both nets --------------------------------------------------
        {
            float acc[4][8];
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int c = 0; c < 8; ++c) acc[r][c] = sm[L::B0 + tx * 8 + c];
#pragma unroll 4
            for (int k = 0; k < IN; ++k) {
                const float4 w0 = *reinterpret_cast<const float4*>(&sm[L::W0T + k * 128 + tx * 8]);
                const float4 w1 = *reinterpret_cast<const float4*>(&sm[L::W0T + k * 128 + tx * 8 + 4]);
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    const float x = sm[L::X + (ty * 4 + r) * L::XS + k];
                    acc[r][0] = fmaf(x, w0.x, acc[r][0]); acc[r][1] = fmaf(x, w0.y, acc[r][1]);
                    acc[r][2] = fmaf(x, w0.z, acc[r][2]); acc[r][3] = fmaf(x, w0.w, acc[r][3]);
                    acc[r][4] = fmaf(x, w1.x, acc[r][4]); acc[r][5] = fmaf(x, w1.y, acc[r][5]);
                    acc[r][6] = fmaf(x, w1.z, acc[r][6]); acc[r][7] = fmaf(x, w1.w, acc[r][7]);
                }
            }
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                float* dst = &sm[L::H1 + (ty * 4 + r) * HS + tx * 8];
                *reinterpret_cast<float4*>(dst) = make_float4(tanhf(acc[r][0]), tanhf(acc[r][1]), tanhf(acc[r][2]), tanhf(acc[r][3]));
                *reinterpret_cast<float4*>(dst + 4) = make_float4(tanhf(acc[r][4]), tanhf(acc[r][5]), tanhf(acc[r][6]), tanhf(acc[r][7]));
            }
        }
        __syncthreads();
        // ---- layer 2: H2 = tanh(H1 W1^T + b1), block diagonal over the two nets -----------------------------
        {
            float acc[4][8];
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int c = 0; c < 8; ++c) acc[r][c] = sm[L::B1 + net_col + ucol + c];
            const float* wT = &sm[L::W1T + net_id * 4096];
#pragma unroll 4
            for (int k = 0; k < 64; ++k) {
                const float4 w0 = *reinterpret_cast<const float4*>(&wT[k * 64 + ucol]);
                const float4 w1 = *reinterpret_cast<const float4*>(&wT[k * 64 + ucol + 4]);
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    const float x = sm[L::H1 + (ty * 4 + r) * HS + net_col + k];
                    acc[r][0] = fmaf(x, w0.x, acc[r][0]); acc[r][1] = fmaf(x, w0.y, acc[r][1]);
                    acc[r][2] = fmaf(x, w0.z, acc[r][2]); acc[r][3] = fmaf(x, w0.w, acc[r][3]);
                    acc[r][4] = fmaf(x, w1.x, acc[r][4]); acc[r][5] = fmaf(x, w1.y, acc[r][5]);
                    acc[r][6] = fmaf(x, w1.z, acc[r][6]); acc[r][7] = fmaf(x, w1.w, acc[r][7]);
                }
            }
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                float* dst = &sm[L::H2 + (ty * 4 + r) * HS + net_col + ucol];
                *reinterpret_cast<float4*>(dst) = make_float4(tanhf(acc[r][0]), tanhf(acc[r][1]), tanhf(acc[r][2]), tanhf(acc[r][3]));
                *reinterpret_cast<float4*>(dst + 4) = make_float4(tanhf(acc[r][4]), tanhf(acc[r][5]), tanhf(acc[r][6]), tanhf(acc[r][7]));
            }
        }
        __syncthreads();
        // ---- layer 3: 7 action means + 1 value per sample (2 outputs per thread) --------------------------
        {
            const int s = tid >> 2, d0 = (tid & 3) * 2;
#pragma unroll
            for (int dd = 0; dd < 2; ++dd) {
                const int d = d0 + dd;
                const float* w = d < 7 ? &sm[L::WOA + d * 64] : &sm[L::WOC];
                const float* h = &sm[L::H2 + s * HS + (d < 7 ? 0 : 64)];
                float a0 = sm[L::BO + d], a1 = 0.0f;
#pragma unroll 8
                for (int k = 0; k < 64; k += 2) { a0 = fmaf(h[k], w[k], a0); a1 = fmaf(h[k + 1], w[k + 1], a1); }
                sm[L::OUT8 + s * 8 + d] = a0 + a1;
            }
        }
        __syncthreads();
        // ---- loss and d(loss)/d(outputs), one thread per sample (ppo.py train()) -----------------------------
        if (tid < TS) {
            const int s = tid;
            const size_t g = base + s;
            float lp = 0.0f, ent = 0.0f, z[7], inv_sig[7];
#pragma unroll
            for (int d = 0; d < 7; ++d) {
                const float ls = sm[L::LS + d];
                inv_sig[d] = expf(-ls);
                z[d] = (__ldg(action + g * 7 + d) - sm[L::OUT8 + s * 8 + d]) * inv_sig[d];
                lp += gauss_logp_term(z[d], ls);
                ent += gauss_entropy_term(ls);
            }
            const Surrogate sur = clipped_surrogate(__ldg(advantage + g), sm[L::SCAL + 0], sm[L::SCAL + 1], lp, __ldg(old_logp + g), hp);
            const float dpl_dlp = sur.dpl_dlp();
            const float v = sm[L::OUT8 + s * 8 + 7], rt = __ldg(returns + g);
#pragma unroll
            for (int d = 0; d < 7; ++d) {
                sm[L::OUT8 + s * 8 + d] = dloss_dmean(inv_global_batch, dpl_dlp, z[d], inv_sig[d]);
                z[d] = dloss_dlog_std(inv_global_batch, dpl_dlp, z[d], hp);
            }
            sm[L::OUT8 + s * 8 + 7] = dloss_dvalue(inv_global_batch, v, rt, hp);
            // statistics: sums over samples (divided by the global batch at the end)
            float st[5];
            st[KIN_PPO_STAT_POLICY_LOSS] = sur.loss();
            st[KIN_PPO_STAT_VALUE_LOSS] = value_loss(v, rt);
            st[KIN_PPO_STAT_ENTROPY] = ent;
            st[KIN_PPO_STAT_APPROX_KL] = sur.approx_kl();
            st[KIN_PPO_STAT_CLIP_FRACTION] = sur.clipped(hp);
#pragma unroll
            for (int q = 0; q < 5; ++q) {
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) st[q] += __shfl_xor_sync(0xffffffffu, st[q], off);
            }
#pragma unroll
            for (int d = 0; d < 7; ++d) {
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) z[d] += __shfl_xor_sync(0xffffffffu, z[d], off);
            }
            if ((tid & 31) == 0) {      // each loss warp into its own row: the sums are taken in a fixed order
                float* r = &sm[L::RED + (tid >> 5) * 12];
#pragma unroll
                for (int q = 0; q < 5; ++q) r[q] += st[q];
#pragma unroll
                for (int d = 0; d < 7; ++d) r[5 + d] += z[d];
            }
        }
        __syncthreads();
        // ---- dZ2 = (dOut Wo) * (1 - H2^2) -> G --------------------------------------------------------------
        {
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const int s = ty * 4 + r;
                float g[8];
                if (net_id == 0) {
#pragma unroll
                    for (int c = 0; c < 8; ++c) g[c] = 0.0f;
#pragma unroll
                    for (int d = 0; d < 7; ++d) {
                        const float dm = sm[L::OUT8 + s * 8 + d];
#pragma unroll
                        for (int c = 0; c < 8; ++c) g[c] = fmaf(dm, sm[L::WOA + d * 64 + ucol + c], g[c]);
                    }
                } else {
                    const float dv = sm[L::OUT8 + s * 8 + 7];
#pragma unroll
                    for (int c = 0; c < 8; ++c) g[c] = dv * sm[L::WOC + ucol + c];
                }
                const float* h = &sm[L::H2 + s * HS + net_col + ucol];
                float* dst = &sm[L::G + s * HS + net_col + ucol];
#pragma unroll
                for (int c = 0; c < 8; ++c) dst[c] = g[c] * (1.0f - h[c] * h[c]);
            }
        }
        __syncthreads();
        // ---- output-layer weight / bias grads, b1 grads -------------------------------------------------------
        {
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                const int e = tid + q * PPO_THREADS;     // 0..447: act_w[d][j]; 448..511: val_w[j]
                const int d = e < 448 ? (e >> 6) : 7, jj = e & 63;
                const int hcol = e < 448 ? jj : 64 + jj;
                float a = 0.0f;
#pragma unroll 8
                for (int s = 0; s < TS; ++s) a = fmaf(sm[L::OUT8 + s * 8 + d], sm[L::H2 + s * HS + hcol], a);
                acc_wo[q] += a;
            }
            if (tid < 8) {
                float a = 0.0f;
                for (int s = 0; s < TS; ++s) a += sm[L::OUT8 + s * 8 + tid];
                acc_bo += a;
            }
            if (tid >= 128) {
                const int u = tid - 128;
                float a = 0.0f;
#pragma unroll 8
                for (int s = 0; s < TS; ++s) a += sm[L::G + s * HS + u];
                acc_b1 += a;
            }
        }
        // ---- dW1 += G^T H1 (per net) ----------------------------------------------------------------------------
        {
            const int gc = w1_net * 64 + w1_u0, hc = w1_net * 64 + w1_i0;
#pragma unroll 2
            for (int s = 0; s < TS; ++s) {
                const float4 g = *reinterpret_cast<const float4*>(&sm[L::G + s * HS + gc]);
                const float4 h0 = *reinterpret_cast<const float4*>(&sm[L::H1 + s * HS + hc]);
                const float4 h1 = *reinterpret_cast<const float4*>(&sm[L::H1 + s * HS + hc + 4]);
                const float gg[4] = {g.x, g.y, g.z, g.w};
                const float hh[8] = {h0.x, h0.y, h0.z, h0.w, h1.x, h1.y, h1.z, h1.w};
#pragma unroll
                for (int a = 0; a < 4; ++a)
#pragma unroll
                    for (int b = 0; b < 8; ++b) acc_w1[a][b] = fmaf(gg[a], hh[b], acc_w1[a][b]);
            }
        }
        // ---- dZ1 = (G W1) * (1 - H1^2) -> H2 tile (H2 itself is dead now for this thread's columns only after the sync) ----
        __syncthreads();
        {
            float acc[4][8];
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int c = 0; c < 8; ++c) acc[r][c] = 0.0f;
            const float* w = &sm[L::W1 + net_id * 4096];
#pragma unroll 4
            for (int u = 0; u < 64; ++u) {
                const float4 w0 = *reinterpret_cast<const float4*>(&w[u * 64 + ucol]);
                const float4 w1 = *reinterpret_cast<const float4*>(&w[u * 64 + ucol + 4]);
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    const float g = sm[L::G + (ty * 4 + r) * HS + net_col + u];
                    acc[r][0] = fmaf(g, w0.x, acc[r][0]); acc[r][1] = fmaf(g, w0.y, acc[r][1]);
                    acc[r][2] = fmaf(g, w0.z, acc[r][2]); acc[r][3] = fmaf(g, w0.w, acc[r][3]);
                    acc[r][4] = fmaf(g, w1.x, acc[r][4]); acc[r][5] = fmaf(g, w1.y, acc[r][5]);
                    acc[r][6] = fmaf(g, w1.z, acc[r][6]); acc[r][7] = fmaf(g, w1.w, acc[r][7]);
                }
            }
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const float* h = &sm[L::H1 + (ty * 4 + r) * HS + net_col + ucol];
                float* dst = &sm[L::H2 + (ty * 4 + r) * HS + net_col + ucol];
#pragma unroll
                for (int c = 0; c < 8; ++c) dst[c] = acc[r][c] * (1.0f - h[c] * h[c]);
            }
        }
        __syncthreads();
        // ---- b0 grads and dW0 += G1^T X --------------------------------------------------------------------------
        {
            if (tid < 128) {
                float a = 0.0f;
#pragma unroll 8
                for (int s = 0; s < TS; ++s) a += sm[L::H2 + s * HS + tid];
                acc_b0 += a;
            }
#pragma unroll 2
            for (int s = 0; s < TS; ++s) {
                const float4 g = *reinterpret_cast<const float4*>(&sm[L::H2 + s * HS + w0_u0]);
#pragma unroll
                for (int a = 0; a < KB; ++a) {
                    const float x = sm[L::X + s * L::XS + w0_k0 + a];
                    acc_w0[a][0] = fmaf(x, g.x, acc_w0[a][0]); acc_w0[a][1] = fmaf(x, g.y, acc_w0[a][1]);
                    acc_w0[a][2] = fmaf(x, g.z, acc_w0[a][2]); acc_w0[a][3] = fmaf(x, g.w, acc_w0[a][3]);
                }
            }
        }
        __syncthreads();
    }

    // ---- write this CTA's partial gradient (flat parameter order) + statistics ------------------------------------------
    float* out = partials + (size_t)blockIdx.x * (P + KIN_PPO_STATS + 8);
    {
        const int w1_base = w1_net ? O.vf_w1 : O.pi_w1;
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int b = 0; b < 8; ++b) out[w1_base + (w1_u0 + a) * 64 + w1_i0 + b] = acc_w1[a][b];
#pragma unroll
        for (int a = 0; a < KB; ++a)
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                const int u = w0_u0 + b, k = w0_k0 + a;
                out[(u < 64 ? O.pi_w0 + u * IN : O.vf_w0 + (u - 64) * IN) + k] = acc_w0[a][b];
            }
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const int e = tid + q * PPO_THREADS;
            out[e < 448 ? O.act_w + e : O.val_w + (e - 448)] = acc_wo[q];
        }
        if (tid < 7) out[O.act_b + tid] = acc_bo;
        if (tid == 7) out[O.val_b] = acc_bo;
        if (tid >= 128) { const int u = tid - 128; out[(u < 64 ? O.pi_b1 + u : O.vf_b1 + u - 64)] = acc_b1; }
        if (tid < 128) out[(tid < 64 ? O.pi_b0 + tid : O.vf_b0 + tid - 64)] = acc_b0;
        if (tid < 7) out[O.log_std + tid] = sm[L::RED + 5 + tid] + sm[L::RED + 12 + 5 + tid];      // loss warp 0 + loss warp 1
        if (tid < 5) out[P + tid] = sm[L::RED + tid] + sm[L::RED + 12 + tid];
    }
}

// grad[p] = sum over CTAs of partials[c][p]; stats likewise.  A block owns 32 consecutive parameters (one 128-byte line per
// partial row); its 8 warps take rows w, w + 8, ... with independent loads in flight, then fold in a fixed order (deterministic).
template <bool POP = false>
__global__ void __launch_bounds__(256)
kin_ppo_reduce_kernel(const float* __restrict__ partials, int n_cta, int P, float* __restrict__ grad, float* __restrict__ stats, float inv_global_batch) {
    if constexpr (POP) {
        const KinPopMember& M = reinterpret_cast<const KinPopMember*>(partials)[blockIdx.y];
        partials = M.partials;
        grad = M.grad;
        stats = M.stats;
    }
    __shared__ float part[8][32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int p = blockIdx.x * 32 + lane;
    const int row = P + KIN_PPO_STATS + 8;
    float a0 = 0.0f, a1 = 0.0f;
    if (p < P + 5) {
        int c = w;
        for (; c + 8 < n_cta; c += 16) {
            a0 += __ldg(partials + (size_t)c * row + p);
            a1 += __ldg(partials + (size_t)(c + 8) * row + p);
        }
        if (c < n_cta) a0 += __ldg(partials + (size_t)c * row + p);
    }
    part[w][lane] = a0 + a1;
    __syncthreads();
    if (w == 0 && p < P + 5) {
        float a = part[0][lane];
#pragma unroll
        for (int k = 1; k < 8; ++k) a += part[k][lane];
        if (p < P) grad[p] = a;
        else if (stats) stats[p - P] = a * inv_global_batch;
    }
}

// adv_normaliser of each minibatch from the per-tile fp64 sums; one CTA per minibatch, minibatch m = tile_ids[m * n_tiles .. (m + 1) * n_tiles)
template <bool POP = false>
__global__ void __launch_bounds__(256)
kin_ppo_adv_stats_kernel(const double* __restrict__ tile_sums, const int* __restrict__ tile_ids, int n_tiles, int normalize, float* __restrict__ out) {
    if constexpr (POP) {
        const KinPopMember& M = reinterpret_cast<const KinPopMember*>(tile_sums)[blockIdx.y];
        tile_sums = M.tile_sums;
        tile_ids = M.tile_ids;
        normalize = M.hyper.normalize_advantage;
        out = M.adv_stats;
    }
    __shared__ double sh[2][8];
    const double2 s = warp_tile_sums(tile_sums, tile_ids + (size_t)blockIdx.x * n_tiles, n_tiles, threadIdx.x, 256);
    if ((threadIdx.x & 31) == 0) { sh[0][threadIdx.x >> 5] = s.x; sh[1][threadIdx.x >> 5] = s.y; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double s1 = 0.0, s2 = 0.0;
        for (int k = 0; k < 8; ++k) { s1 += sh[0][k]; s2 += sh[1][k]; }
        adv_normaliser(s1, s2, (double)n_tiles * TS, normalize, out + 2 * blockIdx.x);
    }
}

// clip_grad_norm_ + Adam.  Every CTA computes the global gradient norm itself (64 KB of L2-resident data, identical summation
// order -> bitwise-identical clip coefficient in every CTA), then updates its own 1024 parameters.
// POP: grad carries the table; bc1 / bc2 come from the one extra (by-value) argument, computed on the host from each member's betas
// and step as kin_ppo_adam computes them.  The standalone instance has no extra argument: its parameter list is unchanged.
struct PopBiasCorrection {
    float bc[KIN_POP_MAX][2];
};

// POP_IMAGE (populations only): keep member.weight_image in step in place (56 inputs); false leaves it alone (the folded route image is
// rebuilt by kin_ppo_pack_weights_kernel<true> afterwards, as the standalone route update calls kin_ppo_adam(NULL) + kin_ppo_pack_weights)
template <bool POP = false, bool POP_IMAGE = true, class... PopArgs>
__global__ void __launch_bounds__(1024)
kin_ppo_adam_kernel(float* __restrict__ params, const float* __restrict__ grad, float* __restrict__ m, float* __restrict__ v, int P,
                    KinPpoHyper hp, float bc1, float bc2, float* __restrict__ stats, float* __restrict__ stats_accum,
                    unsigned short* __restrict__ wimg, int in_dim, const __grid_constant__ PopArgs... pop) {
    static_assert(sizeof...(PopArgs) == (POP ? 1 : 0), "the population instance takes its bias corrections as one extra argument");
    if constexpr (POP) {
        const PopBiasCorrection& B = (pop, ...);
        const KinPopMember& M = reinterpret_cast<const KinPopMember*>(grad)[blockIdx.y];
        params = M.params;
        grad = M.grad;
        m = M.adam_m;
        v = M.adam_v;
        hp = M.hyper;
        bc1 = B.bc[blockIdx.y][0];
        bc2 = B.bc[blockIdx.y][1];
        stats = M.stats;
        stats_accum = M.stats_accum;
        wimg = POP_IMAGE ? static_cast<unsigned short*>(M.weight_image) : nullptr;
    }
    __shared__ float red[32];
    __shared__ float coef;
    if (stats && stats[KIN_PPO_STAT_SKIP] != 0.0f) return;      // the gradient exchange timed out (kin_peer.cu): leave the parameters alone
    // this thread's own parameter: fetch its optimiser state now, so the loads fly while the norm is being reduced
    const int own = blockIdx.x * blockDim.x + threadIdx.x;
    const bool has_own = own < P && gridDim.x * blockDim.x >= P;      // the usual launch: one parameter per thread
    float own_m = 0.0f, own_v = 0.0f, own_p = 0.0f;
    if (has_own) { own_m = m[own]; own_v = v[own]; own_p = params[own]; }
    // sum of squares in a fixed order; batches of 8 independent loads (the trip count is a runtime value: unroll by hand)
    float ss = 0.0f;
    for (int p0 = threadIdx.x; p0 < P; p0 += 8 * blockDim.x) {
        float g[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int p = p0 + k * blockDim.x;
            g[k] = p < P ? __ldcg(grad + p) : 0.0f;
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) ss = fmaf(g[k], g[k], ss);
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, off);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ss;
    __syncthreads();
    if (threadIdx.x < 32) {
        float t = red[threadIdx.x];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) t += __shfl_xor_sync(0xffffffffu, t, off);
        if (threadIdx.x == 0) {
            const float norm = sqrtf(t);
            coef = clip_coef(norm, hp);
            if (stats && blockIdx.x == 0) stats[KIN_PPO_STAT_GRAD_NORM] = norm;
            if (stats && stats_accum && blockIdx.x == 0) {          // running sums over the minibatches of an update (slot 7 counts them)
#pragma unroll
                for (int q = 0; q < 5; ++q) stats_accum[q] += stats[q];
                stats_accum[KIN_PPO_STAT_GRAD_NORM] += norm;
                stats_accum[7] += 1.0f;
            }
        }
    }
    __syncthreads();
    const float cf = coef;
    for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < P; p += gridDim.x * blockDim.x) {
        const AdamMoments mv = adam_moments(__ldcg(grad + p), cf, has_own ? own_m : m[p], has_own ? own_v : v[p], hp);
        m[p] = mv.m;
        v[p] = mv.v;
        const float np = adam_param(has_own ? own_p : params[p], mv, bc1, bc2, hp);
        params[p] = np;
        if (wimg) {      // keep the bf16 operand image of the weights in step with the parameters
            const int off = wimg_offset(ppo_offsets(in_dim), in_dim, p);
            if (off >= 0) wimg[off >> 1] = __bfloat16_as_ushort(__float2bfloat16_rn(np));
        }
    }
}

// full (re)build of the bf16 operand image from the flat parameters
// POP (kin_pop_route_adam): params carries the KinPopMember table, member blockIdx.y's parameters and image replace the arguments.  The
// standalone entry zeroes the image before the launch; here the kernel writes those zeros itself: the only image bytes no parameter
// maps to are the padding rows of the two WO blocks (actor rows 7..15, critic rows 0..6 and 8..15).
template <bool POP = false>
__global__ void __launch_bounds__(256)
kin_ppo_pack_weights_kernel(const float* __restrict__ params, int in_dim, unsigned short* __restrict__ wimg) {
    if constexpr (POP) {
        const KinPopMember& M = reinterpret_cast<const KinPopMember*>(params)[blockIdx.y];
        params = M.params;
        wimg = static_cast<unsigned short*>(M.weight_image);
    }
    const PpoOffsets O = ppo_offsets(in_dim);
    const int i = blockIdx.x * 256 + threadIdx.x;
    if constexpr (POP) {
        if (i < 2 * 16 * 64) {
            const int blk = i >> 10, r = (i >> 6) & 15;
            if (blk == 0 ? r >= 7 : r != 7) wimg[(KIN_WIMG_WO + blk * 2048 + wimg_elem(r, i & 63)) >> 1] = 0;
        }
    }
    if (in_dim == 80) {       // folded layer 1: one thread per image element of the two W0 blocks; the rest as for 56 inputs
        if (i < 2 * 64 * 64) {
            const int net = i >> 12, u = (i >> 6) & 63, k = i & 63;
            const int w0 = net ? O.vf_w0 : O.pi_w0, b0 = net ? O.vf_b0 : O.pi_b0;
            float v = 0.0f;
            if (k < KIN_ROUTE_DYN) v = params[w0 + u * 80 + route_unfold_col(k)];
            else if (k == KIN_ROUTE_DYN) v = params[b0 + u] + params[w0 + u * 80 + KIN_ROUTE_ONE_A] + params[w0 + u * 80 + KIN_ROUTE_ONE_B];
            wimg[(KIN_WIMG_W0 + net * 8192 + wimg_elem(u, k)) >> 1] = __bfloat16_as_ushort(__float2bfloat16_rn(v));
        }
        if (i < O.total) {
            const bool layer1 = (i >= O.pi_w0 && i < O.pi_w1) || (i >= O.vf_w0 && i < O.vf_w1);
            if (!layer1) {
                // the 56-input offsets of the blocks behind layer 1 are the same image positions: map through a 56-layout twin
                const PpoOffsets T = ppo_offsets(56);
                const int twin = i < O.vf_w0 ? i - (O.pi_w1 - T.pi_w1) : i - (O.vf_w1 - T.vf_w1);
                const int off = wimg_offset(T, 56, twin);
                if (off >= 0) wimg[off >> 1] = __bfloat16_as_ushort(__float2bfloat16_rn(params[i]));
            }
        }
        return;
    }
    if (i < O.total) {
        const int off = wimg_offset(O, in_dim, i);
        if (off >= 0) wimg[off >> 1] = __bfloat16_as_ushort(__float2bfloat16_rn(params[i]));
    }
}

// route observations [n_rows][80] fp32 -> folded bf16 operand images [n_rows / 128][16 KB] ([60 live columns | 1 | 0 0 0] rows,
// SWIZZLE_128B): what kin_ppo_grad_tc(in_dim = 80, obs_is_image = 1) stages with one bulk copy per tile.  One thread per 16-byte chunk.
// POP (kin_pop_route_obs_images): obs carries the KinPopRouteMember table and img the KinPopMember table; member blockIdx.y's fp32 rows go
// to its folded images.
template <bool POP = false>
__global__ void __launch_bounds__(256)
kin_route_obs_images_kernel(const float* __restrict__ obs, long long n_rows, unsigned char* __restrict__ img) {
    if constexpr (POP) {
        obs = reinterpret_cast<const KinPopRouteMember*>(obs)[blockIdx.y].obs;
        img = static_cast<unsigned char*>(reinterpret_cast<const KinPopMember*>(img)[blockIdx.y].obs_tiles);
    }
    const long long i = (long long)blockIdx.x * 256 + threadIdx.x;      // row * 8 + chunk
    if (i >= n_rows * 8) return;
    const long long row = i >> 3;
    const int ch = (int)(i & 7), r = (int)(row & 127);
    const float* o = obs + row * 80;
    unsigned short h[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        const int k = ch * 8 + e;
        const float v = k < KIN_ROUTE_DYN ? __ldg(o + route_unfold_col(k)) : (k == KIN_ROUTE_DYN ? 1.0f : 0.0f);
        h[e] = __bfloat16_as_ushort(__float2bfloat16_rn(v));
    }
    uint4 w;
    w.x = h[0] | ((unsigned)h[1] << 16); w.y = h[2] | ((unsigned)h[3] << 16); w.z = h[4] | ((unsigned)h[5] << 16); w.w = h[6] | ((unsigned)h[7] << 16);
    *reinterpret_cast<uint4*>(img + (row >> 7) * 16384 + r * 128 + ((ch ^ (r & 7)) << 4)) = w;
}

int kin_ppo_reduce_launch(const float* partials, int n_cta, int P, float* grad, float* stats, float inv_global_batch, cudaStream_t st) {
    kin_ppo_reduce_kernel<<<(P + 5 + 31) / 32, 256, 0, st>>>(partials, n_cta, P, grad, stats, inv_global_batch);
    return KIN_OK;
}

int kin_pop_reduce_launch(const KinPopMember* members, int n_members, int n_cta, int P, float inv_global_batch, cudaStream_t st) {
    kin_ppo_reduce_kernel<true><<<dim3((unsigned)((P + 5 + 31) / 32), (unsigned)n_members), 256, 0, st>>>(reinterpret_cast<const float*>(members), n_cta, P,
                                                                                                          nullptr, nullptr, inv_global_batch);
    return KIN_OK;
}

static ActW actor_w(const KinPolicyWeights* w) { return ActW{w->pi_w0, w->pi_b0, w->pi_w1, w->pi_b1, w->act_w, w->act_b}; }
static ActW critic_w(const KinPolicyWeights* w) { return ActW{w->vf_w0, w->vf_b0, w->vf_w1, w->vf_b1, w->val_w, w->val_b}; }

// ---- per-sample permutation of the rollout buffer (SB3's RolloutBuffer.get: np.random.permutation over ALL samples) -------------------
// The gradient kernels consume minibatches as unions of 64-sample tiles; to run them on SB3's per-sample minibatches the rollout is
// physically permuted: destination sample d = source sample perm[d] for the observation (a 128-byte row of a bf16 operand image, moved
// between the swizzle phases of the two rows, or `in_dim` fp32 values), the action, old log-prob, advantage and return; the per-tile
// advantage sums of the NEW order come out of the same pass.  One CTA per 128 destination samples; an image row is moved by 8 lanes
// (16 bytes each), so a warp reads 4 whole source rows and writes 512 contiguous bytes per instruction.
template <bool IMG>
__global__ void __launch_bounds__(128)
kin_ppo_shuffle_kernel(const unsigned char* __restrict__ obs, int in_dim, const float* __restrict__ action, const float* __restrict__ logp,
                       const float* __restrict__ adv, const float* __restrict__ ret, const int* __restrict__ perm, unsigned char* __restrict__ obs_out,
                       float* __restrict__ action_out, float* __restrict__ logp_out, float* __restrict__ adv_out, float* __restrict__ ret_out,
                       double* __restrict__ tile_sums_out) {
    __shared__ int src[128];
    __shared__ double wsum[4][2];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const size_t d0 = (size_t)blockIdx.x * 128;
    const int g = __ldg(perm + d0 + tid);
    src[tid] = g;
    const float a = __ldg(adv + g);
    logp_out[d0 + tid] = __ldg(logp + g);
    adv_out[d0 + tid] = a;
    ret_out[d0 + tid] = __ldg(ret + g);
    double s1 = (double)a, s2 = (double)a * (double)a;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        s1 += __shfl_xor_sync(0xffffffffu, s1, off);
        s2 += __shfl_xor_sync(0xffffffffu, s2, off);
    }
    if (lane == 0) { wsum[warp][0] = s1; wsum[warp][1] = s2; }
    __syncthreads();
    if (tid < 4) {      // tile t of this CTA = warps 2t, 2t + 1
        const int t = tid >> 1, q = tid & 1;
        tile_sums_out[(d0 / 64 + t) * 2 + q] = wsum[2 * t][q] + wsum[2 * t + 1][q];
    }
    for (int f = tid; f < 128 * 7; f += 128) {
        const int r = f / 7, c = f - r * 7;
        action_out[d0 * 7 + f] = __ldg(action + (size_t)src[r] * 7 + c);
    }
    if (IMG) {
        const int c = tid & 7;
#pragma unroll
        for (int pass = 0; pass < 8; ++pass) {
            const int r = pass * 16 + (tid >> 3);
            const int sg = src[r], sr = sg & 127;
            const uint4 v = __ldg(reinterpret_cast<const uint4*>(obs + (size_t)(sg >> 7) * 16384 + sr * 128 + ((c ^ (sr & 7)) << 4)));
            *reinterpret_cast<uint4*>(obs_out + (size_t)blockIdx.x * 16384 + r * 128 + ((c ^ (r & 7)) << 4)) = v;
        }
    } else {
        const float* o = reinterpret_cast<const float*>(obs);
        float* oo = reinterpret_cast<float*>(obs_out);
        for (int f = tid; f < 128 * in_dim; f += 128) {
            const int r = f / in_dim, c = f - r * in_dim;
            oo[d0 * in_dim + f] = __ldg(o + (size_t)src[r] * in_dim + c);
        }
    }
}

}  // namespace kin

using namespace kin;

extern "C" int kin_ppo_param_count(int in_dim) { return ppo_offsets(in_dim).total; }

extern "C" int kin_policy_act(const KinPolicyWeights* w, const float* obs, float* action, float* logp, float* value, int n, uint64_t seed,
                              uint32_t step, int deterministic, void* stream) {
    if (!w || !w->pi_w0 || !w->log_std || !obs || !action || !logp || n <= 0) return kin_fail(KIN_ERR_INVALID_ARG, "kin_policy_act: bad arguments");
    if (value && !(w->has_value && w->vf_w0)) return kin_fail(KIN_ERR_INVALID_ARG, "kin_policy_act: value requested but the policy has no critic");
    if (((uintptr_t)obs & 15u)) return kin_fail(KIN_ERR_INVALID_ARG, "kin_policy_act: obs must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    const int blocks = (n + 127) / 128;
    cudaError_t e;
    if (w->in_dim == 56) {
        const size_t smem = (size_t)(MlpSmem<56>::FLOATS + HID * 128) * sizeof(float);
        e = cudaFuncSetAttribute(kin_policy_act_kernel<56>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return kin_fail_cuda(e, "kin_policy_act: smem attribute");
        kin_policy_act_kernel<56><<<blocks, 128, smem, st>>>(actor_w(w), critic_w(w), w->log_std, obs, action, logp, value, n, seed, step, deterministic);
    } else if (w->in_dim == 80) {
        const size_t smem = (size_t)(MlpSmem<80>::FLOATS + HID * 128) * sizeof(float);
        e = cudaFuncSetAttribute(kin_policy_act_kernel<80>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return kin_fail_cuda(e, "kin_policy_act: smem attribute");
        kin_policy_act_kernel<80><<<blocks, 128, smem, st>>>(actor_w(w), critic_w(w), w->log_std, obs, action, logp, value, n, seed, step, deterministic);
    } else {
        return kin_fail(KIN_ERR_UNSUPPORTED, "kin_policy_act: in_dim must be 56 or 80");
    }
    e = cudaGetLastError();
    return e == cudaSuccess ? KIN_OK : kin_fail_cuda(e, "kin_policy_act");
}

extern "C" int kin_ppo_bootstrap(const KinPolicyWeights* w, const float* terminal_obs, const uint8_t* done, float* reward, float gamma, int n,
                                 void* stream) {
    if (!w || !w->vf_w0 || !terminal_obs || !done || !reward || n <= 0) return kin_fail(KIN_ERR_INVALID_ARG, "kin_ppo_bootstrap: bad arguments");
    if (w->in_dim != 56 && w->in_dim != 80) return kin_fail(KIN_ERR_UNSUPPORTED, "kin_ppo_bootstrap: in_dim must be 56 or 80");
    cudaError_t e;
    if (w->in_dim == 56) {
        const size_t smem = (size_t)(MlpSmem<56>::FLOATS + HID * 128) * sizeof(float);
        e = cudaFuncSetAttribute(kin_ppo_bootstrap_kernel<56>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return kin_fail_cuda(e, "kin_ppo_bootstrap: smem attribute");
        kin_ppo_bootstrap_kernel<56><<<(n + 127) / 128, 128, smem, (cudaStream_t)stream>>>(critic_w(w), terminal_obs, done, reward, gamma, n);
    } else {       // the 80-input route policy
        const size_t smem = (size_t)(MlpSmem<80>::FLOATS + HID * 128) * sizeof(float);
        e = cudaFuncSetAttribute(kin_ppo_bootstrap_kernel<80>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return kin_fail_cuda(e, "kin_ppo_bootstrap: smem attribute");
        kin_ppo_bootstrap_kernel<80><<<(n + 127) / 128, 128, smem, (cudaStream_t)stream>>>(critic_w(w), terminal_obs, done, reward, gamma, n);
    }
    e = cudaGetLastError();
    return e == cudaSuccess ? KIN_OK : kin_fail_cuda(e, "kin_ppo_bootstrap");
}

extern "C" int kin_ppo_gae(const float* reward, const float* value, const uint8_t* episode_start, const float* last_value, const uint8_t* last_done,
                           float gamma, float gae_lambda, int T, int n, float* advantage, float* returns, double* tile_sums, void* stream) {
    if (!reward || !value || !episode_start || !last_value || !last_done || !advantage || !returns || T <= 0 || n <= 0)
        return kin_fail(KIN_ERR_INVALID_ARG, "kin_ppo_gae: bad arguments");
    if (tile_sums && (((size_t)T * n) % TS) != 0) return kin_fail(KIN_ERR_INVALID_ARG, "kin_ppo_gae: T*n must be a multiple of 64 for tile sums");
    cudaStream_t st = (cudaStream_t)stream;
    kin_ppo_gae_kernel<<<(n + 255) / 256, 256, 0, st>>>(reward, value, episode_start, last_value, last_done, gamma, gae_lambda, T, n, advantage, returns);
    if (tile_sums) kin_ppo_tile_sums_kernel<<<(unsigned)(((size_t)T * n) / TS), TS, 0, st>>>(advantage, tile_sums);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KIN_OK : kin_fail_cuda(e, "kin_ppo_gae");
}

extern "C" int kin_ppo_grad(const float* params, int in_dim, const KinPpoHyper* hp, const float* obs, const float* action, const float* old_logp,
                            const float* advantage, const float* returns, const double* tile_sums, const int* tile_ids, int n_tiles,
                            long long global_batch, float* partials, int grid, float* grad, float* stats, const float* adv_stats, void* stream) {
    if (!params || !hp || !obs || !action || !old_logp || !advantage || !returns || (!tile_sums && !adv_stats) || !tile_ids || !partials || n_tiles <= 0 ||
        grid <= 0 || global_batch <= 0)
        return kin_fail(KIN_ERR_INVALID_ARG, "kin_ppo_grad: bad arguments");
    if (in_dim != 56) return kin_fail(KIN_ERR_UNSUPPORTED, "kin_ppo_grad: in_dim must be 56 (the route policy's 80-input update is not built yet)");
    const int P = ppo_offsets(in_dim).total;
    const size_t smem = (size_t)GradSmem<56>::FLOATS * sizeof(float);
    cudaError_t e = cudaFuncSetAttribute(kin_ppo_grad_kernel<56>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return kin_fail_cuda(e, "kin_ppo_grad: smem attribute");
    cudaStream_t st = (cudaStream_t)stream;
    const int g = grid < n_tiles ? grid : n_tiles;
    const float inv = 1.0f / (float)global_batch;
    kin_ppo_grad_kernel<56><<<g, PPO_THREADS, smem, st>>>(params, *hp, obs, action, old_logp, advantage, returns, tile_sums, tile_ids, n_tiles, inv, partials, adv_stats);
    if (grad) kin_ppo_reduce_launch(partials, g, P, grad, stats, inv, st);      // grad == NULL: the caller reduces `partials` (kin_peer_grad_push)
    e = cudaGetLastError();
    return e == cudaSuccess ? KIN_OK : kin_fail_cuda(e, "kin_ppo_grad");
}

extern "C" int kin_ppo_adv_stats(const double* tile_sums, const int* tile_ids, int n_tiles_per_minibatch, int n_minibatches, int normalize,
                                 float* adv_stats, void* stream) {
    if (!tile_sums || !tile_ids || !adv_stats || n_tiles_per_minibatch <= 0 || n_minibatches <= 0)
        return kin_fail(KIN_ERR_INVALID_ARG, "kin_ppo_adv_stats: bad arguments");
    kin_ppo_adv_stats_kernel<<<n_minibatches, 256, 0, (cudaStream_t)stream>>>(tile_sums, tile_ids, n_tiles_per_minibatch, normalize, adv_stats);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KIN_OK : kin_fail_cuda(e, "kin_ppo_adv_stats");
}

extern "C" int kin_ppo_shuffle(const void* obs, int obs_is_image, int in_dim, const float* action, const float* old_logp, const float* advantage,
                               const float* returns, const int* perm, long long n_samples, void* obs_out, float* action_out, float* old_logp_out,
                               float* advantage_out, float* returns_out, double* tile_sums_out, void* stream) {
    if (!obs || !action || !old_logp || !advantage || !returns || !perm || !obs_out || !action_out || !old_logp_out || !advantage_out || !returns_out ||
        !tile_sums_out)
        return kin_fail(KIN_ERR_INVALID_ARG, "kin_ppo_shuffle: null argument");
    if (n_samples <= 0 || (n_samples & 127)) return kin_fail(KIN_ERR_INVALID_ARG, "kin_ppo_shuffle: n_samples must be a positive multiple of 128");
    if (!obs_is_image && in_dim != 56 && in_dim != 80) return kin_fail(KIN_ERR_UNSUPPORTED, "kin_ppo_shuffle: in_dim must be 56 or 80");
    if (obs == obs_out || action == action_out) return kin_fail(KIN_ERR_INVALID_ARG, "kin_ppo_shuffle: the permutation is not in place");
    if (obs_is_image && (((uintptr_t)obs | (uintptr_t)obs_out) & 15u)) return kin_fail(KIN_ERR_INVALID_ARG, "kin_ppo_shuffle: images must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned grid = (unsigned)(n_samples / 128);
    if (obs_is_image)
        kin_ppo_shuffle_kernel<true><<<grid, 128, 0, st>>>(static_cast<const unsigned char*>(obs), in_dim, action, old_logp, advantage, returns, perm,
                                                            static_cast<unsigned char*>(obs_out), action_out, old_logp_out, advantage_out, returns_out, tile_sums_out);
    else
        kin_ppo_shuffle_kernel<false><<<grid, 128, 0, st>>>(static_cast<const unsigned char*>(obs), in_dim, action, old_logp, advantage, returns, perm,
                                                             static_cast<unsigned char*>(obs_out), action_out, old_logp_out, advantage_out, returns_out, tile_sums_out);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KIN_OK : kin_fail_cuda(e, "kin_ppo_shuffle");
}

extern "C" int kin_ppo_pack_weights(const float* params, int in_dim, void* weight_image, void* stream) {
    if (!params || !weight_image) return kin_fail(KIN_ERR_INVALID_ARG, "kin_ppo_pack_weights: bad arguments");
    if (in_dim != 56 && in_dim != 80) return kin_fail(KIN_ERR_UNSUPPORTED, "kin_ppo_pack_weights: in_dim must be 56 or 80");
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(weight_image, 0, KIN_WIMG_BYTES, st);
    if (e != cudaSuccess) return kin_fail_cuda(e, "kin_ppo_pack_weights: memset");
    const int P = ppo_offsets(in_dim).total;
    kin_ppo_pack_weights_kernel<<<(P + 255) / 256, 256, 0, st>>>(params, in_dim, static_cast<unsigned short*>(weight_image));
    e = cudaGetLastError();
    return e == cudaSuccess ? KIN_OK : kin_fail_cuda(e, "kin_ppo_pack_weights");
}

extern "C" int kin_route_obs_images(const float* obs, long long n_rows, void* images, void* stream) {
    if (!obs || !images || n_rows <= 0 || (n_rows % 128) != 0) return kin_fail(KIN_ERR_INVALID_ARG, "kin_route_obs_images: n_rows must be a positive multiple of 128");
    if (((uintptr_t)images & 15u)) return kin_fail(KIN_ERR_INVALID_ARG, "kin_route_obs_images: images must be 16-byte aligned");
    const long long chunks = n_rows * 8;
    kin_route_obs_images_kernel<<<(unsigned)((chunks + 255) / 256), 256, 0, (cudaStream_t)stream>>>(obs, n_rows, static_cast<unsigned char*>(images));
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KIN_OK : kin_fail_cuda(e, "kin_route_obs_images");
}

extern "C" int kin_ppo_adam(float* params, const float* grad, float* adam_m, float* adam_v, int n_params, const KinPpoHyper* hp, int step,
                            float* stats, float* stats_accum, void* weight_image, int in_dim, void* stream) {
    if (weight_image && in_dim != 56)
        return kin_fail(KIN_ERR_UNSUPPORTED, "kin_ppo_adam: only the 56-input image is kept current in place; the folded route image is rebuilt with kin_ppo_pack_weights");
    if (!params || !grad || !adam_m || !adam_v || !hp || n_params <= 0 || step < 1) return kin_fail(KIN_ERR_INVALID_ARG, "kin_ppo_adam: bad arguments");
    const float2 bc = adam_bias_corrections(*hp, step);
    kin_ppo_adam_kernel<<<(n_params + 1023) / 1024, 1024, 0, (cudaStream_t)stream>>>(params, grad, adam_m, adam_v, n_params, *hp, bc.x, bc.y, stats, stats_accum,
                                                              static_cast<unsigned short*>(weight_image), in_dim);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KIN_OK : kin_fail_cuda(e, "kin_ppo_adam");
}

static bool pop_args_ok(const KinPopMember* members, int n_members) { return members && n_members > 0 && n_members <= KIN_POP_MAX; }

extern "C" int kin_pop_gae(const KinPopMember* members, int n_members, int n_envs, int n_steps, void* stream) {
    if (!pop_args_ok(members, n_members) || n_envs <= 0 || n_steps <= 0) return kin_fail(KIN_ERR_INVALID_ARG, "kin_pop_gae: bad arguments");
    if ((((size_t)n_steps * n_envs) % TS) != 0) return kin_fail(KIN_ERR_INVALID_ARG, "kin_pop_gae: n_steps * n_envs must be a multiple of 64 for tile sums");
    cudaStream_t st = (cudaStream_t)stream;
    kin_ppo_gae_kernel<true><<<dim3((unsigned)((n_envs + 255) / 256), (unsigned)n_members), 256, 0, st>>>(
        reinterpret_cast<const float*>(members), nullptr, nullptr, nullptr, nullptr, 0.0f, 0.0f, n_steps, n_envs, nullptr, nullptr);
    kin_ppo_tile_sums_kernel<true><<<dim3((unsigned)(((size_t)n_steps * n_envs) / TS), (unsigned)n_members), TS, 0, st>>>(
        reinterpret_cast<const float*>(members), nullptr);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KIN_OK : kin_fail_cuda(e, "kin_pop_gae");
}

extern "C" int kin_pop_adv_stats(const KinPopMember* members, int n_members, int n_tiles_per_minibatch, int n_minibatches, void* stream) {
    if (!pop_args_ok(members, n_members) || n_tiles_per_minibatch <= 0 || n_minibatches <= 0) return kin_fail(KIN_ERR_INVALID_ARG, "kin_pop_adv_stats: bad arguments");
    kin_ppo_adv_stats_kernel<true><<<dim3((unsigned)n_minibatches, (unsigned)n_members), 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const double*>(members), nullptr, n_tiles_per_minibatch, 0, nullptr);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KIN_OK : kin_fail_cuda(e, "kin_pop_adv_stats");
}

extern "C" int kin_pop_adam(const KinPopMember* members, int n_members, const KinPpoHyper* host_hypers, const int* host_steps, void* stream) {
    if (!pop_args_ok(members, n_members) || !host_hypers || !host_steps) return kin_fail(KIN_ERR_INVALID_ARG, "kin_pop_adam: bad arguments");
    PopBiasCorrection B{};
    for (int k = 0; k < n_members; ++k) {
        if (host_steps[k] < 1) return kin_fail(KIN_ERR_INVALID_ARG, "kin_pop_adam: steps count optimiser steps from 1");
        const float2 bc = adam_bias_corrections(host_hypers[k], host_steps[k]);
        B.bc[k][0] = bc.x;
        B.bc[k][1] = bc.y;
    }
    const int P = ppo_offsets(56).total;
    kin_ppo_adam_kernel<true><<<dim3((unsigned)((P + 1023) / 1024), (unsigned)n_members), 1024, 0, (cudaStream_t)stream>>>(
        nullptr, reinterpret_cast<const float*>(members), nullptr, nullptr, P, KinPpoHyper{}, 0.0f, 0.0f, nullptr, nullptr, nullptr, 56, B);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KIN_OK : kin_fail_cuda(e, "kin_pop_adam");
}

extern "C" int kin_pop_route_obs_images(const KinPopMember* members, const KinPopRouteMember* route_members, int n_members, long long n_rows, void* stream) {
    if (!pop_args_ok(members, n_members) || !route_members || n_rows <= 0 || (n_rows % 128) != 0)
        return kin_fail(KIN_ERR_INVALID_ARG, "kin_pop_route_obs_images: bad arguments (n_rows must be a positive multiple of 128)");
    const long long chunks = n_rows * 8;
    kin_route_obs_images_kernel<true><<<dim3((unsigned)((chunks + 255) / 256), (unsigned)n_members), 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const float*>(route_members), n_rows, reinterpret_cast<unsigned char*>(const_cast<KinPopMember*>(members)));
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KIN_OK : kin_fail_cuda(e, "kin_pop_route_obs_images");
}

extern "C" int kin_pop_route_adam(const KinPopMember* members, int n_members, const KinPpoHyper* host_hypers, const int* host_steps, void* stream) {
    if (!pop_args_ok(members, n_members) || !host_hypers || !host_steps) return kin_fail(KIN_ERR_INVALID_ARG, "kin_pop_route_adam: bad arguments");
    PopBiasCorrection B{};
    for (int k = 0; k < n_members; ++k) {
        if (host_steps[k] < 1) return kin_fail(KIN_ERR_INVALID_ARG, "kin_pop_route_adam: steps count optimiser steps from 1");
        const float2 bc = adam_bias_corrections(host_hypers[k], host_steps[k]);
        B.bc[k][0] = bc.x;
        B.bc[k][1] = bc.y;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int P = ppo_offsets(80).total;
    kin_ppo_adam_kernel<true, false><<<dim3((unsigned)((P + 1023) / 1024), (unsigned)n_members), 1024, 0, st>>>(
        nullptr, reinterpret_cast<const float*>(members), nullptr, nullptr, P, KinPpoHyper{}, 0.0f, 0.0f, nullptr, nullptr, nullptr, 80, B);
    kin_ppo_pack_weights_kernel<true><<<dim3((unsigned)((P + 255) / 256), (unsigned)n_members), 256, 0, st>>>(reinterpret_cast<const float*>(members), 80, nullptr);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KIN_OK : kin_fail_cuda(e, "kin_pop_route_adam");
}
