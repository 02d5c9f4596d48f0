// kin_collect_policy.cuh -- the policy half of the fused PPO collection kernels K4 (kin_collect.cu, 56 inputs) and K4-route
// (kin_route_collect.cu, 80 inputs): bf16 weight staging, tile setup, the actor + critic forward on tcgen05 (kind::f16), the
// Gaussian action sample with its log-prob, and the TimeLimit bootstrap list.
//
// One env <-> one thread <-> one row of the A operand <-> one TMEM lane; a CTA holds TILES (1, 2 or 4) independent 128-env tiles
// on named barriers sharing one bf16 copy of the weights, so one tile's FP32 env arithmetic overlaps another's GEMMs.  Per step
// and tile:
//   X = [obs | 1 | 0]  bf16, KT SWIZZLE_128B K-major tiles (K = 64 per tile)
//   Z = X [W0a;W0c]^T            128 x 128 x 16 ceil((IN + 1) / 16) -> tanh -> H1 (actor half over operand tile 0, critic half
//                                                                       over operand tile 1)
//   Z = H1a W1a^T | H1c W1c^T    2 x (128 x 64 x 64) -> tanh(+b1) -> H2 in place
//   O = H2a WOa^T + H2c WOc^T    128 x 16 x 64    -> 7 action means + value
// With KT = 1 (K4) operand tile 1 holds only the critic's activations; with KT = 2 (K4-route) it is also X's second K tile.
#pragma once

#include "kin_ppo_layout.cuh"
#include "kin_state.cuh"
#include "kin_umma.cuh"

namespace kin {

constexpr int AC_ROWS = 128;                       // envs per tile == UMMA M == TMEM lanes
constexpr int AC_TILE_BYTES = AC_ROWS * 128;       // one [128][64 bf16] operand tile

// both nets as bf16 B operands, plus the fp32 vectors of the epilogues and the sampler
template <int KT>
struct AcWeights {
    unsigned char W0[KT][AC_TILE_BYTES];   // [k tile][128 rows: actor 0..63 | critic 64..127][64 cols]; column IN = b0
    unsigned char W1[2][64 * 128];
    unsigned char WO[2][16 * 128];         // [0] rows 0..6 = act_w, [1] row 7 = val_w
    float b1[128];
    float bo[8];
    float ls[8];
    float sig[8];
};

// The kernels' shared-memory structs provide XH[TILES][2][AC_TILE_BYTES] (the per-tile operand tiles), AcWeights<KT> w,
// mbar[TILES][NB] (NB = 2: separate layer-1 barrier, see policy_forward) and tmem_base.

// W0 | W1 | WO converted from the flat fp32 parameters (all NT threads of the CTA)
template <int IN, int KT, int NT>
__device__ __forceinline__ void convert_weights(AcWeights<KT>& W, const float* __restrict__ params, int tid) {
    static_assert(16 * ((IN + 1 + 15) / 16) <= 64 * KT, "layer 1 needs ceil((IN + 1) / 16) K steps of 16");
    using namespace umma;
    const PpoOffsets O = ppo_offsets(IN);
    {
        uint4* zw = reinterpret_cast<uint4*>(W.WO);
        for (int i = tid; i < 2 * 16 * 128 / 16; i += NT) zw[i] = make_uint4(0u, 0u, 0u, 0u);
    }
    for (int i = tid; i < KT * 128 * 64; i += NT) {
        const int kt = i >> 13, nn = (i >> 6) & 127, kc = i & 63, k = kt * 64 + kc, u = nn & 63;
        const int wbase = (nn < 64) ? O.pi_w0 : O.vf_w0, bbase = (nn < 64) ? O.pi_b0 : O.vf_b0;
        st_bf16(W.W0[kt], nn, kc, k < IN ? __ldg(params + wbase + u * IN + k) : (k == IN ? __ldg(params + bbase + u) : 0.0f));
    }
    for (int i = tid; i < 2 * 4096; i += NT) {
        const int nt = i >> 12, u = (i >> 6) & 63, k = i & 63;
        st_bf16(W.W1[nt], u, k, __ldg(params + (nt ? O.vf_w1 : O.pi_w1) + u * 64 + k));
    }
    __syncthreads();
    for (int i = tid; i < 7 * 64; i += NT) st_bf16(W.WO[0], i >> 6, i & 63, __ldg(params + O.act_w + i));
    if (tid < 64) st_bf16(W.WO[1], 7, tid, __ldg(params + O.val_w + tid));
}

// b1, output biases, log_std and sigma (fp32)
template <int IN, int KT>
__device__ __forceinline__ void load_vectors(AcWeights<KT>& W, const float* __restrict__ params, int tid) {
    const PpoOffsets O = ppo_offsets(IN);
    if (tid < 128) W.b1[tid] = __ldg(params + (tid < 64 ? O.pi_b1 + tid : O.vf_b1 + tid - 64));
    if (tid < 8) {
        const float ls = tid < 7 ? __ldg(params + O.log_std + tid) : 0.0f;
        W.bo[tid] = tid < 7 ? __ldg(params + O.act_b + tid) : __ldg(params + O.val_b);
        W.ls[tid] = ls;
        W.sig[tid] = expf(ls);
    }
}

// TMEM (128 columns per tile) and the per-tile mbarriers; ends on a CTA barrier after which the staged weights are visible to the
// tensor core.  With NB = 2, barrier [0] takes two arrivals: the layer-1 MMA commit and the X image store.
template <int TILES, int NB, class Smem>
__device__ __forceinline__ void init_tiles(Smem& S, int tid) {
    using namespace umma;
    if ((tid >> 5) == 0) tmem_alloc(smem_u32(&S.tmem_base), TILES * 128);
    if (tid < TILES) {
        mbar_init(smem_u32(&S.mbar[tid][0]), NB);
        if (NB == 2) mbar_init(smem_u32(&S.mbar[tid][1]), 1);
        fence_mbar_init();
    }
    fence_async_smem();
    fence_before();
    __syncthreads();
    fence_after();
}

template <int TILES, class Smem>
__device__ __forceinline__ void release_tiles(Smem& S, int tid) {
    umma::fence_before();
    __syncthreads();
    if ((tid >> 5) == 0) umma::tmem_dealloc(S.tmem_base, TILES * 128);
}

// this thread's view of its tile: operand tiles, weight, barrier and TMEM addresses, barrier phases
template <int KT>
struct AcTile {
    unsigned char *X0, *X1;
    unsigned aX0, aX1, aW0[KT], aW1a, aW1c, aWOa, aWOc, mb1, mb2, tz_mma, tz_row;
    unsigned par1, par2;
    int tile, row;
};

template <int KT, int NB, class Smem>
__device__ __forceinline__ AcTile<KT> tile_of(Smem& S, int tid) {
    using namespace umma;
    AcTile<KT> c;
    c.tile = tid >> 7;
    c.row = tid & 127;
    c.X0 = S.XH[c.tile][0];
    c.X1 = S.XH[c.tile][1];
    c.aX0 = smem_u32(c.X0);
    c.aX1 = smem_u32(c.X1);
#pragma unroll
    for (int kt = 0; kt < KT; ++kt) c.aW0[kt] = smem_u32(S.w.W0[kt]);
    c.aW1a = smem_u32(S.w.W1[0]);
    c.aW1c = smem_u32(S.w.W1[1]);
    c.aWOa = smem_u32(S.w.WO[0]);
    c.aWOc = smem_u32(S.w.WO[1]);
    c.mb1 = smem_u32(&S.mbar[c.tile][0]);
    c.mb2 = smem_u32(&S.mbar[c.tile][NB - 1]);
    c.tz_mma = S.tmem_base + c.tile * 128;
    c.tz_row = c.tz_mma + ((unsigned)(((tid >> 5) & 3) * 32) << 16);
    c.par1 = c.par2 = 0u;
    return c;
}

// 64 accumulator columns of this thread's lane -> tanh(. + b) -> bf16 -> its row of operand tiles X0 (columns 0..63: actor) and
// X1 (64..127: critic)
template <bool BIAS, int KT>
__device__ __forceinline__ void hidden_epilogue(const AcTile<KT>& c, const float* b1) {
    using namespace umma;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        float v[32];
        tmem_ld32(c.tz_row + q * 32, v);
        unsigned char* dst = (q < 2) ? c.X0 : c.X1;
        const float* b = b1 + q * 32;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            unsigned p[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                if (BIAS) p[e] = pack_bf16(tanh_fast(v[8 * j + 2 * e] + b[8 * j + 2 * e]), tanh_fast(v[8 * j + 2 * e + 1] + b[8 * j + 2 * e + 1]));
                else p[e] = pack_bf16(tanh_fast(v[8 * j + 2 * e]), tanh_fast(v[8 * j + 2 * e + 1]));
            }
            *reinterpret_cast<uint4*>(dst + sw_chunk(c.row, (q & 1) * 4 + j)) = make_uint4(p[0], p[1], p[2], p[3]);
        }
    }
}

// Actor + critic forward of the tile's 128 observations (IN floats each); collective over the tile's 128 threads.
// out[0..6] = action means, out[7] = value.
// STORE_X: the TMA engine also copies the X image (the tile's 16 KB operand, IN <= 63) to `img` when it is not null; layer 1 then
// waits on its own barrier for both the MMA commit and the copy having read the image, which the actor H1 overwrites next.
// Without STORE_X all three layers complete on one barrier.
template <int IN, bool STORE_X, int KT>
__device__ __forceinline__ void policy_forward(const AcWeights<KT>& W, AcTile<KT>& c, const float* o, unsigned char* img, float* out) {
    using namespace umma;
    constexpr int K1 = (IN + 1 + 15) / 16;     // layer-1 MMAs of K = 16
    static_assert(IN % 8 == 0 && 2 * K1 <= 8 * KT && (!STORE_X || KT == 1), "X image layout");
    // ---- X image: IN obs | 1 | zeros up to 16 K1 columns (16-byte chunk ch of the row lives in operand tile ch / 8)
#pragma unroll
    for (int ch = 0; ch < 2 * K1; ++ch) {
        unsigned char* t = ch < 8 ? c.X0 : c.X1;
        uint4 v = make_uint4(0u, 0u, 0u, 0u);
        if (ch < IN / 8)
            v = make_uint4(pack_bf16(o[8 * ch], o[8 * ch + 1]), pack_bf16(o[8 * ch + 2], o[8 * ch + 3]), pack_bf16(o[8 * ch + 4], o[8 * ch + 5]),
                           pack_bf16(o[8 * ch + 6], o[8 * ch + 7]));
        else if (ch == IN / 8)
            v.x = 0x00003F80u;      // column IN = 1 (bias carrier)
        *reinterpret_cast<uint4*>(t + sw_chunk(c.row, ch & 7)) = v;
    }
    fence_async_smem();
    fence_before();
    bar_sync(c.tile + 1, AC_ROWS);
    if (c.row < 32 && elect_one()) {      // one lane of the tile's first (converged) warp: uniform-register descriptors
        fence_after();
        constexpr unsigned id = idesc_bf16(128, 128, false, false);
#pragma unroll
        for (int k = 0; k < K1; ++k) mma_bf16(c.tz_mma, desc_k((k < 4 ? c.aX0 : c.aX1) + (k & 3) * 32), desc_k(c.aW0[k >> 2] + (k & 3) * 32), id, k > 0);
        commit(c.mb1);
        if constexpr (STORE_X) {
            if (img) {
                bulk_store(img, c.aX0, AC_TILE_BYTES);
                bulk_commit();
                bulk_wait_read();      // the actor H1 half overwrites the image next
            }
            mbar_arrive(c.mb1);
        }
    }
    mbar_wait(c.mb1, c.par1);
    c.par1 ^= 1u;
    fence_after();
    unsigned& par23 = STORE_X ? c.par2 : c.par1;
    // ---- H1 = tanh(Z): columns 0..63 actor -> X0's place, 64..127 critic -> X1's place
    hidden_epilogue<false>(c, W.b1);
    fence_async_smem();
    fence_before();
    bar_sync(c.tile + 1, AC_ROWS);
    if (c.row < 32 && elect_one()) {
        fence_after();
        constexpr unsigned id = idesc_bf16(128, 64, false, false);
#pragma unroll
        for (int k = 0; k < 4; ++k) mma_bf16(c.tz_mma, desc_k(c.aX0 + k * 32), desc_k(c.aW1a + k * 32), id, k > 0);
#pragma unroll
        for (int k = 0; k < 4; ++k) mma_bf16(c.tz_mma + 64, desc_k(c.aX1 + k * 32), desc_k(c.aW1c + k * 32), id, k > 0);
        commit(c.mb2);
    }
    mbar_wait(c.mb2, par23);
    par23 ^= 1u;
    fence_after();
    hidden_epilogue<true>(c, W.b1);
    fence_async_smem();
    fence_before();
    bar_sync(c.tile + 1, AC_ROWS);
    if (c.row < 32 && elect_one()) {
        fence_after();
        constexpr unsigned id = idesc_bf16(128, 16, false, false);
#pragma unroll
        for (int k = 0; k < 4; ++k) mma_bf16(c.tz_mma, desc_k(c.aX0 + k * 32), desc_k(c.aWOa + k * 32), id, k > 0);
#pragma unroll
        for (int k = 0; k < 4; ++k) mma_bf16(c.tz_mma, desc_k(c.aX1 + k * 32), desc_k(c.aWOc + k * 32), id, 1u);
        commit(c.mb2);
    }
    mbar_wait(c.mb2, par23);
    par23 ^= 1u;
    fence_after();
    float r[16];
    tmem_ld16(c.tz_row, r);
    fence_before();
#pragma unroll
    for (int d = 0; d < 8; ++d) out[d] = r[d] + W.bo[d];
}

// a = mean + sigma * eps (DiagGaussianDistribution; SB3 stores the unclipped sample) -> a[7] and action_out[7]; returns log N(a).
// The draws are kin_policy_act's.
template <int KT>
__device__ __forceinline__ float sample_action(const AcWeights<KT>& W, uint64_t seed, unsigned env, uint32_t step, const float* mean, float* a,
                                               float* action_out) {
    Philox rng(seed, env, step);
    float eps[8], lp = 0.0f;
#pragma unroll
    for (int k = 0; k < 8; k += 2) eps[k] = gauss_pair(rng, &eps[k + 1]);
#pragma unroll
    for (int k = 0; k < NJ; ++k) {
        a[k] = fmaf(W.sig[k], eps[k], mean[k]);
        lp += -0.5f * eps[k] * eps[k] - W.ls[k] - kHalfLog2Pi;
        action_out[k] = a[k];
    }
    return lp;
}

template <int N>
__device__ __forceinline__ void store_row(float* dst, const float* v) {
    float4* d4 = reinterpret_cast<float4*>(dst);
#pragma unroll
    for (int k = 0; k < N / 4; ++k) d4[k] = make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
}

// TimeLimit bootstrap list: a truncated (not terminated) episode appends (t * n + env, terminal observation); kin_ppo_bootstrap_list
// adds gamma * V(terminal_obs) to its reward afterwards.  observe(float[N]) writes the terminal observation.
template <int N, class Out, class Observe>
__device__ __forceinline__ void push_truncated(const Out& out, unsigned done, size_t idx, Observe observe) {
    if ((done & KIN_DONE_TRUNCATED) && !(done & KIN_DONE_TERMINATED)) {
        const int slot = atomicAdd(out.boot_count, 1);
        if (slot < out.boot_cap) {
            float o[N];
            observe(o);
            out.boot_index[slot] = (int)idx;
            store_row<N>(out.boot_obs + (size_t)slot * N, o);
        }
    }
}

// tiles per CTA: the requested count, or (requested <= 0) the fewest that still fit the batch in one wave of CTAs (one CTA per SM)
inline int collect_tiles_per_cta(int requested, int n_envs) {
    if (requested > 0) return requested;
    int sms = 148, dev = 0;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int n_tiles = n_envs / AC_ROWS;
    return n_tiles <= sms ? 1 : (n_tiles <= 2 * sms ? 2 : 4);
}

// one CTA of TILES * 128 threads per TILES tiles, with `smem` bytes of dynamic shared memory
template <int TILES, class... Params, class... Args>
cudaError_t launch_tiles(void (*kernel)(Params...), size_t smem, int n_envs, cudaStream_t st, Args&&... args) {
    const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    const int n_tiles = n_envs / AC_ROWS;
    kernel<<<(n_tiles + TILES - 1) / TILES, TILES * AC_ROWS, smem, st>>>(static_cast<Args&&>(args)...);
    return cudaGetLastError();
}

}  // namespace kin
