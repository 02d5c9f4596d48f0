// kin_ppo_tc.cu -- K3-TC: the PPO minibatch gradient with EVERY GEMM on the 5th-generation tensor cores
// (tcgen05.mma kind::f16, bf16 operands, fp32 accumulation in TMEM).
//
// Same contract as kin_ppo_grad (kin_ppo.cu; SB3 2.8.0 ppo.py train()), different arithmetic engine:
//   * the actor and the critic are independent networks with independent parameter gradients, so each CTA works on ONE
//     of them (blockIdx.y): 256 threads, threads r and r + 128 <-> sample row r of a 128-sample GEMM tile <-> TMEM lane r (each
//     owns 32 of the row's 64 accumulator columns, halving every epilogue on the per-tile dependency chain).  A CTA needs
//     112 KB of shared memory and 256 TMEM columns, so an actor CTA and a critic CTA (or two of a kind) share every SM and
//     one's epilogue arithmetic overlaps the other's GEMMs and barrier round trips.
//   * every operand lives in shared memory as a [rows][64 bf16] SWIZZLE_128B tile (kin_umma.cuh).  The tiles written for
//     the forward pass (X, H1, H2 as K-major A operands with M = sample) are re-read UNCHANGED as MN-major operands
//     (K = sample) by the weight-gradient GEMMs  dW = G^T H, so nothing is ever transposed; W1 is likewise read K-major by
//     the forward pass and MN-major by the data-gradient GEMM  dH1 = G2 W1.
//   * GEMMs per 128-sample tile and net (M x N x K):
//       forward   Z  = X W0^T      128 x 64 x 64   (bias b0 rides on the constant-one column 56 of X)
//                 Z  = H1 W1^T     128 x 64 x 64
//                 O  = H2 WO^T     128 x 16 x 64   (actor: cols 0-6 action means; critic: col 7 value)
//       backward  Z  = dO WO       128 x 64 x 16   + dWO += H2^T dO          (H2's last readers: G2 then replaces H2 in place)
//                 Z  = G2 W1       128 x 64 x 64   + dW1|db1 += G2^T [H1 | dO(ones col)]   64 x 80 x 128: ONE GEMM, the B operand
//                                                    spans the adjacent H1 and dO tiles     (G1 then replaces H1 in place)
//       weights   dW0|db0 += G1^T X                  M = 64, K = 128 samples
//     The weight-gradient accumulators (and the bias gradients b0 / b1, which fall out of the constant-one columns) stay in TMEM
//     across all tiles of the CTA: 224 of 256 columns = Z/O 64 | dWO 16 | dW1 64 + db1 16 | dW0 64; the last 32 columns hold the bf16
//     A operand of the next chain GEMM (H1, H2, G2: written by the epilogue threads with tcgen05.st, read by TS-mode MMAs -- the kernel
//     is bound by the shared-memory data pipe, and this removes a quarter of the tensor core's operand fetch).  The output-bias gradient is
//     a per-thread fp32 sum of dO, reduced once per CTA.
//   * a dedicated ninth warp issues the MMAs from warp-uniform control flow (one elected lane executes the tcgen05 instructions,
//     descriptors stay in uniform registers); the 256 epilogue threads never issue and never block on a CTA-wide barrier: they
//     `bar.arrive` on a named barrier when an operand tile is written and go on to wait for the next accumulator, the issuer
//     `bar.sync`s on it.  Issuing from `if (tid == 0)` inside an epilogue warp cost ~70 cycles per MMA (R2UR round trips in a
//     divergent branch) on the critical path of every tile -- 4 000 of 11 000 cycles per tile (tools/ppo_trace.py).
//   * completion is tracked with mbarriers: `main` (the forward/backward chain GEMM the epilogue threads wait for), `ride` (the
//     weight-gradient GEMMs that ride behind a chain GEMM and read a tile the next epilogue overwrites in place: the epilogue
//     does its arithmetic first and waits for `ride` only before its stores), `wg` (the trailing dW0 batch, which must drain
//     before the X buffer it reads is refilled) and the X image buffers.
//   * image mode (the rollout buffer kin_ppo_collect wrote): the X operand is one 16 KB bulk copy (TMA engine) per tile,
//     double-buffered so the next tile's image lands while this one is processed.  The loss inputs of the tile (actions,
//     advantages, old log-probs / returns) ride on the same mbarrier into small shared-memory buffers, so the epilogue threads
//     hold no global loads in flight (their registers and latency were on the per-tile chain before).
//   * the elementwise work (tanh, 1 - h^2, the loss and its derivative, log_std gradient, statistics) is fp32 in registers;
//     each thread keeps packed bf16 copies of its H1 / H2 rows in registers for the backward pass.
//
// Numerics: bf16 operands (8-bit mantissa) + fp32 accumulation + tanh.approx -> gradients agree with fp32 autograd to ~1e-2
// relative per tensor (tests/test_gpu_ppo.py::test_minibatch_gradient_tc_*); log-probs move by O(1e-3), so a trainer whose
// rollout sampled with the fp32 policy refreshes old_logp with THIS kernel's forward (forward_only); the fused collection
// (kin_collect.cu) samples with the same bf16 arithmetic, so there the first-epoch ratio is 1 by construction.
#include "kin_peer.cuh"
#include "kin_ppo_layout.cuh"
#include "kin_umma.cuh"

namespace kin {

using namespace umma;

constexpr int TCG_EPI_THREADS = 256;   // 128 sample rows x 2 column halves (32 accumulator columns per thread and epilogue)
constexpr int TCG_THREADS = TCG_EPI_THREADS + 32;   // + the MMA issuer warp
constexpr int TCG_ISSUER_WARP = TCG_EPI_THREADS / 32;
constexpr int TCG_ROWS = 128;
constexpr int TILE_BYTES = TCG_ROWS * 128;        // [128][64 bf16]

// TMEM column map (fp32 columns)
constexpr unsigned COL_Z = 0;         // 64 (layer 3's O aliases columns 0..15)
constexpr unsigned COL_WO = 64;       // 16
constexpr unsigned COL_W1 = 80;       // 64 + 16: the N = 80 GEMM's columns 64..79 come from the dO tile, column 64 + 8 = db1
constexpr unsigned COL_W0 = 160;      // 64 (column 56 = db0)
constexpr unsigned COL_A = 224;       // 32: the A operand of the next chain GEMM (H1, then H2, then G2: bf16 pairs, 8 columns per K = 16 step)
constexpr unsigned TMEM_COLS_G = 256;
// Chain GEMMs whose A operand the epilogue threads have just produced (layer 2: H1, layer 3: H2, Z = G2 W1: G2) take it from tensor
// memory: the kernel is bound by the shared-memory data pipe (tensor-core operand fetch 37 % + epilogue LDS / STS 30 % of its peak,
// profiles/r2_ppo_tc3_raw.csv), and an SS-mode N = 64 MMA fetches 4 KB of A + 2 KB of B per 32 cycles of math.  The tiles are still
// stored to shared memory -- the weight-gradient GEMMs read them MN-major -- so this removes 48 of ~196 KB of operand fetch per tile.
#ifndef KIN_PPO_A_TMEM
#define KIN_PPO_A_TMEM 1
#endif

#ifdef KIN_PPO_TRACE
// phase profiler (debug builds only, tools/ppo_trace.py): cycles per phase of the per-tile chain, summed over the tiles of a CTA,
// for thread 256 (the MMA issuer warp) and thread 32 (an epilogue thread) of CTAs (0, 0) and (1, 1)
__device__ unsigned long long kin_ppo_trace_buf[4][16];
#define TRACE_DECL unsigned long long tr_acc[13] = {}; long long tr_t = clock64(); const bool tr_on = (tid == TCG_EPI_THREADS || tid == 32) && blockIdx.x == blockIdx.y && blockIdx.x < 2;
#define TRACE_MARK(i) do { if (tr_on) { const long long t_ = clock64(); tr_acc[i] += (unsigned long long)(t_ - tr_t); tr_t = t_; } } while (0)
#define TRACE_FLUSH(ntiles) do { if (tr_on) { unsigned long long* o_ = kin_ppo_trace_buf[blockIdx.x * 2 + (tid == 32)]; for (int i_ = 0; i_ < 13; ++i_) o_[i_] = tr_acc[i_]; o_[15] = (unsigned long long)(ntiles); } } while (0)
#else
#define TRACE_DECL
#define TRACE_MARK(i)
#define TRACE_FLUSH(n)
#endif

// Layer 1 always runs K = 64 on ONE operand tile: the 56-input policies as [obs56 | 1 | 0..], the 80-input route policy constant-folded
// to its 60 live columns ([live60 | 1 | 0 0 0], kin_ppo_layout.cuh) -- so both take the same image path, two CTAs per SM.
template <int KT>
struct __align__(1024) TcGradSmem {
    unsigned char X[2][TILE_BYTES];      // double-buffered in image mode (the next tile's image is prefetched by the TMA engine)
    unsigned char H2[TILE_BYTES];        // H2, later G2 = dL/dZ2
    unsigned char H1[TILE_BYTES];        // H1, later G1 = dL/dZ1
    unsigned char DO[TILE_BYTES];        // cols 0..7 dL/d(mean, value), col 8 = 1, rest 0.  MUST follow H1: [H1 | DO] is one MN-major operand
    unsigned char W0[KT][64 * 128];      // col IN = b0
    unsigned char W1[64 * 128];
    unsigned char WO[16 * 128];          // actor: rows 0..6 = act_w; critic: row 7 = val_w
    float act[2][TCG_ROWS * 7];         // loss inputs of the tile, staged by the TMA engine next to the X image (double-buffered)
    float adv[2][TCG_ROWS];
    float olp[2][TCG_ROWS];
    float ret[2][TCG_ROWS];
    float b1[64];
    float bo[8];
    float ls[8];
    float inv_sig[8];
    float scal[32];                      // 0 adv mean, 1 1/(std+eps), 2..5 statistics, 8..14 d log_std, 16..23 d output bias
    float red[4][20];                    // per-warp partial sums of the loss-side reductions (folded in a fixed order: deterministic)
    unsigned long long mbar[6];          // 0 main (chain GEMMs), 1 wg (trailing dW0 batch), 2/3 staged inputs (X image + loss inputs), 4 weights, 5 ride
    unsigned tmem_base;
};

// named barrier 1: the epilogue threads arrive when an operand tile (or a TMEM read) is complete, the issuer warp waits for it
__device__ __forceinline__ void ready_arrive() { bar_arrive(1, TCG_THREADS); }
__device__ __forceinline__ void ready_sync() { bar_sync(1, TCG_THREADS); }

// this thread's 32 accumulator columns [32 * half, 32 * half + 32) of its row -> f -> packed bf16 in p[16].
// MODE 0: tanh; 1: tanh(x + b1); 2: x * (1 - h^2), h = keep[] (the packed copy of the same columns from the forward pass)
template <int MODE>
__device__ __forceinline__ void epilogue_math(unsigned tz, int half, const float* bias, unsigned* keep, unsigned* p) {
    float v[32];
    tmem_ld32(tz + half * 32, v);
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        float a = v[2 * i], b = v[2 * i + 1];
        if (MODE == 0) {
            p[i] = pack_bf16(tanh_fast(a), tanh_fast(b));
        } else if (MODE == 1) {
            p[i] = pack_bf16(tanh_fast(a + bias[half * 32 + 2 * i]), tanh_fast(b + bias[half * 32 + 2 * i + 1]));
        } else {
            const unsigned h = keep[i];
            const float hl = bf16_lo(h), hh = bf16_hi(h);
            p[i] = pack_bf16(a * fmaf(-hl, hl, 1.0f), b * fmaf(-hh, hh, 1.0f));
        }
        if (MODE != 2) keep[i] = p[i];
    }
}
__device__ __forceinline__ void epilogue_store(unsigned char* tile, int row, int half, const unsigned* p) {
#pragma unroll
    for (int j = 0; j < 4; ++j)
        *reinterpret_cast<uint4*>(tile + sw_chunk(row, half * 4 + j)) = make_uint4(p[4 * j], p[4 * j + 1], p[4 * j + 2], p[4 * j + 3]);
}

// IMG: obs is the rollout buffer of bf16 operand images written by kin_ppo_collect (one 16 KB image per 128 consecutive samples)
// PEER: the kernel ends with the in-kernel gradient exchange over NVLink peer memory (kin_peer.cuh::peer_exchange_tail): grid barrier,
// per-CTA column slices reduced over the partial rows and pushed to every rank, rank-ordered sum into px.grad -- no separate push /
// gather launches between this kernel and Adam.
// POP (population launch, kin_pop_grad_tc): params carries the KinPopMember table and the one extra argument is the minibatch index;
// member blockIdx.z's descriptor supplies every per-run pointer and hyper-parameter, its tile ids and advantage statistics are those of
// that minibatch.  blockIdx.y stays the net and blockIdx.x the member's CTA, so the tile loop, the partial rows and their reduction
// order are the standalone launch's.  The standalone instances have no extra argument: their parameter lists are unchanged.
template <bool IMG, int IN, bool PEER = false, bool POP = false, class... PopArgs>
__global__ void __launch_bounds__(TCG_THREADS, 2)
kin_ppo_grad_tc_kernel(const float* __restrict__ params, KinPpoHyper hp, const float* __restrict__ obs, const float* __restrict__ action,
                       const float* __restrict__ old_logp, const float* __restrict__ advantage, const float* __restrict__ returns,
                       const double* __restrict__ tile_sums, const int* __restrict__ tile_ids, int n_pairs, float inv_global_batch,
                       float* __restrict__ partials, float* __restrict__ logp_out, float* __restrict__ value_out, int forward_only, int net_base,
                       const float* __restrict__ adv_stats, const unsigned char* __restrict__ wimg, const PeerFused px, PopArgs... pop) {
    static_assert(IN == 56 || (IN == 80 && IMG), "56-input policies (fp32 observations or images) or the 80-input route policy (folded images)");
    static_assert(sizeof...(PopArgs) == (POP ? 1 : 0) && (!POP || (IMG && IN == 56 && !PEER)), "population: 56-input images, one extra argument");
    if constexpr (POP) {
        const int minibatch = (pop, ...);
        const KinPopMember& M = reinterpret_cast<const KinPopMember*>(params)[blockIdx.z];
        params = M.params;
        hp = M.hyper;
        obs = static_cast<const float*>(M.obs_tiles);
        action = M.action;
        old_logp = M.logp;
        advantage = M.advantage;
        returns = M.returns;
        tile_sums = M.tile_sums;
        tile_ids = M.tile_ids + (size_t)minibatch * 2 * n_pairs;
        partials = M.partials;
        adv_stats = M.adv_stats + 2 * minibatch;
        wimg = static_cast<const unsigned char*>(M.weight_image);
    }
    constexpr int KT = 1;                            // K tiles of layer 1
    constexpr int K1 = 64;                           // padded reduction width of layer 1 (live inputs | 1 | zeros)
    constexpr bool FOLD = IN == 80;                  // route policy: layer 1 sees its 60 live columns, the constants are folded into the bias
    constexpr int INE = FOLD ? KIN_ROUTE_DYN : IN;   // live columns of the X tile; column INE carries the bias
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    // round up to 1024 bytes WITHOUT leaving the shared address space (pointer + offset, not an integer round trip), so every
    // access below compiles to LDS / STS rather than generic LD / ST with 64-bit address arithmetic
    TcGradSmem<KT>& S = *reinterpret_cast<TcGradSmem<KT>*>(smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u));
    const PpoOffsets O = ppo_offsets(IN);
    const int P = O.total;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int row = tid & 127, half = (tid >> 7) & 1;    // two threads per sample row: columns 0..31 / 32..63 of every activation
    const bool issuer = warp == TCG_ISSUER_WARP;         // warp-uniform
    const int net = net_base + (int)blockIdx.y;    // 0 actor, 1 critic
    const int o_w0 = net ? O.vf_w0 : O.pi_w0, o_b0 = net ? O.vf_b0 : O.pi_b0, o_w1 = net ? O.vf_w1 : O.pi_w1, o_b1 = net ? O.vf_b1 : O.pi_b1;

    // ---- prologue: this net's weights -> bf16 operand tiles -------------------------------------------------------------
    {
        uint4* z = reinterpret_cast<uint4*>(S.DO);
        for (int i = tid; i < TILE_BYTES / 16; i += TCG_THREADS) z[i] = make_uint4(0u, 0u, 0u, 0u);
        if (!wimg && tid < 16 * 128 / 16) reinterpret_cast<uint4*>(S.WO)[tid] = make_uint4(0u, 0u, 0u, 0u);   // the image carries its own zero rows
    }
    if (!wimg) {       // no prebuilt operand image: convert this net's weights here (latency-bound; the trainer passes the image)
        for (int i = tid; i < 64 * KT * 64; i += TCG_THREADS) {
            const int u = i / (KT * 64), k = i - u * (KT * 64);
            float v = 0.0f;
            if (k < INE) v = __ldg(params + o_w0 + u * IN + (FOLD ? route_unfold_col(k) : k));
            else if (k == INE) {    // summed left to right, as kin_ppo_pack_weights does: both weight paths round the same fp32 bias
                v = __ldg(params + o_b0 + u);
                if (FOLD) v = (v + __ldg(params + o_w0 + u * IN + KIN_ROUTE_ONE_A)) + __ldg(params + o_w0 + u * IN + KIN_ROUTE_ONE_B);
            }
            st_bf16(S.W0[k >> 6], u, k & 63, v);
        }
        for (int i = tid; i < 64 * 64; i += TCG_THREADS) st_bf16(S.W1, i >> 6, i & 63, __ldg(params + o_w1 + i));
    }
    __syncthreads();   // WO / DO zero fill is complete before the real rows go in
    if (!wimg) {
        if (net == 0) {
            for (int i = tid; i < 7 * 64; i += TCG_THREADS) st_bf16(S.WO, i >> 6, i & 63, __ldg(params + O.act_w + i));
        } else if (tid < 64) {
            st_bf16(S.WO, 7, tid, __ldg(params + O.val_w + tid));
        }
    }
    if (tid < 64) S.b1[tid] = __ldg(params + o_b1 + tid);
    if (tid < 128) *reinterpret_cast<uint4*>(S.DO + sw_chunk(tid, 1)) = make_uint4(0x00003F80u, 0u, 0u, 0u);   // col 8 = 1.0 (bf16)
    if (tid < 8) {
        const float ls = tid < 7 ? __ldg(params + O.log_std + tid) : 0.0f;
        S.bo[tid] = tid < 7 ? __ldg(params + O.act_b + tid) : __ldg(params + O.val_b);
        S.ls[tid] = ls;
        S.inv_sig[tid] = expf(-ls);
    }
    if (tid < 32) S.scal[tid] = 0.0f;
    __syncwarp();
    if (adv_stats) {
        if (tid == 0) { S.scal[0] = adv_stats[0]; S.scal[1] = adv_stats[1]; }
    } else if (tid < 32 && !forward_only && net == 0) {
        double s1 = 0.0, s2 = 0.0;
        for (int j = tid; j < 2 * n_pairs; j += 32) {
            const int t = tile_ids[j];
            s1 += tile_sums[2 * t];
            s2 += tile_sums[2 * t + 1];
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            s1 += __shfl_xor_sync(0xffffffffu, s1, off);
            s2 += __shfl_xor_sync(0xffffffffu, s2, off);
        }
        if (tid == 0) {
            const double nsamp = (double)n_pairs * TCG_ROWS;
            const double mean = s1 / nsamp;
            const double var = nsamp > 1.0 ? fmax((s2 - nsamp * mean * mean) / (nsamp - 1.0), 0.0) : 0.0;
            S.scal[0] = hp.normalize_advantage ? (float)mean : 0.0f;
            S.scal[1] = hp.normalize_advantage ? (float)(1.0 / (sqrt(var) + 1e-8)) : 1.0f;
        }
    }
    if (warp == 0) tmem_alloc(smem_u32(&S.tmem_base), TMEM_COLS_G);
    if (tid == 0) {
#pragma unroll
        for (int i = 0; i < 6; ++i) mbar_init(smem_u32(&S.mbar[i]), 1);
        fence_mbar_init();
        if (wimg) {    // this net's W0 | W1 | WO blocks of the prebuilt image: three bulk copies (TMA engine) on one mbarrier
            const unsigned mbw = smem_u32(&S.mbar[4]);
            mbar_expect_tx(mbw, 8192 + 8192 + 2048);
            bulk_load(smem_u32(S.W0[0]), wimg + KIN_WIMG_W0 + net * 8192, 8192, mbw);
            bulk_load(smem_u32(S.W1), wimg + KIN_WIMG_W1 + net * 8192, 8192, mbw);
            bulk_load(smem_u32(S.WO), wimg + KIN_WIMG_WO + net * 2048, 2048, mbw);
        }
    }
    fence_async_smem();
    fence_before();
    __syncthreads();
    fence_after();
    if (wimg) mbar_wait(smem_u32(&S.mbar[4]), 0u);

    const unsigned tb = S.tmem_base;
    const unsigned tlane = tb + ((unsigned)((warp & 3) * 32) << 16);     // this warp's lane quadrant, column 0
    const unsigned tz = tlane + COL_Z;
    const unsigned mb_main = smem_u32(&S.mbar[0]), mb_wg = smem_u32(&S.mbar[1]), mb_ride = smem_u32(&S.mbar[5]);
    const unsigned char* img = reinterpret_cast<const unsigned char*>(obs);
    int it = 0;
    TRACE_DECL

    if (issuer) {
        // ================= MMA issuer warp: warp-uniform control flow, one elected lane executes the tcgen05 / TMA instructions =========
        const bool lead = elect_one();
        const unsigned aX0 = smem_u32(S.X[0]), aH1 = smem_u32(S.H1), aH2 = smem_u32(S.H2), aDO = smem_u32(S.DO);
        const unsigned aW0 = smem_u32(S.W0[0]), aW1 = smem_u32(S.W1), aWO = smem_u32(S.WO);
        const unsigned mb_x0 = smem_u32(&S.mbar[2]);
        constexpr unsigned id_fwd = idesc_bf16(128, 64, false, false), id_out = idesc_bf16(128, 16, false, false);
        constexpr unsigned id_bwd = idesc_bf16(128, 64, false, true);
        constexpr unsigned id_w16 = idesc_bf16(64, 16, true, true), id_w0 = idesc_bf16(64, K1, true, true), id_w80 = idesc_bf16(64, 80, true, true);
        // staged inputs of one tile -> buffer b: the X image (image mode) and the loss inputs of its two 64-sample halves, all on mb_x[b]
        const unsigned loss_bytes = net == 0 ? 2u * 1792u + (forward_only ? 0u : 4u * 256u) : (forward_only ? 0u : 2u * 256u);
        const unsigned stage_bytes = (IMG ? (unsigned)TILE_BYTES : 0u) + loss_bytes;
        const unsigned aAct = smem_u32(S.act[0]), aAdv = smem_u32(S.adv[0]), aOlp = smem_u32(S.olp[0]), aRet = smem_u32(S.ret[0]);
        auto stage = [&](int jj, int b) {       // called by the elected lane only
            const int t0 = __ldg(tile_ids + 2 * jj), t1 = __ldg(tile_ids + 2 * jj + 1);
            const unsigned mb = mb_x0 + 8 * b;
            mbar_expect_tx(mb, stage_bytes);
            if (IMG) bulk_load(aX0 + b * TILE_BYTES, img + (size_t)(t0 >> 1) * TILE_BYTES, TILE_BYTES, mb);
            if (net == 0) {
                bulk_load(aAct + b * 3584, action + (size_t)t0 * 448, 1792u, mb);
                bulk_load(aAct + b * 3584 + 1792, action + (size_t)t1 * 448, 1792u, mb);
                if (!forward_only) {
                    bulk_load(aAdv + b * 512, advantage + (size_t)t0 * 64, 256u, mb);
                    bulk_load(aAdv + b * 512 + 256, advantage + (size_t)t1 * 64, 256u, mb);
                    bulk_load(aOlp + b * 512, old_logp + (size_t)t0 * 64, 256u, mb);
                    bulk_load(aOlp + b * 512 + 256, old_logp + (size_t)t1 * 64, 256u, mb);
                }
            } else if (!forward_only) {
                bulk_load(aRet + b * 512, returns + (size_t)t0 * 64, 256u, mb);
                bulk_load(aRet + b * 512 + 256, returns + (size_t)t1 * 64, 256u, mb);
            }
        };
        if (stage_bytes && lead && (int)blockIdx.x < n_pairs) stage(blockIdx.x, 0);
        for (int j = blockIdx.x; j < n_pairs; j += gridDim.x, ++it) {
            TRACE_MARK(12);
            const int lb = it & 1, xb = IMG ? lb : 0;
            const unsigned aX = aX0 + xb * TILE_BYTES;
            const int jn = j + gridDim.x;
            if (IMG) {
                mbar_wait(mb_x0 + 8 * lb, (unsigned)(it >> 1) & 1u);                // this tile's image has landed
                if (forward_only && it > 0) ready_sync();                           // the previous tile's outputs have left TMEM
            } else {
                ready_sync();                                                       // the threads have written X (after reading O)
            }
            TRACE_MARK(0);
            fence_after();
            if (lead) {
#pragma unroll
                for (int k = 0; k < K1 / 16; ++k)      // K tile k / 4 of X and W0, 32 bytes (16 bf16) per step inside it
                    mma_bf16(tb + COL_Z, desc_k(aX + (k >> 2) * TILE_BYTES + (k & 3) * 32), desc_k(aW0 + (k >> 2) * 8192 + (k & 3) * 32), id_fwd, k > 0);
                commit(mb_main);
            }
            TRACE_MARK(1);
            if (stage_bytes && jn < n_pairs) {
                // the other buffer's last readers were the previous tile's trailing dW0 batch (gradient pass, image mode) / its layer 1
                // (forward only) / its loss threads (all done: they arrived on `ready` since): refill it with the next tile's inputs
                if (IMG && !forward_only && it > 0) mbar_wait(mb_wg, (unsigned)(it - 1) & 1u);
                if (lead) stage(jn, lb ^ 1);
            }
            TRACE_MARK(2);
            // ---- layer 2 -------------------------------------------------------------------------------------------------
            ready_sync();                       // H1 written
            TRACE_MARK(3);
            fence_after();
            if (lead) {
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    if (KIN_PPO_A_TMEM) mma_bf16_ts(tb + COL_Z, tb + COL_A + 8 * k, desc_k(aW1 + k * 32), id_fwd, k > 0);
                    else mma_bf16(tb + COL_Z, desc_k(aH1 + k * 32), desc_k(aW1 + k * 32), id_fwd, k > 0);
                }
                commit(mb_main);
            }
            // ---- layer 3: action means (cols 0..6) or value (col 7) ----------------------------------------------------------
            ready_sync();                       // H2 written
            TRACE_MARK(4);
            fence_after();
            if (lead) {
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    if (KIN_PPO_A_TMEM) mma_bf16_ts(tb + COL_Z, tb + COL_A + 8 * k, desc_k(aWO + k * 32), id_out, k > 0);
                    else mma_bf16(tb + COL_Z, desc_k(aH2 + k * 32), desc_k(aWO + k * 32), id_out, k > 0);
                }
                commit(mb_main);
            }
            if (forward_only) continue;
            const unsigned acc0 = it > 0;
            // ---- Z = dO WO; dWO += H2^T dO rides behind it (H2's last reader) ----------------------------------------------------
            ready_sync();                       // dO written
            TRACE_MARK(5);
            fence_after();
            if (lead) {
                mma_bf16(tb + COL_Z, desc_k(aDO), desc_mn(aWO), id_bwd, 0u);
                commit(mb_main);
#pragma unroll
                for (int k = 0; k < 8; ++k) mma_bf16(tb + COL_WO, desc_mn(aH2 + k * 2048), desc_mn(aDO + k * 2048), id_w16, acc0 | (k > 0));
                commit(mb_ride);
            }
            // ---- Z = G2 W1; dW1|db1 += G2^T [H1 | dO] rides behind it (H1's last reader) ------------------------------------------
            ready_sync();                       // G2 written (over H2)
            TRACE_MARK(6);
            fence_after();
            if (lead) {
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    if (KIN_PPO_A_TMEM) mma_bf16_ts(tb + COL_Z, tb + COL_A + 8 * k, desc_mn(aW1 + k * 2048), id_bwd, k > 0);
                    else mma_bf16(tb + COL_Z, desc_k(aH2 + k * 32), desc_mn(aW1 + k * 2048), id_bwd, k > 0);
                }
                commit(mb_main);
#pragma unroll
                for (int k = 0; k < 8; ++k) mma_bf16(tb + COL_W1, desc_mn(aH2 + k * 2048), desc_mn(aH1 + k * 2048), id_w80, acc0 | (k > 0));
                commit(mb_ride);
            }
            // ---- dW0|db0 += G1^T X: must drain before this X buffer is refilled ----------------------------------------------------
            ready_sync();                       // G1 written (over H1)
            TRACE_MARK(7);
            fence_after();
            if (lead) {
#pragma unroll
                for (int k = 0; k < 8; ++k)            // N = K1: the MN-major B operand spans the adjacent X K tiles
                    mma_bf16(tb + COL_W0, desc_mn(aH1 + k * 2048), desc_mn(aX + k * 2048), id_w0, acc0 | (k > 0));
                commit(mb_wg);
            }
            TRACE_MARK(8);
        }
        if (IMG && forward_only && it > 0) ready_sync();      // pairs with the last tile's output arrive
    } else {
        // ================= epilogue threads ==============================================================================================
        unsigned par_main = 0u;
        unsigned h1p[16] = {}, h2p[16] = {};
        float dls[7] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, dbo[7] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, st[4] = {0.f, 0.f, 0.f, 0.f};
        for (int j = blockIdx.x; j < n_pairs; j += gridDim.x, ++it) {
            TRACE_MARK(12);
            const int lb = it & 1;
            int t0 = 0, t1 = 0;
            if (!IMG || logp_out || value_out) { t0 = __ldg(tile_ids + 2 * j); t1 = __ldg(tile_ids + 2 * j + 1); }
            const size_t g = (size_t)(row < 64 ? t0 : t1) * 64 + (row & 63);      // only used by the X conversion / the forward outputs
            if constexpr (!IMG) {
                // ---- X tile: obs fp32 -> bf16, coalesced float4 reads; column 56 = 1 carries the layer-1 bias ---------------
                if (it > 0 && !forward_only) mbar_wait(mb_wg, (unsigned)(it - 1) & 1u);    // the previous tile's dW0 batch still reads X
                constexpr int Q = IN / 4;                                    // float4 per observation row
#pragma unroll
                for (int i = 0; i < IN / 8; ++i) {
                    const int idx = tid + TCG_EPI_THREADS * i;           // 0 .. 2 * 64 * Q - 1
                    const int hh = idx >= 64 * Q, rem = idx - hh * 64 * Q;
                    const int r = hh * 64 + rem / Q, c4 = (rem % Q) * 4;    // row, first of its four columns
                    const float4 v = __ldg(reinterpret_cast<const float4*>(obs + (size_t)(hh ? t1 : t0) * 64 * IN) + rem);
                    *reinterpret_cast<uint2*>(S.X[c4 >> 6] + sw_chunk(r, (c4 & 63) >> 3) + (c4 & 4) * 2) = make_uint2(pack_bf16(v.x, v.y), pack_bf16(v.z, v.w));
                }
                if (tid < 128) {      // column IN = 1 (carries the bias), zero up to K1
                    *reinterpret_cast<uint4*>(S.X[0] + sw_chunk(tid, IN >> 3)) = make_uint4(0x00003F80u, 0u, 0u, 0u);
                }
                fence_async_smem();
                fence_before();
                ready_arrive();
            }
            TRACE_MARK(0);
            unsigned p[16];
            // ---- layer 1 -------------------------------------------------------------------------------------------------
            mbar_wait(mb_main, par_main);
            par_main ^= 1u;
            fence_after();
            TRACE_MARK(1);
            epilogue_math<0>(tz, half, nullptr, h1p, p);
            epilogue_store(S.H1, row, half, p);
            if (KIN_PPO_A_TMEM) tmem_st16(tlane + COL_A + half * 16, p);
            fence_async_smem();
            fence_before();
            ready_arrive();
            TRACE_MARK(2);
            // ---- layer 2 -------------------------------------------------------------------------------------------------
            mbar_wait(mb_main, par_main);
            par_main ^= 1u;
            fence_after();
            TRACE_MARK(3);
            epilogue_math<1>(tz, half, S.b1, h2p, p);
            epilogue_store(S.H2, row, half, p);
            if (KIN_PPO_A_TMEM) tmem_st16(tlane + COL_A + half * 16, p);
            fence_async_smem();
            fence_before();
            ready_arrive();
            TRACE_MARK(4);
            // ---- layer 3 -> loss and d(loss)/d(outputs), one thread per sample -------------------------------------------------
            mbar_wait(mb_main, par_main);
            par_main ^= 1u;
            fence_after();
            TRACE_MARK(5);
            if (half == 0) {
                float o[16];
                tmem_ld16(tlane + COL_Z, o);
                if (net == 0 || !forward_only) mbar_wait(smem_u32(&S.mbar[2 + lb]), (unsigned)(it >> 1) & 1u);     // staged loss inputs (landed long ago)
                if (net == 0) {
                    const float* act_r = S.act[lb] + row * 7;
                    const float adv_r = S.adv[lb][row], olp_r = S.olp[lb][row];
                    float lp = 0.0f, z[7];
#pragma unroll
                    for (int d = 0; d < 7; ++d) {
                        z[d] = (act_r[d] - (o[d] + S.bo[d])) * S.inv_sig[d];
                        lp += -0.5f * z[d] * z[d] - S.ls[d] - kHalfLog2Pi;
                    }
                    if (logp_out) logp_out[g] = lp;
                    if (!forward_only) {
                        const float adv_n = (adv_r - S.scal[0]) * S.scal[1];
                        const float log_ratio = lp - olp_r;
                        const float ratio = expf(log_ratio);
                        const float pl1 = adv_n * ratio, pl2 = adv_n * fminf(fmaxf(ratio, 1.0f - hp.clip_range), 1.0f + hp.clip_range);
                        const float dpl_dlp = (pl1 <= pl2) ? -adv_n * ratio : 0.0f;
                        float dm[7];
                        float ent = 0.0f;
#pragma unroll
                        for (int d = 0; d < 7; ++d) {
                            dm[d] = inv_global_batch * dpl_dlp * z[d] * S.inv_sig[d];
                            dbo[d] += dm[d];
                            dls[d] += inv_global_batch * dpl_dlp * (z[d] * z[d] - 1.0f) - inv_global_batch * hp.ent_coef;
                            ent += 0.5f + kHalfLog2Pi + S.ls[d];
                        }
                        *reinterpret_cast<uint4*>(S.DO + sw_chunk(row, 0)) =
                            make_uint4(pack_bf16(dm[0], dm[1]), pack_bf16(dm[2], dm[3]), pack_bf16(dm[4], dm[5]), pack_bf16(dm[6], 0.0f));
                        st[0] += -fminf(pl1, pl2);
                        st[1] += ent;
                        st[2] += (ratio - 1.0f) - log_ratio;
                        st[3] += fabsf(ratio - 1.0f) > hp.clip_range ? 1.0f : 0.0f;
                    }
                } else {
                    const float v = o[7] + S.bo[7];
                    if (value_out) value_out[g] = v;
                    if (!forward_only) {
                        const float ret_r = S.ret[lb][row];
                        const float dv = inv_global_batch * hp.vf_coef * 2.0f * (v - ret_r);
                        dbo[0] += dv;
                        *reinterpret_cast<uint4*>(S.DO + sw_chunk(row, 0)) = make_uint4(0u, 0u, 0u, pack_bf16(0.0f, dv));
                        st[0] += (ret_r - v) * (ret_r - v);
                    }
                }
            }
            if (forward_only) {
                if (IMG) {           // Z / O is re-written by the next tile's layer 1 only after everyone has read it
                    fence_before();
                    ready_arrive();
                }
                continue;
            }
            fence_async_smem();
            fence_before();
            ready_arrive();
            TRACE_MARK(6);
            // ---- dZ2 = (dO WO) * (1 - H2^2): G2 replaces H2 once dWO += H2^T dO has read it ---------------------------------------
            mbar_wait(mb_main, par_main);
            par_main ^= 1u;
            fence_after();
            TRACE_MARK(7);
            epilogue_math<2>(tz, half, nullptr, h2p, p);
            if (KIN_PPO_A_TMEM) tmem_st16(tlane + COL_A + half * 16, p);      // (layer 3, the last reader of these columns, has completed)
            mbar_wait(mb_ride, 0u);
            TRACE_MARK(8);
            epilogue_store(S.H2, row, half, p);
            fence_async_smem();
            fence_before();
            ready_arrive();
            // ---- dZ1 = (G2 W1) * (1 - H1^2): G1 replaces H1 once dW1|db1 += G2^T [H1 | dO] has read it ---------------------------
            mbar_wait(mb_main, par_main);
            par_main ^= 1u;
            fence_after();
            TRACE_MARK(9);
            epilogue_math<2>(tz, half, nullptr, h1p, p);
            mbar_wait(mb_ride, 1u);
            TRACE_MARK(10);
            epilogue_store(S.H1, row, half, p);
            fence_async_smem();
            fence_before();
            ready_arrive();
            TRACE_MARK(11);
        }
        if (!forward_only) {
            // log_std / output-bias gradients and statistics: warp shuffle, then one partial row per warp
#pragma unroll
            for (int d = 0; d < 7; ++d) {
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) {
                    dls[d] += __shfl_xor_sync(0xffffffffu, dls[d], off);
                    dbo[d] += __shfl_xor_sync(0xffffffffu, dbo[d], off);
                }
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) {
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) st[q] += __shfl_xor_sync(0xffffffffu, st[q], off);
            }
            if (lane == 0 && half == 0) {       // warps 0..3 own the loss threads
                float* r = S.red[warp];
#pragma unroll
                for (int q = 0; q < 4; ++q) r[q] = st[q];
#pragma unroll
                for (int d = 0; d < 7; ++d) {
                    r[4 + d] = dls[d];
                    r[11 + d] = dbo[d];
                }
            }
        }
    }

    TRACE_FLUSH(it);
    if (!forward_only) {
        if (it > 0) mbar_wait(mb_wg, (unsigned)(it - 1) & 1u);
        fence_after();
        __syncthreads();
        if (tid < 18) {      // statistics -> scal[2..5], d log_std -> scal[8..14], d output bias -> scal[16..22]
            const float a = ((S.red[0][tid] + S.red[1][tid]) + S.red[2][tid]) + S.red[3][tid];
            S.scal[tid < 4 ? 2 + tid : (tid < 11 ? 8 + tid - 4 : 16 + tid - 11)] = a;
        }
        __syncthreads();
        // ---- accumulators (M = 64: row m lives in lane m % 16 + 32 * (m / 16)) -> this CTA's slice of the partial gradient ----------
        float* out = partials + (size_t)blockIdx.x * (P + KIN_PPO_STATS + 8);
        const int u = (warp & 3) * 16 + lane;       // valid for lane < 16
        const bool rowok = lane < 16;
        if (!issuer) {   // warps 0..3 store columns 0..31 of dW1 / dW0, warps 4..7 columns 32..63
            float v[32];
            tmem_ld32(tlane + COL_W1 + half * 32, v);
            if (rowok) {
#pragma unroll
                for (int c = 0; c < 32; ++c) out[o_w1 + u * 64 + half * 32 + c] = v[c];   // flat offsets are not 16-byte aligned
            }
#pragma unroll
            for (int cb = half; cb < K1 / 32; cb += 2) {      // 32-column blocks of dW0 | db0: this half's, plus block 2 for K1 = 96
                tmem_ld32(tlane + COL_W0 + cb * 32, v);
                if (rowok) {
#pragma unroll
                    for (int c = 0; c < 32; ++c) {
                        const int k = cb * 32 + c;
                        if (k < INE) {
                            out[o_w0 + u * IN + (FOLD ? route_unfold_col(k) : k)] = v[c];
                        } else if (k == INE) {
                            out[o_b0 + u] = v[c];
                            if (FOLD) {       // the inputs of these two columns are the constant 1: their gradient is the bias gradient
                                out[o_w0 + u * IN + KIN_ROUTE_ONE_A] = v[c];
                                out[o_w0 + u * IN + KIN_ROUTE_ONE_B] = v[c];
#pragma unroll
                                for (int z = 0; z < IN; ++z)      // ... and the constant-zero inputs give zero gradient
                                    if (route_fold_col(z) < 0 && z != KIN_ROUTE_ONE_A && z != KIN_ROUTE_ONE_B) out[o_w0 + u * IN + z] = 0.0f;
                            }
                        }
                    }
                }
            }
        }
        if (half == 0 && !issuer) {
            float o[16];
            tmem_ld16(tlane + COL_WO, o);
            if (rowok) {
                if (net == 0) {
#pragma unroll
                    for (int d = 0; d < 7; ++d) out[O.act_w + d * 64 + u] = o[d];
                } else {
                    out[O.val_w + u] = o[7];
                }
            }
            tmem_ld16(tlane + COL_W1 + 64, o);
            if (rowok) out[o_b1 + u] = o[8];
        }
        if (net == 0) {
            if (tid < 7) {
                out[O.log_std + tid] = S.scal[8 + tid];
                out[O.act_b + tid] = S.scal[16 + tid];
            }
            // statistics slots: 0 policy loss, 2 entropy, 3 approx_kl, 4 clip fraction (actor CTAs); 1 value loss (critic CTAs)
            if (tid == 0) { out[P + 0] = S.scal[2]; out[P + 2] = S.scal[3]; out[P + 3] = S.scal[4]; out[P + 4] = S.scal[5]; }
        } else if (tid == 0) {
            out[P + 1] = S.scal[2];
            out[O.val_b] = S.scal[16];
        }
        if constexpr (PEER) {       // every tile buffer is dead by now: the exchange borrows the X tile for its 1 KB of scratch
            float(*part)[32] = reinterpret_cast<float(*)[32]>(S.X[0]);
            peer_exchange_tail(px, partials, (int)gridDim.x, P, inv_global_batch, part, reinterpret_cast<int*>(S.X[0] + 2048));
            if (px.adam.params) peer_adam_tail(px, hp, P, reinterpret_cast<float*>(S.X[0] + 4096));      // clip + Adam on this CTA's slice
        }
    }
    fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tb, TMEM_COLS_G);
}

}  // namespace kin

using namespace kin;

#ifdef KIN_PPO_TRACE
extern "C" int kin_debug_peer_trace(unsigned long long* out) {      // 2 x 12 counters of the fused tail, see PT_DECL (this TU's copy: the
    return cudaMemcpyFromSymbol(out, kin_peer_trace_buf, sizeof(kin_peer_trace_buf)) == cudaSuccess ? KIN_OK : KIN_ERR_INVALID_ARG;   // two-chain kernel's)
}
extern "C" int kin_debug_peer_wait(unsigned long long* out) {       // [512][2]: barrier-1 wait cycles (summed over launches), SM id
    return cudaMemcpyFromSymbol(out, kin_peer_trace_wait, sizeof(kin_peer_trace_wait)) == cudaSuccess ? KIN_OK : KIN_ERR_INVALID_ARG;
}
extern "C" int kin_debug_ppo_trace(unsigned long long* out) {      // 4 x 16 counters, see TRACE_DECL
    return cudaMemcpyFromSymbol(out, kin_ppo_trace_buf, sizeof(kin_ppo_trace_buf)) == cudaSuccess ? KIN_OK : KIN_ERR_INVALID_ARG;
}
#endif

static int grad_tc_launch(const float* params, int in_dim, const KinPpoHyper* hp, const void* obs_any, const float* action, const float* old_logp,
                          const float* advantage, const float* returns, const double* tile_sums, const int* tile_ids, int n_tiles,
                          long long global_batch, float* partials, int grid, float* grad, float* stats, float* logp_out, float* value_out,
                          int forward_only, int obs_is_image, const float* adv_stats, const void* weight_image, const PeerFused& px, void* stream) {
    const float* obs = static_cast<const float*>(obs_any);
    if (!params || !hp || !obs || !action || !tile_ids || n_tiles <= 0 || grid <= 0)
        return kin_fail(KIN_ERR_INVALID_ARG, "kin_ppo_grad_tc: bad arguments");
    if (!forward_only && (!old_logp || !advantage || !returns || (!tile_sums && !adv_stats) || !partials || global_batch <= 0))
        return kin_fail(KIN_ERR_INVALID_ARG, "kin_ppo_grad_tc: the gradient pass needs old_logp, advantage, returns, tile_sums, partials and grad");
    if (forward_only && !logp_out && !value_out) return kin_fail(KIN_ERR_INVALID_ARG, "kin_ppo_grad_tc: forward_only without an output");
    if (in_dim != 56 && in_dim != 80) return kin_fail(KIN_ERR_UNSUPPORTED, "kin_ppo_grad_tc: in_dim must be 56 or 80");
    if (in_dim == 80 && !obs_is_image)
        return kin_fail(KIN_ERR_UNSUPPORTED, "kin_ppo_grad_tc: the 80-input route policy takes folded bf16 observation images (kin_route_obs_images)");
    if (n_tiles & 1) return kin_fail(KIN_ERR_INVALID_ARG, "kin_ppo_grad_tc: n_tiles must be even (two 64-sample tiles per 128-row GEMM tile)");
    if (((uintptr_t)obs & 15u)) return kin_fail(KIN_ERR_INVALID_ARG, "kin_ppo_grad_tc: obs must be 16-byte aligned");
    if (((uintptr_t)action | (uintptr_t)old_logp | (uintptr_t)advantage | (uintptr_t)returns) & 15u)      // staged by the TMA engine
        return kin_fail(KIN_ERR_INVALID_ARG, "kin_ppo_grad_tc: action / old_logp / advantage / returns must be 16-byte aligned");
    const int P = ppo_offsets(in_dim).total;
    const size_t smem = sizeof(TcGradSmem<1>) + 1024;
    static bool attr_set[KIN_MAX_DEVICES] = {};
    const int dev_slot = kin_device_slot();
    if (!attr_set[dev_slot]) {
        cudaError_t e = cudaFuncSetAttribute(kin_ppo_grad_tc_kernel<false, 56>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(TcGradSmem<1>) + 1024));
        if (e == cudaSuccess) e = cudaFuncSetAttribute(kin_ppo_grad_tc_kernel<true, 56>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(TcGradSmem<1>) + 1024));
        if (e == cudaSuccess) e = cudaFuncSetAttribute(kin_ppo_grad_tc_kernel<true, 80>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(TcGradSmem<1>) + 1024));
        if (e == cudaSuccess) e = cudaFuncSetAttribute(kin_ppo_grad_tc_kernel<false, 56, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(TcGradSmem<1>) + 1024));
        if (e == cudaSuccess) e = cudaFuncSetAttribute(kin_ppo_grad_tc_kernel<true, 56, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(TcGradSmem<1>) + 1024));
        if (e == cudaSuccess) e = cudaFuncSetAttribute(kin_ppo_grad_tc_kernel<true, 80, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(TcGradSmem<1>) + 1024));
        if (e != cudaSuccess) return kin_fail_cuda(e, "kin_ppo_grad_tc: smem attribute");
        attr_set[dev_slot] = true;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int n_pairs = n_tiles / 2;
    const int g = grid < n_pairs ? grid : n_pairs;
    const float inv = forward_only ? 0.0f : 1.0f / (float)global_batch;
    // forward-only: only the nets whose output is wanted run (log-prob -> actor CTAs, value -> critic CTAs)
    int net_base = 0;
    dim3 dg((unsigned)g, 2u);
    if (forward_only && !(logp_out && value_out)) {
        dg.y = 1u;
        net_base = logp_out ? 0 : 1;
    }
    const unsigned char* wimg = static_cast<const unsigned char*>(weight_image);
    const bool fused = px.world > 0 && !forward_only;
    if (fused && (int)(dg.x * dg.y) > PEER_MAX_CTA) return kin_fail(KIN_ERR_INVALID_ARG, "kin_ppo_grad_tc_exchange: at most 512 CTAs");
    // 56-input policies on operand images, full-size minibatches: the three-streams-per-SM kernel (kin_ppo_tc3.cu)
    int rc3 = KIN_OK;
    const bool tc3_done = !forward_only && obs_is_image && in_dim == 56 &&
                          kin_ppo_grad_tc3_try(params, hp, obs_any, action, old_logp, advantage, returns, tile_sums, tile_ids, n_pairs, inv, partials, grid,
                                               adv_stats, weight_image, px, fused, st, &rc3);
    if (tc3_done && rc3 != KIN_OK) return rc3;
#define KIN_GRAD_TC_LAUNCH(IMG, IN, PEER)                                                                                                        \
    kin_ppo_grad_tc_kernel<IMG, IN, PEER><<<dg, TCG_THREADS, smem, st>>>(params, *hp, obs, action, old_logp, advantage, returns, tile_sums, tile_ids, n_pairs, \
                                                                         inv, partials, logp_out, value_out, forward_only, net_base, adv_stats, wimg, px)
    if (tc3_done) {
    } else if (fused) {
        if (in_dim == 80) KIN_GRAD_TC_LAUNCH(true, 80, true);
        else if (obs_is_image) KIN_GRAD_TC_LAUNCH(true, 56, true);
        else KIN_GRAD_TC_LAUNCH(false, 56, true);
    } else {
        if (in_dim == 80) KIN_GRAD_TC_LAUNCH(true, 80, false);
        else if (obs_is_image) KIN_GRAD_TC_LAUNCH(true, 56, false);
        else KIN_GRAD_TC_LAUNCH(false, 56, false);
    }
#undef KIN_GRAD_TC_LAUNCH
    if (!forward_only && grad && !fused) kin_ppo_reduce_launch(partials, g, P, grad, stats, inv, st);      // grad == NULL: the caller reduces `partials` (kin_peer_grad_push)
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KIN_OK : kin_fail_cuda(e, "kin_ppo_grad_tc");
}

extern "C" int kin_ppo_grad_tc(const float* params, int in_dim, const KinPpoHyper* hp, const void* obs_any, const float* action, const float* old_logp,
                               const float* advantage, const float* returns, const double* tile_sums, const int* tile_ids, int n_tiles,
                               long long global_batch, float* partials, int grid, float* grad, float* stats, float* logp_out, float* value_out,
                               int forward_only, int obs_is_image, const float* adv_stats, const void* weight_image, void* stream) {
    PeerFused none{};
    return grad_tc_launch(params, in_dim, hp, obs_any, action, old_logp, advantage, returns, tile_sums, tile_ids, n_tiles, global_batch, partials, grid, grad,
                          stats, logp_out, value_out, forward_only, obs_is_image, adv_stats, weight_image, none, stream);
}

extern "C" int kin_ppo_grad_tc_exchange(const float* params, int in_dim, const KinPpoHyper* hp, const void* obs_any, const float* action, const float* old_logp,
                                        const float* advantage, const float* returns, const double* tile_sums, const int* tile_ids, int n_tiles,
                                        long long global_batch, float* partials, int grid, float* grad, float* stats, int obs_is_image,
                                        const float* adv_stats, const void* weight_image, void* const* peer_buffers, int rank, int world, unsigned epoch,
                                        int* timed_out, void* stream) {
    if (!peer_buffers || !grad || !timed_out || world < 1 || world > PEER_MAX || rank < 0 || rank >= world || epoch == 0u)
        return kin_fail(KIN_ERR_INVALID_ARG, "kin_ppo_grad_tc_exchange: bad exchange arguments (epoch counts exchanges from 1)");
    PeerFused px{};
    for (int i = 0; i < world; ++i) {
        if (!peer_buffers[i]) return kin_fail(KIN_ERR_INVALID_ARG, "kin_ppo_grad_tc_exchange: null peer buffer");
        px.peers.base[i] = static_cast<unsigned char*>(peer_buffers[i]);
    }
    px.rank = rank;
    px.world = world;
    px.epoch = epoch;
    px.grad = grad;
    px.stats = stats;
    px.timed_out = timed_out;
    px.timeout_cycles = kin_peer_timeout_cycles();
    return grad_tc_launch(params, in_dim, hp, obs_any, action, old_logp, advantage, returns, tile_sums, tile_ids, n_tiles, global_batch, partials, grid, grad,
                          stats, nullptr, nullptr, 0, obs_is_image, adv_stats, weight_image, px, stream);
}

// gradient + exchange + clip + Adam in ONE launch (peer_adam_tail): the optimiser step of kin_ppo_adam runs in the kernel's tail on the
// slice of the summed gradient each CTA owns
extern "C" int kin_ppo_grad_tc_update(const float* params, int in_dim, const KinPpoHyper* hp, const void* obs_any, const float* action, const float* old_logp,
                                      const float* advantage, const float* returns, const double* tile_sums, const int* tile_ids, int n_tiles,
                                      long long global_batch, float* partials, int grid, float* grad, float* stats, int obs_is_image,
                                      const float* adv_stats, void* weight_image, void* const* peer_buffers, int rank, int world, unsigned epoch,
                                      int* timed_out, float* params_rw, float* adam_m, float* adam_v, int step, float* stats_accum, float* norm_scratch,
                                      void* stream) {
    if (!peer_buffers || !grad || !timed_out || world < 1 || world > PEER_MAX || rank < 0 || rank >= world || epoch == 0u)
        return kin_fail(KIN_ERR_INVALID_ARG, "kin_ppo_grad_tc_update: bad exchange arguments (epoch counts exchanges from 1)");
    if (!params_rw || params_rw != params || !adam_m || !adam_v || !norm_scratch || !stats || step < 1 || !hp)
        return kin_fail(KIN_ERR_INVALID_ARG, "kin_ppo_grad_tc_update: bad optimiser arguments (params_rw must be params; norm_scratch holds 2 * grid floats)");
    PeerFused px{};
    for (int i = 0; i < world; ++i) {
        if (!peer_buffers[i]) return kin_fail(KIN_ERR_INVALID_ARG, "kin_ppo_grad_tc_update: null peer buffer");
        px.peers.base[i] = static_cast<unsigned char*>(peer_buffers[i]);
    }
    px.rank = rank;
    px.world = world;
    px.epoch = epoch;
    px.grad = grad;
    px.stats = stats;
    px.timed_out = timed_out;
    px.timeout_cycles = kin_peer_timeout_cycles();
    px.adam.params = params_rw;
    px.adam.m = adam_m;
    px.adam.v = adam_v;
    px.adam.wimg = in_dim == 56 ? static_cast<unsigned short*>(weight_image) : nullptr;      // the folded route image is rebuilt by kin_ppo_pack_weights
    px.adam.stats_accum = stats_accum;
    px.adam.norm_part = norm_scratch;
    px.adam.bc1 = 1.0f - powf(hp->adam_beta1, (float)step);
    px.adam.bc2 = 1.0f - powf(hp->adam_beta2, (float)step);
    px.adam.in_dim = in_dim;
    return grad_tc_launch(params, in_dim, hp, obs_any, action, old_logp, advantage, returns, tile_sums, tile_ids, n_tiles, global_batch, partials, grid, grad,
                          stats, nullptr, nullptr, 0, obs_is_image, adv_stats, weight_image, px, stream);
}


extern "C" int kin_pop_grad_tc(const KinPopMember* members, int n_members, int minibatch, int n_tiles_per_minibatch, long long global_batch, int grid,
                               void* stream) {
    if (!members || n_members <= 0 || n_members > KIN_POP_MAX || minibatch < 0 || n_tiles_per_minibatch <= 0 || global_batch <= 0 || grid <= 0)
        return kin_fail(KIN_ERR_INVALID_ARG, "kin_pop_grad_tc: bad arguments");
    if (n_tiles_per_minibatch & 1) return kin_fail(KIN_ERR_INVALID_ARG, "kin_pop_grad_tc: n_tiles must be even (two 64-sample tiles per 128-row GEMM tile)");
    auto kernel = kin_ppo_grad_tc_kernel<true, 56, false, true, int>;
    const size_t smem = sizeof(TcGradSmem<1>) + 1024;
    static bool attr_set[KIN_MAX_DEVICES] = {};
    const int dev_slot = kin_device_slot();
    if (!attr_set[dev_slot]) {
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return kin_fail_cuda(e, "kin_pop_grad_tc: smem attribute");
        attr_set[dev_slot] = true;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int n_pairs = n_tiles_per_minibatch / 2;
    const int g = grid < n_pairs ? grid : n_pairs;      // kin_ppo_grad_tc's clamp: the same CTAs, tiles per CTA and partial rows per member
    const float inv = 1.0f / (float)global_batch;
    const PeerFused none{};
    kernel<<<dim3((unsigned)g, 2u, (unsigned)n_members), TCG_THREADS, smem, st>>>(reinterpret_cast<const float*>(members), KinPpoHyper{}, nullptr, nullptr,
                                                                                 nullptr, nullptr, nullptr, nullptr, nullptr, n_pairs, inv, nullptr, nullptr,
                                                                                 nullptr, 0, 0, nullptr, nullptr, none, minibatch);
    kin_pop_reduce_launch(members, n_members, g, ppo_offsets(56).total, inv, st);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KIN_OK : kin_fail_cuda(e, "kin_pop_grad_tc");
}
