// kin_ppo_tc3.cu -- K3-TC, three tile streams per SM: the PPO minibatch gradient of kin_ppo_tc.cu re-cut so that THREE 128-sample
// tile chains are in flight on every SM instead of two.
//
// Why: the two-CTAs-per-SM kernel is latency-bound -- a tile is a chain of 5 GEMM round trips and 6 epilogues (~8 700 cycles) and an SM
// holds two chains (tensor pipe 27 %, XU 27 %, issue slots 34 % busy).  Shared memory is what caps the chains per SM (X, H1, H2 tiles
// = 48 KB per chain plus the input prefetch), so this kernel
//   * runs ONE CTA per SM with 3 x 256 epilogue threads + four issuer warps (896 threads, 72 registers: the bf16 copies of H1 / H2
//     the backward epilogues need are re-read from the shared-memory tile they are about to overwrite instead of living in registers);
//   * has no dO tile: the 7 (actor) / 1 (critic) output-gradient values of a sample go into the spare columns 57..63 of its X row
//     (column 56 is the constant one that carries the layer-1 bias).  Z = dO WO is then the K chunk 48..63 of X against a WO tile whose
//     rows 0..8 are zero (they face the observation columns 48..55 and the one), dWO += H2^T dO reads the same 16 columns MN-major, and
//     the layer-2 bias gradient comes from ONE M = 128 GEMM  [G2 | G1]^T X  (the MN-major A operand spans the adjacent H2 and H1 tiles):
//     rows 64..127 = dW0 | db0, row m < 64, column 56 = db1[m];
//   * keeps ONE set of weight-gradient accumulators in TMEM for the three streams (dWO 16 | dW1 64 | [db1 ; dW0|db0] 64 columns, next to
//     3 x 64 chain columns): every MMA of the CTA is issued by the same thread, so the accumulating MMAs execute in issue order;
//   * issue is split over four warps, because one thread issuing all 41 MMAs of three streams was the bottleneck (~60-100 cycles per
//     UTCHMMA while the operand fetch of the previous ones backs up): one CHAIN issuer per stream (the five GEMMs a tile's epilogues wait
//     for, plain blocking waits) and one ACCUMULATE / LOADER warp that issues the weight-gradient batches of all three streams -- in a
//     fixed (tile round, stream) order per accumulator, so the sums are bitwise reproducible whatever the timing -- and the TMA prefetches;
//     the next tile's layer 1 no longer queues behind the trailing dW0 batch (its epilogue's H1 stores wait for that batch instead);
//   * actor and critic CTAs have different chain lengths (the actor's loss stage is longer), so the grid is split unevenly between
//     the nets (KIN_PPO_TC3_ACTOR_PCT); CTA c owns partial row c and zero-fills the other net's columns.
// Image mode, 56-input policies, gradient pass only (kin_ppo_tc.cu keeps the forward-only pass, fp32 observations, the 80-input route
// policy -- 7 dO values do not fit its 3 spare columns -- and minibatches smaller than one tile per CTA).
// Arithmetic per element is the two-chain kernel's (same bf16 roundings, same tanh.approx, same loss code); sums are taken in a
// different order (tile -> CTA assignment), so gradients agree to fp32 rounding, and the kernel is bitwise reproducible run to run.
//
// MEASURED (B200, 524 288-sample minibatches): 134 us per launch under ncu against 126 us for the two-chain kernel, update 19.2 ms vs
// 18.4 ms; with the chain GEMMs' A operands in tensor memory (both kernels): 18.96 ms vs 17.45 ms -- NOT faster, so it is OFF by default (KIN_PPO_TC3=1 / kin_ppo_tc3_config(1, ..) turn it on).  The ncu capture
// (profiles/r2_ppo_tc3_raw.csv) shows why a third chain cannot pay: the kernel is bound by the shared-memory data pipe, which the tensor
// core's operand fetch (l1tex__data_pipe_tc_wavefronts_mem_shared 36.7 % of peak: every activation tile is read 2-3 times, SS-mode MMAs
// with N = 64 fetch 6 KB per 32-cycle MMA) shares with the epilogues' LDS / STS (30.0 %): 67 % busy on average with a per-tile chain of
// 11 dependent phases.  The tensor pipe proper is 26 % busy in both kernels.  Kept as the measured experiment and as the place to start
// from if the operand traffic is cut (A operands from TMEM for the four chain GEMMs would remove 52 of the 196 KB per tile).
#include "kin_peer.cuh"
#include "kin_ppo_layout.cuh"
#include "kin_ppo_math.cuh"
#include "kin_umma.cuh"

namespace kin {

using namespace umma;

namespace tc3 {

constexpr int STREAMS = 3;
constexpr int EPI = 256;                           // epilogue threads per stream: 128 sample rows x 2 column halves
constexpr int THREADS = STREAMS * EPI + 128;       // + three chain-issuer warps (one per stream) + the accumulate / loader warp
constexpr int ISSUER_WARP = STREAMS * EPI / 32;    // first chain-issuer warp
constexpr int ACC_WARP = ISSUER_WARP + STREAMS;
constexpr int ROWS = 128;
constexpr int TILE = ROWS * 128;                   // [128][64 bf16]
constexpr int DO_COL = 57;                         // X columns 57..63 hold dL/d(mean_0..6) (actor) or dL/dvalue (critic, column 57)
constexpr int WO_ROW = DO_COL - 48;                // ... which face rows 9..15 of the WO tile (K chunk 48..63 of X)

// TMEM column map (fp32 columns)
constexpr unsigned COL_Z = 0;          // 3 x 64: the chain accumulator of stream s at 64 s (layer 3's O aliases its columns 0..15)
constexpr unsigned COL_WO = 192;       // 16 (M = 64): columns 9..15 = dWO rows
constexpr unsigned COL_W1 = 208;       // 64 (M = 64)
constexpr unsigned COL_W0 = 272;       // 64 (M = 128): lanes 64..127 = dW0 | db0 (column 56), lanes 0..63 column 56 = db1
constexpr unsigned COL_A = 336;        // 3 x 32: the bf16 A operand of stream s's next chain GEMM (H1, H2, G2) at 336 + 32 s -- TS-mode MMAs, as in
                                       // the two-chain kernel: the tiles are still stored to shared memory for the MN-major readers
constexpr unsigned TMEM_COLS = 512;

struct __align__(1024) StreamTiles {
    unsigned char X[2][TILE];      // double-buffered operand image of the tile's observations (TMA); columns 57..63 receive dO
    unsigned char H2[TILE];        // H2, later G2 = dL/dZ2
    unsigned char H1[TILE];        // H1, later G1 = dL/dZ1.  MUST follow H2: [H2 | H1] is one MN-major M = 128 operand
};

struct __align__(1024) Smem {
    StreamTiles st[STREAMS];
    unsigned char W0[64 * 128];    // col 56 = b0
    unsigned char W1[64 * 128];
    unsigned char WO[16 * 128];    // actor: rows 9..15 = act_w; critic: row 9 = val_w; rows 0..8 zero
    float act[STREAMS][ROWS * 7];  // loss inputs of the stream's current tile (TMA)
    float adv[STREAMS][ROWS];      // critic CTAs: the returns
    float olp[STREAMS][ROWS];
    float b1[64];
    float bo[8];
    float ls[8];
    float inv_sig[8];
    float scal[32];                // 0 adv mean, 1 1/(std+eps), 2..5 statistics, 8..14 d log_std, 16..23 d output bias
    float red[STREAMS * 4][20];    // per loss-warp partial sums, folded in a fixed order
    unsigned long long mbar[STREAMS][8];   // per stream: 0 main, 1 ride, 2 wg, 3 / 4 X buffers, 5 loss inputs, 6 tile written -> chain issuer, 7 -> accumulate warp
    unsigned long long mbar_w;
    unsigned tmem_base;
};
static_assert(sizeof(Smem) + 1024 <= 232448, "one CTA per SM: 227 KB of shared memory");

#ifdef KIN_PPO_TRACE
// phase profiler (debug builds only, tools/ppo_trace.py --tc3): cycles per phase summed over the tiles of a stream, for the issuer warp and
// the accumulate warp and epilogue thread 32 (stream 0) of the first CTA (actor), and thread 32 of the last CTA (critic)
__device__ unsigned long long kin_ppo_trace3_buf[4][16];
#define T3_DECL unsigned long long tr_acc[15] = {}; long long tr_t = clock64(); \
    const bool tr_on = (blockIdx.x == 0 && (tid == 32 || tid == ISSUER_WARP * 32 || tid == ACC_WARP * 32)) || (blockIdx.x == gridDim.x - 1 && tid == 32);
#define T3_MARK(i) do { if (tr_on) { const long long t_ = clock64(); tr_acc[i] += (unsigned long long)(t_ - tr_t); tr_t = t_; } } while (0)
#define T3_FLUSH(ntiles) do { if (tr_on) { unsigned long long* o_ = kin_ppo_trace3_buf[blockIdx.x ? 3 : (tid == 32 ? 1 : (tid == ACC_WARP * 32 ? 2 : 0))]; \
    for (int i_ = 0; i_ < 15; ++i_) o_[i_] = tr_acc[i_]; o_[15] = (unsigned long long)(ntiles); } } while (0)
#else
#define T3_DECL
#define T3_MARK(i)
#define T3_FLUSH(n)
#endif

// an operand tile (or a TMEM read) of this warp is complete: make the generic-proxy writes visible to the tensor core, converge, and let
// one lane arrive on the stream's "tile written" barriers (count 8 = the stream's warps): the chain issuer's, and for the tiles the
// weight-gradient batches read (dO, G2, G1) the accumulate warp's too
template <bool ACC>
__device__ __forceinline__ void tile_written(unsigned mb_rdy, int lane) {
    fence_async_smem();
    fence_before();
    __syncwarp();
    if (lane == 0) {
        mbar_arrive(mb_rdy);
        if (ACC) mbar_arrive(mb_rdy + 8);
    }
}

// forward epilogue, arithmetic part: this thread's 32 accumulator columns -> tanh -> packed bf16
template <bool BIAS>
__device__ __forceinline__ void epilogue_fwd_math(unsigned tz, int half, const float* bias, unsigned* p) {
    float v[32];
    tmem_ld32(tz + half * 32, v);
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        float a = v[2 * i], b = v[2 * i + 1];
        if (BIAS) {
            a += bias[half * 32 + 2 * i];
            b += bias[half * 32 + 2 * i + 1];
        }
        p[i] = pack_bf16(tanh_fast(a), tanh_fast(b));
    }
}
// backward epilogue, arithmetic part: g = z * (1 - h^2) with h re-read from the tile (the bf16 values the forward pass stored)
__device__ __forceinline__ void epilogue_bwd_math(unsigned tz, int half, const unsigned char* tile, int row, unsigned* p) {
    float v[32];
    tmem_ld32(tz + half * 32, v);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const uint4 hq = *reinterpret_cast<const uint4*>(tile + sw_chunk(row, half * 4 + j));
        const unsigned h4[4] = {hq.x, hq.y, hq.z, hq.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float hl = bf16_lo(h4[i]), hh = bf16_hi(h4[i]);
            p[4 * j + i] = pack_bf16(v[8 * j + 2 * i] * fmaf(-hl, hl, 1.0f), v[8 * j + 2 * i + 1] * fmaf(-hh, hh, 1.0f));
        }
    }
}
__device__ __forceinline__ void epilogue_store(unsigned char* tile, int row, int half, const unsigned* p) {
#pragma unroll
    for (int j = 0; j < 4; ++j)
        *reinterpret_cast<uint4*>(tile + sw_chunk(row, half * 4 + j)) = make_uint4(p[4 * j], p[4 * j + 1], p[4 * j + 2], p[4 * j + 3]);
}

template <bool PEER>
__global__ void __launch_bounds__(THREADS, 1)
kin_ppo_grad_tc3_kernel(const float* __restrict__ params, KinPpoHyper hp, const unsigned char* __restrict__ img, const float* __restrict__ action,
                        const float* __restrict__ old_logp, const float* __restrict__ advantage, const float* __restrict__ returns,
                        const double* __restrict__ tile_sums, const int* __restrict__ tile_ids, int n_pairs, float inv_global_batch,
                        float* __restrict__ partials, int actor_ctas, const float* __restrict__ adv_stats, const unsigned char* __restrict__ wimg,
                        const PeerFused px) {
    constexpr int IN = 56;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    Smem& S = *reinterpret_cast<Smem*>(smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u));
    const PpoOffsets O = ppo_offsets(IN);
    const int P = O.total;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const bool issuer = warp >= ISSUER_WARP;                    // warp-uniform
    const int sid = issuer ? 0 : warp >> 3;                     // this thread's stream
    const int row = tid & 127, half = (tid >> 7) & 1;           // two threads per sample row: columns 0..31 / 32..63 of every activation
    const int net = (int)blockIdx.x < actor_ctas ? 0 : 1;       // 0 actor, 1 critic
    const int cl = net ? (int)blockIdx.x - actor_ctas : (int)blockIdx.x;     // index among this net's CTAs
    const int gn = net ? (int)gridDim.x - actor_ctas : actor_ctas;           // CTAs of this net
    const int o_w0 = net ? O.vf_w0 : O.pi_w0, o_b0 = net ? O.vf_b0 : O.pi_b0, o_w1 = net ? O.vf_w1 : O.pi_w1, o_b1 = net ? O.vf_b1 : O.pi_b1;
    const int prow = P + KIN_PPO_STATS + 8;
    float* out = partials + (size_t)blockIdx.x * prow;

    // ---- prologue ----------------------------------------------------------------------------------------------------------------
    for (int i = tid; i < prow; i += THREADS) out[i] = 0.0f;      // this CTA's partial row: the other net's columns stay zero
    if (tid < 16 * 128 / 16) reinterpret_cast<uint4*>(S.WO)[tid] = make_uint4(0u, 0u, 0u, 0u);
    if (tid < 64) S.b1[tid] = __ldg(params + o_b1 + tid);
    if (tid < 8) {
        const float ls = tid < 7 ? __ldg(params + O.log_std + tid) : 0.0f;
        S.bo[tid] = tid < 7 ? __ldg(params + O.act_b + tid) : __ldg(params + O.val_b);
        S.ls[tid] = ls;
        S.inv_sig[tid] = expf(-ls);
    }
    if (tid >= 32 && tid < 64) S.scal[tid - 32] = 0.0f;
    __syncthreads();
    if (net == 0) {
        for (int i = tid; i < 7 * 64; i += THREADS) st_bf16(S.WO, WO_ROW + (i >> 6), i & 63, __ldg(params + O.act_w + i));
    } else if (tid < 64) {
        st_bf16(S.WO, WO_ROW, tid, __ldg(params + O.val_w + tid));
    }
    if (adv_stats) {
        if (tid == 0) { S.scal[0] = adv_stats[0]; S.scal[1] = adv_stats[1]; }
    } else if (tid < 32 && net == 0) {
        const double2 s = warp_tile_sums(tile_sums, tile_ids, 2 * n_pairs, tid, 32);
        if (tid == 0) adv_normaliser(s.x, s.y, (double)n_pairs * ROWS, hp.normalize_advantage, S.scal);
    }
    if (warp == 1) tmem_alloc(smem_u32(&S.tmem_base), TMEM_COLS);
    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < STREAMS; ++s) {
#pragma unroll
            for (int i = 0; i < 6; ++i) mbar_init(smem_u32(&S.mbar[s][i]), 1);
            mbar_init(smem_u32(&S.mbar[s][6]), EPI / 32);
            mbar_init(smem_u32(&S.mbar[s][7]), EPI / 32);
        }
        mbar_init(smem_u32(&S.mbar_w), 1);
        fence_mbar_init();
        const unsigned mbw = smem_u32(&S.mbar_w);      // this net's W0 | W1 blocks of the prebuilt bf16 image: two bulk copies
        mbar_expect_tx(mbw, 8192 + 8192);
        bulk_load(smem_u32(S.W0), wimg + KIN_WIMG_W0 + net * 8192, 8192, mbw);
        bulk_load(smem_u32(S.W1), wimg + KIN_WIMG_W1 + net * 8192, 8192, mbw);
    }
    fence_async_smem();
    fence_before();
    __syncthreads();
    fence_after();
    mbar_wait(smem_u32(&S.mbar_w), 0u);

    const unsigned tb = S.tmem_base;
    int it = 0;
    T3_DECL

    if (issuer) {
        const bool lead = elect_one();
        const unsigned aS0 = smem_u32(&S.st[0]), aW0 = smem_u32(S.W0), aW1 = smem_u32(S.W1), aWO = smem_u32(S.WO);
        const int stride = STREAMS * gn;
        if (warp < ACC_WARP) {
            // ================= chain issuer of stream `cs`: the five GEMMs a tile's epilogues wait for, in order ==========================
            const int cs = warp - ISSUER_WARP;
            const unsigned mb = smem_u32(&S.mbar[cs][0]);       // main +0, X buffers +24 / +32, tile written +48
            const unsigned aT = aS0 + cs * (unsigned)sizeof(StreamTiles), aH2 = aT + 2 * TILE, aH1 = aT + 3 * TILE;
            const unsigned tz = tb + COL_Z + 64 * cs, ta = tb + COL_A + 32 * cs;
            constexpr unsigned id_fwd = idesc_bf16(128, 64, false, false), id_out = idesc_bf16(128, 16, false, false);
            constexpr unsigned id_bwd = idesc_bf16(128, 64, false, true);
            unsigned pr = 0u;
            for (int j = cs * gn + cl; j < n_pairs; j += stride, ++it) {
                const unsigned aX = aT + (it & 1) * TILE;
                T3_MARK(7);
                mbar_wait(mb + 24 + 8 * (it & 1), (unsigned)(it >> 1) & 1u);       // the tile's image has landed (prefetched half a tile ago)
                fence_after();
                T3_MARK(0);
                if (lead) {
#pragma unroll
                    for (int k = 0; k < 4; ++k) mma_bf16(tz, desc_k(aX + k * 32), desc_k(aW0 + k * 32), id_fwd, k > 0);
                    commit(mb);
                }
                T3_MARK(1);
                mbar_wait(mb + 48, pr); pr ^= 1u;        // H1 written -> layer 2
                fence_after();
                T3_MARK(2);
                if (lead) {
#pragma unroll
                    for (int k = 0; k < 4; ++k) mma_bf16_ts(tz, ta + 8 * k, desc_k(aW1 + k * 32), id_fwd, k > 0);
                    commit(mb);
                }
                mbar_wait(mb + 48, pr); pr ^= 1u;        // H2 written -> layer 3: action means (columns 9..15) or value (column 9)
                fence_after();
                T3_MARK(3);
                if (lead) {
#pragma unroll
                    for (int k = 0; k < 4; ++k) mma_bf16_ts(tz, ta + 8 * k, desc_k(aWO + k * 32), id_out, k > 0);
                    commit(mb);
                }
                mbar_wait(mb + 48, pr); pr ^= 1u;        // dO written (X columns 57..63) -> Z = dO WO
                fence_after();
                T3_MARK(4);
                if (lead) {
                    mma_bf16(tz, desc_k(aX + 96), desc_mn(aWO), id_bwd, 0u);
                    commit(mb);
                }
                mbar_wait(mb + 48, pr); pr ^= 1u;        // G2 written (over H2) -> Z = G2 W1
                fence_after();
                T3_MARK(5);
                if (lead) {
#pragma unroll
                    for (int k = 0; k < 4; ++k) mma_bf16_ts(tz, ta + 8 * k, desc_mn(aW1 + k * 2048), id_bwd, k > 0);
                    commit(mb);
                }
                mbar_wait(mb + 48, pr); pr ^= 1u;        // G1 written: the epilogue threads have read Z, the next tile's layer 1 may overwrite it
                fence_after();
                T3_MARK(6);
            }
        } else {
            // ================= accumulate / loader warp: the weight-gradient batches of all three streams and their TMA prefetches ==========
            // The batches into one accumulator are issued in a FIXED order -- tile round by tile round, stream 0, 1, 2 within a round -- whatever
            // the timing, so the fp32 sums (and the whole update) are bitwise reproducible.
            const unsigned mb0 = smem_u32(&S.mbar[0][0]);       // per stream: ride +8, wg +16, X buffers +24 / +32, loss inputs +40, written (acc) +56
            const unsigned aAct = smem_u32(S.act[0]), aAdv = smem_u32(S.adv[0]), aOlp = smem_u32(S.olp[0]);
            constexpr unsigned id_w16 = idesc_bf16(64, 16, true, true), id_w64 = idesc_bf16(64, 64, true, true), id_w0 = idesc_bf16(128, 64, true, true);
            const unsigned loss_bytes = net == 0 ? 2u * 1792u + 4u * 256u : 2u * 256u;
            auto stage_x = [&](int s, int t0, int b) {           // elected lane only
                const unsigned mb = mb0 + s * 64 + 24 + 8 * b;
                mbar_expect_tx(mb, TILE);
                bulk_load(aS0 + s * (unsigned)sizeof(StreamTiles) + b * TILE, img + (size_t)(t0 >> 1) * TILE, TILE, mb);
            };
            auto stage_loss = [&](int s, int t0, int t1) {       // elected lane only
                const unsigned mb = mb0 + s * 64 + 40;
                mbar_expect_tx(mb, loss_bytes);
                if (net == 0) {
                    bulk_load(aAct + s * 3584, action + (size_t)t0 * 448, 1792u, mb);
                    bulk_load(aAct + s * 3584 + 1792, action + (size_t)t1 * 448, 1792u, mb);
                    bulk_load(aAdv + s * 512, advantage + (size_t)t0 * 64, 256u, mb);
                    bulk_load(aAdv + s * 512 + 256, advantage + (size_t)t1 * 64, 256u, mb);
                    bulk_load(aOlp + s * 512, old_logp + (size_t)t0 * 64, 256u, mb);
                    bulk_load(aOlp + s * 512 + 256, old_logp + (size_t)t1 * 64, 256u, mb);
                } else {
                    bulk_load(aAdv + s * 512, returns + (size_t)t0 * 64, 256u, mb);
                    bulk_load(aAdv + s * 512 + 256, returns + (size_t)t1 * 64, 256u, mb);
                }
            };
            int ph[STREAMS], itv[STREAMS], nt[STREAMS], nx0[STREAMS], nx1[STREAMS];      // nx: 64-sample tile ids of the stream's NEXT tile
            unsigned pr[STREAMS];
            int active = 0;
#pragma unroll
            for (int s = 0; s < STREAMS; ++s) {
                const int j0 = s * gn + cl;
                nt[s] = j0 < n_pairs ? (n_pairs - j0 + stride - 1) / stride : 0;
                itv[s] = 0;
                pr[s] = 0u;
                ph[s] = nt[s] > 0 ? 3 : 6;
                nx0[s] = nx1[s] = 0;
                if (nt[s] > 0) {
                    ++active;
                    const int t0 = __ldg(tile_ids + 2 * j0), t1 = __ldg(tile_ids + 2 * j0 + 1);
                    if (lead) { stage_x(s, t0, 0); stage_loss(s, t0, t1); }
                    if (nt[s] > 1) { nx0[s] = __ldg(tile_ids + 2 * (j0 + stride)); nx1[s] = __ldg(tile_ids + 2 * (j0 + stride) + 1); }
                }
            }
            // cursors of the three accumulators: (round, stream) of the batch that goes in next
            int ct3 = 0, cs3 = 0, ct4 = 0, cs4 = 0, ct5 = 0, cs5 = 0;
            unsigned acc_wo = 0u, acc_w1 = 0u, acc_w0 = 0u;      // the first batch into an accumulator overwrites it
            while (active > 0) {
                T3_MARK(6);          // polling
#pragma unroll
                for (int s = 0; s < STREAMS; ++s) {
                    const int k = ph[s];
                    if (k == 6) continue;
                    const int si = itv[s];
                    if (k == 3 ? (ct3 != si || cs3 != s) : (k == 4 ? (ct4 != si || cs4 != s) : (ct5 != si || cs5 != s))) continue;      // not its turn
                    const unsigned mb = mb0 + s * 64;
                    if (!mbar_test_wait(mb + 56, pr[s])) continue;
                    pr[s] ^= 1u;
                    fence_after();
                    T3_MARK(6);
                    const unsigned aT = aS0 + s * (unsigned)sizeof(StreamTiles);
                    const unsigned aX = aT + (si & 1) * TILE, aH2 = aT + 2 * TILE, aH1 = aT + 3 * TILE;
                    if (k == 3) {            // dO written: dWO += H2^T dO (H2's last reader); prefetch the next tile's inputs
                        if (lead) {
#pragma unroll
                            for (int q = 0; q < 8; ++q) mma_bf16(tb + COL_WO, desc_mn(aH2 + q * 2048), desc_mn(aX + 96 + q * 2048), id_w16, acc_wo | (q > 0));
                            commit(mb + 8);
                        }
                        acc_wo = 1u;
                        if (si + 1 < nt[s]) {
                            // the other X buffer's last reader was the previous tile's trailing batch (issued half a tile ago); the loss
                            // threads have consumed this tile's inputs
                            if (si > 0) mbar_wait(mb + 16, (unsigned)(si - 1) & 1u);
                            if (lead) { stage_x(s, nx0[s], (si + 1) & 1); stage_loss(s, nx0[s], nx1[s]); }
                        }
                        ph[s] = 4;
                        if (++cs3 == STREAMS || nt[cs3] <= ct3) { cs3 = 0; ++ct3; }
                        T3_MARK(3);
                    } else if (k == 4) {     // G2 written (over H2): dW1 += G2^T H1 (H1's last reader)
                        if (lead) {
#pragma unroll
                            for (int q = 0; q < 8; ++q) mma_bf16(tb + COL_W1, desc_mn(aH2 + q * 2048), desc_mn(aH1 + q * 2048), id_w64, acc_w1 | (q > 0));
                            commit(mb + 8);
                        }
                        acc_w1 = 1u;
                        ph[s] = 5;
                        if (++cs4 == STREAMS || nt[cs4] <= ct4) { cs4 = 0; ++ct4; }
                        T3_MARK(4);
                    } else {                 // G1 written (over H1): [db1 ; dW0|db0] += [G2 | G1]^T X
                        if (lead) {
#pragma unroll
                            for (int q = 0; q < 8; ++q) mma_bf16(tb + COL_W0, desc_mn(aH2 + q * 2048), desc_mn(aX + q * 2048), id_w0, acc_w0 | (q > 0));
                            commit(mb + 16);
                        }
                        acc_w0 = 1u;
                        if (++cs5 == STREAMS || nt[cs5] <= ct5) { cs5 = 0; ++ct5; }
                        itv[s] = si + 1;
                        if (si + 1 < nt[s]) {
                            ph[s] = 3;
                            if (si + 2 < nt[s]) {        // tile ids of the tile after next: in registers long before they are staged
                                const int jn = s * gn + cl + (si + 2) * stride;
                                nx0[s] = __ldg(tile_ids + 2 * jn);
                                nx1[s] = __ldg(tile_ids + 2 * jn + 1);
                            }
                        } else {
                            ph[s] = 6;
                            --active;
                        }
                        T3_MARK(5);
                        if (s == 0) it = si + 1;
                    }
                }
            }
        }
    } else {
        // ================= epilogue threads of stream `sid` ==============================================================================
        StreamTiles& T = S.st[sid];
        const unsigned tlane = tb + ((unsigned)((warp & 3) * 32) << 16);     // this warp's lane quadrant, column 0
        const unsigned tz = tlane + COL_Z + 64 * sid, ta = tlane + COL_A + 32 * sid + 16 * half;
        const unsigned mb_main = smem_u32(&S.mbar[sid][0]), mb_ride = mb_main + 8, mb_wg = mb_main + 16, mb_loss = mb_main + 40, mb_rdy = mb_main + 48;
        unsigned par_main = 0u;
        float dls[7] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, dbo[7] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, st[4] = {0.f, 0.f, 0.f, 0.f};
        const int stride = STREAMS * gn;
        for (int j = sid * gn + cl; j < n_pairs; j += stride, ++it) {
            unsigned char* X = T.X[it & 1];
            unsigned p[16];
            // ---- layer 1 (issued ahead of the previous tile's trailing [G2 | G1]^T X batch, which still reads H1 / H2: the arithmetic
            //      overlaps that batch, the stores wait for it) -----------------------------------------------------------------------------
            T3_MARK(14);
            mbar_wait(mb_main, par_main);
            par_main ^= 1u;
            fence_after();
            T3_MARK(0);
            epilogue_fwd_math<false>(tz, half, nullptr, p);
            T3_MARK(1);
            if (it > 0) mbar_wait(mb_wg, (unsigned)(it - 1) & 1u);
            epilogue_store(T.H1, row, half, p);
            tmem_st16(ta, p);
            tile_written<false>(mb_rdy, lane);
            T3_MARK(2);
            // ---- layer 2 -------------------------------------------------------------------------------------------------------------
            mbar_wait(mb_main, par_main);
            par_main ^= 1u;
            fence_after();
            T3_MARK(3);
            epilogue_fwd_math<true>(tz, half, S.b1, p);
            epilogue_store(T.H2, row, half, p);
            tmem_st16(ta, p);
            tile_written<false>(mb_rdy, lane);
            T3_MARK(4);
            // ---- layer 3 -> loss and d(loss)/d(outputs), one thread per sample -----------------------------------------------------------
            mbar_wait(mb_main, par_main);
            par_main ^= 1u;
            fence_after();
            T3_MARK(5);
            if (half == 0) {
                float o[16];
                tmem_ld16(tz, o);
                mbar_wait(mb_loss, (unsigned)it & 1u);          // staged loss inputs (landed long ago)
                if (net == 0) {
                    const float* act_r = S.act[sid] + row * 7;
                    const float adv_r = S.adv[sid][row], olp_r = S.olp[sid][row];
                    float lp = 0.0f, z[7];
#pragma unroll
                    for (int d = 0; d < 7; ++d) {
                        z[d] = (act_r[d] - (o[WO_ROW + d] + S.bo[d])) * S.inv_sig[d];
                        lp += gauss_logp_term(z[d], S.ls[d]);
                    }
                    const Surrogate sur = clipped_surrogate(adv_r, S.scal[0], S.scal[1], lp, olp_r, hp);
                    const float dpl_dlp = sur.dpl_dlp();
                    float dm[7];
                    float ent = 0.0f;
#pragma unroll
                    for (int d = 0; d < 7; ++d) {
                        dm[d] = dloss_dmean(inv_global_batch, dpl_dlp, z[d], S.inv_sig[d]);
                        dbo[d] += dm[d];
                        dls[d] += dloss_dlog_std(inv_global_batch, dpl_dlp, z[d], hp);
                        ent += gauss_entropy_term(S.ls[d]);
                    }
                    *reinterpret_cast<uint4*>(X + sw_chunk(row, 7)) =        // columns 56..63: the constant one, then dO
                        make_uint4(pack_bf16(1.0f, dm[0]), pack_bf16(dm[1], dm[2]), pack_bf16(dm[3], dm[4]), pack_bf16(dm[5], dm[6]));
                    st[0] += sur.loss();
                    st[1] += ent;
                    st[2] += sur.approx_kl();
                    st[3] += sur.clipped(hp);
                } else {
                    const float v = o[WO_ROW] + S.bo[7];
                    const float ret_r = S.adv[sid][row];
                    const float dv = dloss_dvalue(inv_global_batch, v, ret_r, hp);
                    dbo[0] += dv;
                    *reinterpret_cast<uint4*>(X + sw_chunk(row, 7)) = make_uint4(pack_bf16(1.0f, dv), 0u, 0u, 0u);
                    st[0] += value_loss(v, ret_r);
                }
            }
            tile_written<true>(mb_rdy, lane);
            T3_MARK(6);
            // ---- dZ2 = (dO WO) * (1 - H2^2): G2 replaces H2 once dWO += H2^T dO has read it ---------------------------------------------
            mbar_wait(mb_main, par_main);
            par_main ^= 1u;
            fence_after();
            T3_MARK(7);
            epilogue_bwd_math(tz, half, T.H2, row, p);
            tmem_st16(ta, p);            // (layer 3, the last reader of these columns, has completed)
            T3_MARK(8);
            mbar_wait(mb_ride, 0u);
            T3_MARK(9);
            epilogue_store(T.H2, row, half, p);
            tile_written<true>(mb_rdy, lane);
            T3_MARK(10);
            // ---- dZ1 = (G2 W1) * (1 - H1^2): G1 replaces H1 once dW1 += G2^T H1 has read it ----------------------------------------------
            mbar_wait(mb_main, par_main);
            par_main ^= 1u;
            fence_after();
            T3_MARK(11);
            epilogue_bwd_math(tz, half, T.H1, row, p);
            T3_MARK(12);
            mbar_wait(mb_ride, 1u);
            epilogue_store(T.H1, row, half, p);
            tile_written<true>(mb_rdy, lane);
            T3_MARK(13);
        }
        // log_std / output-bias gradients and statistics: warp shuffle, then one partial row per loss warp
        if (half == 0) {
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
            if (lane == 0) {
                float* r = S.red[sid * 4 + (warp & 3)];
#pragma unroll
                for (int q = 0; q < 4; ++q) r[q] = st[q];
#pragma unroll
                for (int d = 0; d < 7; ++d) {
                    r[4 + d] = dls[d];
                    r[11 + d] = dbo[d];
                }
            }
        }
        if (it > 0) mbar_wait(smem_u32(&S.mbar[sid][2]), (unsigned)(it - 1) & 1u);      // the stream's last dW0 batch has drained
    }

    T3_FLUSH(it);
    fence_before();
    __syncthreads();
    fence_after();
    if (tid < 18) {      // statistics -> scal[2..5], d log_std -> scal[8..14], d output bias -> scal[16..22]
        float a = 0.0f;
#pragma unroll
        for (int q = 0; q < STREAMS * 4; ++q) a += S.red[q][tid];
        S.scal[tid < 4 ? 2 + tid : (tid < 11 ? 8 + tid - 4 : 16 + tid - 11)] = a;
    }
    __syncthreads();
    // ---- accumulators -> this CTA's partial row (stream 0's eight warps; a warp reads its own TMEM lane quadrant) ------------------------
    if (warp < 8) {
        const unsigned tlane = tb + ((unsigned)((warp & 3) * 32) << 16);
        const int q = warp & 3;
        float v[32];
        // dW1 (M = 64: row m lives in lane m % 16 + 32 * (m / 16)): warps 0..3 columns 0..31, warps 4..7 columns 32..63
        tmem_ld32(tlane + COL_W1 + half * 32, v);
        if (lane < 16) {
            const int u = q * 16 + lane;
#pragma unroll
            for (int c = 0; c < 32; ++c) out[o_w1 + u * 64 + half * 32 + c] = v[c];
        }
        // [db1 ; dW0 | db0] (M = 128: row m in lane m): lanes 64..127 = hidden unit m - 64 of layer 1, lanes 0..63 column 56 = db1
        tmem_ld32(tlane + COL_W0 + half * 32, v);
        if (q >= 2) {
            const int u = (q - 2) * 32 + lane;
#pragma unroll
            for (int c = 0; c < 32; ++c) {
                const int k = half * 32 + c;
                if (k < IN) out[o_w0 + u * IN + k] = v[c];
                else if (k == IN) out[o_b0 + u] = v[c];
            }
        } else if (half == 1) {
            out[o_b1 + q * 32 + lane] = v[IN - 32];
        }
        if (half == 0) {
            float o[16];
            tmem_ld16(tlane + COL_WO, o);
            if (lane < 16) {
                const int u = q * 16 + lane;
                if (net == 0) {
#pragma unroll
                    for (int d = 0; d < 7; ++d) out[O.act_w + d * 64 + u] = o[WO_ROW + d];
                } else {
                    out[O.val_w + u] = o[WO_ROW];
                }
            }
        }
    }
    if (net == 0) {
        if (tid < 7) {
            out[O.log_std + tid] = S.scal[8 + tid];
            out[O.act_b + tid] = S.scal[16 + tid];
        }
        if (tid == 0) {
            out[P + KIN_PPO_STAT_POLICY_LOSS] = S.scal[2];
            out[P + KIN_PPO_STAT_ENTROPY] = S.scal[3];
            out[P + KIN_PPO_STAT_APPROX_KL] = S.scal[4];
            out[P + KIN_PPO_STAT_CLIP_FRACTION] = S.scal[5];
        }
    } else if (tid == 0) {
        out[P + KIN_PPO_STAT_VALUE_LOSS] = S.scal[2];
        out[O.val_b] = S.scal[16];
    }
    if constexpr (PEER) {       // every tile buffer is dead by now: the exchange borrows an X tile for its 1 KB of scratch
        float(*part)[32] = reinterpret_cast<float(*)[32]>(S.st[0].X[0]);
        peer_exchange_tail(px, partials, (int)gridDim.x, P, inv_global_batch, part, reinterpret_cast<int*>(S.st[0].X[0] + 2048));
        if (px.adam.params) peer_adam_tail(px, hp, P, reinterpret_cast<float*>(S.st[0].X[0] + 4096));      // clip + Adam on this CTA's slice
    }
    fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tb, TMEM_COLS);
}

}  // namespace tc3

// actor share of the grid in percent (the actor's chain is the longer one) and the on / off switch; the environment gives the defaults
// (KIN_PPO_TC3_ACTOR_PCT, KIN_PPO_TC3=1), kin_ppo_tc3_config changes them at run time
static int g_tc3_pct = -1, g_tc3_enabled = -1;
static void tc3_defaults() {
    if (g_tc3_pct < 0) {
        const char* e = getenv("KIN_PPO_TC3_ACTOR_PCT");
        const int v = e ? atoi(e) : 0;
        g_tc3_pct = (v >= 10 && v <= 90) ? v : 52;
    }
    if (g_tc3_enabled < 0) {
        const char* e = getenv("KIN_PPO_TC3");
        g_tc3_enabled = (e && e[0] == '1') ? 1 : 0;      // off by default: measured 4 % slower than the two-chain kernel (DESIGN.md, K3-TC)
    }
}

// 1 = handled (launched or failed with *rc set), 0 = not eligible: the caller uses the two-chain kernel
int kin_ppo_grad_tc3_try(const float* params, const KinPpoHyper* hp, const void* images, const float* action, const float* old_logp,
                         const float* advantage, const float* returns, const double* tile_sums, const int* tile_ids, int n_pairs, float inv_global_batch,
                         float* partials, int grid, const float* adv_stats, const void* weight_image, const PeerFused& px, bool fused, cudaStream_t st,
                         int* rc) {
    tc3_defaults();
    if (!g_tc3_enabled || !weight_image || grid < 2 || n_pairs < grid) return 0;
    static int n_sm[KIN_MAX_DEVICES] = {};
    static bool attr_set[KIN_MAX_DEVICES] = {};
    const int dev_slot = kin_device_slot();
    if (!attr_set[dev_slot]) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n_sm[dev_slot], cudaDevAttrMultiProcessorCount, dev);
        const int bytes = (int)(sizeof(tc3::Smem) + 1024);
        cudaError_t e = cudaFuncSetAttribute(tc3::kin_ppo_grad_tc3_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(tc3::kin_ppo_grad_tc3_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
        if (e != cudaSuccess) { *rc = kin_fail_cuda(e, "kin_ppo_grad_tc3: smem attribute"); return 1; }
        attr_set[dev_slot] = true;
    }
    if (grid > n_sm[dev_slot]) return 0;        // one CTA per SM, all co-resident (the fused exchange has a grid barrier)
    int actor = (grid * g_tc3_pct + 50) / 100;
    actor = actor < 1 ? 1 : (actor > grid - 1 ? grid - 1 : actor);
    const size_t smem = sizeof(tc3::Smem) + 1024;
    const unsigned char* img = static_cast<const unsigned char*>(images);
    const unsigned char* wimg = static_cast<const unsigned char*>(weight_image);
    if (fused)
        tc3::kin_ppo_grad_tc3_kernel<true><<<grid, tc3::THREADS, smem, st>>>(params, *hp, img, action, old_logp, advantage, returns, tile_sums, tile_ids, n_pairs,
                                                                             inv_global_batch, partials, actor, adv_stats, wimg, px);
    else
        tc3::kin_ppo_grad_tc3_kernel<false><<<grid, tc3::THREADS, smem, st>>>(params, *hp, img, action, old_logp, advantage, returns, tile_sums, tile_ids, n_pairs,
                                                                              inv_global_batch, partials, actor, adv_stats, wimg, px);
    *rc = KIN_OK;
    return 1;
}

}  // namespace kin

#ifdef KIN_PPO_TRACE
extern "C" int kin_debug_ppo_trace3(unsigned long long* out) {      // 4 x 16 counters, see T3_DECL
    return cudaMemcpyFromSymbol(out, kin::tc3::kin_ppo_trace3_buf, sizeof(kin::tc3::kin_ppo_trace3_buf)) == cudaSuccess ? KIN_OK : KIN_ERR_INVALID_ARG;
}
#endif

extern "C" int kin_ppo_tc3_config(int enabled, int actor_pct) {
    kin::tc3_defaults();
    if (enabled >= 0) kin::g_tc3_enabled = enabled ? 1 : 0;
    if (actor_pct >= 10 && actor_pct <= 90) kin::g_tc3_pct = actor_pct;
    return kin::g_tc3_enabled | (kin::g_tc3_pct << 8);
}
