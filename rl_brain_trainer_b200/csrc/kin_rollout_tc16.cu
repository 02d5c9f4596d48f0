// kin_rollout_tc16.cu -- K2-TC: the fused policy-in-loop Approach -> Finisher rollout, actor MLP on the 5th-generation tensor
// cores (tcgen05.mma kind::f16, fp16 operands, fp32 accumulators in TMEM).  Round-2 rewrite of the earlier TF32 kernel.
//
// Mapping (unchanged): one episode <-> one thread <-> one row of the A operand <-> one TMEM lane; a CTA carries up to four
// independent 128-episode tiles that share one staged copy of the policy; a batch that fits one wave is spread evenly over
// the SMs (65 536 episodes -> 148 CTAs x 14 warps).
//
// What changed, in order of instructions saved per env-step (1 854 warp-instructions before):
//   * the 20 observation columns that are constants of this path (mode_flag, task_type, the four waypoint blocks,
//     progress[2]) never enter the A operand: W0[:, const] . const is folded into the layer-1 bias when the weights are staged,
//     layer 1 runs K = 48 (3 MMAs) instead of K = 64 TF32 (8 MMAs);
//   * fp16 operands: the 36 live observation values are rounded two at a time (cvt.rn.f16x2.f32), clamped two at a time
//     (min/max.f16x2) and stored with 5 STS.128; a hidden layer's epilogue is 32 cvt + 32 tanh.approx.f16x2 + 8 STS.128;
//   * every bias rides on an MMA (the X tile's constant-one column against a bias slice of the weight image);
//   * no CTA / named barrier in the step loop: writers bump a per-tile arrival counter, the warp that arrives last issues the
//     tile's MMAs from one elected lane, everybody waits on the accumulator mbarrier only;
//   * the env step runs the FAST flavour of kin_core.cuh (single-MUFU sqrt / reciprocal, polynomial atan2, previous pose-error
//     norms carried, margins from the normalised joint position);
//   * the first-confirmed handoff snapshot (21 floats per episode) lives in shared memory, not registers.
//
// Numerics: env arithmetic fp32; MLP operands fp16 (11-bit significand, like TF32) with fp32 accumulation and tanh.approx.f16x2:
// actions differ from strict fp32 by O(1e-3) as before; closed-loop agreement is tested in tests/test_gpu_rollout.py and
// tests/test_gpu_fullsize.py (every flipped success flag must sit within a stated band of a threshold).
//
// Replaces the reference loops eval_pipeline_ablation.py:60-147, eval_workspace_expansion.py:126-147 (same as kin_rollout.cu).
#include <cstdlib>

#include "kin_tc16.cuh"

namespace kin {

using namespace tc16;

#ifdef KIN_TC16_TRACE
// cycle trace (debug builds only, tools/tc16_trace.py): SM-clock stamps of every warp of CTA 0 around the three GEMM round trips
// of approach steps 10..17: [step][warp][0..2 = before arrive L1/L2/L3 | 3..5 = after wake L1/L2/L3 | 6..8 = MMAs committed (issuing warp)]
__device__ long long kin_tc16_trace_buf[8][16][12];   // 9..11 = issuer warp woke up for L1/L2/L3 (issuer-warp mode)
#define TC16_STAMP(slot) do { if (blockIdx.x == 0 && c.step_id >= 10 && c.step_id < 18 && (threadIdx.x & 31) == 0) \
        kin_tc16_trace_buf[c.step_id - 10][threadIdx.x >> 5][slot] = clock64(); } while (0)
#else
#define TC16_STAMP(slot)
#endif

struct Tile16 {
    unsigned char *X, *H;
    float* snap;                 // [21][128] floats, column = row
    unsigned x_lo, h_lo, w0_lo, w1_lo, wo_lo, wob_lo;   // descriptor low words (tc16::desc_lo)
    unsigned mbar_saddr, cnt_saddr, full_saddr, tmem_d, tmem_row;
    unsigned x_row, h_row;       // AT: this thread's lane of the X / H operands in tensor memory
    volatile int* stamp;
    int row, n_warps;
    unsigned parity, arrivals;
    int step_id;
};

// The MMAs of one layer of one tile (one elected lane).  layer 0: X . W0^T (K = 48, bias in column 36); layer 1: H . W1^T + b1
// (bias: X[:, 32:48] . W0img[:, 48:64]^T); layer 2: H . WO^T + bo (N = 16; bias: X[:, 32:48] . WOB[:, 32:48]^T).
// AT: the A operands (X, H) live in tensor memory -- x_lo / h_lo are then TMEM addresses (lane 0, first column of the operand) and a
// K slice of 16 halves is 8 columns further on.
template <bool AT>
__device__ __forceinline__ void issue_layer16(int layer, unsigned tmem_d, unsigned x_lo, unsigned h_lo, unsigned w0_lo, unsigned w1_lo,
                                              unsigned wo_lo, unsigned wob_lo, unsigned mbar_saddr) {
    auto mma = [&](unsigned a, int ka, unsigned b_lo, unsigned id, unsigned acc) {
        if constexpr (AT) mma_f16_ts(tmem_d, a + 8u * ka, b_lo, id, acc);
        else mma_f16(tmem_d, a + 2u * ka, b_lo, id, acc);
    };
    if (layer == 0) {
        constexpr unsigned id = idesc_f16(TILE, HID);
#pragma unroll
        for (int k = 0; k < X_K / 16; ++k) mma(x_lo, k, w0_lo + 2 * k, id, k > 0 ? 1u : 0u);
    } else if (layer == 1) {
        constexpr unsigned id = idesc_f16(TILE, HID);
#pragma unroll
        for (int k = 0; k < HID / 16; ++k) mma(h_lo, k, w1_lo + 2 * k, id, k > 0 ? 1u : 0u);
        mma(x_lo, 2, w0_lo + 6, id, 1u);
    } else {
        constexpr unsigned id = idesc_f16(TILE, 16);
#pragma unroll
        for (int k = 0; k < HID / 16; ++k) mma(h_lo, k, wo_lo + 2 * k, id, k > 0 ? 1u : 0u);
        mma(x_lo, 2, wob_lo + 4, id, 1u);
    }
    umma::commit(mbar_saddr);
}

// "My rows of the operand tile are written; wake me when the accumulator is ready."
//   ISS  (dedicated issuer warps): proxy fence, warp converges, lane 0 arrives on the tile's `full` mbarrier -- the issuer warp
//        that sleeps on it issues the MMAs;
//   !ISS (16-warp CTAs, no room for issuer warps): lane 0 bumps the tile's arrival counter and the warp that arrives last issues.
template <bool ISS, bool AT>
__device__ __forceinline__ void tile_sync16(Tile16& c, int layer, int sid) {
    TC16_STAMP(layer);
    if constexpr (AT) tmem_st_wait();      // the operand rows went to tensor memory: no generic -> async proxy fence to pay
    if constexpr (ISS) {
        if constexpr (!AT) umma::fence_async_smem();
        umma::fence_before();
        __syncwarp();
        if ((threadIdx.x & 31) == 0) mbar_arrive(c.full_saddr);
    } else {
        c.arrivals += (unsigned)c.n_warps;
        if (const int last = tile_arrive(c.cnt_saddr, c.arrivals, layer == 0 ? c.stamp : nullptr, sid)) {
            umma::fence_after();
            if (elect_one()) {
                if (last == 1) issue_layer16<AT>(layer, c.tmem_d, c.x_lo, c.h_lo, c.w0_lo, c.w1_lo, c.wo_lo, c.wob_lo, c.mbar_saddr);
                else mbar_arrive(c.mbar_saddr);
            }
            __syncwarp();
            TC16_STAMP(6 + layer);
        }
    }
    mbar_wait_or_trap(c.mbar_saddr, c.parity);
    TC16_STAMP(3 + layer);
    c.parity ^= 1u;
}

// One policy forward for the tile: X row <- observation, three GEMMs, act[7] out.  Collective over the tile's warps.
// Returns false (without running the MLP) once no episode of the tile is still running.
template <bool ISS, bool AT>
__device__ __forceinline__ bool mlp16(Tile16& c, const unsigned* w, float* act, bool running) {
    const int sid = ++c.step_id;
    if (__any_sync(0xffffffffu, running) && (threadIdx.x & 31) == 0) *c.stamp = sid;
    // ---- layer 1: X = [obs36 | 1 | 0 ...]; columns 40..47 stay zero from the prologue
    if constexpr (AT) {
        tmem_st8(c.x_row, w);
        tmem_st8(c.x_row + 8u, w + 8);
        tmem_st4(c.x_row + 16u, w[16], w[17], 0x00003C00u, 0u);
    } else {
        st_chunk(c.X, c.row, 0, w[0], w[1], w[2], w[3]);
        st_chunk(c.X, c.row, 1, w[4], w[5], w[6], w[7]);
        st_chunk(c.X, c.row, 2, w[8], w[9], w[10], w[11]);
        st_chunk(c.X, c.row, 3, w[12], w[13], w[14], w[15]);
        st_chunk(c.X, c.row, 4, w[16], w[17], 0x00003C00u, 0u);
    }
    tile_sync16<ISS, AT>(c, 0, sid);
    if (*c.stamp != sid) return false;
    umma::fence_after();
    if constexpr (AT) epilogue_tanh_tmem(c.tmem_row, c.h_row);
    else epilogue_tanh(c.tmem_row, c.H, c.row);
    // ---- layer 2
    tile_sync16<ISS, AT>(c, 1, sid);
    umma::fence_after();
    if constexpr (AT) epilogue_tanh_tmem(c.tmem_row, c.h_row);
    else epilogue_tanh(c.tmem_row, c.H, c.row);
    // ---- layer 3 (N = 16: 7 action means + zero rows)
    tile_sync16<ISS, AT>(c, 2, sid);
    umma::fence_after();
    {
        float o[8];
        tmem_ld8(c.tmem_row, o);
#pragma unroll
        for (int i = 0; i < NJ; ++i) act[i] = clampf(o[i], -1.0f, 1.0f);
    }
    return true;
}

// ---- issuer warps (ISS mode): warp `iw` (0 / 1) serves tiles 2 iw and 2 iw + 1 of the CTA -------------------------------------
struct IssTile {
    unsigned x_lo, h_lo, tmem_d, full_saddr, mbar_saddr;
    volatile int* stamp;
    unsigned parity;
    int sid, layer, tile;
    bool exists, live;
};

// Serve one tile if its operands are ready.  Sleeps at most ~hint_ns on the tile's `full` mbarrier.
template <bool AT>
__device__ __forceinline__ void issuer_poll(IssTile& t, unsigned w0_lo, unsigned w1_lo, unsigned wo_lo, unsigned wob_lo, unsigned hint_ns) {
    if (!(hint_ns ? mbar_try_wait_hint(t.full_saddr, t.parity, hint_ns) : mbar_test_wait(t.full_saddr, t.parity))) return;
    t.parity ^= 1u;
    umma::fence_after();
    bool go = true;
    if (t.layer == 0) {
        t.sid += 1;
        go = (*t.stamp == t.sid);
    }
#ifdef KIN_TC16_TRACE
    if (blockIdx.x == 0 && t.sid >= 10 && t.sid < 18 && (threadIdx.x & 31) == 0) kin_tc16_trace_buf[t.sid - 10][4 * t.tile][9 + t.layer] = clock64();
#endif
    if (elect_one()) {
        if (go) issue_layer16<AT>(t.layer, t.tmem_d, t.x_lo, t.h_lo, w0_lo, w1_lo, wo_lo, wob_lo, t.mbar_saddr);
        else mbar_arrive(t.mbar_saddr);
#ifdef KIN_TC16_TRACE
        if (blockIdx.x == 0 && t.sid >= 10 && t.sid < 18) kin_tc16_trace_buf[t.sid - 10][4 * t.tile][6 + t.layer] = clock64();
#endif
    }
    __syncwarp();
    if (!go) t.live = false;
    else t.layer = t.layer == 2 ? 0 : t.layer + 1;
}

__device__ unsigned kin_tc16_poll_hint = 32u;   // experiment knob (KIN_TC16_POLL_HINT): 0 = non-blocking test_wait, else nap length in ns

// one phase (approach or finisher): until both tiles have reported "nobody running"
template <bool AT>
__device__ __forceinline__ void issuer_phase(IssTile& a, IssTile& b, unsigned w0_lo, unsigned w1_lo, unsigned wo_lo, unsigned wob_lo) {
    a.live = a.exists;
    b.live = b.exists;
    a.layer = b.layer = 0;
    unsigned spins = 0u;
    while (a.live || b.live) {
        const unsigned hint = (a.live && b.live) ? kin_tc16_poll_hint : 1000u;   // two tiles to watch: probe each in turn
        if (a.live) issuer_poll<AT>(a, w0_lo, w1_lo, wo_lo, wob_lo, hint);
        if (b.live) issuer_poll<AT>(b, w0_lo, w1_lo, wo_lo, wob_lo, hint);
        if (++spins > (1u << 28)) __trap();   // watchdog: a protocol bug must fail the launch, not hang the GPU
    }
}

__device__ __forceinline__ bool ready_pred16(float pos_thr, float ori_thr, float a_thr, float dq_thr, float pos, float ori, float an, float dqn) {
    return pos_thr > 0.0f && ori_thr > 0.0f && pos <= pos_thr && ori <= ori_thr && (a_thr <= 0.0f || an <= a_thr) && (dq_thr <= 0.0f || dqn <= dq_thr);
}

// ISS: the CTA's last two warps are issuer warps (<= 14 env warps, the balanced one-wave shape): blockDim.x = 32 (env warps + 2)
// AT: the activations (X, H) are A operands in TENSOR MEMORY (tcgen05.st from the epilogue, tcgen05.mma with a TMEM A operand) instead of
// swizzled shared-memory images: 128 TMEM columns per tile (64 accumulator | 32 H | 24 X)
template <int FAST, bool ISS, bool AT>
__global__ void __launch_bounds__(MAX_THREADS, 1)
kin_rollout_tc16_kernel(const __grid_constant__ KinEnvParams PA, const __grid_constant__ KinEnvParams PF, DevPolicy pol_a, DevPolicy pol_f,
                        int has_finisher, const float* __restrict__ iq, const float* __restrict__ idq, const float* __restrict__ ipa,
                        const float* __restrict__ gq, const float* __restrict__ gpose, int n, int stride, int confirm,
                        uint32_t* __restrict__ result, unsigned long long* __restrict__ env_steps) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char* base = smem_raw + ((1024u - (umma::smem_u32(smem_raw) & 1023u)) & 1023u);   // stays in the shared address space
    Smem& S = *reinterpret_cast<Smem*>(base);
    const int tid = threadIdx.x;
    const int warp = tid >> 5;
    const int env_threads = (int)blockDim.x - (ISS ? 64 : 0);
    const int n_tiles_cta = (env_threads + TILE - 1) / TILE;
    unsigned char* tiles = base + ((sizeof(Smem) + 1023) / 1024) * 1024;
    float* snaps = reinterpret_cast<float*>(tiles + (size_t)n_tiles_cta * 2 * TILE_BYTES);

    Tile16 c;
    const int tile = tid >> 7;
    c.row = tid & (TILE - 1);
    c.n_warps = (min(TILE, env_threads - tile * TILE) + 31) >> 5;
    c.X = tiles + (size_t)tile * 2 * TILE_BYTES;
    c.H = c.X + TILE_BYTES;
    c.snap = snaps + (size_t)tile * SNAP_FLOATS * TILE + c.row;
    c.parity = 0u;
    c.arrivals = 0u;
    c.step_id = 0;
    c.stamp = &S.run_stamp[tile];

    constexpr unsigned TCOLS = AT ? 128u : 64u;      // TMEM columns per tile
    const unsigned tmem_cols = n_tiles_cta == 1 ? TCOLS : (n_tiles_cta == 2 ? 2u * TCOLS : 4u * TCOLS);
    if (warp == 0) umma::tmem_alloc(umma::smem_u32(&S.tmem_base), tmem_cols);
    if (tid == 0) {
#pragma unroll
        for (int i = 0; i < MAX_TILES; ++i) {
            umma::mbar_init(umma::smem_u32(&S.mbar[i]), 1);
            umma::mbar_init(umma::smem_u32(&S.full[i]), (unsigned)max(1, (min(TILE, env_threads - i * TILE) + 31) >> 5));
            S.arrive[i] = 0u;
            S.run_stamp[i] = 0;
        }
        umma::fence_mbar_init();
    }
    load_weights(S, pol_a, KIN_MODE_APPROACH, tid, (int)blockDim.x);
    const bool env_thread = tid < env_threads;
    // this thread's rows of the X / H images start as zeros (the K padding of X is never written again)
    if (env_thread) {
#pragma unroll
        for (int ch = 0; ch < 8; ++ch) {
            st_chunk(c.X, c.row, ch, 0u, 0u, 0u, 0u);
            st_chunk(c.H, c.row, ch, 0u, 0u, 0u, 0u);
        }
    }
    if (env_thread && c.n_warps < 4) {   // partial tile: the rows nobody owns still feed the M = 128 GEMMs -- keep them finite
        for (int r = c.n_warps * 32 + c.row; r < TILE; r += c.n_warps * 32)
#pragma unroll
            for (int ch = 0; ch < 8; ++ch) {
                st_chunk(c.X, r, ch, 0u, 0u, 0u, 0u);
                st_chunk(c.H, r, ch, 0u, 0u, 0u, 0u);
            }
    }
    umma::fence_async_smem();
    umma::fence_before();
    __syncthreads();
    umma::fence_after();
    const unsigned tmem_base = S.tmem_base;
    c.x_lo = desc_lo(umma::smem_u32(c.X));
    c.h_lo = desc_lo(umma::smem_u32(c.H));
    c.w0_lo = desc_lo(umma::smem_u32(S.W0));
    c.w1_lo = desc_lo(umma::smem_u32(S.W1));
    c.wo_lo = desc_lo(umma::smem_u32(S.WO));
    c.wob_lo = desc_lo(umma::smem_u32(S.WOB));
    c.mbar_saddr = umma::smem_u32(&S.mbar[tile]);
    c.cnt_saddr = umma::smem_u32(&S.arrive[tile]);
    c.full_saddr = umma::smem_u32(&S.full[tile]);
    c.tmem_d = tmem_base + tile * TCOLS;                                      // lane 0, this tile's columns
    c.tmem_row = c.tmem_d + ((unsigned)((warp & 3) * 32) << 16);              // this warp's 32-lane slice
    c.h_row = c.tmem_row + 64u;
    c.x_row = c.tmem_row + 96u;
    if constexpr (AT) {
        c.x_lo = c.tmem_d + 96u;
        c.h_lo = c.tmem_d + 64u;
        if (env_thread) {      // K padding of X (columns 40..47 = words 20..23) and the spare words start as zeros
            tmem_st4(c.x_row + 20u, 0u, 0u, 0u, 0u);
            tmem_st4(c.x_row + 24u, 0u, 0u, 0u, 0u);
            tmem_st4(c.x_row + 28u, 0u, 0u, 0u, 0u);
            tmem_st_wait();
        }
    }

    if constexpr (ISS) {
        if (!env_thread) {   // ---- issuer warp: serve two tiles through both phases, keep step with the CTA barriers
            const int iw = (tid - env_threads) >> 5;
            IssTile it[2];
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int t = 2 * iw + j;
                it[j].exists = t < n_tiles_cta;
                it[j].tile = t;
                unsigned char* X = tiles + (size_t)t * 2 * TILE_BYTES;
                it[j].x_lo = desc_lo(umma::smem_u32(X));
                it[j].h_lo = desc_lo(umma::smem_u32(X + TILE_BYTES));
                it[j].tmem_d = tmem_base + t * TCOLS;
                if constexpr (AT) { it[j].x_lo = it[j].tmem_d + 96u; it[j].h_lo = it[j].tmem_d + 64u; }
                it[j].full_saddr = umma::smem_u32(&S.full[t]);
                it[j].mbar_saddr = umma::smem_u32(&S.mbar[t]);
                it[j].stamp = &S.run_stamp[t];
                it[j].parity = 0u;
                it[j].sid = 0;
            }
            issuer_phase<AT>(it[0], it[1], c.w0_lo, c.w1_lo, c.wo_lo, c.wob_lo);
            __syncthreads();
            if (has_finisher) {
                load_weights(S, pol_f, KIN_MODE_DOCK, tid, (int)blockDim.x);
                umma::fence_async_smem();
                __syncthreads();
                issuer_phase<AT>(it[0], it[1], c.w0_lo, c.w1_lo, c.wo_lo, c.wob_lo);
            }
            umma::fence_before();
            __syncthreads();
            return;
        }
    }

    const int ep = blockIdx.x * env_threads + tid;
    const bool active = ep < n;
    const int epc = active ? ep : n - 1;

    EnvRegs s;
    s.flags = 0u;
    float goal_q[NJ];
    {
        float r_iq[NJ], r_idq[NJ], r_ipa[NJ], r_gq[NJ], r_gp[6];
#pragma unroll
        for (int k = 0; k < NJ; ++k) {
            r_iq[k] = iq[(size_t)epc * NJ + k];
            r_idq[k] = idq ? idq[(size_t)epc * NJ + k] : 0.0f;
            r_ipa[k] = ipa ? ipa[(size_t)epc * NJ + k] : 0.0f;
            r_gq[k] = gq ? gq[(size_t)epc * NJ + k] : 0.0f;
        }
        if (gpose) {
#pragma unroll
            for (int k = 0; k < 6; ++k) r_gp[k] = gpose[(size_t)epc * 6 + k];
        }
        reset_core(PA, s, KIN_MODE_APPROACH, r_iq, r_idq, r_ipa, r_gq, gpose ? r_gp : nullptr, goal_q);
    }

    // ---- approach phase ------------------------------------------------------------------------------
    float min_pos = s.entry[0], min_ori = s.entry[1];
    int steps = 0, streak = 0, max_streak = 0, first_ready = -1;
    bool ready_hit = false, have_snap = false;
    int snap_step = -1;
    float last_an = 0.0f, last_dqn = 0.0f;
    StepOut so;
    prime_step_out(PA, s, so);
    bool running = active;
    while (true) {
        unsigned w[X_DYN / 2];
        float act[NJ];
        obs_pack(PA, s, so, w);
        if (!mlp16<ISS, AT>(c, w, act, running)) break;
        if (running) {
            step_core<KIN_MODE_APPROACH, false, FAST>(PA, s, act, so, nullptr);
            const float an = so.action_l2;
            steps += 1;
            min_pos = fminf(min_pos, so.pos);
            min_ori = fminf(min_ori, so.ori);
            if (ready_pred16(PA.ar_dock_coarse_ready_pos_threshold_m, PA.ar_dock_coarse_ready_ori_threshold_rad,
                             PA.ar_dock_coarse_ready_action_threshold, PA.ar_dock_coarse_ready_dq_threshold, so.pos, so.ori, an, so.dq_l2)) {
                ready_hit = true;
                if (first_ready < 0) first_ready = steps;
                streak += 1;
            } else {
                streak = 0;
            }
            max_streak = max(max_streak, streak);
            if (!have_snap && streak >= confirm) {
                have_snap = true;
                snap_step = steps;
#pragma unroll
                for (int i = 0; i < NJ; ++i) {
                    c.snap[i * TILE] = s.q[i];
                    c.snap[(NJ + i) * TILE] = s.dq[i];
                    c.snap[(2 * NJ + i) * TILE] = s.pa[i];
                }
            }
            last_an = an;
            last_dqn = so.dq_l2;
            running = !(so.done & (KIN_DONE_TERMINATED | KIN_DONE_TRUNCATED));
        }
    }
    if (active) {   // approach-phase motion metrics (eval_workspace_expansion.py:47-66 classifies failures with them)
        result[(size_t)KIN_RES_APPROACH_ACTION * stride + ep] = __float_as_uint(last_an);
        result[(size_t)KIN_RES_APPROACH_DQ * stride + ep] = __float_as_uint(last_dqn);
    }
    const int approach_steps = steps;
    const bool approach_success = (so.done & KIN_DONE_SUCCESS) != 0;
    const float approach_pos = so.pos, approach_ori = so.ori;
    const bool final_ready = ready_pred16(PA.ar_finisher_ready_pos_threshold_m, PA.ar_finisher_ready_ori_threshold_rad,
                                          PA.ar_finisher_ready_action_threshold, PA.ar_finisher_ready_dq_threshold, so.pos, so.ori, last_an, last_dqn);
    const int handoff_kind = final_ready ? 2 : (have_snap ? 1 : 0);
    const int handoff_step = final_ready ? steps : (have_snap ? snap_step : -1);
    bool success = approach_success;
    float final_pos = so.pos, final_ori = so.ori, final_an = last_an, final_dqn = last_dqn;
    int finisher_steps = 0;

    // ---- finisher phase ------------------------------------------------------------------------------
    __syncthreads();   // every tile is out of the approach loop (no MMA in flight reads the approach weights any more)
    if (has_finisher) {
        load_weights(S, pol_f, KIN_MODE_DOCK, tid, (int)blockDim.x);
        umma::fence_async_smem();
        __syncthreads();
        running = active && handoff_kind != 0;
        if (running) {
            float r_iq[NJ], r_idq[NJ], r_ipa[NJ], gq_out[NJ], r_gp[6];
#pragma unroll
            for (int i = 0; i < NJ; ++i) {
                r_iq[i] = (handoff_kind == 2) ? s.q[i] : c.snap[i * TILE];
                r_idq[i] = (handoff_kind == 2) ? s.dq[i] : c.snap[(NJ + i) * TILE];
                r_ipa[i] = (handoff_kind == 2) ? s.pa[i] : c.snap[(2 * NJ + i) * TILE];
            }
#pragma unroll
            for (int k = 0; k < 6; ++k) r_gp[k] = s.goal[k];
            reset_core(PF, s, KIN_MODE_DOCK, r_iq, r_idq, r_ipa, goal_q, r_gp, gq_out);
        }
        steps = 0;
        prime_step_out(PF, s, so);
        if (!running) { so.pos = final_pos; so.ori = final_ori; }
        while (true) {
            unsigned w[X_DYN / 2];
            float act[NJ];
            obs_pack(PF, s, so, w);
            if (!mlp16<ISS, AT>(c, w, act, running)) break;
            if (running) {
                float an2 = 0.0f;   // the policy's own action (the step clips it to the dock limit before it reports action_l2)
#pragma unroll
                for (int i = 0; i < NJ; ++i) an2 = fmaf(act[i], act[i], an2);
                step_core<KIN_MODE_DOCK, false, FAST>(PF, s, act, so, nullptr);
                steps += 1;
                final_an = sqrt_approx(an2);
                running = !(so.done & (KIN_DONE_TERMINATED | KIN_DONE_TRUNCATED));
            }
        }
        if (active && handoff_kind != 0) {
            finisher_steps = steps;
            success = (so.done & KIN_DONE_SUCCESS) != 0;
            final_pos = so.pos; final_ori = so.ori; final_dqn = so.dq_l2;
        }
    }

    if (active) {
        auto put_u = [&](int row, uint32_t v) { result[(size_t)row * stride + ep] = v; };
        auto put_f = [&](int row, float v) { result[(size_t)row * stride + ep] = __float_as_uint(v); };
        put_u(KIN_RES_SUCCESS, success ? 1u : 0u);
        put_u(KIN_RES_FLAGS, (approach_success ? 1u : 0u) | ((ready_hit || final_ready) ? 2u : 0u) |
                                 ((max_streak >= confirm || final_ready) ? 4u : 0u) | (final_ready ? 8u : 0u) | ((uint32_t)handoff_kind << 4));
        put_u(KIN_RES_HANDOFF_STEP, (uint32_t)handoff_step);
        put_u(KIN_RES_FIRST_READY_STEP, (uint32_t)first_ready);
        put_u(KIN_RES_MAX_READY_STREAK, (uint32_t)max_streak);
        put_u(KIN_RES_STEPS, (uint32_t)approach_steps | ((uint32_t)finisher_steps << 16));
        put_f(KIN_RES_FINAL_POS, final_pos); put_f(KIN_RES_FINAL_ORI, final_ori);
        put_f(KIN_RES_APPROACH_POS, approach_pos); put_f(KIN_RES_APPROACH_ORI, approach_ori);
        put_f(KIN_RES_MIN_POS, min_pos); put_f(KIN_RES_MIN_ORI, min_ori);
        put_f(KIN_RES_FINAL_ACTION, final_an); put_f(KIN_RES_FINAL_DQ, final_dqn);
#pragma unroll
        for (int i = 0; i < NJ; ++i) put_f(KIN_RES_FINAL_Q + i, s.q[i]);
    }
    if (env_steps) {
        unsigned long long mine = active ? (unsigned long long)(approach_steps + finisher_steps) : 0ull;
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, off);
        if ((tid & 31) == 0 && mine) atomicAdd(env_steps, mine);
    }
    umma::fence_before();
    __syncthreads();
    if (warp == 0) umma::tmem_dealloc(tmem_base, tmem_cols);
}

}  // namespace kin

using namespace kin;

#ifdef KIN_TC16_TRACE
extern "C" int kin_debug_tc16_trace(long long* out) {
    return cudaMemcpyFromSymbol(out, kin_tc16_trace_buf, sizeof(kin_tc16_trace_buf)) == cudaSuccess ? KIN_OK : KIN_ERR_INVALID_ARG;
}
#endif

int kin_rollout_tc16_launch(const KinHandle* ha, const KinHandle* hf, const KinPolicyWeights* pa, const KinPolicyWeights* pf,
                            const float* iq, const float* idq, const float* ipa, const float* gq, const float* gpose, int n, int stride,
                            int confirm, uint32_t* result, unsigned long long* env_steps, cudaStream_t st) {
    using Kernel = void (*)(KinEnvParams, KinEnvParams, tc16::DevPolicy, tc16::DevPolicy, int, const float*, const float*, const float*, const float*,
                            const float*, int, int, int, uint32_t*, unsigned long long*);
    static const Kernel kernels[2][2][2] = {{{kin_rollout_tc16_kernel<1, false, false>, kin_rollout_tc16_kernel<1, false, true>},
                                             {kin_rollout_tc16_kernel<1, true, false>, kin_rollout_tc16_kernel<1, true, true>}},
                                            {{kin_rollout_tc16_kernel<2, false, false>, kin_rollout_tc16_kernel<2, false, true>},
                                             {kin_rollout_tc16_kernel<2, true, false>, kin_rollout_tc16_kernel<2, true, true>}}};
    static bool attr_set[KIN_MAX_DEVICES] = {};
    const int dev_slot = kin_device_slot();
    if (!attr_set[dev_slot]) {
        for (int i = 0; i < 8; ++i) {
            cudaError_t e = cudaFuncSetAttribute(kernels[i >> 2][(i >> 1) & 1][i & 1], cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc16::smem_bytes(tc16::MAX_TILES));
            if (e != cudaSuccess) return kin_fail_cuda(e, "kin_rollout_approach_finisher(tc16): smem attribute");
        }
        attr_set[dev_slot] = true;
    }
    // KIN_TC16_EXACT_SINCOS=1: polynomial sine / cosine in the FK instead of the MUFU units (the default: 6 % faster, same flip count)
    static const bool exact_sincos = kin_env_flag("KIN_TC16_EXACT_SINCOS");
    static const bool no_issuer = kin_env_flag("KIN_TC16_NO_ISSUER_WARPS");
    static const bool tmem_a = !kin_env_flag("KIN_TC16_SMEM_A");       // default: activations as TMEM A operands (+5 %, bitwise the same results)
    static bool hint_set = false;
    if (!hint_set) {
        if (const char* v = getenv("KIN_TC16_POLL_HINT")) { const unsigned h = (unsigned)atoi(v); cudaMemcpyToSymbol(kin_tc16_poll_hint, &h, sizeof(h)); }
        hint_set = true;
    }
    tc16::DevPolicy da{pa->pi_w0, pa->pi_b0, pa->pi_w1, pa->pi_b1, pa->act_w, pa->act_b};
    tc16::DevPolicy df = pf ? tc16::DevPolicy{pf->pi_w0, pf->pi_b0, pf->pi_w1, pf->pi_b1, pf->act_w, pf->act_b} : da;
    const KinEnvParams& PF = hf ? hf->params : ha->params;
    static int n_sm = 0;
    if (n_sm == 0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n_sm <= 0) n_sm = 148;
    }
    // one wave: spread the warps evenly over the SMs; several waves: full 16-warp CTAs, one per SM.  Up to 14 env warps leave room
    // (registers: 16 warps x 128) for two issuer warps, which then sit on the two schedulers that carry one env warp fewer.
    const int warps = (n + 31) / 32;
    int w_per_cta = (warps + n_sm - 1) / n_sm;
    if (w_per_cta > 16) w_per_cta = 16;
    if (const char* v = getenv("KIN_TC_WARPS")) { const int f = atoi(v); if (f >= 1 && f <= 16) w_per_cta = f; }
    const bool iss = w_per_cta <= 14 && !no_issuer;
    const int env_threads = 32 * w_per_cta;
    const int threads = env_threads + (iss ? 64 : 0);
    const size_t smem = tc16::smem_bytes((env_threads + tc16::TILE - 1) / tc16::TILE);
    kernels[exact_sincos ? 0 : 1][iss ? 1 : 0][tmem_a ? 1 : 0]<<<(n + env_threads - 1) / env_threads, threads, smem, st>>>(
        ha->params, PF, da, df, (hf && pf) ? 1 : 0, iq, idq, ipa, gq, gpose, n, stride, confirm, result, env_steps);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KIN_OK : kin_fail_cuda(e, "kin_rollout_approach_finisher(tc16)");
}
