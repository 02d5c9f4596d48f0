// kin_tc16.cuh -- tcgen05 kind::f16 (fp16 operands, fp32 accumulation in TMEM) building blocks of the policy-in-the-loop
// rollout: operand images, the packed-half epilogue, and a barrier-free "last arriver issues" hand-off between the threads
// that write an operand tile and the one lane that issues the MMAs on it.
//
// Why fp16 operands (not TF32, not bf16): observations, tanh activations and the trained weights all live in [-8, 8] with
// magnitudes >> 6e-5, where fp16 has the SAME 11-bit significand as TF32 -- the products entering the fp32 accumulator are the
// ones the TF32 kernel fed it -- while an operand row is half as many bytes (one 128-byte swizzle row holds K = 64), two
// elements are rounded by ONE cvt.rn.f16x2.f32 (the hidden activations: tanh.approx.f32 on the fp32 accumulator, then that
// convert), clamps are packed min/max, and one MMA consumes K = 16.  Per env-step and thread that is ~300 instructions for the
// three layers instead of ~530.
//
// Operand images are [rows][64 halves] = 128-byte rows, SWIZZLE_128B, K-major (csrc/kin_umma.cuh has the layout helpers).
#pragma once

#include <cuda_fp16.h>

#include "kin_internal.h"
#include "kin_state.cuh"
#include "kin_umma.cuh"

namespace kin {
namespace tc16 {

using namespace umma;

constexpr int TILE = 128;                  // episodes per tile == UMMA M == TMEM lanes
constexpr int MAX_TILES = 4;               // tiles per CTA (the last one may be partial: 1..4 warps)
constexpr int MAX_THREADS = TILE * MAX_TILES;
constexpr int HID = 64;
constexpr int X_DYN = 36;                  // observation columns that change from step to step
constexpr int X_ONE = 36;                  // column holding the constant 1 (bias carrier); 37..47 are zero
constexpr int X_K = 48;                    // layer-1 reduction width (3 MMAs of K = 16)
constexpr int B1_COL = 52;                 // W0 image columns 48..63 = layer-2 bias slice: X[:, 32:48] . W0img[:, 48:64]^T = b1
constexpr int TILE_BYTES = TILE * 128;     // one operand image of a tile: 16 KB
constexpr int SNAP_FLOATS = 3 * KIN_NJ;    // first-confirmed handoff snapshot (q, dq, prev_action) per episode, kept in smem

struct Smem {
    alignas(1024) unsigned char W0[HID * 128];   // [n][k]: k < 36 dynamic obs columns | 36 folded bias | 37..47 zero | 52 = b1[n]
    alignas(1024) unsigned char W1[HID * 128];   // [n][k]
    alignas(1024) unsigned char WO[16 * 128];    // rows 0..6 action head, rows 7..15 zero (N = 16)
    alignas(1024) unsigned char WOB[16 * 128];   // column 36 = action bias (multiplies the X tile's constant-one column)
    unsigned long long mbar[MAX_TILES];          // "accumulator ready", one per tile
    unsigned long long full[MAX_TILES];          // issuer-warp mode: "operand tile written" (one arrival per warp of the tile)
    unsigned arrive[MAX_TILES];                  // monotonically increasing arrival counters ("operand tile written")
    int run_stamp[MAX_TILES];                    // id of the last step in which some episode of the tile was still running
    unsigned tmem_base;
    // followed (1024-aligned) by n_tiles x [X image | H image] and n_tiles x snapshot[21][128] floats, sized at launch
};

struct DevPolicy {
    const float *w0, *b0, *w1, *b1, *wo, *bo;
};

__host__ __device__ constexpr size_t smem_bytes(int n_tiles) {
    return ((sizeof(Smem) + 1023) / 1024) * 1024 + (size_t)n_tiles * (2 * TILE_BYTES + SNAP_FLOATS * TILE * sizeof(float)) + 1024;
}

// instruction descriptor, kind::f16: D fp32 (bit 4), A / B fp16 (format 0), both K-major, N >> 3 at bit 17, M >> 4 at bit 24
__host__ __device__ constexpr unsigned idesc_f16(int M, int N) { return (1u << 4) | ((unsigned)(N >> 3) << 17) | ((unsigned)(M >> 4) << 24); }

// {hi, lo} -> packed halves, round to nearest even (lo = lower address = lower column)
__device__ __forceinline__ unsigned pack_h2(float lo, float hi) {
    unsigned r;
    asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
// both halves clamped to [-1, 1]
__device__ __forceinline__ unsigned clamp1_h2(unsigned x) {
    unsigned y;
    asm("{\n\t.reg .b32 t;\n\tmax.f16x2 t, %1, %2;\n\tmin.f16x2 %0, t, %3;\n\t}" : "=r"(y) : "r"(x), "r"(0xBC00BC00u), "r"(0x3C003C00u));
    return y;
}
__device__ __forceinline__ void st_chunk(unsigned char* img, int row, int chunk, unsigned a, unsigned b, unsigned c, unsigned d) {
    *reinterpret_cast<uint4*>(img + umma::sw_chunk(row, chunk)) = make_uint4(a, b, c, d);
}

// observation column -> column of the [*, 56] layer-1 weight (SB3's alphabetical flattening, kin_core.cuh::build_obs_from):
// dq 0:7 | goal_ori_err 7:10 | goal_pos_err 10:13 | joint_limit_margin 13:20 | prev_action 30:37 | progress 37:39 | q 40:47.
// The other 20 columns are constants of the path (mode_flag one-hot, task_type = [1, 0, 0], the waypoint blocks and progress[2] = 0)
// and are folded into the layer-1 bias when the weights are staged.
__device__ __forceinline__ int dyn_col(int k) { return k < 20 ? k : (k < 27 ? k + 10 : (k < 29 ? k + 10 : k + 11)); }

// Observation of the current state as 18 packed fp16 pairs in X-image column order:
// dq 0:7 | goal_ori_err 7:10 | goal_pos_err 10:13 | joint_limit_margin 13:20 | prev_action 20:27 | progress 27:29 | q 29:36
// (observation_builder.py:29-94; values and clamps as kin_core.cuh::build_obs_from).
__device__ __forceinline__ void obs_pack(const KinEnvParams& P, const EnvRegs& s, const StepOut& so, unsigned* w) {
    float v[X_DYN];
#pragma unroll
    for (int i = 0; i < NJ; ++i) {
        v[i] = s.dq[i] * P.k_inv_delta_limit[i];
        v[13 + i] = so.margin[i];
        v[20 + i] = s.pa[i];
        v[29 + i] = so.qn[i];
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        v[7 + k] = so.oe[k] * P.k_inv_ori_err_scale;
        v[10 + k] = so.pe[k] * P.k_inv_pos_err_scale;
    }
    v[27] = (float)s.step * P.k_inv_episode_length;
    v[28] = (float)s.dwell * P.k_inv_dwell_steps_target;
#pragma unroll
    for (int i = 0; i < X_DYN / 2; ++i) w[i] = pack_h2(v[2 * i], v[2 * i + 1]);
    // margins (columns 14..19) and normalised q (30..35) are inside [0, 1] / [-1, 1] by construction (q is clipped to its limits
    // and kin_core.cuh::qnorm clamps the rounding above 1); everything else gets the reference's clip to [-1, 1] (progress is
    // non-negative, its clip to [0, 1] is the same upper bound)
#pragma unroll
    for (int i = 0; i < X_DYN / 2; ++i)
        if (!((i >= 7 && i <= 9) || i >= 15)) w[i] = clamp1_h2(w[i]);
}

// pose error, margins and normalised joint positions of a freshly reset state (what step_core<FAST> leaves behind after a step)
__device__ __forceinline__ void prime_step_out(const KinEnvParams& P, const EnvRegs& s, StepOut& so) {
    so.done = 0u;
    so.pos = s.entry[0];
    so.ori = s.entry[1];
    so.dq_l2 = 0.0f;
    pose_error(s.ee, s.goal, so.pe, so.oe);
#pragma unroll
    for (int i = 0; i < NJ; ++i) {
        so.qn[i] = qnorm(P, s.q[i], i);
        so.margin[i] = 1.0f - fabsf(so.qn[i]);
    }
}

// stage one policy's actor as fp16 B-operand images (all threads of the CTA); `mode` selects the mode_flag column
__device__ __forceinline__ void load_weights(Smem& S, const DevPolicy& p, int mode, int tid, int nthreads) {
    for (int i = tid; i < HID * 64; i += nthreads) {
        const int n = i >> 6, k = i & 63;
        float v0 = 0.0f;
        if (k < X_DYN) v0 = __ldg(p.w0 + n * KIN_OBS_DIM + dyn_col(k));
        else if (k == X_ONE) v0 = __ldg(p.b0 + n) + __ldg(p.w0 + n * KIN_OBS_DIM + 20 + mode) + __ldg(p.w0 + n * KIN_OBS_DIM + 47);
        else if (k == B1_COL) v0 = __ldg(p.b1 + n);
        *reinterpret_cast<__half*>(S.W0 + umma::sw_elem(n, k)) = __float2half_rn(v0);
        *reinterpret_cast<__half*>(S.W1 + umma::sw_elem(n, k)) = __float2half_rn(__ldg(p.w1 + n * HID + k));
    }
    for (int i = tid; i < 16 * 64; i += nthreads) {
        const int n = i >> 6, k = i & 63;
        *reinterpret_cast<__half*>(S.WO + umma::sw_elem(n, k)) = __float2half_rn(n < KIN_NJ ? __ldg(p.wo + n * HID + k) : 0.0f);
        *reinterpret_cast<__half*>(S.WOB + umma::sw_elem(n, k)) = __float2half_rn((n < KIN_NJ && k == X_ONE) ? __ldg(p.bo + n) : 0.0f);
    }
}

// Low word of a K-major SWIZZLE_128B descriptor (start >> 4 | LBO); the high word is the constant DESC_HI.  A K slice of 16
// halves is 32 bytes further along the row: + 2 in the low word.  Precomputed once per tile so the issue path is a handful of
// uniform adds instead of shift / mask chains per MMA.
constexpr unsigned DESC_HI = 64u | (1u << 14) | (2u << 29);      // SBO = 1024 B >> 4, version 1 (bit 46), SWIZZLE_128B (bits 61..63 = 2)
__device__ __forceinline__ unsigned desc_lo(unsigned saddr) { return ((saddr >> 4) & 0x3FFFu) | (1u << 16); }
__device__ __forceinline__ void mma_f16(unsigned tmem_d, unsigned a_lo, unsigned b_lo, unsigned idesc, unsigned accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "mov.b64 da, {%1, %5};\n\t"
        "mov.b64 db, {%2, %5};\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, p;\n\t}"
        ::"r"(tmem_d), "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(accumulate), "r"(DESC_HI) : "memory");
}
// the same MMA with the A operand in tensor memory (lane = row, each 32-bit column = two consecutive K halves): no shared-memory
// round trip and no generic -> async proxy fence for the activations
__device__ __forceinline__ void mma_f16_ts(unsigned tmem_d, unsigned a_taddr, unsigned b_lo, unsigned idesc, unsigned accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 db;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "mov.b64 db, {%2, %5};\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], db, %3, p;\n\t}"
        ::"r"(tmem_d), "r"(a_taddr), "r"(b_lo), "r"(idesc), "r"(accumulate), "r"(DESC_HI) : "memory");
}
// "My part of the operand tile is written": every lane makes its generic-proxy stores visible to the async proxy, the warp
// converges, lane 0 bumps the tile's counter.  Returns non-zero -- to the whole warp -- on the warp that arrived last;
// that warp issues the tile's MMAs, nobody blocks on a CTA barrier.  With `stamp` the last arriver also reports whether some
// episode of the tile stamped step `sid` as still running (1) or not (2); the stamps were stored before their writers' arrivals.
__device__ __forceinline__ int tile_arrive(unsigned cnt_saddr, unsigned target, const volatile int* stamp = nullptr, int sid = 0) {
    umma::fence_async_smem();
    umma::fence_before();
    __syncwarp();
    int last = 0;
    if ((threadIdx.x & 31) == 0) {
        unsigned old;
        // relaxed: shared-memory operations of one warp are performed in order, and the proxy fence above is what makes the stores
        // visible to the tensor core; an acq_rel atomic costs two MEMBAR.ALL.CTA on the critical path of every GEMM round trip
        asm volatile("atom.relaxed.cta.shared::cta.add.u32 %0, [%1], 1;" : "=r"(old) : "r"(cnt_saddr) : "memory");
        if (old + 1u == target) last = (stamp == nullptr || *stamp == sid) ? 1 : 2;
    }
    return __shfl_sync(0xffffffffu, last, 0);
}

// 16 accumulator columns -> tanh -> two 16-byte chunks (2 * ch2, 2 * ch2 + 1) of this thread's row of the H image
__device__ __forceinline__ void tanh_store16(const unsigned* r, unsigned char* H, int row, int ch2) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        unsigned w[4];
#pragma unroll
        for (int j = 0; j < 4; ++j)   // tanh.approx.f16x2 is two MUFU + a PRMT in SASS: f32 tanh then one packing convert is 3 instructions per pair, not 4
            w[j] = pack_h2(umma::tanh_fast(__uint_as_float(r[8 * h + 2 * j])), umma::tanh_fast(__uint_as_float(r[8 * h + 2 * j + 1])));
        st_chunk(H, row, 2 * ch2 + h, w[0], w[1], w[2], w[3]);
    }
}

// 16 accumulator columns -> tanh -> 8 packed words -> columns [8 * piece, 8 * piece + 8) of this thread's lane of the H operand in TMEM
__device__ __forceinline__ void tanh_store16_tmem(const unsigned* r, unsigned h_taddr, int piece) {
    unsigned w[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) w[j] = pack_h2(umma::tanh_fast(__uint_as_float(r[2 * j])), umma::tanh_fast(__uint_as_float(r[2 * j + 1])));
    tmem_st8(h_taddr + 8u * piece, w);
}
// the epilogue with the H operand in tensor memory
__device__ __forceinline__ void epilogue_tanh_tmem(unsigned tmem_row, unsigned h_taddr) {
    unsigned a[16], b[16];
    tmem_ld16_raw(tmem_row, a);
    tmem_wait16(a);
    tmem_ld16_raw(tmem_row + 16u, b);
    tanh_store16_tmem(a, h_taddr, 0);
    tmem_wait16(b);
    tmem_ld16_raw(tmem_row + 32u, a);
    tanh_store16_tmem(b, h_taddr, 1);
    tmem_wait16(a);
    tmem_ld16_raw(tmem_row + 48u, b);
    tanh_store16_tmem(a, h_taddr, 2);
    tmem_wait16(b);
    tanh_store16_tmem(b, h_taddr, 3);
}

// hidden-layer epilogue: this thread's 64 accumulator columns -> tanh -> fp16 -> its row of the H image, in four 16-column
// pieces; the TMEM load of piece k + 1 is in flight while piece k goes through the XU pipe (32 live registers, not 64)
__device__ __forceinline__ void epilogue_tanh(unsigned tmem_row, unsigned char* H, int row) {
    unsigned a[16], b[16];
    tmem_ld16_raw(tmem_row, a);
    tmem_wait16(a);
    tmem_ld16_raw(tmem_row + 16u, b);
    tanh_store16(a, H, row, 0);
    tmem_wait16(b);
    tmem_ld16_raw(tmem_row + 32u, a);
    tanh_store16(b, H, row, 1);
    tmem_wait16(a);
    tmem_ld16_raw(tmem_row + 48u, b);
    tanh_store16(a, H, row, 2);
    tmem_wait16(b);
    tanh_store16(b, H, row, 3);
}

}  // namespace tc16
}  // namespace kin
