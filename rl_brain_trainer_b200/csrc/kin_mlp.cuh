// kin_mlp.cuh -- the SB3 MultiInputPolicy actor/critic MLP (in -> tanh 64 -> tanh 64 -> out), fp32 FFMA variant.
//
// One thread per env.  Weights live in shared memory (row-major [out][in] exactly as policy.pth stores
// them) and are read as warp-uniform 128-bit loads (one LDS.128 feeds 4 FFMA); each thread's hidden
// activations go through a private column of a shared [64][BLOCK] scratch so the output loop can stay
// rolled (a full unroll of 64x56 FFMA would blow the instruction cache).  This is the strict-fp32 path
// used for parity runs; the tensor-core variant (tcgen05, TMEM accumulators) lives in kin_rollout_tc16.cu.
//
// Replaces `model.predict(obs, deterministic=True)` (eval/eval_three_stage.py:25-27; SURVEY F4).
#pragma once

#include <cuda_runtime.h>

#include "kin_b200.h"

namespace kin {

constexpr int HID = 64;
constexpr int ACT = KIN_NJ;

// smem image of one actor (or critic) network
template <int IN>
struct MlpSmem {
    static constexpr int W0 = 0;
    static constexpr int B0 = W0 + HID * IN;
    static constexpr int W1 = B0 + HID;
    static constexpr int B1 = W1 + HID * HID;
    static constexpr int WO = B1 + HID;            // [OUT][64], OUT <= 8 rows reserved
    static constexpr int BO = WO + 8 * HID;
    static constexpr int FLOATS = BO + 8;
};

template <int IN>
__device__ __forceinline__ void mlp_load_smem(float* s, const float* w0, const float* b0, const float* w1, const float* b1,
                                              const float* wo, const float* bo, int out_dim, int tid, int nthreads) {
    using L = MlpSmem<IN>;
    for (int i = tid; i < HID * IN; i += nthreads) s[L::W0 + i] = __ldg(w0 + i);
    for (int i = tid; i < HID * HID; i += nthreads) s[L::W1 + i] = __ldg(w1 + i);
    for (int i = tid; i < HID; i += nthreads) {
        s[L::B0 + i] = __ldg(b0 + i);
        s[L::B1 + i] = __ldg(b1 + i);
    }
    for (int i = tid; i < 8 * HID; i += nthreads) s[L::WO + i] = i < out_dim * HID ? __ldg(wo + i) : 0.0f;
    for (int i = tid; i < 8; i += nthreads) s[L::BO + i] = i < out_dim ? __ldg(bo + i) : 0.0f;
}

// x[IN] (registers) -> out[OUT] ; scratch = this thread's column of a [64][BLOCK] smem array (stride BLOCK)
template <int IN, int OUT, int BLOCK>
__device__ __forceinline__ void mlp_forward(const float* __restrict__ s, const float* x, float* out, float* scratch) {
    using L = MlpSmem<IN>;
    static_assert(IN % 4 == 0, "input width must be a multiple of 4");
#pragma unroll 2
    for (int o = 0; o < HID; ++o) {
        const float4* w = reinterpret_cast<const float4*>(s + L::W0 + o * IN);
        float a0 = s[L::B0 + o], a1 = 0.0f;
#pragma unroll
        for (int i = 0; i < IN / 4; ++i) {
            float4 ww = w[i];
            a0 = fmaf(ww.x, x[4 * i], a0);
            a1 = fmaf(ww.y, x[4 * i + 1], a1);
            a0 = fmaf(ww.z, x[4 * i + 2], a0);
            a1 = fmaf(ww.w, x[4 * i + 3], a1);
        }
        scratch[o * BLOCK] = tanhf(a0 + a1);
    }
    float h[HID];
#pragma unroll
    for (int o = 0; o < HID; ++o) h[o] = scratch[o * BLOCK];
#pragma unroll 2
    for (int o = 0; o < HID; ++o) {
        const float4* w = reinterpret_cast<const float4*>(s + L::W1 + o * HID);
        float a0 = s[L::B1 + o], a1 = 0.0f;
#pragma unroll
        for (int i = 0; i < HID / 4; ++i) {
            float4 ww = w[i];
            a0 = fmaf(ww.x, h[4 * i], a0);
            a1 = fmaf(ww.y, h[4 * i + 1], a1);
            a0 = fmaf(ww.z, h[4 * i + 2], a0);
            a1 = fmaf(ww.w, h[4 * i + 3], a1);
        }
        scratch[o * BLOCK] = tanhf(a0 + a1);
    }
#pragma unroll
    for (int o = 0; o < HID; ++o) h[o] = scratch[o * BLOCK];
#pragma unroll
    for (int o = 0; o < OUT; ++o) {
        const float4* w = reinterpret_cast<const float4*>(s + L::WO + o * HID);
        float a0 = s[L::BO + o], a1 = 0.0f;
#pragma unroll
        for (int i = 0; i < HID / 4; ++i) {
            float4 ww = w[i];
            a0 = fmaf(ww.x, h[4 * i], a0);
            a1 = fmaf(ww.y, h[4 * i + 1], a1);
            a0 = fmaf(ww.z, h[4 * i + 2], a0);
            a1 = fmaf(ww.w, h[4 * i + 3], a1);
        }
        out[o] = a0 + a1;
    }
}

}  // namespace kin
