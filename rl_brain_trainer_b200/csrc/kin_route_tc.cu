// kin_route_tc.cu -- the dense holder-route sequential probe (evaluate_sequential_route) with the 80-input route policy on the
// 5th-generation tensor cores (tcgen05.mma kind::tf32, accumulators in TMEM); the env / route arithmetic is the code the
// strict-fp32 probe (kin_route.cu) runs.
//
// One replica <-> one thread <-> one row of the A tile <-> one TMEM lane.  The route observation is 80
// floats (+ a constant 1 that carries the layer-1 bias, zero pad to K = 96), so the A tile has three 128-byte K chunks (48 KB) and
// layer 1 is 12 MMAs of K = 8; the hidden layers reuse the first two chunks (K = 64).  A CTA holds up to three tiles (12 warps)
// on named barriers sharing one copy of the weights (42 KB): 186 KB of shared memory, 192 TMEM columns (256 allocated).
// A tile walks the route in lockstep per waypoint: every replica of the tile steps until all of them have finished the waypoint
// (the replicas differ only by start noise, so they finish within a few steps of each other).
//
// Replaces: eval/eval_route_curriculum.py:55-136 (_roll_one) and :188-218 (evaluate_sequential_route), kinematic_phase1/.
// Numerics: TF32 operands + tanh.approx move actions by O(1e-3) like the Approach -> Finisher tensor-core rollout; the strict
// probe stays the parity path (tests/test_gpu_route.py compares the two prefix distributions).
#include "kin_route_core.cuh"
#include "kin_umma.cuh"

namespace kin {

using namespace umma;

// ---- kind::tf32 operands: fp32 words, [rows][32 floats] = 128-byte rows per K chunk, SWIZZLE_128B, K-major
constexpr int TC_TILE = 128;                   // replicas per tile == UMMA M == TMEM lanes
constexpr int TC_K = 64;                       // padded reduction width of the hidden layers
constexpr int TC_HID = 64;
constexpr int CHUNK_FLOATS_A = TC_TILE * 32;   // one 128-byte-wide K chunk of an A tile: 128 rows x 32 floats
constexpr int CHUNK_FLOATS_W = TC_HID * 32;    // 64 rows x 32 floats
constexpr int W_FLOATS = 2 * CHUNK_FLOATS_W;
constexpr int CHUNK_FLOATS_WO = 8 * 32;        // output layer: 8 rows (7 actions + zero row)
constexpr int WO_FLOATS = 2 * CHUNK_FLOATS_WO;

struct DevPolicyTc {
    const float *w0, *b0, *w1, *b1, *wo, *bo;
};

// Round-to-nearest (ties away) TF32: cvt.rna.tf32 is "add half an ulp of the 10-bit mantissa, clear the low 13 bits"; the
// tensor core ignores those 13 bits of a kind::tf32 operand, so the add alone feeds it the same operand (values here are finite
// and far from overflow: observations in [-1, 1], tanh outputs, trained weights).
__device__ __forceinline__ float to_tf32(float x) { return __uint_as_float(__float_as_uint(x) + 0x1000u); }

// float offset of element (row, k) inside a K-major SWIZZLE_128B operand whose K chunks hold `rows` rows each
__device__ __forceinline__ int sw128_offset(int row, int k, int chunk_floats) {
    const int chunk = k >> 5, kk = k & 31;
    return chunk * chunk_floats + row * 32 + ((((kk >> 2) ^ (row & 7)) << 2) | (kk & 3));
}

// instruction descriptor: D fp32, A/B tf32, both K-major, N>>3 at bit 17, M>>4 at bit 24
__host__ __device__ constexpr unsigned idesc_tf32(int M, int N) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((unsigned)(N >> 3) << 17) | ((unsigned)(M >> 4) << 24);
}

// write 4 consecutive K elements [k4*4, k4*4+4) of this thread's A row (already TF32-rounded)
__device__ __forceinline__ void a_store4(float* A, int row, int k4, float x0, float x1, float x2, float x3) {
    const int chunk = k4 >> 3, j = k4 & 7;
    float4* dst = reinterpret_cast<float4*>(A + chunk * CHUNK_FLOATS_A + row * 32 + ((j ^ (row & 7)) << 2));
    *dst = make_float4(x0, x1, x2, x3);
}

constexpr int RTC_TILES = 3;
constexpr int RTC_MAX_THREADS = TC_TILE * RTC_TILES;
constexpr int RTC_K1 = 96;                              // 80 route-observation floats | 1 | zero pad
constexpr int RTC_A_TILE_FLOATS = 3 * CHUNK_FLOATS_A;   // 48 KB
constexpr int RTC_W0_FLOATS = 3 * CHUNK_FLOATS_W;       // 24 KB

struct RtcSmem {
    float W0[RTC_W0_FLOATS];            // [64][96]: 80 inputs | bias column | zero pad
    float W1[W_FLOATS];
    float WO[WO_FLOATS];
    float b1[TC_HID];
    float bo[8];
    unsigned long long mbar[RTC_TILES];
    unsigned tmem_base;
    int run_flags[2][RTC_TILES][4];
    alignas(1024) float A[1][RTC_A_TILE_FLOATS];   // one 48 KB A tile per tile of the CTA (sized at launch)
};

struct RtcTile {
    float* A;
    unsigned a_saddr, w0_saddr, w1_saddr, wo_saddr, mbar_saddr, tmem_d, tmem_row;
    int tile, row, flag_buf, tile_threads;
    unsigned parity;
};

template <int KSTEPS>
__device__ __forceinline__ void issue_layer_k(unsigned a_saddr, unsigned w_saddr, int w_chunk_bytes, unsigned tmem_d, unsigned idesc, unsigned mbar_saddr) {
    fence_after();
#pragma unroll
    for (int k = 0; k < KSTEPS; ++k) {
        const unsigned a_off = (k >> 2) * (CHUNK_FLOATS_A * 4) + (k & 3) * 32;
        const unsigned w_off = (k >> 2) * w_chunk_bytes + (k & 3) * 32;
        mma_tf32(tmem_d, desc_k(a_saddr + a_off), desc_k(w_saddr + w_off), idesc, k > 0 ? 1u : 0u);
    }
    commit(mbar_saddr);
}

// route observation [80] -> action [7]; collective over the tile's threads.  Returns false (without running the MLP) once no
// replica of the tile is still inside the current waypoint episode.
__device__ __forceinline__ bool mlp_tc_route(RtcSmem& S, RtcTile& c, const float* o, float* act, bool running) {
    const int fb = c.flag_buf;
    c.flag_buf ^= 1;
    const unsigned any = __any_sync(0xffffffffu, running);
    if ((threadIdx.x & 31) == 0) S.run_flags[fb][c.tile][(threadIdx.x >> 5) & 3] = (int)any;
#pragma unroll
    for (int k4 = 0; k4 < KIN_ROUTE_OBS_DIM / 4; ++k4)
        a_store4(c.A, c.row, k4, to_tf32(o[4 * k4]), to_tf32(o[4 * k4 + 1]), to_tf32(o[4 * k4 + 2]), to_tf32(o[4 * k4 + 3]));
    a_store4(c.A, c.row, 20, 1.0f, 0.0f, 0.0f, 0.0f);
#pragma unroll
    for (int k4 = 21; k4 < RTC_K1 / 4; ++k4) a_store4(c.A, c.row, k4, 0.0f, 0.0f, 0.0f, 0.0f);
    fence_async_smem();
    fence_before();
    bar_sync(c.tile + 1, c.tile_threads);
    if (!(S.run_flags[fb][c.tile][0] | S.run_flags[fb][c.tile][1] | S.run_flags[fb][c.tile][2] | S.run_flags[fb][c.tile][3])) return false;
    if (c.row < 32 && elect_one()) issue_layer_k<RTC_K1 / 8>(c.a_saddr, c.w0_saddr, CHUNK_FLOATS_W * 4, c.tmem_d, idesc_tf32(TC_TILE, TC_HID), c.mbar_saddr);
    mbar_wait(c.mbar_saddr, c.parity);
    c.parity ^= 1u;
    fence_after();
    float v[32];
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        tmem_ld32(c.tmem_row + half * 32, v);
#pragma unroll
        for (int j = 0; j < 8; ++j)
            a_store4(c.A, c.row, half * 8 + j, to_tf32(tanh_fast(v[4 * j])), to_tf32(tanh_fast(v[4 * j + 1])),
                     to_tf32(tanh_fast(v[4 * j + 2])), to_tf32(tanh_fast(v[4 * j + 3])));
    }
    fence_async_smem();
    fence_before();
    bar_sync(c.tile + 1, c.tile_threads);
    if (c.row < 32 && elect_one()) issue_layer_k<TC_K / 8>(c.a_saddr, c.w1_saddr, CHUNK_FLOATS_W * 4, c.tmem_d, idesc_tf32(TC_TILE, TC_HID), c.mbar_saddr);
    mbar_wait(c.mbar_saddr, c.parity);
    c.parity ^= 1u;
    fence_after();
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        tmem_ld32(c.tmem_row + half * 32, v);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float* b = S.b1 + half * 32 + 4 * j;
            a_store4(c.A, c.row, half * 8 + j, to_tf32(tanh_fast(v[4 * j] + b[0])), to_tf32(tanh_fast(v[4 * j + 1] + b[1])),
                     to_tf32(tanh_fast(v[4 * j + 2] + b[2])), to_tf32(tanh_fast(v[4 * j + 3] + b[3])));
        }
    }
    fence_async_smem();
    fence_before();
    bar_sync(c.tile + 1, c.tile_threads);
    if (c.row < 32 && elect_one()) issue_layer_k<TC_K / 8>(c.a_saddr, c.wo_saddr, CHUNK_FLOATS_WO * 4, c.tmem_d, idesc_tf32(TC_TILE, 8), c.mbar_saddr);
    mbar_wait(c.mbar_saddr, c.parity);
    c.parity ^= 1u;
    fence_after();
    float a8[8];
    tmem_ld8(c.tmem_row, a8);
    fence_before();
#pragma unroll
    for (int i = 0; i < KIN_NJ; ++i) act[i] = clampf(a8[i] + S.bo[i], -1.0f, 1.0f);
    return true;
}

__global__ void __launch_bounds__(RTC_MAX_THREADS, 1)
kin_route_probe_tc_kernel(const __grid_constant__ KinEnvParams P, RouteView R, DevPolicyTc pol, const float* __restrict__ start_q, int start_index,
                          int end_index, int n, int* __restrict__ prefix_out, uint32_t* __restrict__ success_bits, int words,
                          unsigned long long* __restrict__ env_steps) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    RtcSmem& S = *reinterpret_cast<RtcSmem*>(smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u));
    const int tid = threadIdx.x;
    const int warp = tid >> 5;
    RtcTile c;
    c.tile = tid >> 7;
    c.row = tid & (TC_TILE - 1);
    c.tile_threads = min(TC_TILE, (int)blockDim.x - c.tile * TC_TILE);
    c.A = &S.A[0][0] + (size_t)c.tile * RTC_A_TILE_FLOATS;
    c.parity = 0u;
    c.flag_buf = 0;
    const int n_tiles_cta = ((int)blockDim.x + TC_TILE - 1) / TC_TILE;
    const unsigned tmem_cols = n_tiles_cta == 1 ? 64u : (n_tiles_cta == 2 ? 128u : 256u);
    if (warp == 0) tmem_alloc(smem_u32(&S.tmem_base), tmem_cols);
    if (tid == 0) {
#pragma unroll
        for (int i = 0; i < RTC_TILES; ++i) mbar_init(smem_u32(&S.mbar[i]), 1);
        fence_mbar_init();
    }
    if (tid < 2 * RTC_TILES * 4) (&S.run_flags[0][0][0])[tid] = 0;
    // stage the actor into the swizzled B-operand images
    for (int i = tid; i < TC_HID * RTC_K1; i += (int)blockDim.x) {
        const int u = i / RTC_K1, k = i - u * RTC_K1;
        const float v0 = k < KIN_ROUTE_OBS_DIM ? __ldg(pol.w0 + u * KIN_ROUTE_OBS_DIM + k) : (k == KIN_ROUTE_OBS_DIM ? __ldg(pol.b0 + u) : 0.0f);
        S.W0[sw128_offset(u, k, CHUNK_FLOATS_W)] = to_tf32(v0);
    }
    for (int i = tid; i < TC_HID * TC_K; i += (int)blockDim.x) {
        const int u = i >> 6, k = i & 63;
        S.W1[sw128_offset(u, k, CHUNK_FLOATS_W)] = to_tf32(__ldg(pol.w1 + u * TC_HID + k));
    }
    for (int i = tid; i < 8 * TC_K; i += (int)blockDim.x) {
        const int u = i >> 6, k = i & 63;
        S.WO[sw128_offset(u, k, CHUNK_FLOATS_WO)] = u < KIN_NJ ? to_tf32(__ldg(pol.wo + u * TC_HID + k)) : 0.0f;
    }
    for (int i = tid; i < TC_HID; i += (int)blockDim.x) S.b1[i] = __ldg(pol.b1 + i);
    if (tid < 8) S.bo[tid] = tid < KIN_NJ ? __ldg(pol.bo + tid) : 0.0f;
    fence_async_smem();
    fence_before();
    __syncthreads();
    fence_after();
    const unsigned tmem_base = S.tmem_base;
    c.a_saddr = smem_u32(c.A);
    c.w0_saddr = smem_u32(S.W0);
    c.w1_saddr = smem_u32(S.W1);
    c.wo_saddr = smem_u32(S.WO);
    c.mbar_saddr = smem_u32(&S.mbar[c.tile]);
    c.tmem_d = tmem_base + c.tile * TC_HID;
    c.tmem_row = c.tmem_d + ((unsigned)((warp & 3) * 32) << 16);

    const int rep = blockIdx.x * (int)blockDim.x + tid;
    const bool active = rep < n;
    const int repc = active ? rep : n - 1;
    float cq[NJ], cdq[NJ], cpa[NJ];
    {
        const float* q0 = start_q ? start_q + (size_t)repc * NJ : R.q + (size_t)wp_clamp(R, max(start_index - 1, 0)) * NJ;
#pragma unroll
        for (int i = 0; i < NJ; ++i) { cq[i] = q0[i]; cdq[i] = 0.0f; cpa[i] = 0.0f; }
    }
    const int final_end = min(end_index, R.n - 1);
    int prefix = 0;
    bool broken = false;
    unsigned long long steps = 0;
    unsigned word = 0u;
    float o[ROBS];
#pragma unroll
    for (int i = 0; i < ROBS; ++i) o[i] = 0.0f;
    for (int idx = start_index; idx <= final_end; ++idx) {
        EnvRegs s;
        s.flags = 0u;
        float gq_out[NJ], gq[NJ];
        const float* g = R.q + (size_t)wp_clamp(R, idx) * NJ;
#pragma unroll
        for (int i = 0; i < NJ; ++i) gq[i] = __ldg(g + i);
        reset_core(P, s, KIN_MODE_APPROACH, cq, cdq, cpa, gq, nullptr, gq_out);
        RouteRegs rr{idx, 0, idx, 0};
        RouteOut ro;
        ro.done = 0u;
        bool running = active;
        for (;;) {
            float act[KIN_NJ];
            if (running) {          // a finished replica keeps its last row in the A tile while the tile's stragglers step on
                float o56[OBS];
                build_obs(P, s, KIN_MODE_APPROACH, o56);
                build_route_obs(P, R, s, rr.index, o56, o);
            }
            if (!mlp_tc_route(S, c, o, act, running)) break;      // tile-uniform
            if (running) {
                StepOut so;
                route_step_core<false, false>(P, R, nullptr, s, rr, act, true, so, ro, nullptr);   // eval needs no off-route term
                steps += 1;
                running = !(ro.done & (KIN_DONE_TERMINATED | KIN_DONE_TRUNCATED));
            }
        }
        const bool ok = (ro.done & KIN_DONE_SUCCESS) != 0;
        if (ok && !broken) prefix += 1; else broken = true;
        const int k = idx - start_index;
        if (ok) word |= 1u << (k & 31);
        if (success_bits && active && ((k & 31) == 31 || idx == final_end)) {
            success_bits[(size_t)rep * words + (k >> 5)] = word;
            word = 0u;
        }
#pragma unroll
        for (int i = 0; i < NJ; ++i) { cq[i] = s.q[i]; cdq[i] = s.dq[i]; cpa[i] = s.pa[i]; }
    }
    if (active) prefix_out[rep] = prefix;
    if (env_steps) {
        unsigned long long mine = active ? steps : 0ull;
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, off);
        if ((tid & 31) == 0 && mine) atomicAdd(env_steps, mine);
    }
    fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, tmem_cols);
}

}  // namespace kin

using namespace kin;

extern "C" int kin_route_probe_tc(void* handle, const KinRouteTable* host_route, const KinPolicyWeights* w, const float* start_q, int start_index,
                                  int end_index, int n, int* prefix, uint32_t* success_bits, unsigned long long* env_steps, void* stream) {
    KinHandle* h = kin_handle(handle);
    if (!h || !route_ok(host_route)) return kin_fail(KIN_ERR_INVALID_ARG, "kin_route_probe_tc: bad handle or route table");
    if (!w || w->in_dim != ROBS || !w->pi_w0 || !w->pi_b0 || !w->pi_w1 || !w->pi_b1 || !w->act_w || !w->act_b)
        return kin_fail(KIN_ERR_INVALID_ARG, "kin_route_probe_tc: need an 80-input actor");
    if (!prefix || n <= 0 || start_index < 1 || end_index < start_index) return kin_fail(KIN_ERR_INVALID_ARG, "kin_route_probe_tc: bad sizes / indices");
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    // balanced launch: a batch that fits one wave gets one CTA per SM with ceil(warps / SMs) warps
    const int warps = (n + 31) / 32;
    int w_cta = RTC_MAX_THREADS / 32;
    if (warps <= sms * w_cta) w_cta = (warps + sms - 1) / sms;
    const int threads = 32 * w_cta;
    const int blocks = (n + threads - 1) / threads;
    const int tiles = (threads + TC_TILE - 1) / TC_TILE;
    const size_t smem = sizeof(RtcSmem) + (size_t)(tiles - 1) * RTC_A_TILE_FLOATS * sizeof(float) + 1024;
    cudaError_t e = cudaFuncSetAttribute(kin_route_probe_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return kin_fail_cuda(e, "kin_route_probe_tc: smem attribute");
    const int final_end = end_index < host_route->n_waypoints - 1 ? end_index : host_route->n_waypoints - 1;
    const int words = (final_end - start_index + 1 + 31) / 32;
    DevPolicyTc p{w->pi_w0, w->pi_b0, w->pi_w1, w->pi_b1, w->act_w, w->act_b};
    kin_route_probe_tc_kernel<<<blocks, threads, smem, (cudaStream_t)stream>>>(h->params, view_of(host_route), p, start_q, start_index, end_index, n, prefix,
                                                                              success_bits, words, env_steps);
    e = cudaGetLastError();
    return e == cudaSuccess ? KIN_OK : kin_fail_cuda(e, "kin_route_probe_tc");
}
