// kin_peer.cuh -- receive-buffer layout of the NVLink peer-memory gradient exchange and the in-kernel ("fused") form of it:
// the tail every CTA of the gradient kernel runs after its partial row is written (csrc/kin_ppo_tc.cu), replacing the separate
// kin_peer_push_kernel + kin_peer_gather_kernel launches between the gradient kernel and Adam.
//
//   receive buffer of a rank (cudaMalloc'ed by kin_peer_buffer_create, opened by the peers through CUDA IPC):
//     [0]      unsigned arrived[8]            two-kernel form: arrived[s] = pushes of sender s that have fully landed here
//     [64]     unsigned local_count           two-kernel form: CTAs of this rank's push kernel that have finished
//     [68]     unsigned grid_count            fused form: CTAs of this rank's gradient kernel whose partial row is complete (monotonic)
//     [72]     unsigned adam_count            fused update: CTAs whose slice of the summed gradient and its sum of squares are written (monotonic)
//     [128]    unsigned slice_flag[8][512]    fused form: slice_flag[s][c] = last exchange whose slice c sender s has delivered here
//     [16512]  float    slot[2][world][row]   row = n_params + 8 (gradient, then the 5 loss statistics); slot = exchange parity (two-kernel form)
//     [...]    uint2    ll[2][world][row]     fused form: (value bits, exchange number) pairs -- the flag travels IN the 8-byte store that
//                                             carries the value, so the sender needs no release fence and the receiver no flag round trip
#pragma once

#include <cuda_bf16.h>

#include "kin_internal.h"
#include "kin_ppo_layout.cuh"
#include "kin_ppo_math.cuh"

namespace kin {

constexpr int PEER_MAX = 8;
constexpr int PEER_MAX_CTA = 512;
constexpr size_t PEER_FLAGS = 128;
constexpr size_t PEER_HEADER = PEER_FLAGS + sizeof(unsigned) * PEER_MAX * PEER_MAX_CTA;      // 16 512 bytes

struct PeerTable {
    unsigned char* base[PEER_MAX];
};

// optional clip + Adam step in the same tail (params == nullptr: the caller launches kin_ppo_adam)
struct AdamFused {
    float* params;                    // [P] flat parameters, updated in place
    float* m;                         // [P] Adam first moments
    float* v;                         // [P] Adam second moments
    unsigned short* wimg;             // bf16 operand image of the 56-input weights kept in step (nullable)
    float* stats_accum;               // [KIN_PPO_STATS] running sums over the minibatches of an update (nullable)
    float* norm_part;                 // [n_cta] scratch: sum of squares of each CTA's gradient slice
    float bc1, bc2;                   // 1 - beta^step
    int in_dim;
};

// arguments of the fused exchange (world == 0: no exchange, the caller reduces `partials` itself)
struct PeerFused {
    PeerTable peers;
    int rank, world;
    unsigned epoch;
    float* grad;                      // [P] this rank's copy of the summed gradient
    float* stats;                     // [KIN_PPO_STATS] (5 summed loss statistics, slot KIN_PPO_STAT_SKIP on a timeout)
    int* timed_out;                   // sticky device flag
    unsigned long long timeout_cycles;
    AdamFused adam;
};

unsigned long long kin_peer_timeout_cycles();      // kin_peer.cu

#ifdef KIN_PPO_TRACE
// phase profiler of the fused tail (debug builds only, tools/ppo_trace.py --tail): cycles per phase summed over launches, thread 0 of CTAs 0 and 150
static __device__ unsigned long long kin_peer_trace_buf[2][12];
static __device__ unsigned long long kin_peer_trace_wait[PEER_MAX_CTA][2];      // per CTA: cycles spent in grid barrier 1 (summed), SM id
#define PT_DECL long long pt_t = clock64(); const bool pt_on = threadIdx.x == 0 && (cta == 0 || cta == 150); unsigned long long* pt_o = kin_peer_trace_buf[cta ? 1 : 0];
#define PT_MARK(i) do { if (pt_on) { const long long t_ = clock64(); pt_o[i] += (unsigned long long)(t_ - pt_t); pt_t = t_; } } while (0)
#define PT_COUNT() do { if (pt_on) pt_o[11] += 1ull; } while (0)
#else
#define PT_DECL
#define PT_MARK(i)
#define PT_COUNT()
#endif

__host__ __device__ inline int peer_row(int P) { return (P + KIN_PPO_STATS + 3) & ~3; }
// byte offset of the fused form's (value, exchange) pairs behind the two-kernel form's float slots
__host__ __device__ inline size_t peer_ll_offset(int P, int world) { return PEER_HEADER + sizeof(float) * 2 * (size_t)world * peer_row(P); }
__host__ __device__ inline size_t peer_buffer_size(int P, int world) { return peer_ll_offset(P, world) + sizeof(uint2) * 2 * (size_t)world * peer_row(P); }

__device__ __forceinline__ void st_ll(uint2* p, float value, unsigned epoch) {      // one 8-byte store: value and flag land together
    asm volatile("st.volatile.global.v2.u32 [%0], {%1, %2};" ::"l"(p), "r"(__float_as_uint(value)), "r"(epoch) : "memory");
}
__device__ __forceinline__ uint2 ld_ll(const uint2* p) {
    uint2 v;
    asm volatile("ld.volatile.global.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p) : "memory");
    return v;
}

__device__ __forceinline__ unsigned ld_acquire_sys(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned ld_acquire_gpu(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// Tail of the gradient kernel, called by ALL threads of EVERY CTA (blockDim.x >= 256) after the CTA's part of its partial row is in
// global memory.  Needs every CTA of the grid co-resident (it contains a grid barrier): the gradient kernel's grid is <= 2 CTAs / SM.
//   1. grid barrier: all partial rows of this rank are complete;
//   2. CTA c reduces its slice of the P + 5 columns over the rows -- in the order kin_peer_push_kernel / kin_ppo_reduce_kernel use
//      (8 interleaved row groups, folded in warp order), so the result is bitwise the two-kernel path's -- and stores every value
//      TOGETHER WITH THE EXCHANGE NUMBER as one 8-byte word into ll[epoch & 1][rank] of every peer (posted NVLink stores; an aligned
//      8-byte store lands atomically, the protocol NCCL calls LL): no release fence, no separate flag.  A trace of the first version
//      (per-slice flags published with st.release.sys: tools/peer_tail_trace.py) showed 6 us in the release -- it waits for the
//      acknowledgements of all the CTA's peer stores -- and 9 us in the flag wait per minibatch at 2 GPUs;
//   3. polls its own copy of ll[epoch & 1][r][p] until the exchange number matches, for every rank r, and writes grad / stats = sum over
//      ranks in RANK ORDER (bitwise identical on every rank).  A peer that never delivers sets the sticky timeout flag and marks the
//      minibatch to be skipped.  Two parities suffice: a word is rewritten two exchanges later, and a sender only gets there after its own
//      step 3 of the exchange in between, which waited for every rank's step 2 of that exchange.
__device__ __forceinline__ void peer_exchange_tail(const PeerFused& px, const float* __restrict__ partials, int n_rows, int P, float inv_global_batch,
                                                   float (*part)[32], int* flag_smem) {
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int n_cta = (int)(gridDim.x * gridDim.y), cta = (int)(blockIdx.y * gridDim.x + blockIdx.x);
    unsigned char* own = px.peers.base[px.rank];
    PT_DECL
    PT_COUNT();
    // ---- 1. grid barrier (monotonic counter: exchange e completes at e * n_cta)
    __threadfence();
    __syncthreads();
    if (tid == 0) {
        unsigned* cnt = reinterpret_cast<unsigned*>(own + 68);
        atomicAdd(cnt, 1u);
        const unsigned target = px.epoch * (unsigned)n_cta;
        const long long t0 = clock64();
        while ((int)(ld_acquire_gpu(cnt) - target) < 0) {
            if ((unsigned long long)(clock64() - t0) > px.timeout_cycles) { atomicExch(px.timed_out, 1); break; }
        }
    }
    __syncthreads();
#ifdef KIN_PPO_TRACE
    if (tid == 0 && cta < PEER_MAX_CTA) {
        unsigned smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        kin_peer_trace_wait[cta][0] += (unsigned long long)(clock64() - pt_t);
        kin_peer_trace_wait[cta][1] = smid;
    }
#endif
    PT_MARK(0);
    // ---- 2. this CTA's column slice: reduce over the rows, push to every peer
    const int cols = P + 5, prow = P + KIN_PPO_STATS + 8;
    const int per = ((cols + n_cta - 1) / n_cta + 31) & ~31;      // whole 32-column blocks per CTA
    const int p0 = cta * per, p1 = min(p0 + per, cols);
    for (int base = p0; base < p1; base += 32) {
        const int p = base + lane;
        float a0 = 0.0f, a1 = 0.0f;
        if (w < 8 && p < cols) {
            // rows w, w + 16, ... into a0 and w + 8, w + 24, ... into a1, added in that order (kin_ppo_reduce_kernel's order); the loads
            // of a batch are all issued before the first add, so the L2 latency is paid once per batch, not once per row
            constexpr int B = 10;      // 160 rows per pass: the 148 partial rows of a B200 in ONE batch of loads
            int c = w;
            while (c < n_rows) {
                float v0[B], v1[B];
#pragma unroll
                for (int k = 0; k < B; ++k) {
                    const int r0 = c + 16 * k, r1 = r0 + 8;
                    v0[k] = r0 < n_rows ? __ldcg(partials + (size_t)r0 * prow + p) : 0.0f;
                    v1[k] = (r1 < n_rows && r0 + 8 < n_rows) ? __ldcg(partials + (size_t)r1 * prow + p) : 0.0f;
                }
#pragma unroll
                for (int k = 0; k < B; ++k) {
                    const int r0 = c + 16 * k;
                    if (r0 + 8 < n_rows) { a0 += v0[k]; a1 += v1[k]; }
                    else if (r0 < n_rows) a0 += v0[k];
                }
                c += 16 * B;
            }
        }
        if (w < 8) part[w][lane] = a0 + a1;
        __syncthreads();
        if (w < px.world && p < cols) {
            float a = part[0][lane];
#pragma unroll
            for (int k = 1; k < 8; ++k) a += part[k][lane];
            if (p >= P) a *= inv_global_batch;
            uint2* ll = reinterpret_cast<uint2*>(px.peers.base[w] + peer_ll_offset(P, px.world)) + ((size_t)(px.epoch & 1u) * px.world + px.rank) * peer_row(P);
            st_ll(ll + p, a, px.epoch);
        }
        __syncthreads();
    }
    PT_MARK(1);
    PT_MARK(2);
    // ---- 3. every rank's value of this CTA's columns (the exchange number in the same word says it has landed), rank-ordered sum
    (void)flag_smem;
    const uint2* ll = reinterpret_cast<const uint2*>(own + peer_ll_offset(P, px.world)) + (size_t)(px.epoch & 1u) * px.world * peer_row(P);
    for (int p = p0 + tid; p < p1; p += (int)blockDim.x) {
        // all ranks' words are requested at once (independent loads), then only the ones whose exchange number is still old are polled
        uint2 v[PEER_MAX];
        unsigned pending = 0u;
#pragma unroll
        for (int r = 0; r < PEER_MAX; ++r) {
            if (r < px.world) v[r] = ld_ll(ll + (size_t)r * peer_row(P) + p);
        }
#pragma unroll
        for (int r = 0; r < PEER_MAX; ++r) {
            if (r < px.world && v[r].y != px.epoch) pending |= 1u << r;
        }
        if (pending && *reinterpret_cast<volatile int*>(px.timed_out) == 0) {
            const long long t0 = clock64();
            while (pending) {
#pragma unroll
                for (int r = 0; r < PEER_MAX; ++r) {
                    if (pending & (1u << r)) {
                        v[r] = ld_ll(ll + (size_t)r * peer_row(P) + p);
                        if (v[r].y == px.epoch) pending &= ~(1u << r);
                    }
                }
                if (pending && (unsigned long long)(clock64() - t0) > px.timeout_cycles) { atomicExch(px.timed_out, 1); break; }
            }
        }
        float a = 0.0f;
#pragma unroll
        for (int r = 0; r < PEER_MAX; ++r) {
            if (r < px.world) a += __uint_as_float(v[r].x);      // rank order
        }
        if (p < P) px.grad[p] = a;
        else if (px.stats) px.stats[p - P] = a;
    }
    PT_MARK(3);
    if (cta == 0 && tid == 0 && px.stats) px.stats[KIN_PPO_STAT_SKIP] = *reinterpret_cast<volatile int*>(px.timed_out) ? 1.0f : 0.0f;
    PT_MARK(4);
}

// Second half of the fused update, called by ALL threads of EVERY CTA right after peer_exchange_tail when px.adam.params is set:
// clip_grad_norm_ + Adam (kin_ppo_adam's arithmetic) on the slice of the summed gradient this CTA has just written, so a minibatch is ONE
// launch (gradient, reduction, exchange, optimiser step) instead of three.
//   1. every CTA writes the sum of squares of its slice (fixed order) to norm_part[cta]; grid barrier (adam_count);
//   2. every CTA adds the n_cta partial sums in the same fixed order -> the same clip coefficient everywhere (and on every rank: the
//      summed gradient is bitwise identical on all ranks);
//   3. Adam on the slice: m, v, params, and the bf16 weight image the next launch's TMA copies read.
// The parameters are only read in the gradient kernel's prologue and every CTA is past the first grid barrier, so updating them here
// races with nothing.  A timed-out exchange leaves them untouched (same rule as kin_ppo_adam with KIN_PPO_STAT_SKIP).
__device__ __forceinline__ void peer_adam_tail(const PeerFused& px, const KinPpoHyper& hp, int P, float* red /* >= 40 floats of smem */) {
    const AdamFused& A = px.adam;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5, nw = (int)(blockDim.x + 31) >> 5;
    const int n_cta = (int)(gridDim.x * gridDim.y), cta = (int)(blockIdx.y * gridDim.x + blockIdx.x);
    unsigned char* own = px.peers.base[px.rank];
    const int cols = P + 5;
    const int per = ((cols + n_cta - 1) / n_cta + 31) & ~31;
    const int p0 = min(cta * per, P), p1 = min(cta * per + per, P);       // the gradient part of this CTA's slice
    PT_DECL
    // this thread's first parameter: fetch its optimiser state now, so the loads fly while the norm goes through the grid barrier
    const int own_p = p0 + tid;
    float own_m = 0.0f, own_v = 0.0f, own_w = 0.0f;
    if (own_p < p1) { own_m = A.m[own_p]; own_v = A.v[own_p]; own_w = A.params[own_p]; }
    __syncthreads();                 // px.grad[p0 .. p1) was written by this CTA's threads
    float ss = 0.0f;
    for (int p = p0 + tid; p < p1; p += (int)blockDim.x) {
        const float g = px.grad[p];
        ss = fmaf(g, g, ss);
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, off);
    if (lane == 0) red[w] = ss;
    __syncthreads();
    if (tid == 0) {
        float t = 0.0f;
        for (int k = 0; k < nw; ++k) t += red[k];
        A.norm_part[cta] = t;
        __threadfence();
        unsigned* cnt = reinterpret_cast<unsigned*>(own + 72);
        atomicAdd(cnt, 1u);
        const unsigned target = px.epoch * (unsigned)n_cta;
        const long long t0 = clock64();
        while ((int)(ld_acquire_gpu(cnt) - target) < 0) {
            if ((unsigned long long)(clock64() - t0) > px.timeout_cycles) { atomicExch(px.timed_out, 1); break; }
        }
    }
    __syncthreads();
    PT_MARK(5);
    if (w == 0) {
        float t = 0.0f;
        for (int k = lane; k < n_cta; k += 32) t += __ldcg(A.norm_part + k);
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) t += __shfl_xor_sync(0xffffffffu, t, off);
        if (lane == 0) {
            const float norm = sqrtf(t);
            red[32] = clip_coef(norm, hp);
            red[33] = norm;
        }
    }
    __syncthreads();
    const bool skip = *reinterpret_cast<volatile int*>(px.timed_out) != 0;
    if (cta == 0 && tid == 0 && px.stats) {
        px.stats[KIN_PPO_STAT_GRAD_NORM] = red[33];
        px.stats[KIN_PPO_STAT_SKIP] = skip ? 1.0f : 0.0f;
        if (A.stats_accum && !skip) {
#pragma unroll
            for (int q = 0; q < 5; ++q) A.stats_accum[q] += __ldcg(px.stats + q);
            A.stats_accum[KIN_PPO_STAT_GRAD_NORM] += red[33];
            A.stats_accum[7] += 1.0f;
        }
    }
    if (skip) return;
    const float cf = red[32];
    const PpoOffsets O = ppo_offsets(A.in_dim);
    for (int p = p0 + tid; p < p1; p += (int)blockDim.x) {
        const bool first = p == own_p;
        const AdamMoments mv = adam_moments(px.grad[p], cf, first ? own_m : A.m[p], first ? own_v : A.v[p], hp);
        A.m[p] = mv.m;
        A.v[p] = mv.v;
        const float np = adam_param(first ? own_w : A.params[p], mv, A.bc1, A.bc2, hp);
        A.params[p] = np;
        if (A.wimg) {
            const int off = wimg_offset(O, A.in_dim, p);
            if (off >= 0) A.wimg[off >> 1] = __bfloat16_as_ushort(__float2bfloat16_rn(np));
        }
    }
    PT_MARK(6);
}

}  // namespace kin
