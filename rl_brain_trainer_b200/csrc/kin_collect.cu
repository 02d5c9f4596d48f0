// kin_collect.cu -- K4: the fused PPO rollout collection.  ONE launch runs n_steps of
//   actor + critic forward (tcgen05 kind::f16) -> Gaussian action sample + log-prob -> env step (reward, termination)
//   -> in-register auto-reset -> rollout-buffer writes
// for every env, with the env state in registers for the whole rollout (HBM state rows are read once and written once).
//
// Replaces SB3 OnPolicyAlgorithm.collect_rollouts (stable-baselines3 2.8.0 on_policy_algorithm.py; call site
// kinematic_phase1/train_workspace_expansion.py:232 model.learn) over a VecEnv of ArmKinematicEnv
// (kinematic_phase1/envs/arm_kinematic_env.py:213-365) -- the per-step-launch path in ppo.py::collect stays as the
// strict-fp32 restatement this kernel is tested against.
//
// The policy half (weights, forward, sample, bootstrap list) is kin_collect_policy.cuh, shared with K4-route; this file holds the
// env half.  The X operand image of every step (56 obs | 1 | zeros, bf16, SWIZZLE_128B K-major) is copied by the TMA engine
// straight into the rollout buffer: it IS the operand the tensor-core update (kin_ppo_grad_tc, image mode) consumes with one bulk
// copy per tile, so the observation is never written as fp32.  Truncated episodes append their terminal observation (fp32) to a
// short list; kin_ppo_bootstrap_list adds gamma * V(terminal_obs) to their rewards afterwards.
#include "kin_collect_policy.cuh"

namespace kin {

using namespace umma;

template <int TILES>
struct __align__(1024) CollectSmem {
    unsigned char XH[TILES][2][AC_TILE_BYTES];   // [.][0]: X image, then actor H1 / H2; [.][1]: critic H1 / H2
    AcWeights<1> w;
    unsigned long long mbar[TILES][2];           // [0]: layer 1 (MMA commit + image store drained), [1]: layers 2 / 3
    unsigned long long mbar_w;                   // weight image bulk copy
    unsigned tmem_base;
};

struct CollectOut {
    unsigned char* ximg;      // [T][n/128][16 KB]
    float* action;            // [T][n][7]
    float* logp;              // [T][n]
    float* value;             // [T][n]
    float* reward;            // [T][n]
    uint8_t* done;            // [T][n]
    uint8_t* episode_start;   // [T][n]
    uint8_t* start_io;        // [n]
    float* last_value;        // [n]
    int* boot_count;
    int* boot_index;          // [cap]  t * n + env
    float* boot_obs;          // [cap][56]
    int boot_cap;
};

// POP (population launch, kin_pop_collect): SP carries the KinPopMember table and member blockIdx.y's descriptor replaces every other
// per-run argument; P is shared.  A CTA holds one tile of one member (TILES = 1), blockIdx.x is the member-local tile, so env indices --
// and with them the Philox streams -- are the standalone launch's.
template <int TILES, int MODE, bool POP = false>
__global__ void __launch_bounds__(TILES * AC_ROWS, 1)
kin_collect_kernel(const __grid_constant__ KinEnvParams P, const KinSamplerParams* __restrict__ SP, float* __restrict__ state, int stride, int n,
                   const float* __restrict__ params, const unsigned char* __restrict__ wimg, int T, uint64_t noise_seed, uint32_t step0,
                   uint64_t reset_seed, CollectOut out) {
    static_assert(!POP || TILES == 1, "a CTA never mixes members");
    if constexpr (POP) {
        const KinPopMember& M = reinterpret_cast<const KinPopMember*>(SP)[blockIdx.y];
        SP = M.sampler;
        state = M.state;
        stride = M.stride;
        params = M.params;
        wimg = static_cast<const unsigned char*>(M.weight_image);
        noise_seed = M.noise_seed;
        step0 = M.first_step;
        reset_seed = M.reset_seed;
        out = CollectOut{static_cast<unsigned char*>(M.obs_tiles), M.action, M.logp, M.value, M.reward, M.done, M.episode_start, M.start_io,
                         M.last_value, M.boot_count, M.boot_index, M.boot_obs, M.boot_cap};
    }
    constexpr int IN = 56;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    // round up to 1024 bytes WITHOUT leaving the shared address space (pointer + offset, not an integer round trip), so every
    // access below compiles to LDS / STS rather than generic LD / ST with 64-bit address arithmetic
    CollectSmem<TILES>& S = *reinterpret_cast<CollectSmem<TILES>*>(smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u));
    const int tid = threadIdx.x;
    constexpr int NT = TILES * AC_ROWS;

    // ---- weights -> bf16 operand tiles (both nets): one bulk copy of the prebuilt image, or converted here ---------------
    if (wimg) {
        static_assert(offsetof(AcWeights<1>, W1) == offsetof(AcWeights<1>, W0) + 16384 &&
                      offsetof(AcWeights<1>, WO) == offsetof(AcWeights<1>, W0) + 32768, "W0 | W1 | WO must be laid out like the image");
        if (tid == 0) {
            const unsigned mbw = smem_u32(&S.mbar_w);
            mbar_init(mbw, 1);
            fence_mbar_init();
            mbar_expect_tx(mbw, KIN_WIMG_BYTES);
            bulk_load(smem_u32(S.w.W0), wimg, KIN_WIMG_BYTES, mbw);
        }
    } else {
        convert_weights<IN, 1, NT>(S.w, params, tid);
    }
    load_vectors<IN>(S.w, params, tid);
    init_tiles<TILES, 2>(S, tid);
    if (wimg) mbar_wait(smem_u32(&S.mbar_w), 0u);
    AcTile<1> c = tile_of<1, 2>(S, tid);

    const int gtile = blockIdx.x * TILES + c.tile;            // global 128-env tile
    const int n_tiles = n / AC_ROWS;
    const bool live = gtile < n_tiles;                        // tile-uniform
    const int env = (live ? gtile : 0) * AC_ROWS + c.row;

    EnvRegs s;
    load_env<MODE != KIN_MODE_APPROACH>(state, stride, env, s);
    float pe[3], oe[3], margin[NJ];
    pose_error(s.ee, s.goal, pe, oe);
#pragma unroll
    for (int i = 0; i < NJ; ++i) margin[i] = joint_margin(P, s.q[i], i);
    unsigned start = live ? out.start_io[env] : 0u;

    if (live) {
        for (int t = 0; t < T; ++t) {
            float o[OBS], mv[8];
            build_obs_from(P, s, MODE, pe, oe, margin, o);
            policy_forward<IN, true>(S.w, c, o, out.ximg + ((size_t)t * n_tiles + gtile) * AC_TILE_BYTES, mv);
            const size_t idx = (size_t)t * n + env;
            float a[NJ];
            const float lp = sample_action(S.w, noise_seed, (unsigned)env, step0 + (uint32_t)t, mv, a, out.action + idx * NJ);
            out.logp[idx] = lp;
            out.value[idx] = mv[7];
            out.episode_start[idx] = (uint8_t)start;
            // ---- env step
            StepOut so;
            step_core<MODE, false>(P, s, a, so, nullptr);
            unsigned done_bits = so.done;
            const bool finished = (so.done & (KIN_DONE_TERMINATED | KIN_DONE_TRUNCATED)) != 0u;
            if (finished) {
                push_truncated<OBS>(out, so.done, idx, [&](float* to) { build_obs_from(P, s, MODE, so.pe, so.oe, so.margin, to); });
                const unsigned episode = ld_row_u(state, stride, KIN_ROW_EPISODE, env) + 1u;
                Philox rng(reset_seed, (unsigned)env, episode);
                ResetDraw d;
                sample_reset(P, *SP, rng, MODE, d);
                float gq[NJ];
                reset_core(P, s, MODE, d.iq, d.idq, d.ipa, d.gq, d.has_gpose ? d.gpose : nullptr, gq);
                s.flags = (s.flags & ~(0xfu << KIN_FLAG_STAGE_SHIFT)) | ((unsigned)d.stage << KIN_FLAG_STAGE_SHIFT);
                store_env_reset(state, stride, env, s, gq);
                st_row_u(state, stride, KIN_ROW_EPISODE, env, episode);
                done_bits |= KIN_DONE_AUTORESET;
                pose_error(s.ee, s.goal, pe, oe);
#pragma unroll
                for (int i = 0; i < NJ; ++i) margin[i] = joint_margin(P, s.q[i], i);
            } else {
#pragma unroll
                for (int k = 0; k < 3; ++k) { pe[k] = so.pe[k]; oe[k] = so.oe[k]; }
#pragma unroll
                for (int i = 0; i < NJ; ++i) margin[i] = so.margin[i];
            }
            out.reward[idx] = so.reward;
            out.done[idx] = (uint8_t)done_bits;
            start = finished ? 1u : 0u;
        }
        // ---- value of the observation after the last step (GAE bootstrap)
        float o[OBS], mv[8];
        build_obs_from(P, s, MODE, pe, oe, margin, o);
        policy_forward<IN, true>(S.w, c, o, nullptr, mv);
        out.last_value[env] = mv[7];
        out.start_io[env] = (uint8_t)start;
        store_env_step(state, stride, env, s);
    }
    release_tiles<TILES>(S, tid);
}

// r[idx] += gamma * V(terminal_obs) for the truncated episodes the collection kernel listed (strict fp32 critic)
// POP: params carries the KinPopMember table, member blockIdx.y's list, critic, rewards and gamma replace the arguments.  The route
// population passes one extra argument, the element offset of the chunk's first reward row (list indices are relative to the chunk).
template <int IN, bool POP = false, class... PopArgs>
__global__ void __launch_bounds__(128)
kin_bootstrap_list_kernel(const float* __restrict__ params, const float* __restrict__ boot_obs, const int* __restrict__ boot_index,
                          const int* __restrict__ boot_count, int cap, float* __restrict__ reward, float gamma, PopArgs... pop) {
    static_assert(sizeof...(PopArgs) <= (POP ? 1 : 0), "the chunk offset is a population argument");
    if constexpr (POP) {
        const KinPopMember& M = reinterpret_cast<const KinPopMember*>(params)[blockIdx.y];
        params = M.params;
        boot_obs = M.boot_obs;
        boot_index = M.boot_index;
        boot_count = M.boot_count;
        cap = M.boot_cap;
        reward = M.reward;
        gamma = M.hyper.gamma;
        if constexpr (sizeof...(PopArgs) == 1) reward += (pop, ...);
    }
    const PpoOffsets O = ppo_offsets(IN);
    const int count = min(*boot_count, cap);
    const int i = blockIdx.x * 128 + threadIdx.x;
    if (blockIdx.x * 128 >= count) return;       // block-uniform
    __shared__ float h1[128][65];
    const int ic = min(i, count - 1);
    float x[IN];
    const float4* src = reinterpret_cast<const float4*>(boot_obs + (size_t)ic * IN);
#pragma unroll
    for (int k = 0; k < IN / 4; ++k) {
        const float4 v = __ldg(src + k);
        x[4 * k] = v.x; x[4 * k + 1] = v.y; x[4 * k + 2] = v.z; x[4 * k + 3] = v.w;
    }
    float* mine = h1[threadIdx.x];
    for (int u = 0; u < 64; ++u) {
        const float* w = params + O.vf_w0 + u * IN;
        float acc = __ldg(params + O.vf_b0 + u);
#pragma unroll
        for (int k = 0; k < IN; ++k) acc = fmaf(__ldg(w + k), x[k], acc);
        mine[u] = tanhf(acc);
    }
    float v = __ldg(params + O.val_b);
    for (int u = 0; u < 64; ++u) {
        const float* w = params + O.vf_w1 + u * 64;
        float acc = __ldg(params + O.vf_b1 + u);
#pragma unroll 16
        for (int k = 0; k < 64; ++k) acc = fmaf(__ldg(w + k), mine[k], acc);
        v = fmaf(__ldg(params + O.val_w + u), tanhf(acc), v);
    }
    if (i < count) reward[boot_index[i]] += gamma * v;
}

template <int TILES>
static cudaError_t launch_collect(const KinHandle* h, float* state, int stride, int n, int mode, const float* params, const unsigned char* wimg, int T,
                                  uint64_t noise_seed, uint32_t step0, uint64_t reset_seed, const CollectOut& out, cudaStream_t st) {
    auto kernel = mode == KIN_MODE_APPROACH ? kin_collect_kernel<TILES, KIN_MODE_APPROACH> : kin_collect_kernel<TILES, KIN_MODE_DOCK>;
    return launch_tiles<TILES>(kernel, sizeof(CollectSmem<TILES>) + 1024, n, st, h->params, h->d_sampler, state, stride, n, params, wimg, T, noise_seed,
                               step0, reset_seed, out);
}

__global__ void kin_pop_zero_counts_kernel(const KinPopMember* __restrict__ members, int n_members) {
    if ((int)threadIdx.x < n_members) *members[threadIdx.x].boot_count = 0;
}

cudaError_t pop_zero_boot_counts(const KinPopMember* members, int n_members, cudaStream_t st) {
    kin_pop_zero_counts_kernel<<<1, KIN_POP_MAX, 0, st>>>(members, n_members);
    return cudaGetLastError();
}

}  // namespace kin

using namespace kin;

extern "C" int kin_ppo_collect(void* handle, float* state, int stride, int n_envs, int mode, const float* params, const void* weight_image, int in_dim, int n_steps,
                               uint64_t noise_seed, uint32_t first_step, uint64_t reset_seed, void* obs_tiles, float* action, float* logp, float* value,
                               float* reward, uint8_t* done, uint8_t* episode_start, uint8_t* start_io, float* last_value, int* boot_count,
                               int* boot_index, float* boot_obs, int boot_cap, int tiles_per_cta, void* stream) {
    KinHandle* h = kin_handle(handle);
    if (!h) return kin_fail(KIN_ERR_INVALID_ARG, "kin_ppo_collect: bad handle");
    if (!h->d_sampler) return kin_fail(KIN_ERR_INVALID_ARG, "kin_ppo_collect: auto-reset needs kin_params_set_sampler");
    if (!state || !params || !obs_tiles || !action || !logp || !value || !reward || !done || !episode_start || !start_io || !last_value || !boot_count ||
        !boot_index || !boot_obs || boot_cap <= 0 || n_steps <= 0)
        return kin_fail(KIN_ERR_INVALID_ARG, "kin_ppo_collect: null buffer or bad sizes");
    if (in_dim != 56) return kin_fail(KIN_ERR_UNSUPPORTED, "kin_ppo_collect: in_dim must be 56");
    if (n_envs <= 0 || (n_envs % AC_ROWS) != 0 || stride < n_envs || (stride % 32) != 0)
        return kin_fail(KIN_ERR_INVALID_ARG, "kin_ppo_collect: n_envs must be a positive multiple of 128 (one GEMM tile), stride % 32 == 0");
    if (mode != KIN_MODE_APPROACH && mode != KIN_MODE_DOCK) return kin_fail(KIN_ERR_UNSUPPORTED, "kin_ppo_collect: mode must be approach (0) or dock (1)");
    if (((uintptr_t)obs_tiles & 15u) || ((uintptr_t)boot_obs & 15u)) return kin_fail(KIN_ERR_INVALID_ARG, "kin_ppo_collect: obs_tiles / boot_obs must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    const int tiles = collect_tiles_per_cta(tiles_per_cta, n_envs);
    CollectOut out{(unsigned char*)obs_tiles, action, logp, value, reward, done, episode_start, start_io, last_value, boot_count, boot_index, boot_obs, boot_cap};
    cudaError_t e = cudaMemsetAsync(boot_count, 0, sizeof(int), st);
    if (e != cudaSuccess) return kin_fail_cuda(e, "kin_ppo_collect: memset");
    if (tiles == 1) e = launch_collect<1>(h, state, stride, n_envs, mode, params, static_cast<const unsigned char*>(weight_image), n_steps, noise_seed, first_step, reset_seed, out, st);
    else if (tiles == 2) e = launch_collect<2>(h, state, stride, n_envs, mode, params, static_cast<const unsigned char*>(weight_image), n_steps, noise_seed, first_step, reset_seed, out, st);
    else if (tiles == 4) e = launch_collect<4>(h, state, stride, n_envs, mode, params, static_cast<const unsigned char*>(weight_image), n_steps, noise_seed, first_step, reset_seed, out, st);
    else return kin_fail(KIN_ERR_INVALID_ARG, "kin_ppo_collect: tiles_per_cta must be 0 (auto), 1, 2 or 4");
    return e == cudaSuccess ? KIN_OK : kin_fail_cuda(e, "kin_ppo_collect");
}

extern "C" int kin_ppo_bootstrap_list(const float* params, int in_dim, const float* boot_obs, const int* boot_index, const int* boot_count, int boot_cap,
                                      float* reward, float gamma, void* stream) {
    if (!params || !boot_obs || !boot_index || !boot_count || !reward || boot_cap <= 0) return kin_fail(KIN_ERR_INVALID_ARG, "kin_ppo_bootstrap_list: bad arguments");
    if (in_dim != 56 && in_dim != 80) return kin_fail(KIN_ERR_UNSUPPORTED, "kin_ppo_bootstrap_list: in_dim must be 56 or 80");
    if (in_dim == 56) kin_bootstrap_list_kernel<56><<<(boot_cap + 127) / 128, 128, 0, (cudaStream_t)stream>>>(params, boot_obs, boot_index, boot_count, boot_cap, reward, gamma);
    else kin_bootstrap_list_kernel<80><<<(boot_cap + 127) / 128, 128, 0, (cudaStream_t)stream>>>(params, boot_obs, boot_index, boot_count, boot_cap, reward, gamma);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KIN_OK : kin_fail_cuda(e, "kin_ppo_bootstrap_list");
}

extern "C" int kin_pop_collect(void* handle, const KinPopMember* members, int n_members, int n_envs, int mode, int n_steps, void* stream) {
    KinHandle* h = kin_handle(handle);
    if (!h) return kin_fail(KIN_ERR_INVALID_ARG, "kin_pop_collect: bad handle");
    if (!members || n_members <= 0 || n_members > KIN_POP_MAX || n_steps <= 0)
        return kin_fail(KIN_ERR_INVALID_ARG, "kin_pop_collect: need a device member table, 1 <= n_members <= KIN_POP_MAX and n_steps > 0");
    if (n_envs <= 0 || (n_envs % AC_ROWS) != 0) return kin_fail(KIN_ERR_INVALID_ARG, "kin_pop_collect: n_envs must be a positive multiple of 128 (one GEMM tile)");
    if (mode != KIN_MODE_APPROACH && mode != KIN_MODE_DOCK) return kin_fail(KIN_ERR_UNSUPPORTED, "kin_pop_collect: mode must be approach (0) or dock (1)");
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = pop_zero_boot_counts(members, n_members, st);      // kin_ppo_collect's reset of *boot_count
    if (e != cudaSuccess) return kin_fail_cuda(e, "kin_pop_collect: zero counts");
    auto kernel = mode == KIN_MODE_APPROACH ? kin_collect_kernel<1, KIN_MODE_APPROACH, true> : kin_collect_kernel<1, KIN_MODE_DOCK, true>;
    const size_t smem = sizeof(CollectSmem<1>) + 1024;
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return kin_fail_cuda(e, "kin_pop_collect: smem attribute");
    kernel<<<dim3((unsigned)(n_envs / AC_ROWS), (unsigned)n_members), AC_ROWS, smem, st>>>(h->params, reinterpret_cast<const KinSamplerParams*>(members), nullptr, 0,
                                                                                          n_envs, nullptr, nullptr, n_steps, 0, 0u, 0, CollectOut{});
    e = cudaGetLastError();
    return e == cudaSuccess ? KIN_OK : kin_fail_cuda(e, "kin_pop_collect");
}

extern "C" int kin_pop_bootstrap_list(const KinPopMember* members, int n_members, int max_boot_cap, void* stream) {
    if (!members || n_members <= 0 || n_members > KIN_POP_MAX || max_boot_cap <= 0)
        return kin_fail(KIN_ERR_INVALID_ARG, "kin_pop_bootstrap_list: need a device member table, 1 <= n_members <= KIN_POP_MAX and max_boot_cap > 0");
    // blocks past a member's own count return at once (block-uniform), so one grid sized for the largest list serves every member
    kin_bootstrap_list_kernel<56, true><<<dim3((unsigned)((max_boot_cap + 127) / 128), (unsigned)n_members), 128, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const float*>(members), nullptr, nullptr, nullptr, 0, nullptr, 0.0f);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KIN_OK : kin_fail_cuda(e, "kin_pop_bootstrap_list");
}

extern "C" int kin_pop_route_bootstrap_list(const KinPopMember* members, int n_members, int n_envs, int max_boot_cap, int t0, void* stream) {
    if (!members || n_members <= 0 || n_members > KIN_POP_MAX || n_envs <= 0 || max_boot_cap <= 0 || t0 < 0)
        return kin_fail(KIN_ERR_INVALID_ARG, "kin_pop_route_bootstrap_list: need a device member table, 1 <= n_members <= KIN_POP_MAX, n_envs > 0, "
                                             "max_boot_cap > 0 and t0 >= 0");
    kin_bootstrap_list_kernel<80, true, long long><<<dim3((unsigned)((max_boot_cap + 127) / 128), (unsigned)n_members), 128, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const float*>(members), nullptr, nullptr, nullptr, 0, nullptr, 0.0f, (long long)t0 * n_envs);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KIN_OK : kin_fail_cuda(e, "kin_pop_route_bootstrap_list");
}
