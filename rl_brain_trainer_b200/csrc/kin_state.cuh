// kin_state.cuh -- HBM layout helpers: struct-of-arrays state rows, warp-tile staging of the
// row-major [n,56] observation / [n,7] action tensors through shared memory, Philox RNG and the
// device-side reset samplers.
#pragma once

#include <cstdint>

#include "kin_core.cuh"
#include "kin_umma.cuh"

namespace kin {

constexpr int WARP = 32;
constexpr int OBS = KIN_OBS_DIM;
constexpr int OBS_TILE_FLOATS = WARP * OBS;          // 1792 floats = 7168 B per warp
constexpr int OBS_TILE_BYTES = OBS_TILE_FLOATS * 4;

// ---- SoA rows: state[row * stride + env] -------------------------------------------------------
__device__ __forceinline__ float ld_row(const float* __restrict__ st, int stride, int row, int env) { return st[(size_t)row * stride + env]; }
__device__ __forceinline__ unsigned ld_row_u(const float* __restrict__ st, int stride, int row, int env) {
    return __float_as_uint(st[(size_t)row * stride + env]);
}
__device__ __forceinline__ void st_row(float* __restrict__ st, int stride, int row, int env, float v) { st[(size_t)row * stride + env] = v; }
__device__ __forceinline__ void st_row_u(float* __restrict__ st, int stride, int row, int env, unsigned v) {
    st[(size_t)row * stride + env] = __uint_as_float(v);
}

// rows the step reads: q, dq, prev_action, goal pose, ee pose, min_pos, counters, flags (37 words = 148 B),
// + the 4 entry metrics in dock mode (16 B).
template <bool WITH_ENTRY>
__device__ __forceinline__ void load_env(const float* __restrict__ st, int stride, int env, EnvRegs& s) {
#pragma unroll
    for (int i = 0; i < NJ; ++i) {
        s.q[i] = ld_row(st, stride, KIN_ROW_Q + i, env);
        s.dq[i] = ld_row(st, stride, KIN_ROW_DQ + i, env);
        s.pa[i] = ld_row(st, stride, KIN_ROW_PREV_ACTION + i, env);
    }
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        s.goal[k] = ld_row(st, stride, KIN_ROW_GOAL_POSE + k, env);
        s.ee[k] = ld_row(st, stride, KIN_ROW_EE_POSE + k, env);
    }
    s.min_pos = ld_row(st, stride, KIN_ROW_MIN_POS, env);
    unsigned c0 = ld_row_u(st, stride, KIN_ROW_CNT0, env), c1 = ld_row_u(st, stride, KIN_ROW_CNT1, env);
    s.step = (int)(c0 & 0xffffu);
    s.dwell = (int)(c0 >> 16);
    s.entry_cnt = (int)(c1 & 0xffffu);
    s.drift_cnt = (int)(c1 >> 16);
    s.flags = ld_row_u(st, stride, KIN_ROW_FLAGS, env);
    if (WITH_ENTRY) {
#pragma unroll
        for (int k = 0; k < 4; ++k) s.entry[k] = ld_row(st, stride, KIN_ROW_ENTRY + k, env);
    } else {
#pragma unroll
        for (int k = 0; k < 4; ++k) s.entry[k] = 0.0f;
    }
}

// rows the step writes: q, dq, prev_action, ee pose, min_pos, counters, flags (31 words = 124 B)
__device__ __forceinline__ void store_env_step(float* __restrict__ st, int stride, int env, const EnvRegs& s) {
#pragma unroll
    for (int i = 0; i < NJ; ++i) {
        st_row(st, stride, KIN_ROW_Q + i, env, s.q[i]);
        st_row(st, stride, KIN_ROW_DQ + i, env, s.dq[i]);
        st_row(st, stride, KIN_ROW_PREV_ACTION + i, env, s.pa[i]);
    }
#pragma unroll
    for (int k = 0; k < 6; ++k) st_row(st, stride, KIN_ROW_EE_POSE + k, env, s.ee[k]);
    st_row(st, stride, KIN_ROW_MIN_POS, env, s.min_pos);
    st_row_u(st, stride, KIN_ROW_CNT0, env, (unsigned)min(s.step, 0xffff) | ((unsigned)min(s.dwell, 0xffff) << 16));
    st_row_u(st, stride, KIN_ROW_CNT1, env, (unsigned)min(s.entry_cnt, 0xffff) | ((unsigned)min(s.drift_cnt, 0xffff) << 16));
    st_row_u(st, stride, KIN_ROW_FLAGS, env, s.flags);
}

// everything a reset defines (adds goal pose, entry metrics, goal_q)
__device__ __forceinline__ void store_env_reset(float* __restrict__ st, int stride, int env, const EnvRegs& s, const float* goal_q) {
    store_env_step(st, stride, env, s);
#pragma unroll
    for (int k = 0; k < 6; ++k) st_row(st, stride, KIN_ROW_GOAL_POSE + k, env, s.goal[k]);
#pragma unroll
    for (int k = 0; k < 4; ++k) st_row(st, stride, KIN_ROW_ENTRY + k, env, s.entry[k]);
#pragma unroll
    for (int i = 0; i < NJ; ++i) st_row(st, stride, KIN_ROW_GOAL_Q + i, env, goal_q[i]);
}

// ---- warp tiles ---------------------------------------------------------------------------------
// The [n,7] action tensor is row-major: a warp's 32 rows are 224 contiguous floats.  Load them
// coalesced into the warp's smem tile, then each lane reads its 7 (stride 7 words: conflict-free).
__device__ __forceinline__ void load_action_tile(const float* __restrict__ action, int env0, int n, float* tile, int lane, float* a) {
    const int valid = min(WARP, n - env0) * NJ;
    const float* src = action + (size_t)env0 * NJ;
#pragma unroll
    for (int k = 0; k < NJ; ++k) {
        int idx = lane + WARP * k;
        tile[idx] = idx < valid ? __ldg(src + idx) : 0.0f;
    }
    __syncwarp();
#pragma unroll
    for (int k = 0; k < NJ; ++k) a[k] = tile[lane * NJ + k];
    __syncwarp();
}

// The [n,56] observation tensor is row-major: a warp's 32 rows are one contiguous 7168-byte span.
// Lanes write their row into the smem tile with 128-bit stores, then ONE lane hands the whole span
// to the TMA engine (cp.async.bulk shared -> global, SASS UBLKCP) so no LSU store slots are spent
// on the 224 B/env that dominate the kernel's traffic.
__device__ __forceinline__ void stage_obs_row(float* tile, int lane, const float* o) {
    float4* dst = reinterpret_cast<float4*>(tile + lane * OBS);
#pragma unroll
    for (int k = 0; k < OBS / 4; ++k) dst[k] = make_float4(o[4 * k], o[4 * k + 1], o[4 * k + 2], o[4 * k + 3]);
}

__device__ __forceinline__ void bulk_store_tile(float* __restrict__ gdst, const float* tile, int bytes, int lane) {
    // make the generic-proxy smem writes visible to the async proxy, then one elected lane issues the copy
    umma::fence_async_smem();
    __syncwarp();
    if (lane == 0 && bytes > 0) {
        umma::bulk_store(gdst, umma::smem_u32(tile), bytes);
        umma::bulk_commit();
    }
}
// smem may be overwritten / the CTA may exit only after the bulk engine has READ the tile
__device__ __forceinline__ void bulk_store_wait_read(int lane) {
    if (lane == 0) umma::bulk_wait_read();
    __syncwarp();
}

// LSU fallback of the same tile write (kept for A/B measurement)
__device__ __forceinline__ void lsu_store_tile(float* __restrict__ gdst, const float* tile, int bytes, int lane) {
    __syncwarp();
    const float4* src = reinterpret_cast<const float4*>(tile);
    float4* dst = reinterpret_cast<float4*>(gdst);
    const int n16 = bytes >> 4;
#pragma unroll
    for (int k = 0; k < OBS_TILE_BYTES / 16 / WARP; ++k) {
        int idx = lane + WARP * k;
        if (idx < n16) dst[idx] = src[idx];
    }
    __syncwarp();
}

// ---- Philox4x32-10 counter RNG (key = seed ^ env, counter = (episode, draw)) --------------------
struct Philox {
    uint32_t k0, k1;
    uint32_t c0, c1, c2, c3;
    uint32_t out[4];
    int have;
    __device__ __forceinline__ Philox(uint64_t seed, uint32_t env, uint32_t episode)
        : k0((uint32_t)seed ^ (env * 0x9E3779B9u)), k1((uint32_t)(seed >> 32) ^ env), c0(0), c1(episode), c2(env), c3(0x5851F42Du), have(0) {}
    __device__ __forceinline__ void round4() {
        uint32_t a0 = c0, a1 = c1, a2 = c2, a3 = c3, x0 = k0, x1 = k1;
#pragma unroll
        for (int r = 0; r < 10; ++r) {
            uint32_t hi0 = __umulhi(0xD2511F53u, a0), lo0 = 0xD2511F53u * a0;
            uint32_t hi1 = __umulhi(0xCD9E8D57u, a2), lo1 = 0xCD9E8D57u * a2;
            uint32_t n0 = hi1 ^ a1 ^ x0, n1 = lo1, n2 = hi0 ^ a3 ^ x1, n3 = lo0;
            a0 = n0; a1 = n1; a2 = n2; a3 = n3;
            x0 += 0x9E3779B9u; x1 += 0xBB67AE85u;
        }
        out[0] = a0; out[1] = a1; out[2] = a2; out[3] = a3;
        c0 += 1;
        have = 4;
    }
    __device__ __forceinline__ uint32_t next_u32() {
        if (have == 0) round4();
        have -= 1;
        return out[have];
    }
    // uniform in [0, 1): 24 random bits
    __device__ __forceinline__ float uniform() { return (float)(next_u32() >> 8) * (1.0f / 16777216.0f); }
    __device__ __forceinline__ float uniform(float lo, float hi) { return fmaf(hi - lo, uniform(), lo); }
    // uniform integer in [lo, hi] (numpy rng.integers(lo, hi + 1))
    __device__ __forceinline__ int integers(int lo, int hi) {
        if (hi <= lo) return lo;
        uint32_t span = (uint32_t)(hi - lo + 1);
        return lo + (int)__umulhi(next_u32(), span);
    }
};

// two standard normals from one Philox pair (policy noise of the PPO rollout)
__device__ __forceinline__ float gauss_pair(Philox& rng, float* second) {
    // Box-Muller on two 24-bit uniforms in (0, 1]
    const float u1 = ((float)(rng.next_u32() >> 8) + 1.0f) * (1.0f / 16777216.0f);
    const float u2 = (float)(rng.next_u32() >> 8) * (1.0f / 16777216.0f);
    const float r = sqrtf(-2.0f * logf(u1));
    float s, c;
    sincosf(kTwoPi * u2, &s, &c);
    *second = r * s;
    return r * c;
}

// curriculum.py:90-101: base + U(-noise, noise) (only if any noise > 0), clipped to the limits
__device__ __forceinline__ void sample_shell(const KinEnvParams& P, Philox& rng, const float* base, const float* noise, float* q) {
    bool any = false;
#pragma unroll
    for (int i = 0; i < NJ; ++i) any |= noise[i] > 0.0f;
#pragma unroll
    for (int i = 0; i < NJ; ++i) {
        float v = base[i];
        if (any) v += rng.uniform(-noise[i], noise[i]);
        q[i] = clampf(v, P.joint_lower[i], P.joint_upper[i]);
    }
}

// joint_limits.py:124-137: uniform inside the margin-shrunk box
__device__ __forceinline__ void sample_box(const KinEnvParams& P, Philox& rng, float margin_fraction, float* q) {
#pragma unroll
    for (int i = 0; i < NJ; ++i) {
        float span = P.joint_upper[i] - P.joint_lower[i];
        float m = fmaxf(span * margin_fraction, 1e-6f);
        q[i] = rng.uniform(P.joint_lower[i] + m, P.joint_upper[i] - m);
    }
}

__device__ __forceinline__ int clampi(int v, int lo, int hi) { return min(max(v, lo), hi); }

// reset_samplers.py:344-389
__device__ __forceinline__ int sample_stage_index(const KinSamplerParams& S, Philox& rng) {
    const int current = clampi(S.current_stage, 0, max(S.n_stages - 1, 0));
    if (!S.stage_mix_enabled || current <= 0) return current;
    const float cr = fmaxf(S.current_stage_ratio, 0.0f), pr = fmaxf(S.previous_stage_ratio, 0.0f);
    const float orr = fmaxf(S.old_workspace_replay_ratio, 0.0f), fr = fmaxf(S.failure_replay_ratio, 0.0f);
    const float total = cr + pr + orr + fr;
    if (total <= 0.0f) return current;
    float draw = rng.uniform() * total;
    if (draw < cr) return current;
    draw -= cr;
    if (draw < pr) {
        int low = max(S.previous_stage_min_index, 0);
        int high = max(current - 1, low);
        return rng.integers(low, high);
    }
    draw -= pr;
    int old_max = clampi(S.old_workspace_max_stage_index, 0, min(S.n_stages - 1, current));
    if (draw < orr) return rng.integers(0, old_max);
    int replay_max = max(min(old_max, current - 1), 0);
    return replay_max > 0 ? rng.integers(0, replay_max) : current;
}

// reset_samplers.py:312-341
__device__ __forceinline__ int sample_target_stage(const KinSamplerParams& S, Philox& rng, int source, int current) {
    const int last = S.n_stages - 1;
    if (source == 0 || source == 1) return rng.integers(0, clampi(S.known_target_max_stage_index, 0, last));
    if (source == 3) {
        int lo = clampi(S.frontier_target_min_stage_index, 0, last);
        return rng.integers(lo, clampi(S.frontier_target_max_stage_index, lo, last));
    }
    if (source == 5) {
        int lo = clampi(S.stress_target_min_stage_index, 0, last);
        return rng.integers(lo, clampi(S.stress_target_max_stage_index, lo, last));
    }
    (void)current;
    return rng.integers(0, clampi(S.mixed_target_max_stage_index, 0, last));
}

struct ResetDraw {
    float iq[NJ], gq[NJ], idq[NJ], ipa[NJ];
    float gpose[6];      // explicit goal pose (handoff-state replay); otherwise the reset computes FK(goal_q)
    bool has_gpose;
    int stage;
};

// Adaptive frontier target (this project's extension, KinSamplerParams draw order step 3): alias-table bucket, uniform target in it.
// Returns the target's stage (current for a uniform-valid target).
__device__ __forceinline__ int sample_frontier_target(const KinSamplerParams& S, Philox& rng, int current, float* gq) {
    const int k = rng.integers(0, S.frontier_bucket_count - 1);
    const float u = rng.uniform();
    const int b = u < S.frontier_alias_prob[k] ? k : S.frontier_alias_index[k];
    const int j = rng.integers(S.frontier_bucket_offset[b], S.frontier_bucket_offset[b + 1] - 1);
    const float* t = S.frontier_targets + (size_t)j * KIN_FRONTIER_TARGET_FLOATS;
#pragma unroll
    for (int i = 0; i < NJ; ++i) gq[i] = t[i];
    const int st = (int)t[NJ];
    return st < 0 ? current : min(st, S.n_stages - 1);
}

// reset_samplers.py:213-309.  sources: 0 home, 1 old_success, 2 random_valid, 3 frontier, 4 failure_recovery, 5 stress
__device__ __forceinline__ void sample_random_start_pair(const KinEnvParams& P, const KinSamplerParams& S, Philox& rng, ResetDraw& d) {
    const int last = S.n_stages - 1;
    const int current = clampi(S.current_stage, 0, last);
    // the coin is drawn only when the table is armed: an unarmed sampler consumes exactly the reference-parity stream
    const bool from_table = S.frontier_probability > 0.0f && S.frontier_bucket_count > 0 && S.frontier_bucket_offset && S.frontier_alias_prob &&
                            S.frontier_alias_index && S.frontier_targets && rng.uniform() < S.frontier_probability;
    float total = 0.0f;
#pragma unroll
    for (int k = 0; k < 6; ++k) total += fmaxf(S.source_ratio[k], 0.0f);
    int source = 1;
    if (total > 0.0f) {
        float draw = rng.uniform() * total;
        bool found = false;
#pragma unroll
        for (int k = 0; k < 6; ++k) {
            float v = fmaxf(S.source_ratio[k], 0.0f);
            if (!found && draw <= v) { source = k; found = true; }
            if (!found) draw -= v;
        }
    }
    int tstage;
    if (from_table) {
        tstage = sample_frontier_target(S, rng, current, d.gq);
    } else {
        tstage = sample_target_stage(S, rng, source, current);
        sample_shell(P, rng, S.goal_q + tstage * NJ, S.goal_noise + tstage * NJ, d.gq);
    }
    if (source == 0) {
        int st = min(S.home_stage_index, last);
        sample_shell(P, rng, S.start_q + st * NJ, S.start_noise + st * NJ, d.iq);
    } else if (source == 1) {
        int st = rng.integers(0, clampi(S.old_success_max_stage_index, 0, last));
        sample_shell(P, rng, S.goal_q + st * NJ, S.goal_noise + st * NJ, d.iq);
    } else if (source == 3) {
        int lo = clampi(S.frontier_min_stage_index, 0, last);
        int st = rng.integers(lo, clampi(S.frontier_max_stage_index, lo, last));
        sample_shell(P, rng, S.start_q + st * NJ, S.start_noise + st * NJ, d.iq);
    } else if (source == 4) {
#pragma unroll
        for (int i = 0; i < NJ; ++i)
            d.iq[i] = clampf(d.gq[i] + rng.uniform(-S.failure_recovery_q_noise[i], S.failure_recovery_q_noise[i]), P.joint_lower[i], P.joint_upper[i]);
    } else if (source == 5) {
        sample_box(P, rng, S.stress_start_margin_fraction, d.iq);
    } else {
        sample_box(P, rng, S.random_valid_start_margin_fraction, d.iq);
    }
    bool any_dq = false, any_pa = false;
#pragma unroll
    for (int i = 0; i < NJ; ++i) { any_dq |= S.initial_dq_noise[i] > 0.0f; any_pa |= S.initial_prev_action_noise[i] > 0.0f; }
#pragma unroll
    for (int i = 0; i < NJ; ++i) d.idq[i] = any_dq ? rng.uniform(-S.initial_dq_noise[i], S.initial_dq_noise[i]) : 0.0f;
#pragma unroll
    for (int i = 0; i < NJ; ++i) d.ipa[i] = any_pa ? rng.uniform(-S.initial_prev_action_noise[i], S.initial_prev_action_noise[i]) : 0.0f;
    if (S.min_pair_joint_l2 > 0.0f) {
        for (int attempt = 0; attempt < 12; ++attempt) {
            float acc = 0.0f;
#pragma unroll
            for (int i = 0; i < NJ; ++i) acc = fmaf(d.gq[i] - d.iq[i], d.gq[i] - d.iq[i], acc);
            if (sqrtf(acc) >= S.min_pair_joint_l2) break;
            if (from_table) {
                tstage = sample_frontier_target(S, rng, current, d.gq);
            } else {
                tstage = sample_target_stage(S, rng, source, current);
                sample_shell(P, rng, S.goal_q + tstage * NJ, S.goal_noise + tstage * NJ, d.gq);
            }
        }
    }
#pragma unroll
    for (int i = 0; i < NJ; ++i) d.iq[i] = clampf(d.iq[i], P.joint_lower[i], P.joint_upper[i]);
    d.stage = tstage;
}

// sample_approach_reset (reset_samplers.py:168-210) / sample_dock_reset basic branch (:426-471)
__device__ __forceinline__ void sample_reset(const KinEnvParams& P, const KinSamplerParams& S, Philox& rng, int mode, ResetDraw& d) {
#pragma unroll
    for (int i = 0; i < NJ; ++i) { d.idq[i] = 0.0f; d.ipa[i] = 0.0f; }
    d.has_gpose = false;
    d.stage = clampi(S.current_stage, 0, max(S.n_stages - 1, 0));
    if (mode == KIN_MODE_DOCK) {
        // handoff-state replay (reset_samplers.py:434-446)
        if (S.dock_handoff_state_probability > 0.0f && S.dock_handoff_state_count > 0 && S.dock_handoff_states &&
            rng.uniform() < S.dock_handoff_state_probability) {
            const float* st = S.dock_handoff_states + (size_t)rng.integers(0, S.dock_handoff_state_count - 1) * KIN_HANDOFF_STATE_FLOATS;
#pragma unroll
            for (int i = 0; i < NJ; ++i) { d.iq[i] = st[i]; d.idq[i] = st[7 + i]; d.ipa[i] = st[14 + i]; d.gq[i] = st[21 + i]; }
#pragma unroll
            for (int k = 0; k < 6; ++k) d.gpose[k] = st[28 + k];
            d.has_gpose = true;
            return;
        }
        if (S.dock_use_stage_goal && S.curriculum_enabled && S.n_stages > 0)
            sample_shell(P, rng, S.goal_q + d.stage * NJ, S.goal_noise + d.stage * NJ, d.gq);
        else
            sample_shell(P, rng, S.dock_goal_q, S.dock_goal_noise, d.gq);
        // close bucket (reset_samplers.py:452-515): near-success but not-yet-success starts, best miss kept as the fallback
        if (S.dock_close_bucket_probability > 0.0f && rng.uniform() < S.dock_close_bucket_probability) {
            float goal_pose[6], best[NJ];
            fk_pose6(P, d.gq, goal_pose);
            float best_dist = CUDART_INF_F;
            bool have_best = false, found = false;
            const int attempts = max(S.dock_close_bucket_max_attempts, 1);
            for (int a = 0; a < attempts && !found; ++a) {
                float cand[NJ], pose[6], pe[3], oe[3];
#pragma unroll
                for (int i = 0; i < NJ; ++i)
                    cand[i] = clampf(d.gq[i] + rng.uniform(-S.dock_close_init_q_noise[i], S.dock_close_init_q_noise[i]), P.joint_lower[i], P.joint_upper[i]);
                fk_pose6(P, cand, pose);
                pose_error(pose, goal_pose, pe, oe);
                const float pos = norm3(pe[0], pe[1], pe[2]), ori = norm3(oe[0], oe[1], oe[2]);
                if (pos >= S.dock_close_bucket_min_pos_error_m && pos <= S.dock_close_bucket_max_pos_error_m &&
                    ori >= S.dock_close_bucket_min_ori_error_rad && ori <= S.dock_close_bucket_max_ori_error_rad) {
#pragma unroll
                    for (int i = 0; i < NJ; ++i) d.iq[i] = cand[i];
                    found = true;
                } else {
                    float dist;
                    if (pos < S.dock_close_bucket_min_pos_error_m) dist = S.dock_close_bucket_min_pos_error_m - pos;
                    else if (pos > S.dock_close_bucket_max_pos_error_m) dist = pos - S.dock_close_bucket_max_pos_error_m;
                    else dist = fmaxf(fmaxf(S.dock_close_bucket_min_ori_error_rad - ori, ori - S.dock_close_bucket_max_ori_error_rad), 0.0f);
                    if (dist < best_dist) {
                        best_dist = dist;
                        have_best = true;
#pragma unroll
                        for (int i = 0; i < NJ; ++i) best[i] = cand[i];
                    }
                }
            }
            if (!found) {
#pragma unroll
                for (int i = 0; i < NJ; ++i) d.iq[i] = have_best ? best[i] : clampf(d.gq[i], P.joint_lower[i], P.joint_upper[i]);
            }
            return;
        }
#pragma unroll
        for (int i = 0; i < NJ; ++i)
            d.iq[i] = clampf(d.gq[i] + rng.uniform(-S.dock_init_q_noise[i], S.dock_init_q_noise[i]), P.joint_lower[i], P.joint_upper[i]);
        return;
    }
    if (S.random_start_enabled && S.curriculum_enabled && S.n_stages > 0) {
        sample_random_start_pair(P, S, rng, d);
        return;
    }
    if (S.curriculum_enabled && S.n_stages > 0) {
        d.stage = sample_stage_index(S, rng);
        sample_shell(P, rng, S.start_q + d.stage * NJ, S.start_noise + d.stage * NJ, d.iq);
        sample_shell(P, rng, S.goal_q + d.stage * NJ, S.goal_noise + d.stage * NJ, d.gq);
    } else {
        sample_box(P, rng, S.start_sample_margin_fraction, d.iq);
        sample_box(P, rng, S.goal_sample_margin_fraction, d.gq);
    }
}

}  // namespace kin
