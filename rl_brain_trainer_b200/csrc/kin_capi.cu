// kin_capi.cu -- library-level entry points of the C ABI: version, errors, device info, handles.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>

#include "kin_internal.h"

namespace kin {

static thread_local char g_err[512] = "";

int kin_fail(int code, const char* msg) {
    snprintf(g_err, sizeof(g_err), "%s", msg);
    return code;
}

int kin_fail_cuda(cudaError_t e, const char* where) {
    snprintf(g_err, sizeof(g_err), "%s: CUDA error %d (%s)", where, (int)e, cudaGetErrorString(e));
    return KIN_ERR_CUDA;
}

bool kin_env_flag(const char* name) {
    const char* v = getenv(name);
    return v && v[0] && v[0] != '0';
}

}  // namespace kin

using namespace kin;

extern "C" int kin_abi_version(void) { return KIN_ABI_VERSION; }

#ifndef KIN_SOURCE_HASH
#define KIN_SOURCE_HASH "unstamped"
#endif
extern "C" const char* kin_source_hash(void) { return KIN_SOURCE_HASH; }

extern "C" const char* kin_last_error_string(void) { return g_err; }

extern "C" int kin_device_info(int* sm_count, int* cc_major, int* cc_minor, char* name, int name_len) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return kin_fail(KIN_ERR_NO_DEVICE, "kin_device_info: no CUDA device");
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, dev);
    if (e != cudaSuccess) return kin_fail_cuda(e, "kin_device_info");
    if (sm_count) *sm_count = prop.multiProcessorCount;
    if (cc_major) *cc_major = prop.major;
    if (cc_minor) *cc_minor = prop.minor;
    if (name && name_len > 0) snprintf(name, (size_t)name_len, "%s", prop.name);
    return KIN_OK;
}

static bool finite_all(const float* v, int n) {
    for (int i = 0; i < n; ++i)
        if (!std::isfinite(v[i])) return false;
    return true;
}

// ArmKinematicEnv.__init__ raises ValueError when len(joint_specs) != n_joints (arm_kinematic_env.py:76-77);
// here the joint count is fixed at 7 by the struct, so validation is about well-formed limits.
extern "C" int kin_params_create(const KinEnvParams* host_params, void** handle) {
    if (!host_params || !handle) return kin_fail(KIN_ERR_INVALID_ARG, "kin_params_create: null argument");
    const KinEnvParams& p = *host_params;
    if (!finite_all(p.joint_lower, 7) || !finite_all(p.joint_upper, 7) || !finite_all(p.joint_delta_limit, 7) ||
        !finite_all(p.fk_C, 54) || !finite_all(p.fk_t, 15) || !finite_all(p.fk_AT, 9) || !finite_all(p.fk_pbase, 3) || !finite_all(p.fk_pq0, 3))
        return kin_fail(KIN_ERR_INVALID_ARG, "kin_params_create: non-finite joint spec or FK constant");
    for (int i = 0; i < 7; ++i)
        if (!(p.joint_upper[i] > p.joint_lower[i])) return kin_fail(KIN_ERR_INVALID_ARG, "kin_params_create: joint upper must exceed lower");
    if (p.ar_n_milestones < 0 || p.ar_n_milestones > KIN_MAX_MILESTONES) return kin_fail(KIN_ERR_INVALID_ARG, "kin_params_create: too many orientation milestones (max 4)");
    if (p.term_max_episode_steps <= 0 || p.term_max_episode_steps > 65535) return kin_fail(KIN_ERR_INVALID_ARG, "kin_params_create: max_episode_steps must be in [1, 65535]");
    if (!(p.obs_pos_err_scale_m > 0.0f) || !(p.obs_ori_err_scale_rad > 0.0f)) return kin_fail(KIN_ERR_INVALID_ARG, "kin_params_create: observation scales must be positive");
    KinHandle* h = new (std::nothrow) KinHandle();
    if (!h) return kin_fail(KIN_ERR_INVALID_ARG, "kin_params_create: out of host memory");
    h->magic = KIN_HANDLE_MAGIC;
    h->params = p;
    h->d_sampler = nullptr;
    memset(&h->h_sampler, 0, sizeof(h->h_sampler));
    *handle = h;
    return KIN_OK;
}

extern "C" int kin_params_set_sampler(void* handle, const KinSamplerParams* host_sampler) {
    KinHandle* h = kin_handle(handle);
    if (!h || !host_sampler) return kin_fail(KIN_ERR_INVALID_ARG, "kin_params_set_sampler: bad argument");
    if (host_sampler->n_stages < 0 || host_sampler->n_stages > KIN_MAX_STAGES) return kin_fail(KIN_ERR_INVALID_ARG, "kin_params_set_sampler: at most 16 curriculum stages");
    const KinSamplerParams& s = *host_sampler;
    if (!std::isfinite(s.frontier_probability) || s.frontier_probability < 0.0f || s.frontier_probability > 1.0f)
        return kin_fail(KIN_ERR_INVALID_ARG, "kin_params_set_sampler: frontier_probability must be finite and in [0, 1]");
    if (s.frontier_probability > 0.0f) {
        if (s.frontier_bucket_count <= 0 || s.frontier_target_count <= 0)
            return kin_fail(KIN_ERR_INVALID_ARG, "kin_params_set_sampler: frontier_probability > 0 needs positive frontier bucket and target counts");
        if (!s.frontier_bucket_offset || !s.frontier_alias_prob || !s.frontier_alias_index || !s.frontier_targets)
            return kin_fail(KIN_ERR_INVALID_ARG, "kin_params_set_sampler: frontier_probability > 0 needs all four frontier table pointers");
        if (!s.random_start_enabled)
            return kin_fail(KIN_ERR_INVALID_ARG, "kin_params_set_sampler: frontier targets are drawn by the random-start pair sampler: enable random_start");
    }
    if (!h->d_sampler) {
        cudaError_t e = cudaMalloc(&h->d_sampler, sizeof(KinSamplerParams));
        if (e != cudaSuccess) return kin_fail_cuda(e, "kin_params_set_sampler: cudaMalloc");
    }
    h->h_sampler = *host_sampler;
    // stream-ordered against the legacy stream; callers update the sampler between rollouts, not inside them
    cudaError_t e = cudaMemcpy(h->d_sampler, &h->h_sampler, sizeof(KinSamplerParams), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) return kin_fail_cuda(e, "kin_params_set_sampler: cudaMemcpy");
    return KIN_OK;
}

extern "C" int kin_params_device_sampler(void* handle, const void** sampler) {
    KinHandle* h = kin_handle(handle);
    if (!h || !sampler) return kin_fail(KIN_ERR_INVALID_ARG, "kin_params_device_sampler: bad argument");
    *sampler = h->d_sampler;
    return KIN_OK;
}

extern "C" int kin_params_same_env(void* handle_a, void* handle_b, int* same) {
    KinHandle* a = kin_handle(handle_a);
    KinHandle* b = kin_handle(handle_b);
    if (!a || !b || !same) return kin_fail(KIN_ERR_INVALID_ARG, "kin_params_same_env: bad argument");
    *same = std::memcmp(&a->params, &b->params, sizeof(KinEnvParams)) == 0 ? 1 : 0;
    return KIN_OK;
}

extern "C" int kin_params_destroy(void* handle) {
    KinHandle* h = kin_handle(handle);
    if (!h) return kin_fail(KIN_ERR_INVALID_ARG, "kin_params_destroy: bad handle");
    if (h->d_sampler) cudaFree(h->d_sampler);
    h->magic = 0;
    delete h;
    return KIN_OK;
}
