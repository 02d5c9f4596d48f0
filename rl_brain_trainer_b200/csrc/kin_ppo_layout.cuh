// kin_ppo_layout.cuh -- flat parameter layout of the PPO trainer (PARAM_ORDER in ppo.py) shared by the update kernels.
#pragma once

#include "kin_internal.h"

namespace kin {

struct PpoOffsets {
    int pi_w0, pi_b0, pi_w1, pi_b1, act_w, act_b, vf_w0, vf_b0, vf_w1, vf_b1, val_w, val_b, log_std, total;
};
__host__ __device__ inline PpoOffsets ppo_offsets(int in_dim) {
    PpoOffsets o;
    int p = 0;
    o.pi_w0 = p; p += 64 * in_dim;
    o.pi_b0 = p; p += 64;
    o.pi_w1 = p; p += 4096;
    o.pi_b1 = p; p += 64;
    o.act_w = p; p += 7 * 64;
    o.act_b = p; p += 7;
    o.vf_w0 = p; p += 64 * in_dim;
    o.vf_b0 = p; p += 64;
    o.vf_w1 = p; p += 4096;
    o.vf_b1 = p; p += 64;
    o.val_w = p; p += 64;
    o.val_b = p; p += 1;
    o.log_std = p; p += 7;
    o.total = p;
    return o;
}

// ---- constant-folded layer-1 input of the 80-input route policy ---------------------------------------------------------------------
// 20 of the 80 route-observation columns are constants of the path (mode_flag one-hot = approach -> column 20 is 1, task_type = [1, 0, 0]
// -> column 71 is 1, the next_wp / wp blocks, progress[2], mode_flag[1..3], task_type[1..2] are 0).  The tensor-core kernels run layer 1 on
// the 60 live columns + a constant-one column (K = 64, ONE operand tile, like the 56-input policies) with the bias column holding
// b0 + W0[:, 20] + W0[:, 71]; the gradient of that column IS d b0 = d W0[:, 20] = d W0[:, 71], the zero columns get zero gradient --
// exactly what SB3 computes on the full 80 columns.
constexpr int KIN_ROUTE_DYN = 60;
// live column k (0..59) of the folded input -> column of the 80-float route observation
__host__ __device__ inline int route_unfold_col(int k) { return k < 20 ? k : (k < 29 ? k + 10 : k + 11); }
// column c (0..79) of the route observation -> folded column, or -1 for the constant columns
__host__ __device__ inline int route_fold_col(int c) { return c < 20 ? c : (c < 30 ? -1 : (c < 39 ? c - 10 : (c == 39 ? -1 : (c < 71 ? c - 11 : -1)))); }
constexpr int KIN_ROUTE_ONE_A = 20, KIN_ROUTE_ONE_B = 71;       // the two columns that are the constant 1
// effective layer-1 width of the tensor-core kernels (live columns; the bias rides in column `ppo_in_eff`)
__host__ __device__ inline int ppo_in_eff(int in_dim) { return in_dim == 80 ? KIN_ROUTE_DYN : in_dim; }

// ---- bf16 operand image of the weights (the B operands of the tensor-core kernels), 36 KB:
//   [W0 actor 8 KB][W0 critic 8 KB][W1 actor 8 KB][W1 critic 8 KB][WO actor 2 KB][WO critic 2 KB]
// every block a [rows][64 bf16] SWIZZLE_128B tile (kin_umma.cuh): W0 rows = hidden unit, col 56 = its bias, cols 57.. zero (the route
// policy: its 60 live columns, col 60 = the folded bias, see above -- built by kin_ppo_pack_weights only, not by wimg_offset);
// WO actor rows 0..6 = act_w, WO critic row 7 = val_w, other rows zero.  b1 / act_b / val_b / log_std stay fp32 in `params`.
constexpr int KIN_WIMG_BYTES = 36864;
constexpr int KIN_WIMG_W0 = 0, KIN_WIMG_W1 = 16384, KIN_WIMG_WO = 32768;
__host__ __device__ inline int wimg_elem(int row, int col) { return row * 128 + ((((col >> 3) ^ (row & 7)) << 4) | ((col & 7) << 1)); }
// byte offset of flat parameter p inside the image, or -1 when the parameter is not part of it
__host__ __device__ inline int wimg_offset(const PpoOffsets& o, int in_dim, int p) {
    if (p < o.pi_b0) return KIN_WIMG_W0 + wimg_elem((p - o.pi_w0) / in_dim, (p - o.pi_w0) % in_dim);
    if (p < o.pi_w1) return KIN_WIMG_W0 + wimg_elem(p - o.pi_b0, in_dim);
    if (p < o.pi_b1) return KIN_WIMG_W1 + wimg_elem((p - o.pi_w1) >> 6, (p - o.pi_w1) & 63);
    if (p < o.act_w) return -1;
    if (p < o.act_b) return KIN_WIMG_WO + wimg_elem((p - o.act_w) >> 6, (p - o.act_w) & 63);
    if (p < o.vf_w0) return -1;
    if (p < o.vf_b0) return KIN_WIMG_W0 + 8192 + wimg_elem((p - o.vf_w0) / in_dim, (p - o.vf_w0) % in_dim);
    if (p < o.vf_w1) return KIN_WIMG_W0 + 8192 + wimg_elem(p - o.vf_b0, in_dim);
    if (p < o.vf_b1) return KIN_WIMG_W1 + 8192 + wimg_elem((p - o.vf_w1) >> 6, (p - o.vf_w1) & 63);
    if (p < o.val_w) return -1;
    if (p < o.val_b) return KIN_WIMG_WO + 2048 + wimg_elem(7, p - o.val_w);
    return -1;
}

// grad[p] = sum over CTAs of partials[c][p] (rows of P + KIN_PPO_STATS + 8 floats); stats (nullable) likewise, scaled
int kin_ppo_reduce_launch(const float* partials, int n_cta, int P, float* grad, float* stats, float inv_global_batch, cudaStream_t st);
// the same reduction for every member of a population (partials / grad / stats from member blockIdx.y's descriptor)
int kin_pop_reduce_launch(const KinPopMember* members, int n_members, int n_cta, int P, float inv_global_batch, cudaStream_t st);


// kin_ppo_tc3.cu: the three-streams-per-SM form of the tensor-core gradient kernel.  Returns 0 when the call is not eligible (the caller
// launches the two-chain kernel), 1 when it was handled (*rc = KIN_OK or the error)
struct PeerFused;
int kin_ppo_grad_tc3_try(const float* params, const KinPpoHyper* hp, const void* images, const float* action, const float* old_logp,
                         const float* advantage, const float* returns, const double* tile_sums, const int* tile_ids, int n_pairs, float inv_global_batch,
                         float* partials, int grid, const float* adv_stats, const void* weight_image, const PeerFused& px, bool fused, cudaStream_t st,
                         int* rc);

}  // namespace kin
