// kernels.cuh -- parameter blocks and launchers shared between the translation units.
#pragma once
#include "common.cuh"

namespace mmf {

struct ResampleParams {
  int N, M, sd, M_out;
  int estimation, mode;
  float alpha;
  const float* states;
  const float* logw_unnorm;  // ignored when logits_in != null
  const float* logits_in;    // standalone mmf_resample(): logits given directly
  const double* uniforms;
  float* states_out;
  float* logw_out;
  float* est_out;
  float* logw_norm_out;
  float* logits_out;
  long long* idx_out;
  int prefetch = 0;  // k_resample_fast: request the trajectory's particles / uniforms from HBM up front
};

constexpr int EKF_MAX_FILTERS = 4;
constexpr int EKF_MAX_WARPS = 16;

struct EkfParams {
  ChainDev dyn[EKF_MAX_FILTERS];
  TrajRowsDev rows[EKF_MAX_FILTERS];
  float q[EKF_MAX_FILTERS][MMF_MAX_SD * MMF_MAX_SD];
  int F, T, N, cd, jac_only;
  const float* mean0;     // (F, N, sd)
  const float* cov0;      // (F, N, sd, sd)
  const float* controls;  // (T, N, cd)   shared by all filters
  const float* z;         // (F, T, N, sd)
  const float* r_tril;    // (F, T, N, sd, sd)
  float* mean_out;        // (F, T, N, sd)      [jac_only: pred (N, sd)]
  float* cov_out;         // (F, T, N, sd, sd)  [jac_only: jacobian (N, sd, sd)]
  float* pred_out;        // (F, T, N, sd)      tape: mu- of every step   (launch_ekf(..., tape = true) only)
  float* jac_out;         // (F, T, N, sd, sd)  tape: A of every step
};

// Reverse mode of the EKF recursion (k_ekf_loop_bwd); d_means / d_covs may be NULL (= zero).
struct EkfBwdParams {
  float q[EKF_MAX_FILTERS][MMF_MAX_SD * MMF_MAX_SD];
  int F, T, N;
  const float* cov0;      // (F, N, sd, sd)
  const float* z;         // (F, T, N, sd)
  const float* r_tril;    // (F, T, N, sd, sd)
  const float* covs;      // (F, T, N, sd, sd)  posteriors of the forward
  const float* pred;      // (F, T, N, sd)      tape
  const float* jac;       // (F, T, N, sd, sd)  tape
  const float* d_means;   // (F, T, N, sd)
  const float* d_covs;    // (F, T, N, sd, sd)
  float* d_mean0;         // (F, N, sd)
  float* d_cov0;          // (F, N, sd, sd)
  float* d_z;             // (F, T, N, sd)
  float* d_r_tril;        // (F, T, N, sd, sd)
};

int launch_particle_chain_ffma(const mmf_pf_model* model, int N, int M, const float* states_in, const float* eps,
                               const float* rowbias, const float* logw_in, const float* modw, uint32_t enabled,
                               float* states_out, float* logw_out, float* ll_out, cudaStream_t stream,
                               int rb_stride = 0);
int launch_particle_chain_tc(const mmf_pf_model* model, int N, int M, const float* states_in, const float* eps,
                             const float* rowbias, const float* logw_in, const float* modw, uint32_t enabled,
                             int precision, float* states_out, float* logw_out, float* ll_out, cudaStream_t stream,
                             int first_chain = 0, float* act_out = nullptr, int rb_stride = 0);
int launch_traj_rows(const mmf_pf_model* model, int N, const float* controls, const float* const* obs_feats,
                     float* out, cudaStream_t stream);
int launch_fuse_loglik(int N, int M, int K, const float* ll, const float* w, float* out, cudaStream_t stream);
int launch_pf_init(int N, int M, int sd, const float* mean, const float* cov, const float* eps, float* states,
                   float* logw, cudaStream_t stream);
int launch_normalize_resample(const ResampleParams& P, void* workspace, cudaStream_t stream);
size_t resample_workspace_bytes(int N, int M);
int launch_ekf(const EkfParams& P, int sd, cudaStream_t stream, bool tape = false);
int launch_ekf_bwd(const EkfBwdParams& P, int sd, cudaStream_t stream);
int launch_reweight_train(int N, int M, int K, int sd, uint32_t enabled, const float* ll, const float* w, const float* logw_in,
                          const float* states, float* logw_out, float* est_out, const float* d_est, const float* d_logw,
                          float* d_ll, float* d_w, float* d_logw_in, bool backward, cudaStream_t stream);
bool resample_big_applies(int N, int M, bool soft);
size_t resample_big_workspace_bytes(int N, int M);
int launch_resample_big(const ResampleParams& P, void* workspace, cudaStream_t stream);
bool pf_loop_small_applies(int N, int M);
int launch_pf_loop_small(const mmf_pf_model* model, int T, int N, int M, float* states, float* logw, const float* rowbias,
                         const float* modw, uint32_t enabled, int precision, const float* eps, int estimation, int mode,
                         const double* uniforms, float* states_ws, float* logw_ws, float* est_out, cudaStream_t stream);
int launch_kf_fuse_measurements(int K, long long rows, int sd, const float* z, const float* tril, const float* w,
                                float* z_out, float* mat_out, int unimodal, cudaStream_t stream);
int launch_kf_fuse(int K, long long rows, int sd, const float* mu, const float* Pk, const float* beta,
                   float* mean_out, float* cov_out, int unimodal, cudaStream_t stream);
size_t chain_bwd_bytes(const mmf_chain* chain);
int pack_chain_bwd(const mmf_chain* chain, void* dst, cudaStream_t stream);
int launch_head_chain_bwd(const mmf_pf_model* model, int N, int M, const float* act, const float* d_ll, uint32_t enabled,
                          float* delta_out, cudaStream_t stream);
size_t heads_dw_workspace_bytes(int K, int L, long long P);
int launch_heads_dw(int K, int L, long long P, int sd, const float* act, const float* delta, const float* x,
                    const float* d_ll, float* dW, float* db, float* g_in, float* g_out, void* workspace,
                    cudaStream_t stream);
size_t enc_map_bytes_host(int channels);
size_t enc_trunk_weight_bytes();
size_t enc_trunk_scratch_bytes();
int launch_enc_trunk(int n_images, int cout, const float* images, const void* weights, void* scratch, float* out_nchw,
                     cudaStream_t stream);
int launch_enc_stem(int n_images, const float* images, const float* w, void* out_map, cudaStream_t stream);
int launch_enc_conv3x3(int n_images, int cin, int cout, const void* in_map, const void* w_image, const void* res_map,
                       int relu, void* out_map, float* out_nchw, cudaStream_t stream);
int launch_row_mlp(long long rows, const mmf_mlp_op* ops, int n_ops, const float* weights, const float* const* inputs,
                   const int32_t* in_dims, const int32_t* in_slots, int n_inputs, float* const* outputs,
                   const int32_t* out_dims, const int32_t* out_slots, int n_outputs, int scratch, cudaStream_t stream);
size_t chain_mma_bytes(const mmf_chain* chain);
int pack_chain_mma(const mmf_chain* chain, void* dst, cudaStream_t stream);

}  // namespace mmf
