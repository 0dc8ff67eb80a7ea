// api.cu -- the extern "C" surface declared in include/mmf_b200.h.
#include <stdarg.h>
#include <string.h>

#include "kernels.cuh"

namespace mmf {

static thread_local char g_error[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_error, sizeof(g_error), fmt, ap);
  va_end(ap);
}

int cuda_fail(cudaError_t err, const char* what) {
  set_error("CUDA error in %s: %s", what, cudaGetErrorString(err));
  return MMF_E_CUDA;
}

int validate_chain(const mmf_chain& c, int sd, int out_dim, const char* what) {
  MMF_REQUIRE(c.w != nullptr, "%s: packed weights are NULL", what);
  MMF_REQUIRE(((uintptr_t)c.w & 15) == 0, "%s: packed weights must be 16-byte aligned", what);
  MMF_REQUIRE(c.in_dim == sd, "%s: in_dim %d != state_dim %d", what, c.in_dim, sd);
  MMF_REQUIRE(c.out_dim == out_dim, "%s: out_dim %d != %d", what, c.out_dim, out_dim);
  MMF_REQUIRE(c.n_pre_res >= 0 && c.n_pre_res <= 4 && c.n_post_res >= 0 && c.n_post_res <= 8,
              "%s: unsupported resblock counts (%d, %d)", what, c.n_pre_res, c.n_post_res);
  return MMF_OK;
}

static int validate_pf_model(const mmf_pf_model* m) {
  MMF_REQUIRE(m != nullptr, "model is NULL");
  MMF_REQUIRE(m->state_dim >= 1 && m->state_dim <= MMF_MAX_SD, "state_dim %d outside 1..%d", m->state_dim, MMF_MAX_SD);
  MMF_REQUIRE(m->control_dim >= 1 && m->control_dim <= MMF_MAX_CD, "control_dim %d outside 1..%d", m->control_dim,
              MMF_MAX_CD);
  MMF_REQUIRE(m->num_heads >= 1 && m->num_heads <= MMF_MAX_HEADS, "num_heads %d outside 1..%d", m->num_heads,
              MMF_MAX_HEADS);
  int rc = validate_chain(m->dynamics, m->state_dim, m->state_dim + 1, "dynamics chain");
  if (rc) return rc;
  MMF_REQUIRE(m->dynamics_rows.w != nullptr && m->dynamics_rows.in_dim == m->control_dim,
              "dynamics_rows: in_dim %d != control_dim %d (or NULL weights)", m->dynamics_rows.in_dim, m->control_dim);
  for (int k = 0; k < m->num_heads; ++k) {
    rc = validate_chain(m->heads[k], m->state_dim, 1, "measurement head chain");
    if (rc) return rc;
    MMF_REQUIRE(m->head_rows[k].w != nullptr && m->head_rows[k].in_dim >= 1 &&
                    m->head_rows[k].in_dim <= MMF_MAX_OBS_FEATS,
                "head_rows[%d]: bad in_dim %d or NULL weights", k, m->head_rows[k].in_dim);
  }
  return MMF_OK;
}

}  // namespace mmf

using namespace mmf;

extern "C" {

const char* mmf_last_error(void) { return g_error; }

int mmf_abi_version(void) { return MMF_ABI_VERSION; }

int mmf_device_check(void) {
  int dev = 0;
  MMF_CUDA(cudaGetDevice(&dev));
  int major = 0, minor = 0;
  MMF_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  MMF_CUDA(cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev));
  if (major != 10) {
    set_error("libmmf_b200 is built for sm_100a only; device %d is sm_%d%d", dev, major, minor);
    return MMF_E_UNSUPPORTED;
  }
  return MMF_OK;
}

int mmf_pf_init(int32_t N, int32_t M, int32_t sd, const float* mean, const float* cov, const float* eps_MNsd,
                float* states_out, float* logw_out, void* stream) {
  MMF_REQUIRE(N >= 0 && M >= 1 && sd >= 1 && sd <= MMF_MAX_SD, "pf_init: bad shape N=%d M=%d sd=%d", N, M, sd);
  MMF_REQUIRE(N == 0 || (mean && cov && eps_MNsd && states_out && logw_out), "pf_init: NULL buffer");
  return launch_pf_init(N, M, sd, mean, cov, eps_MNsd, states_out, logw_out, (cudaStream_t)stream);
}

int mmf_pf_traj_rows(const mmf_pf_model* model, int32_t N, const float* controls, const float* const* obs_feats,
                     float* rowbias_out, void* stream) {
  int rc = validate_pf_model(model);
  if (rc) return rc;
  MMF_REQUIRE(N >= 0, "traj_rows: N=%d", N);
  MMF_REQUIRE(N == 0 || (controls && rowbias_out), "traj_rows: NULL buffer");
  return launch_traj_rows(model, N, controls, obs_feats, rowbias_out, (cudaStream_t)stream);
}

int mmf_pf_predict_measure(const mmf_pf_model* model, int32_t N, int32_t M, const float* states_in, const float* eps,
                           const float* rowbias, const float* logw_in, const float* modality_logw,
                           uint32_t enabled_mask, int32_t precision, float* states_out, float* logw_unnorm_out,
                           float* ll_out, void* stream) {
  int rc = validate_pf_model(model);
  if (rc) return rc;
  MMF_REQUIRE(N >= 0 && M >= 1, "predict_measure: bad shape N=%d M=%d", N, M);
  if (N == 0) return MMF_OK;
  MMF_REQUIRE(states_in && eps && rowbias && logw_in && states_out && logw_unnorm_out, "predict_measure: NULL buffer");
  const uint32_t all = (1u << model->num_heads) - 1u;
  MMF_REQUIRE((enabled_mask & all) != 0, "predict_measure: no measurement head enabled (mask 0x%x)", enabled_mask);
  enabled_mask &= all;
  if (precision == MMF_PREC_FP32)
    return launch_particle_chain_ffma(model, N, M, states_in, eps, rowbias, logw_in, modality_logw, enabled_mask,
                                      states_out, logw_unnorm_out, ll_out, (cudaStream_t)stream);
  if (precision == MMF_PREC_BF16X3 || precision == MMF_PREC_BF16)
    return launch_particle_chain_tc(model, N, M, states_in, eps, rowbias, logw_in, modality_logw, enabled_mask,
                                    precision, states_out, logw_unnorm_out, ll_out, (cudaStream_t)stream);
  set_error("predict_measure: unknown precision mode %d", precision);
  return MMF_E_INVALID;
}

int mmf_pf_forward_loop(const mmf_pf_model* model, int32_t T, int32_t N, int32_t M, float* states, float* logw,
                        const float* controls, const float* const* obs_feats, const float* modality_logw,
                        uint32_t enabled_mask, int32_t precision, const float* eps, int32_t estimation_method,
                        int32_t resample_mode, const double* uniforms, float* rowbias_ws, float* states_ws,
                        float* logw_ws, float* est_out, void* resample_ws, void* stream_) {
  int rc = validate_pf_model(model);
  if (rc) return rc;
  MMF_REQUIRE(T >= 0 && N >= 0 && M >= 1, "forward_loop: bad shape T=%d N=%d M=%d", T, N, M);
  if (T == 0 || N == 0) return MMF_OK;
  MMF_REQUIRE(states && logw && controls && obs_feats && eps && rowbias_ws && states_ws && logw_ws && est_out,
              "forward_loop: NULL buffer");
  MMF_REQUIRE(estimation_method == MMF_ESTIMATE_WEIGHTED_AVERAGE || estimation_method == MMF_ESTIMATE_ARGMAX,
              "forward_loop: unknown estimation method %d", estimation_method);
  MMF_REQUIRE(resample_mode >= MMF_RESAMPLE_NONE && resample_mode <= MMF_RESAMPLE_SYSTEMATIC_FAST,
              "forward_loop: unknown resample mode %d", resample_mode);
  MMF_REQUIRE(resample_mode == MMF_RESAMPLE_NONE || uniforms != nullptr, "forward_loop: resampling needs uniforms");
  MMF_REQUIRE(precision >= MMF_PREC_FP32 && precision <= MMF_PREC_BF16, "forward_loop: unknown precision mode %d", precision);
  MMF_REQUIRE((long long)T * N <= 0x7fffffffLL, "forward_loop: T * N = %lld rows exceed the hoisting kernel's range",
              (long long)T * N);
  const uint32_t all = (1u << model->num_heads) - 1u;
  MMF_REQUIRE((enabled_mask & all) != 0, "forward_loop: no measurement head enabled (mask 0x%x)", enabled_mask);
  enabled_mask &= all;
  cudaStream_t stream = (cudaStream_t)stream_;
  const int sd = model->state_dim, K = model->num_heads;
  const bool systematic = resample_mode == MMF_RESAMPLE_SYSTEMATIC_STRICT || resample_mode == MMF_RESAMPLE_SYSTEMATIC_FAST;
  // the per-trajectory rows of ALL steps in one launch: they do not depend on the particles
  rc = launch_traj_rows(model, T * N, controls, obs_feats, rowbias_ws, stream);
  if (rc) return rc;
  if (pf_loop_small_applies(N, M))  // small problem: the T steps in ONE launch, a CTA per trajectory (pf_loop_small.cu)
    return launch_pf_loop_small(model, T, N, M, states, logw, rowbias_ws, modality_logw, enabled_mask, precision, eps,
                                estimation_method, resample_mode, uniforms, states_ws, logw_ws, est_out, stream);
  const size_t NM = (size_t)N * M;
  float* cur = states;     // particle set entering the step
  float* moved = states_ws;  // particle set after the dynamics (and, without resampling, after the step)
  for (int t = 0; t < T; ++t) {
    const float* rb = rowbias_ws + (size_t)t * N * MMF_UNITS;
    const float* mw = modality_logw ? modality_logw + (size_t)t * N * K : nullptr;
    const float* e = eps + (size_t)t * NM * sd;
    if (precision == MMF_PREC_FP32)
      rc = launch_particle_chain_ffma(model, N, M, cur, e, rb, logw, mw, enabled_mask, moved, logw_ws, nullptr, stream, T * N);
    else
      rc = launch_particle_chain_tc(model, N, M, cur, e, rb, logw, mw, enabled_mask, precision, moved, logw_ws, nullptr,
                                    stream, 0, nullptr, T * N);
    if (rc) return rc;
    ResampleParams P;
    P.N = N; P.M = M; P.sd = sd; P.M_out = M;
    P.estimation = estimation_method; P.mode = resample_mode; P.alpha = 1.0f;
    P.states = moved; P.logw_unnorm = logw_ws; P.logits_in = nullptr;
    P.uniforms = uniforms ? uniforms + (size_t)t * (systematic ? (size_t)N : NM) : nullptr;
    P.states_out = resample_mode == MMF_RESAMPLE_NONE ? nullptr : cur;  // `cur` is dead once the chain kernel has read it
    P.logw_out = logw; P.est_out = est_out + (size_t)t * N * sd;
    P.logw_norm_out = nullptr; P.logits_out = nullptr; P.idx_out = nullptr;
    rc = launch_normalize_resample(P, resample_ws, stream);
    if (rc) return rc;
    if (resample_mode == MMF_RESAMPLE_NONE) {  // the moved set IS the next step's input: swap the roles of the buffers
      float* tmp = cur; cur = moved; moved = tmp;
    }
  }
  if (cur != states) MMF_CUDA(cudaMemcpyAsync(states, cur, NM * sd * sizeof(float), cudaMemcpyDeviceToDevice, stream));
  return MMF_OK;
}

int mmf_pf_forward_loop_persistent(int32_t N, int32_t M) { return pf_loop_small_applies(N, M) ? 1 : 0; }

size_t mmf_pf_resample_workspace_bytes(int32_t N, int32_t M) {
  if (N <= 0 || M <= 0) return 0;
  return resample_workspace_bytes(N, M);
}

int mmf_pf_normalize_resample(int32_t N, int32_t M, int32_t sd, const float* states, const float* logw_unnorm,
                              int32_t estimation_method, int32_t resample_mode, float soft_resample_alpha,
                              int32_t M_out, const double* uniforms, float* states_out, float* logw_out,
                              float* est_out, float* logw_norm_out, float* logits_out, int64_t* idx_out,
                              void* workspace, void* stream) {
  MMF_REQUIRE(N >= 0 && M >= 1 && sd >= 1 && sd <= MMF_MAX_SD, "normalize_resample: bad shape N=%d M=%d sd=%d", N, M, sd);
  MMF_REQUIRE(estimation_method == MMF_ESTIMATE_WEIGHTED_AVERAGE || estimation_method == MMF_ESTIMATE_ARGMAX,
              "normalize_resample: unknown estimation method %d", estimation_method);
  MMF_REQUIRE(resample_mode >= MMF_RESAMPLE_NONE && resample_mode <= MMF_RESAMPLE_SYSTEMATIC_FAST,
              "normalize_resample: unknown resample mode %d", resample_mode);
  if (N == 0) return MMF_OK;
  MMF_REQUIRE(states && logw_unnorm && est_out && logw_out, "normalize_resample: NULL buffer");
  if (resample_mode != MMF_RESAMPLE_NONE) {
    MMF_REQUIRE(M_out >= 1 && uniforms && states_out, "normalize_resample: resampling needs M_out, uniforms, states_out");
    MMF_REQUIRE(soft_resample_alpha > 0.0f && soft_resample_alpha <= 1.0f, "soft_resample_alpha %f outside (0, 1]",
                (double)soft_resample_alpha);
    MMF_REQUIRE(soft_resample_alpha == 1.0f || M_out == M, "soft resampling keeps the particle count (M=%d, M_out=%d)",
                M, M_out);
  }
  ResampleParams P;
  P.N = N; P.M = M; P.sd = sd; P.M_out = M_out;
  P.estimation = estimation_method; P.mode = resample_mode;
  P.alpha = (resample_mode == MMF_RESAMPLE_NONE) ? 1.0f : soft_resample_alpha;
  P.states = states; P.logw_unnorm = logw_unnorm; P.logits_in = nullptr; P.uniforms = uniforms;
  P.states_out = states_out; P.logw_out = logw_out; P.est_out = est_out;
  P.logw_norm_out = logw_norm_out; P.logits_out = logits_out; P.idx_out = (long long*)idx_out;
  return launch_normalize_resample(P, workspace, (cudaStream_t)stream);
}

int mmf_fuse_loglik(int32_t N, int32_t M, int32_t K, const float* ll, const float* w, float* out, void* stream) {
  MMF_REQUIRE(N >= 0 && M >= 0 && K >= 1, "fuse_loglik: bad shape N=%d M=%d K=%d", N, M, K);
  MMF_REQUIRE((long long)N * M == 0 || (ll && out), "fuse_loglik: NULL buffer");
  return launch_fuse_loglik(N, M, K, ll, w, out, (cudaStream_t)stream);
}

int mmf_resample(int32_t N, int32_t M, int32_t M_out, const float* logits, int32_t resample_mode,
                 const double* uniforms, int64_t* idx_out, void* workspace, void* stream) {
  MMF_REQUIRE(N >= 0 && M >= 1 && M_out >= 1, "resample: bad shape N=%d M=%d M_out=%d", N, M, M_out);
  MMF_REQUIRE(resample_mode > MMF_RESAMPLE_NONE && resample_mode <= MMF_RESAMPLE_SYSTEMATIC_FAST,
              "resample: unknown resample mode %d", resample_mode);
  if (N == 0) return MMF_OK;
  MMF_REQUIRE(logits && uniforms && idx_out, "resample: NULL buffer");
  ResampleParams P;
  memset(&P, 0, sizeof(P));
  P.N = N; P.M = M; P.sd = 1; P.M_out = M_out;
  P.mode = resample_mode; P.alpha = 1.0f;
  P.logits_in = logits; P.uniforms = uniforms; P.idx_out = (long long*)idx_out;
  return launch_normalize_resample(P, workspace, (cudaStream_t)stream);
}

static int fill_ekf(EkfParams& P, const mmf_ekf_model* models, int F) {
  MMF_REQUIRE(models != nullptr && F >= 1 && F <= EKF_MAX_FILTERS, "ekf: num_filters %d outside 1..%d", F, EKF_MAX_FILTERS);
  const int sd = models[0].state_dim, cd = models[0].control_dim;
  MMF_REQUIRE(sd >= 1 && sd <= MMF_MAX_SD && cd >= 1 && cd <= MMF_MAX_CD, "ekf: bad dims sd=%d cd=%d", sd, cd);
  for (int f = 0; f < F; ++f) {
    MMF_REQUIRE(models[f].state_dim == sd && models[f].control_dim == cd, "ekf: filters disagree on dims");
    int rc = validate_chain(models[f].dynamics, sd, sd + 1, "ekf dynamics chain");
    if (rc) return rc;
    MMF_REQUIRE(models[f].dynamics_rows.w && models[f].dynamics_rows.in_dim == cd && models[f].dynamics_rows.has_encoder,
                "ekf dynamics_rows: need the control encoder with in_dim == control_dim");
    P.dyn[f] = to_dev(models[f].dynamics);
    P.rows[f] = to_dev(models[f].dynamics_rows);
    for (int i = 0; i < MMF_MAX_SD * MMF_MAX_SD; ++i) P.q[f][i] = models[f].q_tril[i];
  }
  P.F = F;
  P.cd = cd;
  return MMF_OK;
}

int mmf_ekf_loop_fwd(const mmf_ekf_model* models, int32_t num_filters, int32_t T, int32_t N, const float* mean0,
                     const float* cov0, const float* controls, const float* z, const float* r_tril, float* mean_out,
                     float* cov_out, void* stream) {
  EkfParams P;
  memset(&P, 0, sizeof(P));
  int rc = fill_ekf(P, models, num_filters);
  if (rc) return rc;
  MMF_REQUIRE(T >= 0 && N >= 0, "ekf: bad shape T=%d N=%d", T, N);
  if (T == 0 || N == 0) return MMF_OK;
  MMF_REQUIRE(mean0 && cov0 && controls && z && r_tril && mean_out && cov_out, "ekf: NULL buffer");
  P.T = T; P.N = N; P.jac_only = 0;
  P.mean0 = mean0; P.cov0 = cov0; P.controls = controls; P.z = z; P.r_tril = r_tril;
  P.mean_out = mean_out; P.cov_out = cov_out;
  return launch_ekf(P, models[0].state_dim, (cudaStream_t)stream);
}

int mmf_ekf_loop_train_fwd(const mmf_ekf_model* models, int32_t num_filters, int32_t T, int32_t N, const float* mean0,
                           const float* cov0, const float* controls, const float* z, const float* r_tril,
                           float* mean_out, float* cov_out, float* pred_out, float* jac_out, void* stream) {
  EkfParams P;
  memset(&P, 0, sizeof(P));
  int rc = fill_ekf(P, models, num_filters);
  if (rc) return rc;
  MMF_REQUIRE(T >= 0 && N >= 0, "ekf_train: bad shape T=%d N=%d", T, N);
  if (T == 0 || N == 0) return MMF_OK;
  MMF_REQUIRE(mean0 && cov0 && controls && z && r_tril && mean_out && cov_out && pred_out && jac_out,
              "ekf_train: NULL buffer");
  P.T = T; P.N = N; P.jac_only = 0;
  P.mean0 = mean0; P.cov0 = cov0; P.controls = controls; P.z = z; P.r_tril = r_tril;
  P.mean_out = mean_out; P.cov_out = cov_out; P.pred_out = pred_out; P.jac_out = jac_out;
  return launch_ekf(P, models[0].state_dim, (cudaStream_t)stream, /*tape=*/true);
}

int mmf_ekf_loop_bwd(const mmf_ekf_model* models, int32_t num_filters, int32_t T, int32_t N, const float* mean0,
                     const float* cov0, const float* z, const float* r_tril, const float* means, const float* covs,
                     const float* pred, const float* jac, const float* d_means, const float* d_covs, float* d_mean0,
                     float* d_cov0, float* d_z, float* d_r_tril, void* stream) {
  (void)mean0;  // mu- of every step is on the tape: the posterior means are not read
  (void)means;
  EkfParams F;
  memset(&F, 0, sizeof(F));
  int rc = fill_ekf(F, models, num_filters);
  if (rc) return rc;
  MMF_REQUIRE(T >= 0 && N >= 0, "ekf_bwd: bad shape T=%d N=%d", T, N);
  if (N == 0) return MMF_OK;
  MMF_REQUIRE(cov0 && d_mean0 && d_cov0, "ekf_bwd: NULL buffer");
  MMF_REQUIRE(T == 0 || (z && r_tril && covs && pred && jac && d_z && d_r_tril), "ekf_bwd: NULL buffer");
  EkfBwdParams P;
  memset(&P, 0, sizeof(P));
  memcpy(P.q, F.q, sizeof(P.q));
  P.F = num_filters; P.T = T; P.N = N;
  P.cov0 = cov0; P.z = z; P.r_tril = r_tril; P.covs = covs; P.pred = pred; P.jac = jac;
  P.d_means = d_means; P.d_covs = d_covs;
  P.d_mean0 = d_mean0; P.d_cov0 = d_cov0; P.d_z = d_z; P.d_r_tril = d_r_tril;
  return launch_ekf_bwd(P, models[0].state_dim, (cudaStream_t)stream);
}

int mmf_dynamics_jacobian(const mmf_ekf_model* model, int32_t N, const float* states, const float* controls,
                          float* pred_out, float* jac_out, void* stream) {
  EkfParams P;
  memset(&P, 0, sizeof(P));
  int rc = fill_ekf(P, model, 1);
  if (rc) return rc;
  MMF_REQUIRE(N >= 0, "jacobian: N=%d", N);
  if (N == 0) return MMF_OK;
  MMF_REQUIRE(states && controls && pred_out && jac_out, "jacobian: NULL buffer");
  P.T = 1; P.N = N; P.jac_only = 1;
  P.mean0 = states; P.controls = controls; P.mean_out = pred_out; P.cov_out = jac_out;
  return launch_ekf(P, model->state_dim, (cudaStream_t)stream);
}

int mmf_kf_fuse_crossmodal(int32_t K, int32_t rows, int32_t sd, const float* mu, const float* P, const float* beta,
                           float* mean_out, float* cov_out, void* stream) {
  MMF_REQUIRE(K >= 1 && rows >= 0 && sd >= 1 && sd <= MMF_MAX_SD, "kf_fuse: bad shape K=%d rows=%d sd=%d", K, rows, sd);
  MMF_REQUIRE(rows == 0 || (mu && P && beta && mean_out && cov_out), "kf_fuse: NULL buffer");
  return launch_kf_fuse(K, rows, sd, mu, P, beta, mean_out, cov_out, 0, (cudaStream_t)stream);
}

int mmf_kf_fuse_measurements(int32_t K, int32_t rows, int32_t sd, const float* z, const float* r_tril, const float* weights,
                             float* z_out, float* mat_out, void* stream) {
  MMF_REQUIRE(K >= 1 && rows >= 0 && sd >= 1 && sd <= MMF_MAX_SD, "kf_fuse_measurements: bad shape K=%d rows=%d sd=%d", K, rows, sd);
  MMF_REQUIRE(rows == 0 || (z && r_tril && z_out && mat_out), "kf_fuse_measurements: NULL buffer");
  return launch_kf_fuse_measurements(K, rows, sd, z, r_tril, weights, z_out, mat_out, weights == nullptr ? 1 : 0,
                                     (cudaStream_t)stream);
}

int mmf_kf_fuse_unimodal(int32_t K, int32_t rows, int32_t sd, const float* mu, const float* P, float* mean_out,
                         float* cov_out, void* stream) {
  MMF_REQUIRE(K >= 1 && rows >= 0 && sd >= 1 && sd <= MMF_MAX_SD, "kf_fuse: bad shape K=%d rows=%d sd=%d", K, rows, sd);
  MMF_REQUIRE(rows == 0 || (mu && P && mean_out && cov_out), "kf_fuse: NULL buffer");
  return launch_kf_fuse(K, rows, sd, mu, P, nullptr, mean_out, cov_out, 1, (cudaStream_t)stream);
}

size_t mmf_chain_mma_bytes(const mmf_chain* chain) { return chain ? chain_mma_bytes(chain) : 0; }

int mmf_pack_chain_mma(const mmf_chain* chain, void* dst, void* stream) {
  MMF_REQUIRE(chain && dst, "pack_chain_mma: NULL argument");
  return pack_chain_mma(chain, dst, (cudaStream_t)stream);
}

size_t mmf_chain_bwd_bytes(const mmf_chain* chain) { return chain ? chain_bwd_bytes(chain) : 0; }

int mmf_pack_chain_bwd(const mmf_chain* chain, void* dst, void* stream) {
  MMF_REQUIRE(chain && dst, "pack_chain_bwd: NULL argument");
  return pack_chain_bwd(chain, dst, (cudaStream_t)stream);
}

int mmf_pf_heads_forward_train(const mmf_pf_model* model, int32_t N, int32_t M, const float* states_in,
                               const float* eps, float* states_moved, const float* rowbias, uint32_t enabled_mask,
                               int32_t precision, float* ll_out, float* act_out, float* logw_scratch, void* stream) {
  int rc = validate_pf_model(model);
  if (rc) return rc;
  MMF_REQUIRE(N >= 0 && M >= 1, "heads_forward_train: bad shape N=%d M=%d", N, M);
  if (N == 0) return MMF_OK;
  MMF_REQUIRE(states_moved && rowbias && ll_out && act_out && logw_scratch, "heads_forward_train: NULL buffer");
  MMF_REQUIRE(precision == MMF_PREC_BF16X3 || precision == MMF_PREC_BF16, "heads_forward_train: tensor-core precisions only");
  const uint32_t all = (1u << model->num_heads) - 1u;
  MMF_REQUIRE((enabled_mask & all) != 0, "heads_forward_train: no head enabled");
  MMF_REQUIRE((states_in == nullptr) == (eps == nullptr), "heads_forward_train: states_in and eps go together");
  return launch_particle_chain_tc(model, N, M, states_in, eps, rowbias, logw_scratch, nullptr, enabled_mask & all,
                                  precision, states_moved, logw_scratch, ll_out, (cudaStream_t)stream,
                                  /*first_chain=*/states_in ? 0 : 1, act_out);
}

int mmf_pf_heads_backward(const mmf_pf_model* model, int32_t N, int32_t M, const float* act, const float* d_ll,
                          uint32_t enabled_mask, float* delta_out, void* stream) {
  int rc = validate_pf_model(model);
  if (rc) return rc;
  MMF_REQUIRE(N >= 0 && M >= 1, "heads_backward: bad shape N=%d M=%d", N, M);
  if (N == 0) return MMF_OK;
  MMF_REQUIRE(act && d_ll && delta_out, "heads_backward: NULL buffer");
  const uint32_t all = (1u << model->num_heads) - 1u;
  MMF_REQUIRE((enabled_mask & all) != 0, "heads_backward: no head enabled");
  return launch_head_chain_bwd(model, N, M, act, d_ll, enabled_mask & all, delta_out, (cudaStream_t)stream);
}

size_t mmf_pf_heads_weight_grads_workspace_bytes(int32_t K, int32_t L, int64_t rows) {
  if (K < 1 || K > MMF_MAX_HEADS || L < 1 || rows <= 0) return 0;
  return heads_dw_workspace_bytes(K, L, rows);
}

int mmf_pf_heads_weight_grads(int32_t K, int32_t L, int64_t rows, int32_t sd, const float* act, const float* delta,
                              const float* x, const float* d_ll, float* dW_out, float* db_out, float* g_in_out,
                              float* g_out_out, void* workspace, void* stream) {
  MMF_REQUIRE(K >= 1 && K <= MMF_MAX_HEADS && L >= 1 && rows >= 0 && sd >= 1 && sd <= MMF_MAX_SD,
              "heads_weight_grads: bad shape K=%d L=%d sd=%d", K, L, sd);
  MMF_REQUIRE(rows == 0 || (act && delta && x && d_ll && dW_out && db_out && g_in_out && g_out_out),
              "heads_weight_grads: NULL buffer");
  return launch_heads_dw(K, L, rows, sd, act, delta, x, d_ll, dW_out, db_out, g_in_out, g_out_out, workspace,
                         (cudaStream_t)stream);
}

int mmf_pf_reweight_train_fwd(int32_t N, int32_t M, int32_t K, int32_t sd, uint32_t enabled_mask, const float* ll,
                              const float* modality_logw, const float* logw_in, const float* states, float* logw_out,
                              float* est_out, void* stream) {
  MMF_REQUIRE(N >= 0 && M >= 1 && K >= 1 && K <= MMF_MAX_HEADS && sd >= 1 && sd <= MMF_MAX_SD,
              "reweight_train: bad shape N=%d M=%d K=%d sd=%d", N, M, K, sd);
  MMF_REQUIRE((enabled_mask & ((1u << K) - 1u)) != 0, "reweight_train: no head enabled (mask 0x%x)", enabled_mask);
  MMF_REQUIRE(N == 0 || (ll && logw_in && states && logw_out && est_out), "reweight_train: NULL buffer");
  return launch_reweight_train(N, M, K, sd, enabled_mask & ((1u << K) - 1u), ll, modality_logw, logw_in, states, logw_out,
                               est_out, nullptr, nullptr, nullptr, nullptr, nullptr, false, (cudaStream_t)stream);
}

int mmf_pf_reweight_train_bwd(int32_t N, int32_t M, int32_t K, int32_t sd, uint32_t enabled_mask, const float* ll,
                              const float* modality_logw, const float* logw_in, const float* states, const float* d_est,
                              const float* d_logw, float* d_ll, float* d_modality_logw, float* d_logw_in, void* stream) {
  MMF_REQUIRE(N >= 0 && M >= 1 && K >= 1 && K <= MMF_MAX_HEADS && sd >= 1 && sd <= MMF_MAX_SD,
              "reweight_train: bad shape N=%d M=%d K=%d sd=%d", N, M, K, sd);
  MMF_REQUIRE((enabled_mask & ((1u << K) - 1u)) != 0, "reweight_train: no head enabled (mask 0x%x)", enabled_mask);
  MMF_REQUIRE(N == 0 || (ll && logw_in && states && d_ll && d_logw_in), "reweight_train: NULL buffer");
  MMF_REQUIRE((modality_logw == nullptr) == (d_modality_logw == nullptr) || d_modality_logw == nullptr,
              "reweight_train: d_modality_logw given without modality_logw");
  return launch_reweight_train(N, M, K, sd, enabled_mask & ((1u << K) - 1u), ll, modality_logw, logw_in, states, nullptr,
                               nullptr, d_est, d_logw, d_ll, d_modality_logw, d_logw_in, true, (cudaStream_t)stream);
}

int mmf_row_mlp(int64_t rows, const mmf_mlp_op* ops, int32_t n_ops, const float* weights, const float* const* inputs,
                const int32_t* in_dims, const int32_t* in_slots, int32_t n_inputs, float* const* outputs,
                const int32_t* out_dims, const int32_t* out_slots, int32_t n_outputs, int32_t scratch_floats,
                void* stream) {
  MMF_REQUIRE(rows >= 0, "row_mlp: rows = %lld", (long long)rows);
  MMF_REQUIRE(inputs && in_dims && in_slots && outputs && out_dims && out_slots, "row_mlp: NULL argument array");
  return launch_row_mlp(rows, ops, n_ops, weights, inputs, in_dims, in_slots, n_inputs, outputs, out_dims, out_slots,
                        n_outputs, scratch_floats, (cudaStream_t)stream);
}

size_t mmf_enc_map_bytes(int32_t channels) { return enc_map_bytes_host(channels); }

int mmf_enc_stem(int32_t n_images, const float* images, const float* w, void* out_map, void* stream) {
  MMF_REQUIRE(n_images >= 0, "enc_stem: negative image count");
  MMF_REQUIRE(n_images == 0 || (images && w && out_map), "enc_stem: NULL buffer");
  MMF_REQUIRE(((uintptr_t)out_map & 15) == 0, "enc_stem: map must be 16-byte aligned");
  return launch_enc_stem(n_images, images, w, out_map, (cudaStream_t)stream);
}

int mmf_enc_conv3x3(int32_t n_images, int32_t cin, int32_t cout, const void* in_map, const void* w_image,
                    const void* res_map, int32_t relu, void* out_map, float* out_nchw, void* stream) {
  MMF_REQUIRE(n_images >= 0, "enc_conv3x3: negative image count");
  MMF_REQUIRE(n_images == 0 || (in_map && w_image), "enc_conv3x3: NULL input");
  MMF_REQUIRE(out_map || out_nchw, "enc_conv3x3: no output requested");
  MMF_REQUIRE((((uintptr_t)in_map | (uintptr_t)w_image | (uintptr_t)res_map | (uintptr_t)out_map) & 15) == 0,
              "enc_conv3x3: maps and the operand image must be 16-byte aligned");
  return launch_enc_conv3x3(n_images, cin, cout, in_map, w_image, res_map, relu, out_map, out_nchw, (cudaStream_t)stream);
}

size_t mmf_enc_trunk_scratch_bytes(void) { return enc_trunk_scratch_bytes(); }
size_t mmf_enc_trunk_weight_bytes(void) { return enc_trunk_weight_bytes(); }

int mmf_enc_trunk(int32_t n_images, int32_t cout, const float* images, const void* weights, void* scratch,
                  float* out_nchw, void* stream) {
  MMF_REQUIRE(n_images >= 0 && cout >= 1 && cout <= 16, "enc_trunk: bad shape n=%d cout=%d", n_images, cout);
  MMF_REQUIRE(n_images == 0 || (images && weights && scratch && out_nchw), "enc_trunk: NULL buffer");
  MMF_REQUIRE((((uintptr_t)weights | (uintptr_t)scratch) & 15) == 0, "enc_trunk: weights and scratch must be 16-byte aligned");
  return launch_enc_trunk(n_images, cout, images, weights, scratch, out_nchw, (cudaStream_t)stream);
}

}  // extern "C"
