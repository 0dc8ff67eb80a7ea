/* mmf_b200.h -- C ABI of the B200 (sm_100a) filtering-recursion library `libmmf_b200.so`.
 *
 * Drop-in boundary for ONE hot path of brentyi/multimodalfilter: the particle-filter /
 * extended-Kalman-filter step and the crossmodal fusion around it.  The reference is pure Python
 * (torchfilter + crossmodal on eager PyTorch) and has no FFI of its own; each entry point below
 * therefore cites the Python interface whose arithmetic it replaces.  "ref:" = /root/reference,
 * "A.n" = SURVEY.md Appendix A (normative restatement of the un-vendored torchfilter dependency).
 *
 * Conventions
 *  - every pointer is a DEVICE pointer to C-contiguous fp32 unless stated otherwise; the caller
 *    owns all buffers (the library never allocates device memory and keeps no global state
 *    besides a thread-local error string);
 *  - every call is asynchronous on `stream` (a cudaStream_t passed as void*), re-entrant, and may
 *    be issued from several host threads on different streams / devices;
 *  - return value 0 = OK, negative = error (MMF_E_*); `mmf_last_error()` gives the message;
 *  - N = trajectories, M = particles per trajectory, sd = state_dim (<= MMF_MAX_SD),
 *    cd = control_dim (<= MMF_MAX_CD), K = measurement heads (<= MMF_MAX_HEADS), U = 64 hidden units.
 */
#ifndef MMF_B200_H
#define MMF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MMF_ABI_VERSION 3
#define MMF_UNITS 64
#define MMF_MAX_SD 4
#define MMF_MAX_CD 16
#define MMF_MAX_HEADS 4
#define MMF_MAX_OBS_FEATS 256

#define MMF_OK 0
#define MMF_E_INVALID (-1)   /* bad argument / unsupported shape */
#define MMF_E_CUDA (-2)      /* CUDA runtime error (message has the cudaError string) */
#define MMF_E_UNSUPPORTED (-3)

/* resampling modes (R7).  *_STRICT reproduces torch.multinomial's CPU arithmetic (sequential fp32
 * running sum); *_FAST uses the blocked summation order specified in DESIGN.md; SYSTEMATIC is the
 * north-star low-variance variant (one uniform per trajectory). */
#define MMF_RESAMPLE_NONE 0
#define MMF_RESAMPLE_MULTINOMIAL_STRICT 1
#define MMF_RESAMPLE_MULTINOMIAL_FAST 2
#define MMF_RESAMPLE_SYSTEMATIC_STRICT 3
#define MMF_RESAMPLE_SYSTEMATIC_FAST 4

#define MMF_ESTIMATE_WEIGHTED_AVERAGE 0
#define MMF_ESTIMATE_ARGMAX 1

/* arithmetic of the per-particle MLP chain */
#define MMF_PREC_FP32 0      /* CUDA-core FFMA, fp32 throughout (parity build)               */
#define MMF_PREC_BF16X3 1    /* tcgen05, bf16 hi/lo split operands, 3 MMAs/layer, fp32 accum  */
#define MMF_PREC_BF16 2      /* tcgen05, single-pass bf16 operands (fast, NOT parity grade)   */

/* One MLP "chain" over 64-wide activations (all 64x64 matrices stored TRANSPOSED, Wt[k][j] =
 * W[j][k], i.e. input-major, so 4 consecutive outputs share a 16-byte word):
 *
 *   h  = relu(in_W x + in_b)                                  x: in_dim inputs
 *   h  = res(h)                       x n_pre_res             res(h) = relu(W2 relu(W1 h + b1) + b2 + h)
 *   h  = act_mid(mid_W h + rowbias[trajectory])               act_mid = relu or identity
 *   h  = res(h)                       x n_post_res
 *   y  = out_W h + out_b                                      out_dim outputs
 *
 * `rowbias` is the per-trajectory part of the reference's concatenated Linear (control features
 * for the dynamics, observation features for a measurement head) plus that Linear's bias, hoisted
 * out of the particle loop (computed by mmf_pf_traj_rows).
 *
 * Packed fp32 layout of `w` (floats, in this order):
 *   in_Wt[in_dim][64], in_b[64],
 *   pre_res[r]  : W1t[64][64], b1[64], W2t[64][64], b2[64]        r < n_pre_res
 *   mid_Wt[64][64]                                                 (no bias: it lives in rowbias)
 *   post_res[r] : W1t[64][64], b1[64], W2t[64][64], b2[64]        r < n_post_res
 *   out_W[out_dim][64] (row-major, NOT transposed), out_b[out_dim]
 *
 * Dynamics chain  = ref: crossmodal/push_models/dynamics.py:22-31,44-63 (state branch + shared);
 * measurement head = ref: crossmodal/push_models/pf.py:52-61,97-105.
 */
typedef struct mmf_chain {
  int32_t in_dim;       /* = sd */
  int32_t n_pre_res;    /* 1 */
  int32_t mid_relu;     /* 0 for dynamics (ref: dynamics.py:26 no activation), 1 for heads (pf.py:55-56) */
  int32_t n_post_res;   /* 3 dynamics, 2 heads */
  int32_t out_dim;      /* sd+1 dynamics, 1 heads */
  int32_t reserved;
  const float* w;       /* packed fp32 weights, layout above */
  const void* w_mma;    /* optional tcgen05 operand pack built by mmf_pack_chain_mma (NULL => FP32 only) */
  const void* w_bwd;    /* optional backward operand pack built by mmf_pack_chain_bwd (training only) */
} mmf_chain;

/* Per-trajectory (hoisted) part of a chain's mid layer:
 *   feats = (has_encoder ? res(relu(enc_W u + enc_b)) : u)        u: in_dim raw inputs
 *   rowbias = traj_W feats + mid_b
 * Packed fp32 layout of `w`:
 *   [has_encoder: enc_Wt[in_dim][64], enc_b[64], W1t, b1, W2t, b2]   (ref: layers.py:27-40 control_layers)
 *   traj_Wt[feat_dim][64], mid_b[64]      feat_dim = 64 if has_encoder else in_dim
 */
typedef struct mmf_traj_rows {
  int32_t in_dim;       /* cd for the dynamics (controls), 64*k for a head (observation features) */
  int32_t has_encoder;  /* 1: dynamics control branch; 0: heads (features come from the encoders) */
  const float* w;
} mmf_traj_rows;

typedef struct mmf_pf_model {
  int32_t state_dim, control_dim, num_heads, reserved;
  mmf_chain dynamics;
  mmf_traj_rows dynamics_rows;
  mmf_chain heads[MMF_MAX_HEADS];
  mmf_traj_rows head_rows[MMF_MAX_HEADS];
  float q_tril[MMF_MAX_SD * MMF_MAX_SD]; /* row-major sd x sd lower-triangular process-noise factor
                                            (ref: dynamics.py:17-20,63; door dynamics.py:85-88,131-133) */
} mmf_pf_model;

const char* mmf_last_error(void);
int mmf_abi_version(void);
/* 0 if the current device is a compute-capability-10.x part and the kernels load, else MMF_E_UNSUPPORTED. */
int mmf_device_check(void);

/* R2  ParticleFilter.initialize_beliefs (A.3; call site ref: crossmodal/eval_helpers.py:128-131)
 *   states[n,m,:] = mean[n] + chol(cov[n]) eps[m,n,:]   (eps laid out (M,N,sd), the draw order of
 *   MultivariateNormal.sample((M,)), A.6);   logw[n,m] = -log M */
int mmf_pf_init(int32_t N, int32_t M, int32_t sd, const float* mean, const float* cov,
                const float* eps_MNsd, float* states_out, float* logw_out, void* stream);

/* Hoisted per-trajectory rows for one step: rowbias_out is (1+K, N, 64): plane 0 = dynamics,
 * plane 1+k = head k.  controls (N,cd); obs_feats[k] (N, head_rows[k].in_dim) or NULL for a
 * disabled head. */
int mmf_pf_traj_rows(const mmf_pf_model* model, int32_t N, const float* controls,
                     const float* const* obs_feats, float* rowbias_out, void* stream);

/* R3+R4+R5 and the first half of R6: predict every particle, evaluate the enabled measurement
 * heads on the moved particle, fuse, add to the incoming log-weight.
 *   x'  = x + h[:sd] * sigmoid(h[sd]) + q_tril eps          (A.3 predict; ref: dynamics.py:55-63)
 *   ll_k = head_k(x')                                        (ref: pf.py:91-109)
 *   fused = logsumexp_k(w[n,k] + ll_k) over enabled k        (ref: base_models/crossmodal_pf.py:132-139;
 *           w == NULL => plain logsumexp_k, the "unimodal" fusion)
 *   logw_unnorm = logw_in + fused
 * enabled_mask bit k = head k enabled (ref: crossmodal_pf.py:106-121, quirk Q4).
 * modality_logw is (N, K) over ALL heads (disabled columns ignored).  ll_out (optional, may be
 * NULL) receives the per-head log-likelihoods as (K, N*M) planes for the parity tests. */
int mmf_pf_predict_measure(const mmf_pf_model* model, int32_t N, int32_t M, const float* states_in,
                           const float* eps, const float* rowbias, const float* logw_in,
                           const float* modality_logw, uint32_t enabled_mask, int32_t precision,
                           float* states_out, float* logw_unnorm_out, float* ll_out, void* stream);

/* R1: the whole T-step recursion of a recognised particle filter, enqueued by ONE call (replaces the Python loop of
 * A.2 `Filter.forward_loop` over A.3 `ParticleFilter.forward`; call site ref: crossmodal/eval_helpers.py:139-142).
 * The observation encoders are hoisted: `obs_feats[k]` is (T, N, F_k) (NULL for a disabled head), `modality_logw`
 * (T, N, K) or NULL, `controls` (T, N, cd), `eps` (T, N*M, sd) process noise, `uniforms` float64 (T, N, M)
 * [multinomial*] / (T, N) [systematic*] / NULL [MMF_RESAMPLE_NONE].  Hard resampling that keeps the particle count.
 *   states (N, M, sd), logw (N, M): IN the particle set entering step 0, OUT the set after step T-1;
 *   est_out (T, N, sd): the state estimate of every step;
 *   workspaces (caller-owned): rowbias_ws (1+K, T*N, 64) floats, states_ws (N, M, sd), logw_ws (N, M),
 *   resample_ws of mmf_pf_resample_workspace_bytes(N, M) bytes (may be NULL when that is 0).
 * Launches: 1 (per-trajectory rows of all T steps) + 2 per step (per-particle chain, normalise/estimate/resample).
 * Small problems (M <= 64 particles and N <= one CTA per SM; mmf_pf_forward_loop_persistent(N, M) == 1) run the T steps
 * in ONE further launch instead: a CTA carries a trajectory through the whole sequence, particle set in shared memory
 * (MMF_PREC_FP32: CUDA-core arithmetic, identical bits to the per-step fp32 kernels; MMF_PREC_BF16X3 / BF16: the layers
 * on mma.sync with the same split bf16 operands as the per-step tcgen05 kernel).  Environment MMF_PF_LOOP_SMALL, read
 * once when the library is loaded: 0 = never, 1 = whenever M <= 128. */
int mmf_pf_forward_loop(const mmf_pf_model* model, int32_t T, int32_t N, int32_t M, float* states, float* logw,
                        const float* controls, const float* const* obs_feats, const float* modality_logw,
                        uint32_t enabled_mask, int32_t precision, const float* eps, int32_t estimation_method,
                        int32_t resample_mode, const double* uniforms, float* rowbias_ws, float* states_ws,
                        float* logw_ws, float* est_out, void* resample_ws, void* stream);

/* 1 when mmf_pf_forward_loop runs this shape through the one-launch whole-sequence kernel, else 0. */
int mmf_pf_forward_loop_persistent(int32_t N, int32_t M);

/* Second half of R6, and R7 (A.3): per trajectory
 *   logw = logw_unnorm - logsumexp_m(logw_unnorm);  est = sum_m exp(logw) x  (or argmax particle)
 *   resample_mode != NONE: logits = logw (alpha == 1) or log(alpha e^logw + (1-alpha)/M);
 *     idx = inverse CDF of the uniforms (pinned arithmetic: DESIGN.md "Resampling arithmetic");
 *     states_out[n,j,:] = states[n,idx[n,j],:];  logw_out = -log M  (alpha<1: logw[idx]-logits[idx])
 *   resample_mode == NONE: states_out may be NULL (states stay where they are), logw_out (N,M).
 * uniforms: float64, (N, M_out) for MULTINOMIAL_*, (N) for SYSTEMATIC_*.
 * Optional outputs (NULL to skip): logw_norm_out (N,M), logits_out (N,M), idx_out (N,M_out) int64.
 * workspace: mmf_pf_resample_workspace_bytes(N, M) bytes, 16-byte aligned; 0 (workspace may be NULL) for M <= 2048, where a
 * warp owns a trajectory in shared memory.  Longer trajectories take a multi-pass path over (chunk of 4096 particles,
 * trajectory) grids whose CDF lives in the workspace (4 (M + ~0.1 M) + 32 K bytes per trajectory; resample_big.cu);
 * environment MMF_RESAMPLE_BIG, read once when the library is loaded: 0 = CTA-per-trajectory kernels instead, n > 1 =
 * multi-pass from M > n. */
size_t mmf_pf_resample_workspace_bytes(int32_t N, int32_t M);
int mmf_pf_normalize_resample(int32_t N, int32_t M, int32_t sd, const float* states,
                              const float* logw_unnorm, int32_t estimation_method,
                              int32_t resample_mode, float soft_resample_alpha, int32_t M_out,
                              const double* uniforms, float* states_out, float* logw_out,
                              float* est_out, float* logw_norm_out, float* logits_out,
                              int64_t* idx_out, void* workspace, void* stream);

/* Individually testable pieces of the above.
 * mmf_fuse_loglik: ll (N,M,K) interleaved as torch.stack(dim=2) gives it, w (N,K) or NULL -> (N,M). */
int mmf_fuse_loglik(int32_t N, int32_t M, int32_t K, const float* ll, const float* w, float* out,
                    void* stream);
/* mmf_resample: logits (N,M) -> idx (N,M_out) int64, same pinned arithmetic as the fused kernel. */
int mmf_resample(int32_t N, int32_t M, int32_t M_out, const float* logits, int32_t resample_mode,
                 const double* uniforms, int64_t* idx_out, void* workspace, void* stream);

/* ---- extended Kalman filter (R8), T steps in one launch --------------------------------------
 * One VirtualSensorExtendedKalmanFilter (A.5; ref: crossmodal/door_models/kf.py:14-28) whose
 * dynamics is the gated residual MLP (ref: crossmodal/door_models/dynamics.py:37-67):
 *   mu- = f(mu,u);  A = df/dx at mu (forward-mode tangents == the reference's autograd Jacobian, A.4)
 *   P-  = A P A^T + Q Q^T;  S = P- + R R^T;  Kg = P- S^-1;  mu = mu- + Kg (z - mu-);  P = (I - Kg) P-
 * z (T,N,sd) and r_tril (T,N,sd,sd) come from the virtual sensor (R9), controls (T,N,cd).
 * mean_out (T,N,sd), cov_out (T,N,sd,sd) receive every step's posterior.  num_filters independent
 * filters can be advanced by one launch: all arrays then carry a leading filter axis F and
 * `dynamics` / `dynamics_rows` / q_tril are arrays of F entries. */
typedef struct mmf_ekf_model {
  int32_t state_dim, control_dim;
  mmf_chain dynamics;
  mmf_traj_rows dynamics_rows;
  float q_tril[MMF_MAX_SD * MMF_MAX_SD];
} mmf_ekf_model;

int mmf_ekf_loop_fwd(const mmf_ekf_model* models, int32_t num_filters, int32_t T, int32_t N,
                     const float* mean0, const float* cov0, const float* controls, const float* z,
                     const float* r_tril, float* mean_out, float* cov_out, void* stream);

/* Training forward of the same recursion: mmf_ekf_loop_fwd's arithmetic (bit-identical mean_out / cov_out) that also
 * records the tape mmf_ekf_loop_bwd needs, pred_out (F,T,N,sd) = mu- and jac_out (F,T,N,sd,sd) = A of every step. */
int mmf_ekf_loop_train_fwd(const mmf_ekf_model* models, int32_t num_filters, int32_t T, int32_t N,
                           const float* mean0, const float* cov0, const float* controls, const float* z,
                           const float* r_tril, float* mean_out, float* cov_out, float* pred_out,
                           float* jac_out, void* stream);

/* Reverse mode of mmf_ekf_loop_train_fwd with frozen dynamics.  A = df/dx is evaluated at a detached state (A.4),
 * so it is a constant of the recursion and one step's adjoint is SD x SD algebra given the tape.  Going backwards in
 * t, with mb / Pb the gradient reaching posterior t (d_means[t] / d_covs[t] plus what step t+1 sent back), P the
 * posterior covariance of step t-1 (cov0 at t = 0), Pp, S, Sinv = S^-1, Kg recomputed as in the forward, r = z - mu-:
 *   d_z[t]   = Kg^T mb;                  mb-  = mb - d_z[t]
 *   Kg_bar   = mb r^T - Pb Pp^T;         S_bar = -Sinv^T Pp^T Kg_bar Sinv^T
 *   Pp_bar   = (I - Kg)^T Pb + Kg_bar Sinv^T + S_bar
 *   d_r_tril[t] = (S_bar + S_bar^T) r_tril[t]   (full sd x sd, upper entries included)
 *   Pb(t-1)  = A^T Pp_bar A;             mb(t-1) = A^T mb-
 * and d_mean0 = mb(-1), d_cov0 = Pb(-1).  means / covs / pred / jac are the forward's outputs; mean0 and means are
 * not read (mu- is on the tape) and may be NULL.  d_means and d_covs may each be NULL (= zero).  One thread per
 * (filter, trajectory), no atomics: the gradients are bit-reproducible run to run.  No workspace. */
int mmf_ekf_loop_bwd(const mmf_ekf_model* models, int32_t num_filters, int32_t T, int32_t N,
                     const float* mean0, const float* cov0, const float* z, const float* r_tril,
                     const float* means, const float* covs, const float* pred, const float* jac,
                     const float* d_means, const float* d_covs, float* d_mean0, float* d_cov0, float* d_z,
                     float* d_r_tril, void* stream);

/* Dynamics Jacobian alone (A.4 DynamicsModel.jacobian): states (N,sd), controls (N,cd) ->
 * pred (N,sd), jac (N,sd,sd). */
int mmf_dynamics_jacobian(const mmf_ekf_model* model, int32_t N, const float* states,
                          const float* controls, float* pred_out, float* jac_out, void* stream);

/* ---- dynamics training: open-loop rollout with a tape, and its reverse mode ---------------------------------------
 * DynamicsModel.forward_loop (A.4; ref: crossmodal/eval_helpers.py:135-137) of the gated-residual dynamics `chain`
 * (in_dim = sd, out_dim = sd + 1), T steps in ONE launch, a warp per trajectory:
 *   h = chain(x_t, rowbias[t]);   x_{t+1} = x_t + h[:sd] * sigmoid(h[sd]);   states_out[t] = x_{t+1}   (x_0 = x0)
 * x0 (N,sd), states_out (T,N,sd).  rowbias (T,N,64) = the hoisted control rows (mmf_chain's `rowbias`) given by the
 * caller, or NULL: then `rows` (with the control encoder) and controls (T,N,cd) compute them inside the kernel.
 * act_out (L+1, 16, T*N, 4), NULL = no tape, L = 2 n_pre_res + 1 + 2 n_post_res: chunk-major planes in the layout of
 * mmf_pf_heads_weight_grads (element [l][c][p][j] = column 4c+j of row p, rows p = t*N + n): plane l = the input of
 * 64x64 layer l, plane L = the input of the output layer.  The arithmetic is the same with and without the tape, so
 * states_out is bit-identical either way. */
int mmf_dyn_rollout_fwd(const mmf_chain* chain, const mmf_traj_rows* rows, int32_t T, int32_t N, const float* x0,
                        const float* controls, const float* rowbias, float* states_out, float* act_out, void* stream);

/* Reverse mode of mmf_dyn_rollout_fwd from its tape, one warp per trajectory walking t = T-1 ... 0.  With xb the gradient
 * reaching states[t] (d_states[t] plus what step t+1 sent back), y = the output layer recomputed from plane L,
 * g = sigmoid(y[sd]):
 *   d_y[t]  = yb:   yb_i = xb_i g (i < sd),   yb_sd = g (1 - g) sum_i xb_i y_i
 *   delta through W_out, the resblocks, the mid layer and the input layer, each ReLU mask read from the tape (the output
 *   of layer l is plane l+1, that of the input layer plane 0; the mid layer is masked only when mid_relu);
 *   d rowbias[t] = delta of the mid layer (plane 2 n_pre_res);   xb(t-1) = xb + in_W^T delta_in;   d_x0 = xb(-1).
 * d_states (T,N,sd) may be NULL (= zero).  delta_out (L+1, 16, T*N, 4) in the tape's layout: plane l = delta of 64x64
 * layer l, plane L = delta of the input layer (the convention of mmf_pf_heads_backward, so mmf_pf_heads_weight_grads with
 * K = 1 and x = the step inputs (x0, states[0 .. T-2]) reduces the parameter gradients); d_y_out (T*N, sd+1) = delta of
 * the output layer; d_x0_out (N,sd).  Every element is written by one lane, no atomics: bit-reproducible. */
int mmf_dyn_rollout_bwd(const mmf_chain* chain, int32_t T, int32_t N, const float* act, const float* d_states,
                        float* delta_out, float* d_y_out, float* d_x0_out, void* stream);

/* R10  CrossmodalKalmanFilter.calculate_weighted_states (ref: base_models/crossmodal_kf.py:153-167,
 * utility.py:4-11): rows = T*N independent fusions.
 *   mean = sum_k (beta_k / (sum_k beta_k + 1e-9)) * mu_k ;  cov = sum_k (beta_k beta_k^T) o P_k
 * mu (K,rows,sd), P (K,rows,sd,sd), beta (K,rows,sd). */
int mmf_kf_fuse_crossmodal(int32_t K, int32_t rows, int32_t sd, const float* mu, const float* P,
                           const float* beta, float* mean_out, float* cov_out, void* stream);
/* R11  UnimodalKalmanFilter.forward fusion (ref: base_models/unimodal_kf.py:199-242):
 *   Lk = inv(P_k + 1e-9);  cov = inv(sum_k Lk + 1e-9);  mean = cov sum_k Lk mu_k   (+1e-9 elementwise) */
int mmf_kf_fuse_unimodal(int32_t K, int32_t rows, int32_t sd, const float* mu, const float* P,
                         float* mean_out, float* cov_out, void* stream);

/* R12  measurement-level fusion of K virtual sensors (ref: crossmodal/base_models/crossmodal_kf.py:219-235,337-354
 * CrossmodalVirtualSensorModel.forward; crossmodal/base_models/unimodal_kf.py:56-115 UnimodalVirtualSensorModel.forward):
 * rows independent fusions, z (K,rows,sd), r_tril (K,rows,sd,sd) lower factors, weights (K,rows,sd) or NULL.
 *   weights != NULL (crossmodal): z_out = sum_k (w_k / (sum_k w_k + 1e-9)) z_k ;
 *                                 mat_out = cholesky((prod_k prod_d w_k[d]) * sum_k L_k L_k^T)          (a lower factor)
 *   weights == NULL (unimodal):   K == 1: z_0 and L_0 L_0^T; else Pr_k = 1 / (L_k + 1e-9) elementwise, w_k = diag Pr_k,
 *                                 z_out as above, mat_out = inverse(sum_k Pr_k + 1e-9)                  (a covariance) */
int mmf_kf_fuse_measurements(int32_t K, int32_t rows, int32_t sd, const float* z, const float* r_tril, const float* weights,
                             float* z_out, float* mat_out, void* stream);

/* Build the tcgen05 operand pack of a chain (bf16 hi/lo copies of every 64x64 matrix in the
 * UMMA shared-memory layout).  dst must hold mmf_chain_mma_bytes(chain) bytes. */
size_t mmf_chain_mma_bytes(const mmf_chain* chain);
int mmf_pack_chain_mma(const mmf_chain* chain, void* dst, void* stream);

/* ---- BPTT training support (BASELINE config C4) ------------------------------------------------
 * Backward of the measurement heads for the case every reference curriculum trains
 * (ref: scripts/push_task/train_push.py:154,213: dynamics frozen, no resampling in train mode, A.3/A.7):
 * the particle states then carry no gradient to a trainable leaf, so one filter step needs
 *   d loss / d (pre-activation) of every head layer, from which dW = delta^T a, db = sum delta,
 *   d rowbias = sum over the trajectory's particles of delta_mid.
 * mmf_pf_heads_forward_train: the forward step with the heads' activations saved.  states_in/eps non-NULL:
 *   the particles are first moved through the dynamics (as in mmf_pf_predict_measure) into states_moved;
 *   states_in == NULL: states_moved is an input (heads only).
 *   ll_out (K, N*M) per-head log-likelihoods; act_out (K, L+1, N*M, 64): plane l = input of 64x64 layer l,
 *   plane L = input of the output layer (L = 2 n_pre_res + 1 + 2 n_post_res); logw_scratch (N*M) is clobbered.
 * mmf_pf_heads_backward: d_ll (K, N*M) -> delta_out (K, L+1, N*M, 64): plane l = delta of 64x64 layer l,
 *   plane L = delta of the input layer (Linear(sd, 64) + ReLU). */
size_t mmf_chain_bwd_bytes(const mmf_chain* chain);
int mmf_pack_chain_bwd(const mmf_chain* chain, void* dst, void* stream);
int mmf_pf_heads_forward_train(const mmf_pf_model* model, int32_t N, int32_t M, const float* states_in,
                               const float* eps, float* states_moved, const float* rowbias, uint32_t enabled_mask,
                               int32_t precision, float* ll_out, float* act_out, float* logw_scratch, void* stream);
int mmf_pf_heads_backward(const mmf_pf_model* model, int32_t N, int32_t M, const float* act, const float* d_ll,
                          uint32_t enabled_mask, float* delta_out, void* stream);
/* ---- image observation encoder: convolutional trunk (SURVEY.md 8(f)-1) ------------------------------------
 * Replaces the Conv2d layers of observation_image_layers (ref: crossmodal/push_models/layers.py:93-101,
 * crossmodal/door_models/layers.py:43-57) for 32x32 single-channel images:
 *   x = relu(stem(image)), t = relu(block1(x)), y = relu(block2(t) + x), z = relu(conv3(y)), out = conv4(z)
 * with stem = Conv2d(1, 32, 5, padding=2), block1, block2 = Conv2d(32, 32, 3, padding=1),
 * conv3 = Conv2d(32, 16, 3, padding=1), conv4 = Conv2d(16, cout, 3, padding=1), cout <= 16.
 *   mmf_enc_trunk     the whole trunk of every image in ONE launch: a persistent CTA carries an image through all
 *                     layers, the 3x3 layers on the tensor cores (bf16 hi/lo split operands, fp32 accumulation).  Its
 *                     activation maps live in `scratch` (mmf_enc_trunk_scratch_bytes() bytes, stays L2-resident), which
 *                     MUST be zero-initialised once by the caller: the kernel relies on zero guard regions it never writes.
 *                     out_nchw = (n_images, cout, 32, 32) fp32.
 *                     weights = [w_image block1 | w_image block2 | w_image conv3 | w_image conv4 | stem w]
 *                     (mmf_enc_trunk_weight_bytes() bytes in total), where
 *                     w_image of a Conv2d(cin, c, 3) = bf16 [tap 9][cin/8][2 npad rows: hi then lo][8] then fp32
 *                       bias[npad], npad = 32 if c > 16 else 16: row n, element j of (tap, chunk k) holds
 *                       weight[n][8k + j][tap / 3][tap % 3] split as hi = rn_bf16(w), lo = rn_bf16(w - hi); rows >= c
 *                       and bias entries >= c are zero;
 *                     stem w = fp32 weight as [tap 25][32] (element [5 ky + kx][c] = weight[c][0][ky][kx]) then bias[32]. */
size_t mmf_enc_trunk_scratch_bytes(void);
size_t mmf_enc_trunk_weight_bytes(void);
int mmf_enc_trunk(int32_t n_images, int32_t cout, const float* images, const void* weights, void* scratch,
                  float* out_nchw, void* stream);

/* Parameter gradients of the heads from the saved activations and the deltas (both (K, L+1, 16, rows, 4)
 * chunk-major planes: element [k][l][c][p][j] = column 4c+j of row p), fp32 reductions over the N*M rows:
 *   dW_out   (K, L, 64, 64)  = delta[k][l]^T act[k][l]               the L 64x64 layers
 *   db_out   (K, L+1, 64)    = column sums of delta[k][l]            (plane L = the input layer)
 *   g_in_out (K, 64, sd)     = delta[k][L]^T x,  x = states (rows, sd)    input-layer weight
 *   g_out_out(K, 64)         = act[k][L]^T d_ll[k],  d_ll (K, rows)       output-layer weight
 * The outputs are OVERWRITTEN.  The rows are split over CTAs that write partial sums into `workspace`
 * (mmf_pf_heads_weight_grads_workspace_bytes() bytes, 16-byte aligned, caller-owned); a second kernel adds the
 * partials in a fixed order: no floating-point atomics, the gradients are bit-reproducible from run to run. */
size_t mmf_pf_heads_weight_grads_workspace_bytes(int32_t K, int32_t L, int64_t rows);
int mmf_pf_heads_weight_grads(int32_t K, int32_t L, int64_t rows, int32_t sd, const float* act, const float* delta,
                              const float* x, const float* d_ll, float* dW_out, float* db_out, float* g_in_out,
                              float* g_out_out, void* workspace, void* stream);

/* R5 + R6 of the BPTT step (no resampling, particle states without gradient) as one forward and one backward kernel:
 *   fused = logsumexp_k(ll[k] + modality_logw[n,k]) over the enabled heads   (ref: crossmodal/base_models/crossmodal_pf.py:132-139)
 *   logw_out = (logw_in + fused) - logsumexp_m(logw_in + fused);  est_out = sum_m exp(logw_out) states[n,m,:]   (A.3)
 * ll (K,N,M) planes as mmf_pf_heads_forward_train writes them, modality_logw (N,K) or NULL, logw_in (N,M), states (N,M,sd).
 * _bwd: given d_est (N,sd) and d_logw (N,M) (either may be NULL = zero) writes d_ll (K,N,M) (zeros for disabled heads),
 * d_modality_logw (N,K) (may be NULL) and d_logw_in (N,M).  Nothing is saved between the calls: _bwd recomputes. */
int mmf_pf_reweight_train_fwd(int32_t N, int32_t M, int32_t K, int32_t sd, uint32_t enabled_mask, const float* ll,
                              const float* modality_logw, const float* logw_in, const float* states, float* logw_out,
                              float* est_out, void* stream);
int mmf_pf_reweight_train_bwd(int32_t N, int32_t M, int32_t K, int32_t sd, uint32_t enabled_mask, const float* ll,
                              const float* modality_logw, const float* logw_in, const float* states, const float* d_est,
                              const float* d_logw, float* d_ll, float* d_modality_logw, float* d_logw_in, void* stream);

/* Per-trajectory MLP stacks (observation encoders of positions / sensors, crossmodal weight models, virtual-sensor heads:
 * ref: crossmodal/push_models/layers.py:107-136, crossmodal/push_models/crossmodal_pf.py:72-104,
 * crossmodal/door_models/crossmodal_kf.py:134-167, crossmodal/door_models/kf.py:81-126) as ONE launch: the host
 * compiles the nn.Sequential into a program of fused ops over per-row scratch slots,
 *     scratch[dst : dst + out_dim] = act(W scratch[src : src + in_dim] + b [+ scratch[res : res + out_dim]])
 * with W stored input-major, Wt[in_dim][out_dim], followed by b[out_dim], at float offset `w_off` of `weights`.
 * A resblock is two ops (the second with res = the block's input).  `inputs[i]` (rows, in_dims[i]) is copied to slot
 * in_slots[i] before the program; `outputs[i]` (rows, out_dims[i]) is read from slot out_slots[i] after it.
 * `ops`, `inputs`, `outputs` and the dims / slots arrays are HOST arrays; `weights` and the tensors are device memory.
 * dst must not overlap src or res.  fp32 FFMA, inputs summed in index order. */
#define MMF_MLP_MAX_OPS 24
#define MMF_MLP_MAX_IO 4
#define MMF_MLP_NONE 0
#define MMF_MLP_RELU 1
#define MMF_MLP_SIGMOID 2
typedef struct mmf_mlp_op {
  int32_t in_dim, out_dim, act;
  int32_t src, dst, res; /* scratch slots (float offsets); res < 0: no residual */
  int64_t w_off;
} mmf_mlp_op;
int mmf_row_mlp(int64_t rows, const mmf_mlp_op* ops, int32_t n_ops, const float* weights, const float* const* inputs,
                const int32_t* in_dims, const int32_t* in_slots, int32_t n_inputs, float* const* outputs,
                const int32_t* out_dims, const int32_t* out_slots, int32_t n_outputs, int32_t scratch_floats,
                void* stream);

/* Training of an mmf_row_mlp program (reverse mode of the ops above).  Rows are taken in groups of 8 (G = ceil(rows/8)
 * groups, the last one padded); per-row planes are stored group-major and feature-major inside a group:
 *     element (row, f) of a plane with F floats per row is at  [(row / 8) * F + f] * 8 + row % 8
 * so the 8 rows a warp owns are 32 contiguous bytes per feature.
 *   tape    F_tape = sum over ops of (in_dim + out_dim) floats per row, G * 8 * F_tape floats in all: op o's input
 *           (src) at f = T_o, its post-activation output (dst) at f = T_o + in_dim, T_o = sum_{p<o} (in_dim + out_dim).
 *   delta   F_delta = sum over ops of out_dim, G * 8 * F_delta floats: g_o = d loss / d (pre-activation of op o)
 *           at f = sum_{p<o} out_dim.  Rows past the end of the padded last group hold zeros.
 * mmf_row_mlp_train_sizes: the float counts of both planes and the byte size of the weight-gradient workspace.
 * mmf_row_mlp_train_fwd: mmf_row_mlp (bit-identical outputs) that also writes the tape.
 * mmf_row_mlp_bwd: the reverse program `bops` (usually the ops in reverse order) over a per-row delta scratch of
 *   scratch_floats floats, laid out like the forward scratch.  d_outputs[i] (rows, out_dims[i]) seed slot dout_slots[i].
 *   For each reverse op (forward op o = ops[bop.op], y = its output from the tape):
 *       g        = delta[g : g + out_dim] * act'(y)      (ReLU: y > 0; Sigmoid: y (1 - y); none: 1)
 *       delta[g] = g, and g -> the delta planes
 *       delta[dres : + out_dim]  = g          or += g         (dres >= 0: the op has a residual; MMF_MLP_DRES_ACC)
 *       delta[dsrc : + in_dim]   = W^T g      or += W^T g     (dsrc >= 0; MMF_MLP_DSRC_ACC), fp32 FFMA over j in order
 *   then d_inputs[i] (rows, din_dims[i]) = delta[din_slots[i] ...].  weights_t holds, at each op's w_off, the torch
 *   layout W (out_dim, in_dim) row-major followed by b (out_dim).
 * mmf_row_mlp_weight_grads: grads at each op's w_off, torch layout like weights_t:
 *       dW (out_dim, in_dim) = sum_rows g x^T,   db (out_dim) = sum_rows g,   x = the op's input from the tape.
 *   The rows are split into fixed chunks whose partial sums go to `workspace` (mmf_row_mlp_train_sizes bytes); a second
 *   kernel adds them in a fixed order: no floating-point atomics, bit-reproducible.  All outputs are overwritten. */
/* mmf_row_mlp_weight_grads takes programs of at most MMF_MLP_MAX_DW_TILES 64 x 64 tiles, summed over the ops:
 * ceil(out_dim / 64) * ceil(in_dim / 64). */
#define MMF_MLP_MAX_DW_TILES 512
#define MMF_MLP_DSRC_ACC 1
#define MMF_MLP_DRES_ACC 2
typedef struct mmf_mlp_bwd_op {
  int32_t op;   /* forward op index */
  int32_t g;    /* delta slot of the op's output: d loss / d dst on entry, g afterwards */
  int32_t dsrc; /* delta slot of the op's input, < 0: not needed */
  int32_t dres; /* delta slot of the op's residual, < 0: no residual */
  int32_t flags;
  int32_t reserved;
} mmf_mlp_bwd_op;
int mmf_row_mlp_train_sizes(int64_t rows, const mmf_mlp_op* ops, int32_t n_ops, int64_t* tape_floats,
                            int64_t* delta_floats, size_t* workspace_bytes);
int mmf_row_mlp_train_fwd(int64_t rows, const mmf_mlp_op* ops, int32_t n_ops, const float* weights,
                          const float* const* inputs, const int32_t* in_dims, const int32_t* in_slots, int32_t n_inputs,
                          float* const* outputs, const int32_t* out_dims, const int32_t* out_slots, int32_t n_outputs,
                          int32_t scratch_floats, float* tape, void* stream);
int mmf_row_mlp_bwd(int64_t rows, const mmf_mlp_op* ops, int32_t n_ops, const float* weights_t, const float* tape,
                    const mmf_mlp_bwd_op* bops, int32_t n_bops, const float* const* d_outputs, const int32_t* out_dims,
                    const int32_t* dout_slots, int32_t n_outputs, float* const* d_inputs, const int32_t* din_dims,
                    const int32_t* din_slots, int32_t n_dinputs, int32_t scratch_floats, float* delta, void* stream);
int mmf_row_mlp_weight_grads(int64_t rows, const mmf_mlp_op* ops, int32_t n_ops, const float* tape, const float* delta,
                             float* grads, void* workspace, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MMF_B200_H */
