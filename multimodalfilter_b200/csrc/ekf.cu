// ekf.cu -- R8 (EKF predict/update with forward-mode dynamics Jacobian), R10/R11 fusion, and the
// per-trajectory hoisted rows of the particle filter (control branch / observation-feature bias).
//
// EKF: one warp owns one (filter, trajectory) pair for ALL T steps (the recursion is serial in t);
// the dynamics chain's weights sit in shared memory once per CTA.  Each 64-wide layer is evaluated
// for 1 + sd rows at once: the primal row and one tangent row per state dimension, the tangents
// being masked by the primal's ReLU pattern -- mathematically the reference's autograd Jacobian
// (A.4; ref: crossmodal/door_models/dynamics.py:37-67) without the (N*sd)-row backward pass.
// Then A P A^T + Q Q^T, S = P- + R R^T, K = P- S^-1, mean/covariance update (A.5), all in registers.
#include "kernels.cuh"

namespace mmf {

// Gauss-Jordan with partial pivoting on an SD x SD matrix held in registers.
template <int SD>
__device__ __forceinline__ void invert(const float (&A)[SD][SD], float (&inv)[SD][SD]) {
  float a[SD][SD];
#pragma unroll
  for (int i = 0; i < SD; ++i)
#pragma unroll
    for (int j = 0; j < SD; ++j) {
      a[i][j] = A[i][j];
      inv[i][j] = (i == j) ? 1.0f : 0.0f;
    }
#pragma unroll
  for (int c = 0; c < SD; ++c) {
    // bring the largest |pivot| of rows >= c to row c (compare-and-swap keeps indices static)
#pragma unroll
    for (int r = c + 1; r < SD; ++r) {
      const bool sw = fabsf(a[r][c]) > fabsf(a[c][c]);
#pragma unroll
      for (int j = 0; j < SD; ++j) {
        const float t0 = a[c][j], t1 = a[r][j];
        a[c][j] = sw ? t1 : t0;
        a[r][j] = sw ? t0 : t1;
        const float u0 = inv[c][j], u1 = inv[r][j];
        inv[c][j] = sw ? u1 : u0;
        inv[r][j] = sw ? u0 : u1;
      }
    }
    const float piv = 1.0f / a[c][c];
#pragma unroll
    for (int j = 0; j < SD; ++j) {
      a[c][j] *= piv;
      inv[c][j] *= piv;
    }
#pragma unroll
    for (int r = 0; r < SD; ++r) {
      if (r != c) {
        const float f = a[r][c];
#pragma unroll
        for (int j = 0; j < SD; ++j) {
          a[r][j] = fmaf(-f, a[c][j], a[r][j]);
          inv[r][j] = fmaf(-f, inv[c][j], inv[r][j]);
        }
      }
    }
  }
}

// Q Q^T of one filter's process-noise factor (row-major SD x SD in q).
template <int SD>
__device__ __forceinline__ void ekf_qqt(const float* q, float (&Q)[SD][SD]) {
#pragma unroll
  for (int i = 0; i < SD; ++i)
#pragma unroll
    for (int j = 0; j < SD; ++j) {
      float s = 0.0f;
#pragma unroll
      for (int k = 0; k < SD; ++k) s = fmaf(q[i * SD + k], q[j * SD + k], s);
      Q[i][j] = s;
    }
}

// The covariance half of one EKF step, shared by the forward (k_ekf_loop) and its reverse mode (k_ekf_loop_bwd),
// which recomputes these from the stored posteriors and the tape instead of saving them:
//   Pp = A Pm A^T + Q Q^T;  S = Pp + Rt Rt^T;  Sinv = S^-1;  Kg = Pp Sinv
template <int SD>
__device__ __forceinline__ void ekf_gain(const float (&A)[SD][SD], const float (&Pm)[SD][SD], const float (&Q)[SD][SD],
                                         const float (&Rt)[SD][SD], float (&Pp)[SD][SD], float (&Sinv)[SD][SD],
                                         float (&Kg)[SD][SD]) {
  float AP[SD][SD], S[SD][SD];
#pragma unroll
  for (int i = 0; i < SD; ++i)
#pragma unroll
    for (int j = 0; j < SD; ++j) {
      float s = 0.0f;
#pragma unroll
      for (int k = 0; k < SD; ++k) s = fmaf(A[i][k], Pm[k][j], s);
      AP[i][j] = s;
    }
#pragma unroll
  for (int i = 0; i < SD; ++i)
#pragma unroll
    for (int j = 0; j < SD; ++j) {
      float s = 0.0f;
#pragma unroll
      for (int k = 0; k < SD; ++k) s = fmaf(AP[i][k], A[j][k], s);
      Pp[i][j] = s + Q[i][j];
    }
#pragma unroll
  for (int i = 0; i < SD; ++i)
#pragma unroll
    for (int j = 0; j < SD; ++j) {
      float s = 0.0f;
#pragma unroll
      for (int k = 0; k < SD; ++k) s = fmaf(Rt[i][k], Rt[j][k], s);
      S[i][j] = Pp[i][j] + s;
    }
  invert<SD>(S, Sinv);
#pragma unroll
  for (int i = 0; i < SD; ++i)
#pragma unroll
    for (int j = 0; j < SD; ++j) {
      float s = 0.0f;
#pragma unroll
      for (int k = 0; k < SD; ++k) s = fmaf(Pp[i][k], Sinv[k][j], s);
      Kg[i][j] = s;
    }
}

// One 64x64 layer for R rows held in shared memory.  Lane computes outputs `lane` and `lane+32`.
// mode: 0 = first half of a resblock (bias, relu), 1 = second half (bias + residual rows, relu),
//       2 = mid layer (rowbias given in `bias`, relu optional)
template <int R>
__device__ __forceinline__ void warp_dense(const float* __restrict__ Wt, const float* __restrict__ bias,
                                           const float* __restrict__ in, const float* __restrict__ resid,
                                           float* __restrict__ out, bool relu, int lane) {
  float acc[R][2];
#pragma unroll
  for (int r = 0; r < R; ++r) acc[r][0] = acc[r][1] = 0.0f;
#pragma unroll 4
  for (int k = 0; k < U; k += 4) {
    float4 hv[R];
#pragma unroll
    for (int r = 0; r < R; ++r) hv[r] = *reinterpret_cast<const float4*>(in + r * U + k);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float w0 = Wt[(k + i) * U + lane], w1 = Wt[(k + i) * U + lane + 32];
#pragma unroll
      for (int r = 0; r < R; ++r) {
        const float h = (i == 0) ? hv[r].x : (i == 1) ? hv[r].y : (i == 2) ? hv[r].z : hv[r].w;
        acc[r][0] = fmaf(w0, h, acc[r][0]);
        acc[r][1] = fmaf(w1, h, acc[r][1]);
      }
    }
  }
#pragma unroll
  for (int half = 0; half < 2; ++half) {
    const int j = lane + 32 * half;
    float a = acc[0][half] + bias[j];
    if (resid != nullptr) a += resid[j];
    const bool on = !relu || a > 0.0f;
    float outv[R];
    outv[0] = on ? a : 0.0f;
#pragma unroll
    for (int r = 1; r < R; ++r) {
      float t = acc[r][half];
      if (resid != nullptr) t += resid[r * U + j];
      outv[r] = on ? t : 0.0f;
    }
    __syncwarp();
#pragma unroll
    for (int r = 0; r < R; ++r) out[r * U + j] = outv[r];
  }
  __syncwarp();
}

// Control branch + hoisted mid-layer row for ONE trajectory, computed by one warp with weights
// read through the read-only path (they are shared by every warp => L1 resident).
// buf: >= max(in_dim, 64) + 64 floats of per-warp shared memory.  Result left in rowbias[64] (smem).
__device__ __forceinline__ void warp_traj_row(const TrajRowsDev& tr, const float* __restrict__ input,
                                              float* __restrict__ buf, float* __restrict__ rowbias, int lane) {
  const float* w = tr.w;
  int feat_dim = tr.in_dim;
  float* a = buf;             // current features
  float* b = buf + 256;       // scratch (64)
  for (int i = lane; i < tr.in_dim; i += 32) a[i] = input[i];
  __syncwarp();
  if (tr.has_encoder) {
    // h = relu(enc_W u + enc_b)
    float h0 = __ldg(w + tr.in_dim * U + lane), h1 = __ldg(w + tr.in_dim * U + lane + 32);
    for (int i = 0; i < tr.in_dim; ++i) {
      h0 = fmaf(__ldg(w + i * U + lane), a[i], h0);
      h1 = fmaf(__ldg(w + i * U + lane + 32), a[i], h1);
    }
    w += tr.in_dim * U + U;
    __syncwarp();
    b[lane] = fmaxf(h0, 0.0f);
    b[lane + 32] = fmaxf(h1, 0.0f);
    __syncwarp();
    // resblock: t = relu(W1 h + b1); y = relu(W2 t + b2 + h)
    float t0 = __ldg(w + U * U + lane), t1 = __ldg(w + U * U + lane + 32);
    for (int k = 0; k < U; ++k) {
      t0 = fmaf(__ldg(w + k * U + lane), b[k], t0);
      t1 = fmaf(__ldg(w + k * U + lane + 32), b[k], t1);
    }
    w += U * U + U;
    a[lane] = fmaxf(t0, 0.0f);
    a[lane + 32] = fmaxf(t1, 0.0f);
    __syncwarp();
    float y0 = __ldg(w + U * U + lane) + b[lane], y1 = __ldg(w + U * U + lane + 32) + b[lane + 32];
    for (int k = 0; k < U; ++k) {
      y0 = fmaf(__ldg(w + k * U + lane), a[k], y0);
      y1 = fmaf(__ldg(w + k * U + lane + 32), a[k], y1);
    }
    w += U * U + U;
    __syncwarp();
    a[lane] = fmaxf(y0, 0.0f);
    a[lane + 32] = fmaxf(y1, 0.0f);
    __syncwarp();
    feat_dim = U;
  }
  float r0 = __ldg(w + feat_dim * U + lane), r1 = __ldg(w + feat_dim * U + lane + 32);
  for (int k = 0; k < feat_dim; ++k) {
    r0 = fmaf(__ldg(w + k * U + lane), a[k], r0);
    r1 = fmaf(__ldg(w + k * U + lane + 32), a[k], r1);
  }
  __syncwarp();
  rowbias[lane] = r0;
  rowbias[lane + 32] = r1;
  __syncwarp();
}

// ---- mmf_pf_traj_rows: (1+K) planes x N trajectories, one warp each ----------------------------------
struct TrajRowsParams {
  TrajRowsDev rows[1 + MMF_MAX_HEADS];
  const float* inputs[1 + MMF_MAX_HEADS];
  int planes, N;
  float* out;  // (planes, N, 64)
};

__global__ void __launch_bounds__(256) k_traj_rows(const __grid_constant__ TrajRowsParams P) {
  __shared__ __align__(16) float sm[8][256 + 64 + 64];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const long long total = (long long)P.planes * P.N;
  for (long long item = (long long)blockIdx.x * 8 + wid; item < total; item += (long long)gridDim.x * 8) {
    const int plane = (int)(item / P.N), n = (int)(item % P.N);
    if (P.inputs[plane] == nullptr) continue;
    const TrajRowsDev tr = P.rows[plane];
    float* buf = sm[wid];
    warp_traj_row(tr, P.inputs[plane] + (size_t)n * tr.in_dim, buf, buf + 320, lane);
    float* dst = P.out + ((size_t)plane * P.N + n) * U;
    dst[lane] = buf[320 + lane];
    dst[lane + 32] = buf[320 + lane + 32];
    __syncwarp();
  }
}

int launch_traj_rows(const mmf_pf_model* model, int N, const float* controls, const float* const* obs_feats,
                     float* out, cudaStream_t stream) {
  TrajRowsParams P;
  P.planes = 1 + model->num_heads;
  P.N = N;
  P.out = out;
  P.rows[0] = to_dev(model->dynamics_rows);
  P.inputs[0] = controls;
  for (int k = 0; k < model->num_heads; ++k) {
    P.rows[1 + k] = to_dev(model->head_rows[k]);
    P.inputs[1 + k] = obs_feats ? obs_feats[k] : nullptr;
    MMF_REQUIRE(model->head_rows[k].in_dim <= MMF_MAX_OBS_FEATS, "head %d: %d observation features > %d", k,
                model->head_rows[k].in_dim, MMF_MAX_OBS_FEATS);
  }
  const long long total = (long long)P.planes * N;
  if (total == 0) return MMF_OK;
  long long blocks = (total + 7) / 8;
  if (blocks > 148 * 8) blocks = 148 * 8;
  k_traj_rows<<<(int)blocks, 256, 0, stream>>>(P);
  MMF_LAUNCH_CHECK("k_traj_rows");
  return MMF_OK;
}

// ---- EKF loop ------------------------------------------------------------------------------------------
// TAPE: also record mu- (pred_out) and A (jac_out) of every step for k_ekf_loop_bwd.  The arithmetic is the same
// with and without it, so both instantiations produce the same posteriors bit for bit.
template <int SD, bool TAPE>
__global__ void __launch_bounds__(EKF_MAX_WARPS * 32, 1) k_ekf_loop(const __grid_constant__ EkfParams P, int wpc) {
  constexpr int R = 1 + SD;
  extern __shared__ __align__(16) float sm[];
  const int f = blockIdx.y;
  const ChainDev ch = P.dyn[f];
  const int nf = ch.floats();
  float* wsm = sm;
  float* warp_base = sm + ((nf + 3) & ~3);
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  // per-warp scratch: rows A (R*64), rows B (R*64), residual rows (R*64), traj buffers (256+64+64)
  constexpr int WARP_FLOATS = 3 * R * U + 384;
  float* rowsA = warp_base + (size_t)wid * WARP_FLOATS;
  float* rowsB = rowsA + R * U;
  float* rowsX = rowsB + R * U;
  float* tbuf = rowsX + R * U;
  float* rowbias = tbuf + 320;

  {
    const float4* src = reinterpret_cast<const float4*>(ch.w);
    float4* dst = reinterpret_cast<float4*>(wsm);
    for (int i = tid; i < nf / 4; i += blockDim.x) dst[i] = __ldg(src + i);
    for (int i = (nf & ~3) + tid; i < nf; i += blockDim.x) wsm[i] = __ldg(ch.w + i);
  }
  __syncthreads();

  const int N = P.N, T = P.T;
  float Q[SD][SD];  // Q Q^T
  ekf_qqt<SD>(P.q[f], Q);

  for (int n = blockIdx.x * wpc + wid; n < N && wid < wpc; n += gridDim.x * wpc) {
    float mu[SD], Pm[SD][SD];
#pragma unroll
    for (int i = 0; i < SD; ++i) {
      mu[i] = P.jac_only ? 0.0f : P.mean0[((size_t)f * N + n) * SD + i];
#pragma unroll
      for (int j = 0; j < SD; ++j) Pm[i][j] = P.jac_only ? 0.0f : P.cov0[(((size_t)f * N + n) * SD + i) * SD + j];
    }
    for (int t = 0; t < T; ++t) {
      if (P.jac_only) {
#pragma unroll
        for (int i = 0; i < SD; ++i) mu[i] = P.mean0[(size_t)n * SD + i];
      }
      // ---- hoisted row: control branch -> mid-layer bias --------------------------------------------
      warp_traj_row(P.rows[f], P.controls + ((size_t)t * N + n) * P.cd, tbuf, rowbias, lane);

      // ---- input layer with tangents -----------------------------------------------------------------
      const float* w = wsm;
      {
        const float* inb = w + SD * U;
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          const int j = lane + 32 * half;
          float a = inb[j];
#pragma unroll
          for (int i = 0; i < SD; ++i) a = fmaf(w[i * U + j], mu[i], a);
          const bool on = a > 0.0f;
          rowsA[j] = on ? a : 0.0f;
#pragma unroll
          for (int i = 0; i < SD; ++i) rowsA[(1 + i) * U + j] = on ? w[i * U + j] : 0.0f;
        }
        __syncwarp();
        w += SD * U + U;
      }
      float* cur = rowsA;
      float* nxt = rowsB;
      // ---- 64x64 layers ----------------------------------------------------------------------------------
      const int n_dense = 2 * ch.n_pre + 1 + 2 * ch.n_post;
      const int mid_at = 2 * ch.n_pre;
      for (int s = 0; s < n_dense; ++s) {
        const bool is_mid = (s == mid_at);
        const int rel = (s < mid_at) ? s : s - mid_at - 1;
        const bool first_half = !is_mid && ((rel & 1) == 0);
        if (is_mid) {
          warp_dense<R>(w, rowbias, cur, nullptr, nxt, ch.mid_relu != 0, lane);
          w += U * U;
        } else if (first_half) {
          for (int i = lane; i < R * U; i += 32) rowsX[i] = cur[i];
          __syncwarp();
          warp_dense<R>(w, w + U * U, cur, nullptr, nxt, true, lane);
          w += U * U + U;
        } else {
          warp_dense<R>(w, w + U * U, cur, rowsX, nxt, true, lane);
          w += U * U + U;
        }
        float* tmp = cur;
        cur = nxt;
        nxt = tmp;
      }
      // ---- output layer: y (SD+1) and its tangents ------------------------------------------------------
      float y[SD + 1], dy[SD + 1][SD];
#pragma unroll
      for (int o = 0; o < SD + 1; ++o) {
        const float w0 = w[o * U + lane], w1 = w[o * U + lane + 32];
        float part = fmaf(w0, cur[lane], w1 * cur[lane + 32]);
        y[o] = warp_sum(part) + w[(SD + 1) * U + o];
#pragma unroll
        for (int i = 0; i < SD; ++i) {
          part = fmaf(w0, cur[(1 + i) * U + lane], w1 * cur[(1 + i) * U + lane + 32]);
          dy[o][i] = warp_sum(part);
        }
      }
      __syncwarp();
      // ---- gate, prediction, Jacobian A = I + g dy[:sd] + y[:sd] g(1-g) dy[sd]^T --------------------------
      const float g = 1.0f / (1.0f + expf(-y[SD]));
      const float gp = g * (1.0f - g);
      float pred[SD], A[SD][SD];
#pragma unroll
      for (int i = 0; i < SD; ++i) {
        pred[i] = mu[i] + y[i] * g;
#pragma unroll
        for (int j = 0; j < SD; ++j) A[i][j] = ((i == j) ? 1.0f : 0.0f) + g * dy[i][j] + y[i] * gp * dy[SD][j];
      }
      if (P.jac_only) {
        if (lane == 0) {
#pragma unroll
          for (int i = 0; i < SD; ++i) {
            P.mean_out[(size_t)n * SD + i] = pred[i];
#pragma unroll
            for (int j = 0; j < SD; ++j) P.cov_out[((size_t)n * SD + i) * SD + j] = A[i][j];
          }
        }
        continue;
      }
      // ---- predict covariance, update (C = I) -----------------------------------------------------------------
      const size_t ft = ((size_t)f * T + t) * N + n;
      float Rt[SD][SD], Pp[SD][SD], Sinv[SD][SD], Kg[SD][SD], zt[SD];
#pragma unroll
      for (int i = 0; i < SD; ++i) {
        zt[i] = P.z[ft * SD + i];
#pragma unroll
        for (int j = 0; j < SD; ++j) Rt[i][j] = P.r_tril[(ft * SD + i) * SD + j];
      }
      if constexpr (TAPE) {
        if (lane == 0) {
#pragma unroll
          for (int i = 0; i < SD; ++i) {
            P.pred_out[ft * SD + i] = pred[i];
#pragma unroll
            for (int j = 0; j < SD; ++j) P.jac_out[(ft * SD + i) * SD + j] = A[i][j];
          }
        }
      }
      ekf_gain<SD>(A, Pm, Q, Rt, Pp, Sinv, Kg);
#pragma unroll
      for (int i = 0; i < SD; ++i) {
        float s = 0.0f;
#pragma unroll
        for (int k = 0; k < SD; ++k) s = fmaf(Kg[i][k], zt[k] - pred[k], s);
        mu[i] = pred[i] + s;
      }
#pragma unroll
      for (int i = 0; i < SD; ++i)
#pragma unroll
        for (int j = 0; j < SD; ++j) {
          float s = 0.0f;
#pragma unroll
          for (int k = 0; k < SD; ++k) s = fmaf(((i == k) ? 1.0f : 0.0f) - Kg[i][k], Pp[k][j], s);
          Pm[i][j] = s;
        }
      if (lane == 0) {
#pragma unroll
        for (int i = 0; i < SD; ++i) {
          P.mean_out[ft * SD + i] = mu[i];
#pragma unroll
          for (int j = 0; j < SD; ++j) P.cov_out[(ft * SD + i) * SD + j] = Pm[i][j];
        }
      }
    }
  }
}

template <int SD, bool TAPE>
static int launch_ekf_sd(const EkfParams& P, cudaStream_t stream) {
  int dev = 0, sms = 148;
  MMF_CUDA(cudaGetDevice(&dev));
  MMF_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  int nf = 0;
  for (int f = 0; f < P.F; ++f) nf = nf > P.dyn[f].floats() ? nf : P.dyn[f].floats();
  // spread (filter, trajectory) pairs over the SMs: few warps per CTA => low per-step latency
  const long long pairs = (long long)P.F * P.N;
  int wpc = (int)((pairs + sms - 1) / sms);
  wpc = wpc < 1 ? 1 : (wpc > EKF_MAX_WARPS ? EKF_MAX_WARPS : wpc);
  constexpr int WARP_FLOATS = 3 * (1 + SD) * U + 384;
  static thread_local int configured_dev = -1;
  static thread_local size_t window = 0;
  if (configured_dev != dev) {
    int rc = opt_in_shared_memory(k_ekf_loop<SD, TAPE>, &window);
    if (rc) return rc;
    configured_dev = dev;
  }
  size_t smem = ((size_t)((nf + 3) & ~3) + (size_t)wpc * WARP_FLOATS) * sizeof(float);
  while (smem > window && wpc > 1) {
    --wpc;
    smem = ((size_t)((nf + 3) & ~3) + (size_t)wpc * WARP_FLOATS) * sizeof(float);
  }
  MMF_REQUIRE(smem <= window, "ekf: %zu B of shared memory needed (window %zu B)", smem, window);
  int ctas = (P.N + wpc - 1) / wpc;
  const int max_ctas = (sms + P.F - 1) / P.F > 0 ? (sms / P.F > 0 ? sms / P.F : 1) : 1;
  if (ctas > max_ctas) ctas = max_ctas;
  dim3 grid(ctas, P.F);
  k_ekf_loop<SD, TAPE><<<grid, wpc * 32, smem, stream>>>(P, wpc);
  MMF_LAUNCH_CHECK("k_ekf_loop");
  return MMF_OK;
}

int launch_ekf(const EkfParams& P, int sd, cudaStream_t stream, bool tape) {
  switch (sd) {
    case 1: return tape ? launch_ekf_sd<1, true>(P, stream) : launch_ekf_sd<1, false>(P, stream);
    case 2: return tape ? launch_ekf_sd<2, true>(P, stream) : launch_ekf_sd<2, false>(P, stream);
    case 3: return tape ? launch_ekf_sd<3, true>(P, stream) : launch_ekf_sd<3, false>(P, stream);
    case 4: return tape ? launch_ekf_sd<4, true>(P, stream) : launch_ekf_sd<4, false>(P, stream);
  }
  set_error("ekf: state_dim %d unsupported (1..%d)", sd, MMF_MAX_SD);
  return MMF_E_INVALID;
}

// ---- reverse mode of the EKF loop: one thread per (filter, trajectory), t = T-1 ... 0 in registers ---------------
// The dynamics Jacobian A is a constant of the recursion (the reference differentiates f at a detached state, A.4) and
// the dynamics are frozen, so one step's adjoint is SD x SD algebra given A and mu- from the tape.  With mb / Pb the
// gradient reaching posterior t (the caller's d_means[t] / d_covs[t] plus what step t+1 sent back), r = z - mu-:
//   z_bar  = Kg^T mb;                       mb-  = mb - z_bar
//   Kg_bar = mb r^T - Pb Pp^T;              S_bar = -Sinv^T Pp^T Kg_bar Sinv^T
//   Pp_bar = (I - Kg)^T Pb + Kg_bar Sinv^T + S_bar;    R_bar = (S_bar + S_bar^T) Rt
//   Pb(t-1) = A^T Pp_bar A;                 mb(t-1) = A^T mb-
// Every output element is written by exactly one thread: no atomics, bit-reproducible.
template <int SD>
__global__ void __launch_bounds__(128) k_ekf_loop_bwd(const __grid_constant__ EkfBwdParams P) {
  const int N = P.N, T = P.T;
  const long long total = (long long)P.F * N;
  for (long long item = blockIdx.x * (long long)blockDim.x + threadIdx.x; item < total;
       item += (long long)gridDim.x * blockDim.x) {
    const int f = (int)(item / N), n = (int)(item % N);
    float Q[SD][SD];
    ekf_qqt<SD>(P.q[f], Q);
    float mb[SD], Pb[SD][SD];
#pragma unroll
    for (int i = 0; i < SD; ++i) {
      mb[i] = 0.0f;
#pragma unroll
      for (int j = 0; j < SD; ++j) Pb[i][j] = 0.0f;
    }
    for (int t = T - 1; t >= 0; --t) {
      const size_t ft = ((size_t)f * T + t) * N + n;
      const float* prev = t > 0 ? P.covs + (ft - N) * SD * SD : P.cov0 + ((size_t)f * N + n) * SD * SD;
      float A[SD][SD], Pm[SD][SD], Rt[SD][SD], r[SD];
#pragma unroll
      for (int i = 0; i < SD; ++i) {
        r[i] = P.z[ft * SD + i] - P.pred[ft * SD + i];
#pragma unroll
        for (int j = 0; j < SD; ++j) {
          A[i][j] = P.jac[(ft * SD + i) * SD + j];
          Pm[i][j] = prev[i * SD + j];
          Rt[i][j] = P.r_tril[(ft * SD + i) * SD + j];
        }
      }
      float Pp[SD][SD], Sinv[SD][SD], Kg[SD][SD];
      ekf_gain<SD>(A, Pm, Q, Rt, Pp, Sinv, Kg);
      if (P.d_means != nullptr) {
#pragma unroll
        for (int i = 0; i < SD; ++i) mb[i] += P.d_means[ft * SD + i];
      }
      if (P.d_covs != nullptr) {
#pragma unroll
        for (int i = 0; i < SD; ++i)
#pragma unroll
          for (int j = 0; j < SD; ++j) Pb[i][j] += P.d_covs[(ft * SD + i) * SD + j];
      }
      // z_bar, mb-
      float mbp[SD];
#pragma unroll
      for (int i = 0; i < SD; ++i) {
        float s = 0.0f;
#pragma unroll
        for (int k = 0; k < SD; ++k) s = fmaf(Kg[k][i], mb[k], s);
        P.d_z[ft * SD + i] = s;
        mbp[i] = mb[i] - s;
      }
      // Kg_bar = mb r^T - Pb Pp^T
      float Kb[SD][SD];
#pragma unroll
      for (int i = 0; i < SD; ++i)
#pragma unroll
        for (int j = 0; j < SD; ++j) {
          float s = 0.0f;
#pragma unroll
          for (int k = 0; k < SD; ++k) s = fmaf(Pb[i][k], Pp[j][k], s);
          Kb[i][j] = mb[i] * r[j] - s;
        }
      // S_bar = -Sinv^T (Pp^T Kg_bar) Sinv^T
      float M1[SD][SD], M2[SD][SD], Sb[SD][SD];
#pragma unroll
      for (int i = 0; i < SD; ++i)
#pragma unroll
        for (int j = 0; j < SD; ++j) {
          float s = 0.0f;
#pragma unroll
          for (int k = 0; k < SD; ++k) s = fmaf(Pp[k][i], Kb[k][j], s);
          M1[i][j] = s;
        }
#pragma unroll
      for (int i = 0; i < SD; ++i)
#pragma unroll
        for (int j = 0; j < SD; ++j) {
          float s = 0.0f;
#pragma unroll
          for (int k = 0; k < SD; ++k) s = fmaf(Sinv[k][i], M1[k][j], s);
          M2[i][j] = s;
        }
#pragma unroll
      for (int i = 0; i < SD; ++i)
#pragma unroll
        for (int j = 0; j < SD; ++j) {
          float s = 0.0f;
#pragma unroll
          for (int k = 0; k < SD; ++k) s = fmaf(M2[i][k], Sinv[j][k], s);
          Sb[i][j] = -s;
        }
      // R_bar = (S_bar + S_bar^T) Rt: every entry, the upper ones included (as autograd of r_tril @ r_tril^T)
#pragma unroll
      for (int i = 0; i < SD; ++i)
#pragma unroll
        for (int j = 0; j < SD; ++j) {
          float s = 0.0f;
#pragma unroll
          for (int k = 0; k < SD; ++k) s = fmaf(Sb[i][k] + Sb[k][i], Rt[k][j], s);
          P.d_r_tril[(ft * SD + i) * SD + j] = s;
        }
      // Pp_bar = (I - Kg)^T Pb + Kg_bar Sinv^T + S_bar   (into M1)
#pragma unroll
      for (int i = 0; i < SD; ++i)
#pragma unroll
        for (int j = 0; j < SD; ++j) {
          float s = Sb[i][j];
#pragma unroll
          for (int k = 0; k < SD; ++k) s = fmaf(((k == i) ? 1.0f : 0.0f) - Kg[k][i], Pb[k][j], s);
#pragma unroll
          for (int k = 0; k < SD; ++k) s = fmaf(Kb[i][k], Sinv[j][k], s);
          M1[i][j] = s;
        }
      // Pb <- A^T Pp_bar A,  mb <- A^T mb-
#pragma unroll
      for (int i = 0; i < SD; ++i)
#pragma unroll
        for (int j = 0; j < SD; ++j) {
          float s = 0.0f;
#pragma unroll
          for (int k = 0; k < SD; ++k) s = fmaf(A[k][i], M1[k][j], s);
          M2[i][j] = s;
        }
#pragma unroll
      for (int i = 0; i < SD; ++i) {
        float s = 0.0f;
#pragma unroll
        for (int k = 0; k < SD; ++k) s = fmaf(A[k][i], mbp[k], s);
        mb[i] = s;
#pragma unroll
        for (int j = 0; j < SD; ++j) {
          float u = 0.0f;
#pragma unroll
          for (int k = 0; k < SD; ++k) u = fmaf(M2[i][k], A[k][j], u);
          Pb[i][j] = u;
        }
      }
    }
    const size_t fn = (size_t)f * N + n;
#pragma unroll
    for (int i = 0; i < SD; ++i) {
      P.d_mean0[fn * SD + i] = mb[i];
#pragma unroll
      for (int j = 0; j < SD; ++j) P.d_cov0[(fn * SD + i) * SD + j] = Pb[i][j];
    }
  }
}

int launch_ekf_bwd(const EkfBwdParams& P, int sd, cudaStream_t stream) {
  const long long total = (long long)P.F * P.N;
  if (total == 0) return MMF_OK;
  long long blocks = (total + 127) / 128;
  if (blocks > 148 * 16) blocks = 148 * 16;
  switch (sd) {
    case 1: k_ekf_loop_bwd<1><<<(int)blocks, 128, 0, stream>>>(P); break;
    case 2: k_ekf_loop_bwd<2><<<(int)blocks, 128, 0, stream>>>(P); break;
    case 3: k_ekf_loop_bwd<3><<<(int)blocks, 128, 0, stream>>>(P); break;
    case 4: k_ekf_loop_bwd<4><<<(int)blocks, 128, 0, stream>>>(P); break;
    default: set_error("ekf_bwd: state_dim %d unsupported (1..%d)", sd, MMF_MAX_SD); return MMF_E_INVALID;
  }
  MMF_LAUNCH_CHECK("k_ekf_loop_bwd");
  return MMF_OK;
}

// ---- R10 / R11 fusion: one thread per (t, n) row ---------------------------------------------------------
template <int SD>
__global__ void k_kf_fuse(int K, long long rows, const float* __restrict__ mu, const float* __restrict__ Pk,
                          const float* __restrict__ beta, float* __restrict__ mean_out,
                          float* __restrict__ cov_out, int unimodal) {
  for (long long r = blockIdx.x * (long long)blockDim.x + threadIdx.x; r < rows;
       r += (long long)gridDim.x * blockDim.x) {
    float mean[SD], cov[SD][SD];
    if (!unimodal) {
      // ref: base_models/utility.py:4-11 + crossmodal_kf.py:153-167
      float bsum[SD];
#pragma unroll
      for (int d = 0; d < SD; ++d) {
        bsum[d] = 0.0f;
        mean[d] = 0.0f;
#pragma unroll
        for (int e = 0; e < SD; ++e) cov[d][e] = 0.0f;
      }
      for (int k = 0; k < K; ++k)
#pragma unroll
        for (int d = 0; d < SD; ++d) bsum[d] += beta[((size_t)k * rows + r) * SD + d];
      for (int k = 0; k < K; ++k) {
        float b[SD];
#pragma unroll
        for (int d = 0; d < SD; ++d) b[d] = beta[((size_t)k * rows + r) * SD + d];
#pragma unroll
        for (int d = 0; d < SD; ++d) {
          mean[d] += (b[d] / (bsum[d] + 1e-9f)) * mu[((size_t)k * rows + r) * SD + d];
#pragma unroll
          for (int e = 0; e < SD; ++e) cov[d][e] += (b[d] * b[e]) * Pk[(((size_t)k * rows + r) * SD + d) * SD + e];
        }
      }
    } else {
      // ref: base_models/unimodal_kf.py:199-242 (information form; +1e-9 is elementwise)
      float Lsum[SD][SD], info[SD];
#pragma unroll
      for (int d = 0; d < SD; ++d) {
        info[d] = 0.0f;
#pragma unroll
        for (int e = 0; e < SD; ++e) Lsum[d][e] = 0.0f;
      }
      for (int k = 0; k < K; ++k) {
        float Pm[SD][SD], L[SD][SD];
#pragma unroll
        for (int d = 0; d < SD; ++d)
#pragma unroll
          for (int e = 0; e < SD; ++e) Pm[d][e] = Pk[(((size_t)k * rows + r) * SD + d) * SD + e] + 1e-9f;
        invert<SD>(Pm, L);
#pragma unroll
        for (int d = 0; d < SD; ++d) {
          float s = 0.0f;
#pragma unroll
          for (int e = 0; e < SD; ++e) {
            Lsum[d][e] += L[d][e];
            s = fmaf(L[d][e], mu[((size_t)k * rows + r) * SD + e], s);
          }
          info[d] += s;
        }
      }
#pragma unroll
      for (int d = 0; d < SD; ++d)
#pragma unroll
        for (int e = 0; e < SD; ++e) Lsum[d][e] += 1e-9f;
      invert<SD>(Lsum, cov);
#pragma unroll
      for (int d = 0; d < SD; ++d) {
        float s = 0.0f;
#pragma unroll
        for (int e = 0; e < SD; ++e) s = fmaf(cov[d][e], info[e], s);
        mean[d] = s;
      }
    }
#pragma unroll
    for (int d = 0; d < SD; ++d) {
      mean_out[r * SD + d] = mean[d];
#pragma unroll
      for (int e = 0; e < SD; ++e) cov_out[(r * SD + d) * SD + e] = cov[d][e];
    }
  }
}

int launch_kf_fuse(int K, long long rows, int sd, const float* mu, const float* Pk, const float* beta,
                   float* mean_out, float* cov_out, int unimodal, cudaStream_t stream) {
  if (rows == 0) return MMF_OK;
  long long blocks = (rows + 127) / 128;
  if (blocks > 148 * 16) blocks = 148 * 16;
  switch (sd) {
    case 1: k_kf_fuse<1><<<(int)blocks, 128, 0, stream>>>(K, rows, mu, Pk, beta, mean_out, cov_out, unimodal); break;
    case 2: k_kf_fuse<2><<<(int)blocks, 128, 0, stream>>>(K, rows, mu, Pk, beta, mean_out, cov_out, unimodal); break;
    case 3: k_kf_fuse<3><<<(int)blocks, 128, 0, stream>>>(K, rows, mu, Pk, beta, mean_out, cov_out, unimodal); break;
    case 4: k_kf_fuse<4><<<(int)blocks, 128, 0, stream>>>(K, rows, mu, Pk, beta, mean_out, cov_out, unimodal); break;
    default: set_error("kf_fuse: state_dim %d unsupported", sd); return MMF_E_INVALID;
  }
  MMF_LAUNCH_CHECK("k_kf_fuse");
  return MMF_OK;
}

// ---- R12 measurement-level fusion of K virtual sensors: one thread per (t, n) row ---------------------------
// crossmodal (ref: crossmodal/base_models/crossmodal_kf.py:219-235, 337-354, utility.py:4-11):
//   z = sum_k (w_k / (sum_k w_k + 1e-9)) z_k ;  C = (prod_k prod_d w_k[d]) * sum_k L_k L_k^T ;  out = cholesky(C)
// unimodal (ref: crossmodal/base_models/unimodal_kf.py:56-115; returns a covariance, as the reference does):
//   K == 1: (z_0, L_0 L_0^T);  else  Pr_k = 1 / (L_k + 1e-9) ELEMENTWISE (the reference's arithmetic, zeros above the
//   diagonal included), w_k = diag(Pr_k), z as above, out = inverse(sum_k Pr_k + 1e-9)
template <int SD>
__global__ void k_kf_fuse_measurements(int K, long long rows, const float* __restrict__ z, const float* __restrict__ tril,
                                       const float* __restrict__ w, float* __restrict__ z_out,
                                       float* __restrict__ mat_out, int unimodal) {
  for (long long r = blockIdx.x * (long long)blockDim.x + threadIdx.x; r < rows;
       r += (long long)gridDim.x * blockDim.x) {
    float wsum[SD], mean[SD], acc[SD][SD], out[SD][SD];
    float mult = 1.0f;
#pragma unroll
    for (int d = 0; d < SD; ++d) {
      wsum[d] = 0.0f;
      mean[d] = 0.0f;
#pragma unroll
      for (int e = 0; e < SD; ++e) acc[d][e] = 0.0f;
    }
    auto weight = [&](int k, int d) -> float {
      if (!unimodal) return w[((size_t)k * rows + r) * SD + d];
      return 1.0f / (tril[(((size_t)k * rows + r) * SD + d) * SD + d] + 1e-9f);
    };
    for (int k = 0; k < K; ++k)
#pragma unroll
      for (int d = 0; d < SD; ++d) {
        const float wk = weight(k, d);
        wsum[d] += wk;
        mult *= wk;
      }
    for (int k = 0; k < K; ++k) {
      float L[SD][SD];
#pragma unroll
      for (int d = 0; d < SD; ++d)
#pragma unroll
        for (int e = 0; e < SD; ++e) L[d][e] = tril[(((size_t)k * rows + r) * SD + d) * SD + e];
#pragma unroll
      for (int d = 0; d < SD; ++d) {
        mean[d] += (weight(k, d) / (wsum[d] + 1e-9f)) * z[((size_t)k * rows + r) * SD + d];
#pragma unroll
        for (int e = 0; e < SD; ++e) {
          if (unimodal && K > 1) {
            acc[d][e] += 1.0f / (L[d][e] + 1e-9f);
          } else {
            float s = 0.0f;
#pragma unroll
            for (int j = 0; j < SD; ++j) s = fmaf(L[d][j], L[e][j], s);
            acc[d][e] += s;
          }
        }
      }
    }
    if (unimodal) {
      if (K > 1) {
#pragma unroll
        for (int d = 0; d < SD; ++d)
#pragma unroll
          for (int e = 0; e < SD; ++e) acc[d][e] += 1e-9f;
        invert<SD>(acc, out);
      } else {
#pragma unroll
        for (int d = 0; d < SD; ++d) {
          mean[d] = z[(size_t)r * SD + d];
#pragma unroll
          for (int e = 0; e < SD; ++e) out[d][e] = acc[d][e];
        }
      }
    } else {
      // Cholesky factor (lower) of mult * sum_k L_k L_k^T; a non-positive pivot gives NaN like torch.linalg.cholesky raises
#pragma unroll
      for (int d = 0; d < SD; ++d)
#pragma unroll
        for (int e = 0; e < SD; ++e) {
          acc[d][e] *= mult;
          out[d][e] = 0.0f;
        }
#pragma unroll
      for (int j = 0; j < SD; ++j) {
        float s = acc[j][j];
#pragma unroll
        for (int q = 0; q < SD; ++q)
          if (q < j) s -= out[j][q] * out[j][q];
        const float piv = sqrtf(s);
        out[j][j] = piv;
#pragma unroll
        for (int i = 0; i < SD; ++i) {
          if (i > j) {
            float t = acc[i][j];
#pragma unroll
            for (int q = 0; q < SD; ++q)
              if (q < j) t -= out[i][q] * out[j][q];
            out[i][j] = t / piv;
          }
        }
      }
    }
#pragma unroll
    for (int d = 0; d < SD; ++d) {
      z_out[(size_t)r * SD + d] = mean[d];
#pragma unroll
      for (int e = 0; e < SD; ++e) mat_out[((size_t)r * SD + d) * SD + e] = out[d][e];
    }
  }
}

int launch_kf_fuse_measurements(int K, long long rows, int sd, const float* z, const float* tril, const float* w,
                                float* z_out, float* mat_out, int unimodal, cudaStream_t stream) {
  if (rows == 0) return MMF_OK;
  long long blocks = (rows + 127) / 128;
  if (blocks > 148 * 16) blocks = 148 * 16;
  switch (sd) {
    case 1: k_kf_fuse_measurements<1><<<(int)blocks, 128, 0, stream>>>(K, rows, z, tril, w, z_out, mat_out, unimodal); break;
    case 2: k_kf_fuse_measurements<2><<<(int)blocks, 128, 0, stream>>>(K, rows, z, tril, w, z_out, mat_out, unimodal); break;
    case 3: k_kf_fuse_measurements<3><<<(int)blocks, 128, 0, stream>>>(K, rows, z, tril, w, z_out, mat_out, unimodal); break;
    case 4: k_kf_fuse_measurements<4><<<(int)blocks, 128, 0, stream>>>(K, rows, z, tril, w, z_out, mat_out, unimodal); break;
    default: set_error("kf_fuse_measurements: state_dim %d unsupported", sd); return MMF_E_INVALID;
  }
  MMF_LAUNCH_CHECK("k_kf_fuse_measurements");
  return MMF_OK;
}

}  // namespace mmf
