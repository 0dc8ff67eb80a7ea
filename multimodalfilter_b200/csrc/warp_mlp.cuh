// warp_mlp.cuh -- one warp evaluates the 64-wide MLP layers of one trajectory from shared memory: shared by the EKF
// recursion (ekf.cu) and the dynamics rollout (dyn_rollout.cu).
#pragma once
#include "common.cuh"

namespace mmf {

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

}  // namespace mmf
