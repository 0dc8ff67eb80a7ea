// dyn_rollout.cu -- open-loop rollout of the gated-residual dynamics (ref: crossmodal/push_models/dynamics.py:44-63) over
// T steps in ONE launch (k_dyn_rollout), optionally recording a tape of every layer's input, and its reverse mode in one
// more (k_dyn_rollout_bwd), which walks t = T-1 ... 0 carrying the state gradient.
//
// A warp owns one trajectory for all T steps (the rollout is serial in t).  The forward keeps the packed chain in shared
// memory and evaluates it with warp_dense<1>, the arithmetic of k_ekf_loop's primal row.  The backward's products are
// W^T delta: the packed 64x64 matrices are input-major (Wt[k][o]), where lane k reading Wt[k*64 + o] would put all 32
// lanes on one bank, so each CTA stages them output-major (W[o][k]) once and lane k reads W[o*64 + k].
#include "kernels.cuh"
#include "warp_mlp.cuh"

namespace mmf {

constexpr int DYN_MAX_WARPS = 32;
constexpr int DYN_MIN_THREADS = 256;  // extra warps only help stage the weights when few trajectories share a CTA

// Float offset of 64x64 layer s (0 ... L-1, in evaluation order) inside the packed chain, and of the output layer.
__host__ __device__ __forceinline__ int dense_offset(const ChainDev& ch, int s) {
  const int base = ch.in_dim * U + U, mid_at = 2 * ch.n_pre;
  if (s < mid_at) return base + (s >> 1) * RES_FLOATS + (s & 1) * (U * U + U);
  if (s == mid_at) return base + ch.n_pre * RES_FLOATS;
  const int r = s - mid_at - 1;
  return base + ch.n_pre * RES_FLOATS + U * U + (r >> 1) * RES_FLOATS + (r & 1) * (U * U + U);
}
__host__ __device__ __forceinline__ int out_offset(const ChainDev& ch) {
  return ch.in_dim * U + U + ch.n_pre * RES_FLOATS + U * U + ch.n_post * RES_FLOATS;
}

// Element (row p, column col) of plane l of a chunk-major (L+1, 16, P, 4) tape / delta tensor.
__device__ __forceinline__ size_t plane_at(int l, int col, long long P, long long p) {
  return (((size_t)l * (U / 4) + (size_t)(col >> 2)) * (size_t)P + (size_t)p) * 4 + (size_t)(col & 3);
}

template <int SD, bool TAPE>
__global__ void __launch_bounds__(DYN_MAX_WARPS * 32, 1) k_dyn_rollout(const __grid_constant__ DynRolloutParams P, int wpc) {
  extern __shared__ __align__(16) float sm[];
  const ChainDev ch = P.ch;
  const int nf = ch.floats();
  float* wsm = sm;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  // per-warp scratch: rows A, B, residual (64 each), traj buffers (256 + 64) and the hoisted row (64)
  constexpr int WARP_FLOATS = 3 * U + 384;
  float* rowsA = sm + ((nf + 3) & ~3) + (size_t)(wid < wpc ? wid : 0) * WARP_FLOATS;
  float* rowsB = rowsA + U;
  float* rowsX = rowsB + U;
  float* tbuf = rowsX + U;
  float* rbs = tbuf + 320;
  {
    const float4* src = reinterpret_cast<const float4*>(ch.w);
    float4* dst = reinterpret_cast<float4*>(wsm);
    for (int i = tid; i < nf / 4; i += blockDim.x) dst[i] = __ldg(src + i);
    for (int i = (nf & ~3) + tid; i < nf; i += blockDim.x) wsm[i] = __ldg(ch.w + i);
  }
  __syncthreads();

  const int N = P.N, T = P.T;
  const long long rows_total = (long long)T * N;
  const int n_dense = 2 * ch.n_pre + 1 + 2 * ch.n_post;
  const int mid_at = 2 * ch.n_pre;
  for (int n = blockIdx.x * wpc + wid; n < N && wid < wpc; n += gridDim.x * wpc) {
    float x[SD];
#pragma unroll
    for (int i = 0; i < SD; ++i) x[i] = P.x0[(size_t)n * SD + i];
    for (int t = 0; t < T; ++t) {
      const long long p = (long long)t * N + n;
      const float* rb = rbs;
      if (P.rowbias != nullptr)
        rb = P.rowbias + (size_t)p * U;
      else
        warp_traj_row(P.rows, P.controls + (size_t)p * P.cd, tbuf, rbs, lane);

      const float* w = wsm;
      {
        const float* inb = w + SD * U;
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          const int j = lane + 32 * half;
          float a = inb[j];
#pragma unroll
          for (int i = 0; i < SD; ++i) a = fmaf(w[i * U + j], x[i], a);
          rowsA[j] = a > 0.0f ? a : 0.0f;
        }
        __syncwarp();
        w += SD * U + U;
      }
      float* cur = rowsA;
      float* nxt = rowsB;
      for (int s = 0; s < n_dense; ++s) {
        if constexpr (TAPE) {  // plane s = the input of layer s
          P.act_out[plane_at(s, lane, rows_total, p)] = cur[lane];
          P.act_out[plane_at(s, lane + 32, rows_total, p)] = cur[lane + 32];
        }
        const bool is_mid = (s == mid_at);
        const int rel = (s < mid_at) ? s : s - mid_at - 1;
        if (is_mid) {
          warp_dense<1>(w, rb, cur, nullptr, nxt, ch.mid_relu != 0, lane);
          w += U * U;
        } else if ((rel & 1) == 0) {
          rowsX[lane] = cur[lane];
          rowsX[lane + 32] = cur[lane + 32];
          __syncwarp();
          warp_dense<1>(w, w + U * U, cur, nullptr, nxt, true, lane);
          w += U * U + U;
        } else {
          warp_dense<1>(w, w + U * U, cur, rowsX, nxt, true, lane);
          w += U * U + U;
        }
        float* tmp = cur;
        cur = nxt;
        nxt = tmp;
      }
      if constexpr (TAPE) {  // plane L = the input of the output layer
        P.act_out[plane_at(n_dense, lane, rows_total, p)] = cur[lane];
        P.act_out[plane_at(n_dense, lane + 32, rows_total, p)] = cur[lane + 32];
      }
      float y[SD + 1];
#pragma unroll
      for (int o = 0; o < SD + 1; ++o) {
        const float w0 = w[o * U + lane], w1 = w[o * U + lane + 32];
        y[o] = warp_sum(fmaf(w0, cur[lane], w1 * cur[lane + 32])) + w[(SD + 1) * U + o];
      }
      __syncwarp();
      const float g = 1.0f / (1.0f + expf(-y[SD]));
#pragma unroll
      for (int i = 0; i < SD; ++i) x[i] = x[i] + y[i] * g;
      if (lane == 0) {
#pragma unroll
        for (int i = 0; i < SD; ++i) P.states_out[(size_t)p * SD + i] = x[i];
      }
    }
  }
}

// out_j = sum_o S[o*64 + j] d[o] for j = lane, lane + 32: W^T d with S the output-major copy of a 64x64 layer.
__device__ __forceinline__ void warp_dense_t(const float* __restrict__ S, const float* __restrict__ d, float& o0, float& o1,
                                             int lane) {
  float a0 = 0.0f, a1 = 0.0f;
#pragma unroll 4
  for (int o = 0; o < U; o += 4) {
    const float4 dv = *reinterpret_cast<const float4*>(d + o);
    a0 = fmaf(S[(o + 0) * U + lane], dv.x, a0);
    a1 = fmaf(S[(o + 0) * U + lane + 32], dv.x, a1);
    a0 = fmaf(S[(o + 1) * U + lane], dv.y, a0);
    a1 = fmaf(S[(o + 1) * U + lane + 32], dv.y, a1);
    a0 = fmaf(S[(o + 2) * U + lane], dv.z, a0);
    a1 = fmaf(S[(o + 2) * U + lane + 32], dv.z, a1);
    a0 = fmaf(S[(o + 3) * U + lane], dv.w, a0);
    a1 = fmaf(S[(o + 3) * U + lane + 32], dv.w, a1);
  }
  o0 = a0;
  o1 = a1;
}

// Reverse mode, one warp per trajectory, t = T-1 ... 0.  xb = the gradient reaching states[t] (d_states[t] plus what step
// t+1 sent back).  y is recomputed from tape plane L with the forward's arithmetic (same bits), every ReLU mask is read
// from the saved activations (layer s's output is plane s+1, the input layer's is plane 0):
//   g = sigmoid(y_sd);  yb_i = xb_i g (i < sd);  yb_sd = g (1 - g) sum_i xb_i y_i            -> d_y
//   through W_out, the resblocks and the mid layer: delta_s = mask_s o (W_{s+1}^T delta_{s+1} [+ the block's residual])
//   delta of the input layer (plane L) = mask_0 o W_0^T delta_0 (+ residual);  xb(t-1) = xb + W_in^T delta_in
// Every output element is written by exactly one lane: no atomics, bit-reproducible.
template <int SD>
__global__ void __launch_bounds__(DYN_MAX_WARPS * 32, 1) k_dyn_rollout_bwd(const __grid_constant__ DynRolloutBwdParams P,
                                                                         int wpc) {
  extern __shared__ __align__(16) float sm[];
  const ChainDev ch = P.ch;
  const int L = 2 * ch.n_pre + 1 + 2 * ch.n_post, mid_at = 2 * ch.n_pre;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  float* wt = sm;  // L x W[o][k]
  float* dbuf = sm + (size_t)L * U * U + (size_t)(wid < wpc ? wid : 0) * U;
  for (int i = tid; i < L * U * U; i += blockDim.x) {
    const int s = i / (U * U), e = i % (U * U);  // e = k * 64 + o in the packed (input-major) layer
    wt[(size_t)s * U * U + (e % U) * U + e / U] = __ldg(ch.w + dense_offset(ch, s) + e);
  }
  __syncthreads();
  const float* w_in = ch.w;                   // in_Wt[SD][64]
  const float* w_out = ch.w + out_offset(ch);  // out_W[SD+1][64], out_b[SD+1]

  const int N = P.N, T = P.T;
  const long long rows_total = (long long)T * N;
  for (int n = blockIdx.x * wpc + wid; n < N && wid < wpc; n += gridDim.x * wpc) {
    float xb[SD];
#pragma unroll
    for (int i = 0; i < SD; ++i) xb[i] = 0.0f;
    for (int t = T - 1; t >= 0; --t) {
      const long long p = (long long)t * N + n;
      // ReLU masks of every layer output (bit l = plane l > 0) for this lane's two columns, loads issued up front
      uint32_t mk0 = 0, mk1 = 0;
      for (int l = 0; l <= L; ++l) {
        mk0 |= (uint32_t)(__ldg(P.act + plane_at(l, lane, rows_total, p)) > 0.0f) << l;
        mk1 |= (uint32_t)(__ldg(P.act + plane_at(l, lane + 32, rows_total, p)) > 0.0f) << l;
      }
      const float aL0 = __ldg(P.act + plane_at(L, lane, rows_total, p));
      const float aL1 = __ldg(P.act + plane_at(L, lane + 32, rows_total, p));
      float y[SD + 1];
#pragma unroll
      for (int o = 0; o < SD + 1; ++o) {
        const float w0 = __ldg(w_out + o * U + lane), w1 = __ldg(w_out + o * U + lane + 32);
        y[o] = warp_sum(fmaf(w0, aL0, w1 * aL1)) + __ldg(w_out + (SD + 1) * U + o);
      }
      if (P.d_states != nullptr) {
#pragma unroll
        for (int i = 0; i < SD; ++i) xb[i] += P.d_states[(size_t)p * SD + i];
      }
      const float g = 1.0f / (1.0f + expf(-y[SD]));
      float yb[SD + 1], sy = 0.0f;
#pragma unroll
      for (int i = 0; i < SD; ++i) {
        yb[i] = xb[i] * g;
        sy = fmaf(xb[i], y[i], sy);
      }
      yb[SD] = g * (1.0f - g) * sy;
      if (lane == 0) {
#pragma unroll
        for (int o = 0; o < SD + 1; ++o) P.d_y_out[(size_t)p * (SD + 1) + o] = yb[o];
      }
      // gradient of the output layer's input
      float g0 = 0.0f, g1 = 0.0f;
#pragma unroll
      for (int o = 0; o < SD + 1; ++o) {
        g0 = fmaf(__ldg(w_out + o * U + lane), yb[o], g0);
        g1 = fmaf(__ldg(w_out + o * U + lane + 32), yb[o], g1);
      }
      float r0 = 0.0f, r1 = 0.0f;  // delta of the resblock's second half: it also reaches the block input directly
      for (int s = L - 1; s >= 0; --s) {
        const bool is_mid = (s == mid_at);
        const int rel = (s < mid_at) ? s : s - mid_at - 1;
        const bool first_half = !is_mid && ((rel & 1) == 0);
        float d0 = g0, d1 = g1;
        if (!is_mid || ch.mid_relu) {
          d0 = ((mk0 >> (s + 1)) & 1u) ? d0 : 0.0f;
          d1 = ((mk1 >> (s + 1)) & 1u) ? d1 : 0.0f;
        }
        P.delta_out[plane_at(s, lane, rows_total, p)] = d0;
        P.delta_out[plane_at(s, lane + 32, rows_total, p)] = d1;
        __syncwarp();  // the previous layer's product has finished reading dbuf
        dbuf[lane] = d0;
        dbuf[lane + 32] = d1;
        __syncwarp();
        warp_dense_t(wt + (size_t)s * U * U, dbuf, g0, g1, lane);
        if (first_half) {
          g0 += r0;
          g1 += r1;
        } else if (!is_mid) {
          r0 = d0;
          r1 = d1;
        }
      }
      // input layer: Linear(sd, 64) + ReLU
      const float d0 = (mk0 & 1u) ? g0 : 0.0f, d1 = (mk1 & 1u) ? g1 : 0.0f;
      P.delta_out[plane_at(L, lane, rows_total, p)] = d0;
      P.delta_out[plane_at(L, lane + 32, rows_total, p)] = d1;
#pragma unroll
      for (int i = 0; i < SD; ++i) xb[i] += warp_sum(fmaf(__ldg(w_in + i * U + lane), d0, __ldg(w_in + i * U + lane + 32) * d1));
    }
    if (lane == 0) {
#pragma unroll
      for (int i = 0; i < SD; ++i) P.d_x0_out[(size_t)n * SD + i] = xb[i];
    }
  }
}

// Few warps per CTA keep the per-step latency low; wpc is shrunk until the weights and the per-warp scratch fit.
// `configured_dev` / `window` are the caller's per-kernel cache of the shared-memory opt-in.
template <typename Kernel>
static int dyn_launch_shape(Kernel kernel, int* configured_dev, size_t* window, int N, size_t fixed_floats,
                            size_t warp_floats, int* wpc_out, int* ctas_out, int* threads_out, size_t* smem_out) {
  int dev = 0, sms = 148;
  MMF_CUDA(cudaGetDevice(&dev));
  MMF_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  if (*configured_dev != dev) {
    int rc = opt_in_shared_memory(kernel, window);
    if (rc) return rc;
    *configured_dev = dev;
  }
  int wpc = (N + sms - 1) / sms;
  wpc = wpc < 1 ? 1 : (wpc > DYN_MAX_WARPS ? DYN_MAX_WARPS : wpc);
  size_t smem = (fixed_floats + (size_t)wpc * warp_floats) * sizeof(float);
  while (smem > *window && wpc > 1) {
    --wpc;
    smem = (fixed_floats + (size_t)wpc * warp_floats) * sizeof(float);
  }
  MMF_REQUIRE(smem <= *window, "dyn_rollout: %zu B of shared memory needed (window %zu B)", smem, *window);
  int ctas = (N + wpc - 1) / wpc;
  if (ctas > sms) ctas = sms;
  *wpc_out = wpc;
  *ctas_out = ctas;
  *threads_out = wpc * 32 > DYN_MIN_THREADS ? wpc * 32 : DYN_MIN_THREADS;
  *smem_out = smem;
  return MMF_OK;
}

template <int SD, bool TAPE>
static int launch_dyn_rollout_sd(const DynRolloutParams& P, cudaStream_t stream) {
  int wpc, ctas, threads;
  size_t smem;
  static thread_local int configured_dev = -1;
  static thread_local size_t window = 0;
  int rc = dyn_launch_shape(k_dyn_rollout<SD, TAPE>, &configured_dev, &window, P.N, (size_t)((P.ch.floats() + 3) & ~3), 3 * U + 384, &wpc, &ctas,
                            &threads, &smem);
  if (rc) return rc;
  k_dyn_rollout<SD, TAPE><<<ctas, threads, smem, stream>>>(P, wpc);
  MMF_LAUNCH_CHECK("k_dyn_rollout");
  return MMF_OK;
}

int launch_dyn_rollout(const DynRolloutParams& P, cudaStream_t stream) {
  if (P.T == 0 || P.N == 0) return MMF_OK;
  const bool tape = P.act_out != nullptr;
  switch (P.ch.in_dim) {
    case 1: return tape ? launch_dyn_rollout_sd<1, true>(P, stream) : launch_dyn_rollout_sd<1, false>(P, stream);
    case 2: return tape ? launch_dyn_rollout_sd<2, true>(P, stream) : launch_dyn_rollout_sd<2, false>(P, stream);
    case 3: return tape ? launch_dyn_rollout_sd<3, true>(P, stream) : launch_dyn_rollout_sd<3, false>(P, stream);
    case 4: return tape ? launch_dyn_rollout_sd<4, true>(P, stream) : launch_dyn_rollout_sd<4, false>(P, stream);
  }
  set_error("dyn_rollout: state_dim %d unsupported (1..%d)", P.ch.in_dim, MMF_MAX_SD);
  return MMF_E_INVALID;
}

template <int SD>
static int launch_dyn_rollout_bwd_sd(const DynRolloutBwdParams& P, cudaStream_t stream) {
  const int L = 2 * P.ch.n_pre + 1 + 2 * P.ch.n_post;
  int wpc, ctas, threads;
  size_t smem;
  static thread_local int configured_dev = -1;
  static thread_local size_t window = 0;
  int rc = dyn_launch_shape(k_dyn_rollout_bwd<SD>, &configured_dev, &window, P.N, (size_t)L * U * U, U, &wpc, &ctas, &threads, &smem);
  if (rc) return rc;
  k_dyn_rollout_bwd<SD><<<ctas, threads, smem, stream>>>(P, wpc);
  MMF_LAUNCH_CHECK("k_dyn_rollout_bwd");
  return MMF_OK;
}

int launch_dyn_rollout_bwd(const DynRolloutBwdParams& P, cudaStream_t stream) {
  if (P.N == 0) return MMF_OK;
  switch (P.ch.in_dim) {
    case 1: return launch_dyn_rollout_bwd_sd<1>(P, stream);
    case 2: return launch_dyn_rollout_bwd_sd<2>(P, stream);
    case 3: return launch_dyn_rollout_bwd_sd<3>(P, stream);
    case 4: return launch_dyn_rollout_bwd_sd<4>(P, stream);
  }
  set_error("dyn_rollout_bwd: state_dim %d unsupported (1..%d)", P.ch.in_dim, MMF_MAX_SD);
  return MMF_E_INVALID;
}

}  // namespace mmf
