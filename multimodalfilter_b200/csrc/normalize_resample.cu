// normalize_resample.cu -- second half of R6 (normalise, estimate) and R7 (resample + gather).
// HBM-bound: per particle it reads logw (4 B) + state (4*sd B) [+ uniform 8 B] and writes the
// resampled state (4*sd B) + log-weight (4 B) [+ index 8 B].
//
// One CTA per trajectory; the trajectory's log-weights / CDF live in shared memory.
// Replaces A.3 `logw - logsumexp`, `sum(exp(logw) * states)`, `_resample()` (Categorical.sample
// -> torch.multinomial inverse CDF -> gather); call site ref: crossmodal/eval_helpers.py:139-142.
//
// Resampling arithmetic is PINNED (DESIGN.md): max is exact; e_j = exp_pinned(l_j - max);
//   *_STRICT: c_j = sequential fp32 running sum (what torch.multinomial does on CPU, A.6);
//   *_FAST  : segments of 8 (serial) -> groups of 32 segments (Kogge-Stone over segment totals)
//             -> serial over group totals; c_j = (G_excl[g] + S_excl[s]) + local_j;
//   idx = lower_bound over fl(c_j / c_{M-1}) compared as double with u; clamped to M-1.
#include <stdlib.h>
#include "normalize_resample.cuh"

namespace mmf {

template <bool GLOBAL_WS, int COOP>
__global__ void __launch_bounds__(COOP == 32 ? NR_WARP_TPB : NR_TPB, COOP == 32 ? NR_WARP_CTAS_PER_SM : 1) k_normalize_resample(const __grid_constant__ ResampleParams P, float* workspace) {
  extern __shared__ __align__(16) float sm[];
  __shared__ float scratch[32];
  __shared__ int cand_w[NR_TPB / 32];
  constexpr int UNITS_PER_CTA = (COOP == 32 ? NR_WARP_TPB : NR_TPB) / COOP;
  const int tid = threadIdx.x;
  const int unit = blockIdx.x * UNITS_PER_CTA + tid / COOP;
  const int units = gridDim.x * UNITS_PER_CTA;
  const size_t slice = trajectory_scratch_floats(P.M, P.alpha < 1.0f);
  float* cdf = GLOBAL_WS ? workspace + (size_t)blockIdx.x * slice : sm + (size_t)(tid / COOP) * slice;  // log-weights first, CDF later

  for (int n = unit; n < P.N; n += units) {
    coop_sync<COOP>();
    nr_trajectory<COOP>(P, n, cdf, scratch, cand_w);
  }
}

// ---- *_FAST modes, hard resampling, M <= 2048: one warp per trajectory, the CDF built in registers ------------------
// The generic kernel above spends ~470 warp instructions per particle (three exponentials per particle, CDF and search
// through shared memory) and reaches 0.2 of the HBM roofline (ncu r01).  The FAST modes are free to choose their
// arithmetic, so this kernel does the least it can per particle:
//   * ONE exponential: e_j = EXP(l_j - max l) on the UN-normalised log-weights serves the estimate
//     (sum_j e_j x_j / total), the normalisation (lse = max + log total, only materialised on request) and the CDF.
//     The logits of the FAST modes are therefore the un-normalised log-weights themselves (softmax is shift
//     invariant); `logits_out` reports exactly what the CDF was built from, so the pinned arithmetic applied to it
//     reproduces the indices bit for bit.
//   * lane L holds segments L, L + 32, ... (8 consecutive particles each) in registers: the blocked summation order
//     of the FAST definition (segments of 8 -> Kogge-Stone over the 32 segment totals of a 256-group -> serial over
//     groups) is a register / shuffle computation, the CDF touches shared memory once, on its way to the search;
//   * inverse CDF through the guide table (expected O(1) probes); the systematic positions are formed in fp32
//     ((u0 + j) * total / S) -- the key only has to be within a few ulp of the exact threshold, draws that land within
//     8 ulp of a CDF entry are re-decided with the exact fp64 predicate, so the indices are those of the definition.
template <typename ExactU>
__device__ __forceinline__ int guided_search(const float* cdf, const uint16_t* guide, int M, int K, float scale,
                                             float total, float c0, bool degenerate, ExactU exact_u) {
  int b = (int)(c0 * scale);
  b = b < 0 ? 0 : (b > K ? K : b);
  int lo = guide[b], hi = guide[b + 1];
  while (hi - lo > 4) {  // crowded bucket: bisect down to a short run first
    const int mid = lo + ((hi - lo) >> 1);
    if (cdf[mid] < c0) lo = mid + 1; else hi = mid;
  }
  while (lo < hi && cdf[lo] < c0) ++lo;
  const float band = fmaxf(c0 * 9.6e-7f, 1e-37f);  // >= 8 ulp: fp32 key (<= 3 ulp off) + distance key..c* (<= 2 ulp)
  bool near = degenerate;
  if (lo < M) near |= fabsf(cdf[lo] - c0) <= band;
  if (lo > 0) near |= fabsf(cdf[lo - 1] - c0) <= band;
  if (near) {
    const float cstar = cdf_threshold(total, exact_u());
    lo = 0;
    hi = M;
    while (lo < hi) {
      const int mid = lo + ((hi - lo) >> 1);
      if (cdf[mid] < cstar) lo = mid + 1; else hi = mid;
    }
  }
  return lo < M - 1 ? lo : M - 1;
}

constexpr int RF_TPB = 128;  // 4 trajectories per CTA
__host__ __device__ inline size_t fast_slice_floats(int NG) { return (size_t)NG * GROUP + ((size_t)NG * GROUP + 8) / 2; }

template <int NG>
__global__ void __launch_bounds__(RF_TPB, NG <= 4 ? 7 : 4) k_resample_fast(const __grid_constant__ ResampleParams P) {
  extern __shared__ __align__(16) float sm[];
  constexpr int MPAD = NG * GROUP;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  float* cdf = sm + (size_t)wid * fast_slice_floats(NG);
  uint16_t* guide = reinterpret_cast<uint16_t*>(cdf + MPAD);  // MPAD + 2 entries
  const int M = P.M, sd = P.sd, S = P.M_out;
  const bool systematic = P.mode == MMF_RESAMPLE_SYSTEMATIC_FAST;
  const float uniform_lw = -logf((float)M);
  const int K = ((M + 31) / 32) * 32;  // guide buckets (<= MPAD)

  for (int n = blockIdx.x * (RF_TPB / 32) + wid; n < P.N; n += gridDim.x * (RF_TPB / 32)) {
    const float* lw = (P.logits_in ? P.logits_in : P.logw_unnorm) + (size_t)n * M;
    // Optional (MMF_RESAMPLE_PREFETCH=1, off by default): request everything this trajectory will read later (its
    // particles for the estimate and the gather, its uniforms) from HBM now.  The grid is ONE wave of warps that all sit
    // in the same phase -- load, compute, load, compute -- so the memory system idles half of the time; measured on B200
    // at C3's shape the prefetch changes nothing (multinomial_fast 57.3 -> 61.4 us, systematic_fast 51.2 -> 51.2 us):
    // the kernel is bound by its 33 M warp instructions (issue slots 50 % busy at 7 warps per scheduler), not by the
    // exposed load latency.
    if (P.prefetch) {
      if (P.logits_in == nullptr || P.states_out != nullptr) {
        const char* xs = reinterpret_cast<const char*>(P.states + (size_t)n * M * sd);
        for (int off = lane * 128; off < M * sd * 4; off += 32 * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(xs + off));
      }
      const char* un = reinterpret_cast<const char*>(P.uniforms + (systematic ? (size_t)n : (size_t)n * S));
      for (int off = lane * 128; off < (systematic ? 8 : S * 8); off += 32 * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(un + off));
    }
    // ---- log-weights of my segments -> registers; max -----------------------------------------------------------
    float e[NG][SEG];
    const bool vec = (M & 3) == 0 && ((uintptr_t)lw & 15) == 0;
    float mx = -INFINITY;
#pragma unroll
    for (int g = 0; g < NG; ++g) {
      const int base = g * GROUP + lane * SEG;
      if (vec && base + SEG <= M) {
        const float4 a = __ldg(reinterpret_cast<const float4*>(lw + base));
        const float4 b = __ldg(reinterpret_cast<const float4*>(lw + base + 4));
        e[g][0] = a.x; e[g][1] = a.y; e[g][2] = a.z; e[g][3] = a.w;
        e[g][4] = b.x; e[g][5] = b.y; e[g][6] = b.z; e[g][7] = b.w;
      } else {
#pragma unroll
        for (int i = 0; i < SEG; ++i) e[g][i] = base + i < M ? __ldg(lw + base + i) : -INFINITY;
      }
#pragma unroll
      for (int i = 0; i < SEG; ++i) mx = fmaxf(mx, e[g][i]);
    }
    mx = warp_max(mx);
    // ---- the one exponential per particle; un-normalised weights to shared memory for the estimate ---------------
    __syncwarp();  // the previous trajectory's searches are done with cdf[]
#pragma unroll
    for (int g = 0; g < NG; ++g) {
#pragma unroll
      for (int i = 0; i < SEG; ++i) e[g][i] = exp_pinned(__fsub_rn(e[g][i], mx));
      float4* dst = reinterpret_cast<float4*>(cdf + g * GROUP + lane * SEG);
      dst[0] = make_float4(e[g][0], e[g][1], e[g][2], e[g][3]);
      dst[1] = make_float4(e[g][4], e[g][5], e[g][6], e[g][7]);
    }
    __syncwarp();
    // ---- estimate: sum_j e_j x_j (divided by the total below); the arg max waits for the total --------------------
    float acc[MMF_MAX_SD] = {0.f, 0.f, 0.f, 0.f};
    if (P.logits_in == nullptr) {
      const float* xs = P.states + (size_t)n * M * sd;
      if (P.estimation == MMF_ESTIMATE_WEIGHTED_AVERAGE) {
        if (sd == 2 && (M & 1) == 0 && ((uintptr_t)xs & 15) == 0) {
          for (int j = 2 * lane; j < M; j += 64) {  // two particles per lane per step: coalesced 16-byte loads
            const float4 x = __ldg(reinterpret_cast<const float4*>(xs + (size_t)j * 2));
            const float2 w = *reinterpret_cast<const float2*>(cdf + j);
            acc[0] = fmaf(w.x, x.x, acc[0]);
            acc[1] = fmaf(w.x, x.y, acc[1]);
            acc[0] = fmaf(w.y, x.z, acc[0]);
            acc[1] = fmaf(w.y, x.w, acc[1]);
          }
        } else {
          for (int j = lane; j < M; j += 32) {
            const float w = cdf[j];
#pragma unroll
            for (int d = 0; d < MMF_MAX_SD; ++d)
              if (d < sd) acc[d] = fmaf(w, __ldg(xs + (size_t)j * sd + d), acc[d]);
          }
        }
#pragma unroll
        for (int d = 0; d < MMF_MAX_SD; ++d) acc[d] = warp_sum(acc[d]);
      }
    }
    // ---- CDF in registers: the blocked order of the FAST definition ------------------------------------------------
    float gbase = 0.0f;  // exclusive running sum over the group totals (every lane carries it)
    float segx[NG];      // exclusive offset of my segment inside its group
#pragma unroll
    for (int g = 0; g < NG; ++g) {
      float run = 0.0f;
#pragma unroll
      for (int i = 0; i < SEG; ++i) {
        run = __fadd_rn(run, e[g][i]);
        e[g][i] = run;
      }
      float t = run;  // Kogge-Stone inclusive scan of the 32 segment totals
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const float v = __shfl_up_sync(0xffffffffu, t, d);
        if (lane >= d) t = __fadd_rn(v, t);
      }
      const float excl = __shfl_up_sync(0xffffffffu, t, 1);
      segx[g] = __fadd_rn(gbase, lane == 0 ? 0.0f : excl);
      gbase = __fadd_rn(gbase, __shfl_sync(0xffffffffu, t, 31));
    }
    __syncwarp();  // the estimate has read its weights
#pragma unroll
    for (int g = 0; g < NG; ++g) {
#pragma unroll
      for (int i = 0; i < SEG; ++i) e[g][i] = __fadd_rn(segx[g], e[g][i]);
      float4* dst = reinterpret_cast<float4*>(cdf + g * GROUP + lane * SEG);
      dst[0] = make_float4(e[g][0], e[g][1], e[g][2], e[g][3]);
      dst[1] = make_float4(e[g][4], e[g][5], e[g][6], e[g][7]);
    }
    __syncwarp();
    const float total = cdf[M - 1];
    const float scale = (float)K / total;
    const float lse = mx + logf(total);
    // ---- per-trajectory outputs ------------------------------------------------------------------------------------
    if (P.logits_in == nullptr) {
      if (P.estimation == MMF_ESTIMATE_WEIGHTED_AVERAGE) {
        if (lane < sd) {
          float v = acc[0];
#pragma unroll
          for (int d = 1; d < MMF_MAX_SD; ++d)
            if (lane == d) v = acc[d];
          P.est_out[(size_t)n * sd + lane] = __fdiv_rn(v, total);
        }
      } else {
        // first arg max of the normalised log-weights fl(l_j - lse), as every other path takes it.  Not of e_j: two
        // log-weights less than half an ulp of lse apart normalise to the same value (the first one wins), while their
        // exponentials on the un-normalised scale still differ.
        float best = -INFINITY;
        int best_i = 0x7fffffff;
        for (int j = lane; j < M; j += 32) {
          const float l = __fsub_rn(__ldg(lw + j), lse);
          if (l > best) { best = l; best_i = j; }
        }
        const float gbest = warp_max(best);
        int cand = best == gbest ? best_i : 0x7fffffff;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) cand = min(cand, __shfl_xor_sync(0xffffffffu, cand, o));
        best_i = cand == 0x7fffffff ? 0 : cand;
        if (lane < sd) P.est_out[(size_t)n * sd + lane] = P.states[((size_t)n * M + best_i) * sd + lane];
      }
    }
    if (P.logits_out || P.logw_norm_out) {  // debug / introspection only
      for (int j = lane; j < M; j += 32) {
        const float l = lw[j];
        if (P.logits_out) P.logits_out[(size_t)n * M + j] = l;
        if (P.logw_norm_out) P.logw_norm_out[(size_t)n * M + j] = __fsub_rn(l, lse);
      }
    }
    // ---- guide table: guide[b] = number of CDF entries whose bucket is < b = first entry whose bucket is >= b ----------
    // Built without data-dependent loops (a heavy particle spans hundreds of buckets: filling its range from one lane
    // serialised the warp -- a third of this kernel's instructions in the first ncu capture): every particle that opens
    // a new bucket writes ITSELF at the first bucket of its range, then a prefix maximum over the buckets forward-fills
    // the ranges (entries increase with the bucket index).
    {
      const int words = (K + 2 + 1) / 2;
      uint32_t* g32 = reinterpret_cast<uint32_t*>(guide);
      for (int w = lane; w < words; w += 32) g32[w] = 0u;
      __syncwarp();
      for (int i = lane; i < M; i += 32) {
        int fi = (int)(cdf[i] * scale);
        fi = fi < 0 ? 0 : (fi > K ? K : fi);
        int fp = -1;
        if (i > 0) {
          fp = (int)(cdf[i - 1] * scale);
          fp = fp < 0 ? 0 : (fp > K ? K : fp);
        }
        if (fi > fp) guide[fp + 1] = (uint16_t)i;  // bucket fp + 1 is opened by this particle only
      }
      if (lane == 0) {
        int fl = (int)(total * scale);
        fl = fl < 0 ? 0 : (fl > K ? K : fl);
        guide[fl + 1] = (uint16_t)M;  // buckets past the total mass (fl + 1 <= K + 1)
      }
      __syncwarp();
      const int per = (K + 2 + 31) / 32;  // consecutive buckets per lane
      const int b0 = lane * per, b1 = min(b0 + per, K + 2);
      int mx_chunk = 0;
      for (int b = b0; b < b1; ++b) mx_chunk = max(mx_chunk, (int)guide[b]);
      int incl = mx_chunk;  // inclusive prefix maximum over the lanes' chunks
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl = max(incl, v);
      }
      int run = __shfl_up_sync(0xffffffffu, incl, 1);
      if (lane == 0) run = 0;
      for (int b = b0; b < b1; ++b) {
        run = max(run, (int)guide[b]);
        guide[b] = (uint16_t)run;
      }
    }
    __syncwarp();
    // ---- inverse CDF + gather ------------------------------------------------------------------------------------
    const double u0 = systematic ? P.uniforms[n] : 0.0;
    const float u0f = (float)u0, step = __fdiv_rn(total, (float)S);
    const double* un = P.uniforms + (size_t)n * S;
    for (int base = 0; base < S; base += 32 * NB) {
      int idx[NB];
      if (systematic) {
#pragma unroll
        for (int b = 0; b < NB; ++b) {
          const int j = base + b * 32 + lane;
          const float c0 = (u0f + (float)j) * step;
          idx[b] = j < S ? guided_search(cdf, guide, M, K, scale, total, c0, !(c0 > 0.0f),
                                         [&] { return (u0 + (double)j) / (double)S; }) : 0;
        }
      } else {
        double u[NB];
#pragma unroll
        for (int b = 0; b < NB; ++b) {
          const int j = base + b * 32 + lane;
          u[b] = j < S ? un[j] : 0.5;
        }
#pragma unroll
        for (int b = 0; b < NB; ++b) {
          const float uf = (float)u[b];
          const double ub = u[b];
          idx[b] = guided_search(cdf, guide, M, K, scale, total, uf * total, !(uf > 0.0f), [&] { return ub; });
        }
      }
      if (P.states_out) {
        if (sd == 2) {
          float2 sv[NB];
#pragma unroll
          for (int b = 0; b < NB; ++b)
            sv[b] = __ldg(reinterpret_cast<const float2*>(P.states + ((size_t)n * M + idx[b]) * 2));
#pragma unroll
          for (int b = 0; b < NB; ++b) {
            const int j = base + b * 32 + lane;
            if (j < S) *reinterpret_cast<float2*>(P.states_out + ((size_t)n * S + j) * 2) = sv[b];
          }
        } else {
#pragma unroll
          for (int b = 0; b < NB; ++b) {
            const int j = base + b * 32 + lane;
            if (j < S) {
              const float* src = P.states + ((size_t)n * M + idx[b]) * sd;
              float* dst = P.states_out + ((size_t)n * S + j) * sd;
              for (int d = 0; d < sd; ++d) dst[d] = __ldg(src + d);
            }
          }
        }
      }
#pragma unroll
      for (int b = 0; b < NB; ++b) {
        const int j = base + b * 32 + lane;
        if (j < S) {
          if (P.idx_out) P.idx_out[(size_t)n * S + j] = idx[b];
          if (P.logw_out) P.logw_out[(size_t)n * S + j] = uniform_lw;
        }
      }
    }
  }
}

static bool resample_prefetch_enabled() {
  static const bool on = [] {
    const char* env = getenv("MMF_RESAMPLE_PREFETCH");
    return env != nullptr && atoi(env) != 0;
  }();
  return on;
}

template <int NG>
static int launch_resample_fast(const ResampleParams& P_in, int sms, cudaStream_t stream) {
  ResampleParams P = P_in;
  P.prefetch = resample_prefetch_enabled() ? 1 : 0;
  static thread_local int configured_dev = -1;
  static thread_local size_t window = 0;
  int dev = 0;
  MMF_CUDA(cudaGetDevice(&dev));
  if (configured_dev != dev) {
    int rc = opt_in_shared_memory(k_resample_fast<NG>, &window);
    if (rc) return rc;
    configured_dev = dev;
  }
  const size_t smem = fast_slice_floats(NG) * sizeof(float) * (RF_TPB / 32);
  int per_sm = (int)((window + 1024) / (smem + 1024));
  per_sm = per_sm < 1 ? 1 : (per_sm > 8 ? 8 : per_sm);
  long long ctas = ((long long)P.N + RF_TPB / 32 - 1) / (RF_TPB / 32);
  long long grid = (long long)sms * per_sm;
  if (grid > ctas) grid = ctas;
  k_resample_fast<NG><<<(int)grid, RF_TPB, smem, stream>>>(P);
  MMF_LAUNCH_CHECK("k_resample_fast");
  return MMF_OK;
}

constexpr int NR_WARP_MAX_M = 2048;

// MMF_RESAMPLE_FAST_KERNEL=0 (read once when the library is loaded) sends the FAST modes through the generic kernel:
// the two produce identical indices from identical logits, the switch exists for A/B timing.
static bool fast_kernel_enabled() {
  static const bool on = [] {
    const char* env = getenv("MMF_RESAMPLE_FAST_KERNEL");
    return env == nullptr || atoi(env) != 0;
  }();
  return on;
}
  // warp-per-trajectory path: 8 slices of <= ~20 KB per CTA

static size_t resample_smem_bytes(int M, bool soft) { return trajectory_scratch_floats(M, soft) * sizeof(float); }

static int resample_window(size_t* window_out) {
  static thread_local int configured_dev = -1;
  static thread_local size_t window = 0;
  int dev = 0;
  MMF_CUDA(cudaGetDevice(&dev));
  if (configured_dev != dev) {
    int rc = opt_in_shared_memory(k_normalize_resample<false, NR_TPB>, &window);
    if (rc) return rc;
    size_t w2 = 0;
    rc = opt_in_shared_memory(k_normalize_resample<false, 32>, &w2);
    if (rc) return rc;
    configured_dev = dev;
  }
  *window_out = window;
  return MMF_OK;
}

constexpr int WS_CTAS_PER_SM = 4;

// bytes of global workspace mmf_pf_normalize_resample / mmf_resample need for (N, M): 0 when a trajectory
// fits shared memory, else one scratch slice per resident CTA
size_t resample_workspace_bytes(int N, int M) {
  size_t window = 0;
  if (resample_window(&window) != MMF_OK) window = 200 * 1024;
  const size_t big = resample_big_applies(N, M, false) ? resample_big_workspace_bytes(N, M) : 0;  // multi-pass path (resample_big.cu)
  if (resample_smem_bytes(M, true) <= window) return big;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  long long grid = (long long)sms * WS_CTAS_PER_SM;
  if (grid > N) grid = N;
  const size_t per_cta = (size_t)grid * trajectory_scratch_floats(M, true) * sizeof(float);  // (soft resampling stays there)
  return per_cta > big ? per_cta : big;
}

int launch_normalize_resample(const ResampleParams& P, void* workspace, cudaStream_t stream) {
  const bool soft = P.alpha < 1.0f;
  const bool fast_mode = P.mode == MMF_RESAMPLE_MULTINOMIAL_FAST || P.mode == MMF_RESAMPLE_SYSTEMATIC_FAST;
  if (fast_mode && !soft && P.M <= NR_WARP_MAX_M && fast_kernel_enabled()) {
    int dev = 0, sms = 148;
    MMF_CUDA(cudaGetDevice(&dev));
    MMF_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    if (P.M <= 256) return launch_resample_fast<1>(P, sms, stream);
    if (P.M <= 512) return launch_resample_fast<2>(P, sms, stream);
    if (P.M <= 1024) return launch_resample_fast<4>(P, sms, stream);
    return launch_resample_fast<8>(P, sms, stream);
  }
  if (resample_big_applies(P.N, P.M, soft)) return launch_resample_big(P, workspace, stream);  // long trajectories: multi-pass
  const size_t smem = resample_smem_bytes(P.M, soft);
  size_t window = 0;
  int rc = resample_window(&window);
  if (rc) return rc;
  int dev = 0, sms = 148;
  MMF_CUDA(cudaGetDevice(&dev));
  MMF_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  if (smem > window) {
    MMF_REQUIRE(workspace != nullptr,
                "normalize_resample: M=%d does not fit shared memory; pass a workspace of mmf_pf_resample_workspace_bytes() bytes",
                P.M);
    long long grid = (long long)sms * WS_CTAS_PER_SM;
    if (grid > P.N) grid = P.N;
    k_normalize_resample<true, NR_TPB><<<(int)grid, NR_TPB, 0, stream>>>(P, static_cast<float*>(workspace));
    MMF_LAUNCH_CHECK("k_normalize_resample<global>");
    return MMF_OK;
  }
  if (P.M <= NR_WARP_MAX_M && P.M_out <= 4 * NR_WARP_MAX_M) {
    // warp per trajectory, 4 trajectories per CTA; the kernel is bound by the latency of one warp walking its
    // trajectory, so what matters is that all trajectories are resident at once (no second, half-empty wave)
    constexpr int per_cta = NR_WARP_TPB / 32;
    const size_t smem4 = smem * per_cta;
    int per_sm = (int)((200 * 1024) / (smem4 + 1024));
    per_sm = per_sm < 1 ? 1 : (per_sm > NR_WARP_CTAS_PER_SM ? NR_WARP_CTAS_PER_SM : per_sm);
    long long ctas = ((long long)P.N + per_cta - 1) / per_cta;
    long long grid = (long long)sms * per_sm;
    if (grid > ctas) grid = ctas;
    k_normalize_resample<false, 32><<<(int)grid, NR_WARP_TPB, smem4, stream>>>(P, nullptr);
    MMF_LAUNCH_CHECK("k_normalize_resample<warp>");
    return MMF_OK;
  }
  // enough CTAs per SM to hide the serial CDF chain of one trajectory behind the others
  int per_sm = (int)((200 * 1024) / (smem + 1024));
  per_sm = per_sm < 1 ? 1 : (per_sm > 8 ? 8 : per_sm);
  long long grid = (long long)sms * per_sm;
  if (grid > P.N) grid = P.N;
  k_normalize_resample<false, NR_TPB><<<(int)grid, NR_TPB, smem, stream>>>(P, nullptr);
  MMF_LAUNCH_CHECK("k_normalize_resample");
  return MMF_OK;
}

// ---- mmf_fuse_loglik: (N,M,K) x (N,K) -> (N,M), torch.logsumexp semantics ------------------------
__global__ void k_fuse_loglik(int N, int M, int K, const float* __restrict__ ll, const float* __restrict__ w,
                              float* __restrict__ out) {
  const long long total = (long long)N * M;
  for (long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x; p < total;
       p += (long long)gridDim.x * blockDim.x) {
    const int n = (int)(p / M);
    float mx = -INFINITY;
    for (int k = 0; k < K; ++k) mx = fmaxf(mx, ll[p * K + k] + (w ? w[(size_t)n * K + k] : 0.0f));
    const float shift = (mx == -INFINITY || mx == INFINITY) ? 0.0f : mx;
    float s = 0.0f;
    for (int k = 0; k < K; ++k) s += expf(ll[p * K + k] + (w ? w[(size_t)n * K + k] : 0.0f) - shift);
    out[p] = shift + logf(s);
  }
}

int launch_fuse_loglik(int N, int M, int K, const float* ll, const float* w, float* out, cudaStream_t stream) {
  const long long total = (long long)N * M;
  if (total == 0) return MMF_OK;
  long long blocks = (total + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  k_fuse_loglik<<<(int)blocks, 256, 0, stream>>>(N, M, K, ll, w, out);
  MMF_LAUNCH_CHECK("k_fuse_loglik");
  return MMF_OK;
}

// ---- mmf_pf_init (R2) ------------------------------------------------------------------------------------
__global__ void k_pf_init(int N, int M, int sd, const float* __restrict__ mean, const float* __restrict__ cov,
                          const float* __restrict__ eps, float* __restrict__ states, float* __restrict__ logw) {
  const long long total = (long long)N * M;
  const float lw = -logf((float)M);
  for (long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x; p < total;
       p += (long long)gridDim.x * blockDim.x) {
    const int n = (int)(p / M), m = (int)(p % M);
    // Cholesky of the small sd x sd covariance (lower factor), recomputed per thread (sd <= 4)
    float L[MMF_MAX_SD][MMF_MAX_SD];
    const float* C = cov + (size_t)n * sd * sd;
    for (int i = 0; i < sd; ++i) {
      for (int j = 0; j <= i; ++j) {
        float s = C[i * sd + j];
        for (int k = 0; k < j; ++k) s -= L[i][k] * L[j][k];
        L[i][j] = (i == j) ? sqrtf(s) : s / L[j][j];
      }
    }
    const float* e = eps + ((size_t)m * N + n) * sd;
    for (int i = 0; i < sd; ++i) {
      float v = 0.0f;
      for (int j = 0; j <= i; ++j) v = fmaf(L[i][j], e[j], v);
      states[p * sd + i] = mean[(size_t)n * sd + i] + v;
    }
    logw[p] = lw;
  }
}

int launch_pf_init(int N, int M, int sd, const float* mean, const float* cov, const float* eps, float* states,
                   float* logw, cudaStream_t stream) {
  const long long total = (long long)N * M;
  if (total == 0) return MMF_OK;
  long long blocks = (total + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  k_pf_init<<<(int)blocks, 256, 0, stream>>>(N, M, sd, mean, cov, eps, states, logw);
  MMF_LAUNCH_CHECK("k_pf_init");
  return MMF_OK;
}

}  // namespace mmf
