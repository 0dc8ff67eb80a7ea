// row_mlp.cu -- the per-trajectory MLPs of the path as ONE kernel per module (SURVEY.md section 8f rank 1; R9):
// position / sensor observation encoders (ref: crossmodal/push_models/layers.py:107-136), the particle-filter and
// Kalman-filter crossmodal weight models (ref: crossmodal/push_models/crossmodal_pf.py:72-104,
// crossmodal/door_models/crossmodal_kf.py:134-167) and the virtual-sensor head (ref: crossmodal/door_models/kf.py:81-126).
//
// These are stacks of Linear / ReLU / Sigmoid / residual blocks, 3 ... 192 inputs wide, evaluated once per (step,
// trajectory) row: 10-90 k MAC per row, all weights L2 resident.  As torch modules each stack is 10-40 library
// launches (cuBLAS SIMT sgemm + ATen elementwise) per call; here the host compiles a stack into a short program of
// fused ops   dst = act(W src + b [+ residual])   over per-row scratch slots and one launch runs the whole program:
// a warp owns R = 8 rows, lane j computes output features j, j + 32, ... for its rows (weights are read once per 8 rows,
// coalesced, through L1; the rows' activations sit row-minor in shared memory, S[slot][row], so the 8 rows' value of
// one input is two broadcast LDS.128: 4 loads per 16 FFMA), fp32 FFMA in the reference's summation order over the
// inputs -- so the results are torch's to rounding (parity tests: 2e-5).  First version (4 rows per warp, row-major
// scratch: 6 loads per 8 FFMA): 0.57 ms per 16,384 rows of the virtual-sensor program (ncu launch list of C2).
//
// Training (include/mmf_b200.h, mmf_row_mlp_train_fwd / _bwd / _weight_grads): k_row_mlp_train is the same program
// with every op's input and output copied to a tape; k_row_mlp_bwd walks a host-compiled reverse program with the same
// tile loop (rm_op) fed the torch-layout (out, in) weights, so   delta_src (+)= W^T g   is the forward product of the
// transposed matrix; k_row_mlp_dw / k_row_mlp_dw_sum reduce dW = sum_rows g x^T and db = sum_rows g over fixed row
// ranges and then in a fixed order (no floating-point atomics: bit-reproducible).
#include "kernels.cuh"

namespace mmf {

constexpr int RM_ROWS = 8;       // rows per warp
constexpr int RM_WARPS = 16;     // most warps per CTA (fewer when the program's scratch is large)
constexpr int RM_MAX_OUT = 256;  // widest layer output
constexpr int RM_MAX_TILES = MMF_MLP_MAX_DW_TILES;  // 64 x 64 tiles of all dW matrices of one program (k_row_mlp_dw)

struct RowMlpParams {
  mmf_mlp_op ops[MMF_MLP_MAX_OPS];
  int n_ops, n_inputs, n_outputs, scratch;
  long long rows;
  const float* weights;
  const float* inputs[MMF_MLP_MAX_IO];
  int in_dims[MMF_MLP_MAX_IO], in_slots[MMF_MLP_MAX_IO];
  float* outputs[MMF_MLP_MAX_IO];
  int out_dims[MMF_MLP_MAX_IO], out_slots[MMF_MLP_MAX_IO];
  float* tape;     // k_row_mlp_train only
  int tape_floats;  // per row: sum over ops of in_dim + out_dim
};

constexpr int RM_KC = 64;                      // input rows of a staged weight tile
constexpr int RM_TILE = RM_KC * 64;            // floats of a weight tile: RM_KC inputs x 64 output features

__device__ __forceinline__ void rm_cp_async4(float* dst, const float* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src) : "memory");
}

// Weight tile (k0 .. k0 + RM_KC) x (j0 .. j0 + 64) of an op -> shared memory, by all threads of the CTA.
__device__ __forceinline__ void rm_stage(float* buf, const float* Wt, int in_dim, int out_dim, int k0, int j0) {
  const int cols = min(64, out_dim - j0), rows = min(RM_KC, in_dim - k0);
  for (int e = threadIdx.x; e < rows * 64; e += blockDim.x) {
    const int kk = e >> 6, c = e & 63;
    if (c < cols) rm_cp_async4(buf + e, Wt + (size_t)(k0 + kk) * out_dim + j0 + c);
  }
  asm volatile("cp.async.commit_group;" ::: "memory");
}

// One op over the warp's 8 rows:  S[dst] = act(Wt^T S[src] + b [+ S[res]])  with Wt = [in_dim][out_dim] input-major and
// b = NULL meaning zero.  The CTA's warps run it in lock step (CTA-uniform arguments: barriers inside): a weight tile is
// fetched from L2 ONCE per CTA (cp.async, double buffered) and read by every warp from shared memory.  (First version:
// every warp streamed the program's ~300 KB of weights through L1 for its own 4 rows -- 1.4 GB of L2 traffic per
// launch, 0.57 ms per 16,384 rows.)  res may equal dst (accumulation: a lane reads a feature before it writes it);
// dst must not overlap src.
__device__ __forceinline__ void rm_op(float* S, float* wbuf, const float* Wt, const float* b, int in_dim, int out_dim,
                                      int src, int dst, int res, int act, int lane) {
  const int kchunks = (in_dim + RM_KC - 1) / RM_KC;
  const int tiles = ((out_dim + 63) / 64) * kchunks;
  __syncthreads();  // every warp is done with the previous op's last tile
  rm_stage(wbuf, Wt, in_dim, out_dim, 0, 0);
  float acc_a[RM_ROWS], acc_b[RM_ROWS];
  for (int t = 0; t < tiles; ++t) {
    const int j0 = (t / kchunks) * 64, k0 = (t % kchunks) * RM_KC;
    if (t + 1 < tiles) {
      rm_stage(wbuf + ((t + 1) & 1) * RM_TILE, Wt, in_dim, out_dim, ((t + 1) % kchunks) * RM_KC, ((t + 1) / kchunks) * 64);
      asm volatile("cp.async.wait_group 1;" ::: "memory");
    } else {
      asm volatile("cp.async.wait_group 0;" ::: "memory");
    }
    __syncthreads();  // tile t has landed for everybody
    const float* w = wbuf + (t & 1) * RM_TILE;
    const int ja = j0 + lane, jb = j0 + 32 + lane;
    const bool va = ja < out_dim, vb = jb < out_dim;
    if (k0 == 0) {
      const float ba = va && b ? __ldg(b + ja) : 0.0f, bb = vb && b ? __ldg(b + jb) : 0.0f;
#pragma unroll
      for (int r = 0; r < RM_ROWS; ++r) {
        acc_a[r] = ba;
        acc_b[r] = bb;
      }
    }
    const float4* src4 = reinterpret_cast<const float4*>(S + (size_t)(src + k0) * RM_ROWS);
    const int kn = min(RM_KC, in_dim - k0);
#pragma unroll 4
    for (int k = 0; k < kn; ++k) {
      const float wa = va ? w[k * 64 + lane] : 0.0f;
      const float wb = vb ? w[k * 64 + 32 + lane] : 0.0f;
      const float4 x0 = src4[2 * k], x1 = src4[2 * k + 1];  // the 8 rows' input k: two broadcast loads
      const float x[RM_ROWS] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
#pragma unroll
      for (int r = 0; r < RM_ROWS; ++r) {
        acc_a[r] = fmaf(wa, x[r], acc_a[r]);
        acc_b[r] = fmaf(wb, x[r], acc_b[r]);
      }
    }
    if (k0 + RM_KC >= in_dim) {
      // residual, activation, store: the 8 rows of a feature are 32 contiguous bytes -> vector accesses, conflict-free
      float4* dst_a = reinterpret_cast<float4*>(S + (size_t)(dst + ja) * RM_ROWS);
      float4* dst_b = reinterpret_cast<float4*>(S + (size_t)(dst + jb) * RM_ROWS);
      if (res >= 0) {
        if (va) {
          const float4* r4 = reinterpret_cast<const float4*>(S + (size_t)(res + ja) * RM_ROWS);
          const float4 r0 = r4[0], r1 = r4[1];
          acc_a[0] += r0.x; acc_a[1] += r0.y; acc_a[2] += r0.z; acc_a[3] += r0.w;
          acc_a[4] += r1.x; acc_a[5] += r1.y; acc_a[6] += r1.z; acc_a[7] += r1.w;
        }
        if (vb) {
          const float4* r4 = reinterpret_cast<const float4*>(S + (size_t)(res + jb) * RM_ROWS);
          const float4 r0 = r4[0], r1 = r4[1];
          acc_b[0] += r0.x; acc_b[1] += r0.y; acc_b[2] += r0.z; acc_b[3] += r0.w;
          acc_b[4] += r1.x; acc_b[5] += r1.y; acc_b[6] += r1.z; acc_b[7] += r1.w;
        }
      }
#pragma unroll
      for (int r = 0; r < RM_ROWS; ++r) {
        if (act == MMF_MLP_RELU) {
          acc_a[r] = fmaxf(acc_a[r], 0.0f);
          acc_b[r] = fmaxf(acc_b[r], 0.0f);
        } else if (act == MMF_MLP_SIGMOID) {
          acc_a[r] = 1.0f / (1.0f + expf(-acc_a[r]));
          acc_b[r] = 1.0f / (1.0f + expf(-acc_b[r]));
        }
      }
      if (va) {
        dst_a[0] = make_float4(acc_a[0], acc_a[1], acc_a[2], acc_a[3]);
        dst_a[1] = make_float4(acc_a[4], acc_a[5], acc_a[6], acc_a[7]);
      }
      if (vb) {
        dst_b[0] = make_float4(acc_b[0], acc_b[1], acc_b[2], acc_b[3]);
        dst_b[1] = make_float4(acc_b[4], acc_b[5], acc_b[6], acc_b[7]);
      }
    }
    __syncthreads();  // tile t's buffer may be refilled (tile t + 2)
  }
}

// The warp's 8 rows of `dim` features at slot `slot` -> tape 8-row block (both are feature-major over 8 rows: a straight
// copy of dim * 32 contiguous bytes).
__device__ __forceinline__ void rm_to_tape(float* tape, const float* S, int slot, int dim, int lane) {
  float4* t4 = reinterpret_cast<float4*>(tape);
  const float4* s4 = reinterpret_cast<const float4*>(S + (size_t)slot * RM_ROWS);
  for (int e = lane; e < 2 * dim; e += 32) t4[e] = s4[e];
}

// The forward program; TAPE: also every op's input and output -> P.tape (layout: include/mmf_b200.h).
template <bool TAPE>
__device__ __forceinline__ void rm_forward(const RowMlpParams& P) {
  extern __shared__ __align__(16) float sm[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, warps = blockDim.x >> 5;
  float* wbuf = sm;                                                        // [2][RM_TILE]
  float* S = sm + 2 * RM_TILE + (size_t)warp * RM_ROWS * P.scratch;        // S[slot * RM_ROWS + r]: a slot's rows are contiguous
  const long long cta_rows = (long long)warps * RM_ROWS;
  const long long passes = (P.rows + cta_rows - 1) / cta_rows;
  for (long long pass = blockIdx.x; pass < passes; pass += gridDim.x) {  // CTA-uniform trip count (barriers inside)
    const long long row0 = pass * cta_rows + (long long)warp * RM_ROWS;
    __syncwarp();
    // ---- inputs -> scratch (rows past the end read row P.rows - 1: computed, never written) -------------------------
    for (int i = 0; i < P.n_inputs; ++i) {
      const int d = P.in_dims[i];
      for (int e = lane; e < RM_ROWS * d; e += 32) {
        const int r = e / d, k = e - r * d;
        long long row = row0 + r;
        row = row < P.rows ? row : P.rows - 1;
        S[(P.in_slots[i] + k) * RM_ROWS + r] = __ldg(P.inputs[i] + row * d + k);
      }
    }
    __syncwarp();
    // ---- the program -------------------------------------------------------------------------------------------------
    float* tape = TAPE ? P.tape + (size_t)(row0 / RM_ROWS) * P.tape_floats * RM_ROWS : nullptr;
    for (int o = 0; o < P.n_ops; ++o) {
      const mmf_mlp_op op = P.ops[o];
      const float* Wt = P.weights + op.w_off;              // [in_dim][out_dim], input-major
      const float* b = Wt + (size_t)op.in_dim * op.out_dim;  // [out_dim]
      rm_op(S, wbuf, Wt, b, op.in_dim, op.out_dim, op.src, op.dst, op.res, op.act, lane);
      if (TAPE) {  // rm_op ends with a barrier: the op's output is in S
        if (row0 < P.rows) {
          rm_to_tape(tape, S, op.src, op.in_dim, lane);
          rm_to_tape(tape + (size_t)op.in_dim * RM_ROWS, S, op.dst, op.out_dim, lane);
        }
        tape += (size_t)(op.in_dim + op.out_dim) * RM_ROWS;
      }
    }
    __syncwarp();
    // ---- outputs -----------------------------------------------------------------------------------------------------
    for (int i = 0; i < P.n_outputs; ++i) {
      const int d = P.out_dims[i];
      for (int e = lane; e < RM_ROWS * d; e += 32) {
        const int r = e / d, k = e - r * d;
        if (row0 + r < P.rows) P.outputs[i][(row0 + r) * d + k] = S[(P.out_slots[i] + k) * RM_ROWS + r];
      }
    }
  }
}

__global__ void __launch_bounds__(RM_WARPS * 32) k_row_mlp(const __grid_constant__ RowMlpParams P) { rm_forward<false>(P); }

__global__ void __launch_bounds__(RM_WARPS * 32) k_row_mlp_train(const __grid_constant__ RowMlpParams P) {
  rm_forward<true>(P);
}

// ---- reverse program ---------------------------------------------------------------------------------------------------
struct RowMlpBwdParams {
  mmf_mlp_op ops[MMF_MLP_MAX_OPS];
  mmf_mlp_bwd_op bops[MMF_MLP_MAX_OPS];
  int tape_dst[MMF_MLP_MAX_OPS], goff[MMF_MLP_MAX_OPS];  // per forward op: tape offset of its output, delta-plane offset
  int n_bops, n_outputs, n_dinputs, scratch, tape_floats, delta_floats;
  long long rows;
  const float* weights_t;
  const float* tape;
  float* delta;
  const float* d_outputs[MMF_MLP_MAX_IO];
  int out_dims[MMF_MLP_MAX_IO], dout_slots[MMF_MLP_MAX_IO];
  float* d_inputs[MMF_MLP_MAX_IO];
  int din_dims[MMF_MLP_MAX_IO], din_slots[MMF_MLP_MAX_IO];
};

__global__ void __launch_bounds__(RM_WARPS * 32, 1) k_row_mlp_bwd(const __grid_constant__ RowMlpBwdParams P) {
  extern __shared__ __align__(16) float sm[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, warps = blockDim.x >> 5;
  float* wbuf = sm;
  float* D = sm + 2 * RM_TILE + (size_t)warp * RM_ROWS * P.scratch;  // delta slots, same layout as the forward scratch
  float4* D4 = reinterpret_cast<float4*>(D);
  const long long cta_rows = (long long)warps * RM_ROWS;
  const long long passes = (P.rows + cta_rows - 1) / cta_rows;
  for (long long pass = blockIdx.x; pass < passes; pass += gridDim.x) {
    const long long row0 = pass * cta_rows + (long long)warp * RM_ROWS;
    const bool live = row0 < P.rows;  // a warp past the end only keeps the CTA's barriers company
    __syncwarp();
    // ---- d outputs -> delta slots (rows past the end: zero, so that they add nothing to dW / db) ----------------------
    for (int i = 0; i < P.n_outputs; ++i) {
      const int d = P.out_dims[i];
      for (int e = lane; e < RM_ROWS * d; e += 32) {
        const int r = e / d, k = e - r * d;
        const long long row = row0 + r;
        D[(P.dout_slots[i] + k) * RM_ROWS + r] = row < P.rows ? __ldg(P.d_outputs[i] + row * d + k) : 0.0f;
      }
    }
    __syncwarp();
    const size_t grp = live ? (size_t)(row0 / RM_ROWS) : 0;
    const float4* tape4 = reinterpret_cast<const float4*>(P.tape + grp * P.tape_floats * RM_ROWS);
    float4* delta4 = reinterpret_cast<float4*>(P.delta + grp * P.delta_floats * RM_ROWS);
    for (int q = 0; q < P.n_bops; ++q) {
      const mmf_mlp_bwd_op bo = P.bops[q];
      const mmf_mlp_op op = P.ops[bo.op];
      // g = delta_dst * act'(y), y = the op's output from the tape; g -> the delta planes; delta_res (+)= g
      if (live) {
        const float4* y4 = tape4 + (size_t)P.tape_dst[bo.op] * 2;
        float4* p4 = delta4 + (size_t)P.goff[bo.op] * 2;
        for (int e = lane; e < 2 * op.out_dim; e += 32) {
          float4 g = D4[bo.g * 2 + e];
          if (op.act != MMF_MLP_NONE) {
            const float4 y = y4[e];
            if (op.act == MMF_MLP_RELU) {
              g.x = y.x > 0.0f ? g.x : 0.0f; g.y = y.y > 0.0f ? g.y : 0.0f;
              g.z = y.z > 0.0f ? g.z : 0.0f; g.w = y.w > 0.0f ? g.w : 0.0f;
            } else {
              g.x *= y.x * (1.0f - y.x); g.y *= y.y * (1.0f - y.y);
              g.z *= y.z * (1.0f - y.z); g.w *= y.w * (1.0f - y.w);
            }
          }
          D4[bo.g * 2 + e] = g;
          p4[e] = g;
          if (bo.dres >= 0) {
            float4 r = g;
            if (bo.flags & MMF_MLP_DRES_ACC) {
              const float4 old = D4[bo.dres * 2 + e];
              r = make_float4(old.x + g.x, old.y + g.y, old.z + g.z, old.w + g.w);
            }
            D4[bo.dres * 2 + e] = r;
          }
        }
      }
      __syncwarp();
      // delta_src (+)= W^T g: the forward tile loop over W in torch layout (out_dim, in_dim) = input-major for the transpose
      if (bo.dsrc >= 0)
        rm_op(D, wbuf, P.weights_t + op.w_off, nullptr, op.out_dim, op.in_dim, bo.g, bo.dsrc,
              (bo.flags & MMF_MLP_DSRC_ACC) ? bo.dsrc : -1, MMF_MLP_NONE, lane);
      __syncwarp();
    }
    // ---- delta slots -> d inputs ----------------------------------------------------------------------------------------
    for (int i = 0; i < P.n_dinputs; ++i) {
      const int d = P.din_dims[i];
      for (int e = lane; e < RM_ROWS * d; e += 32) {
        const int r = e / d, k = e - r * d;
        if (row0 + r < P.rows) P.d_inputs[i][(row0 + r) * d + k] = D[(P.din_slots[i] + k) * RM_ROWS + r];
      }
    }
  }
}

// ---- weight gradients ----------------------------------------------------------------------------------------------------
// CTA (tile, chunk): the 64 x 64 block (j0.., k0..) of dW of one op over the row groups of one chunk, 32 rows at a time
// from the tape (x) and the delta planes (g), 16 outputs per thread; the k0 == 0 tiles also sum db.  Partials ->
// workspace[chunk][pack index]; k_row_mlp_dw_sum adds the chunks in order (compensated, like the per-group sums).
struct RmTile {
  int op, j0, k0, reserved;
};

struct RowMlpDwParams {
  mmf_mlp_op ops[MMF_MLP_MAX_OPS];
  int tape_src[MMF_MLP_MAX_OPS], goff[MMF_MLP_MAX_OPS];
  RmTile tiles[RM_MAX_TILES];
  int tape_floats, delta_floats, groups_per_chunk;
  long long groups, pack_floats;
  const float* tape;
  const float* delta;
  float* workspace;
};

// s + c += x with the running compensation c (Kahan); __fadd_rn / __fsub_rn keep the compiler from contracting it away
__device__ __forceinline__ void kahan_add(float& s, float& c, float x) {
  const float y = __fsub_rn(x, c);
  const float t = __fadd_rn(s, y);
  c = __fsub_rn(__fsub_rn(t, s), y);
  s = t;
}

constexpr int RM_DW_ROWS = 32;
constexpr int RM_DW_LD = 68;  // padded row of the staged blocks: conflict-free transposing stores

__global__ void __launch_bounds__(256) k_row_mlp_dw(const __grid_constant__ RowMlpDwParams P) {
  __shared__ __align__(16) float Gs[RM_DW_ROWS * RM_DW_LD], Xs[RM_DW_ROWS * RM_DW_LD];
  const RmTile tl = P.tiles[blockIdx.x];
  const mmf_mlp_op op = P.ops[tl.op];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int jn = min(64, op.out_dim - tl.j0), kn = min(64, op.in_dim - tl.k0);
  const long long g_lo = (long long)blockIdx.y * P.groups_per_chunk;
  const long long g_hi = min(P.groups, g_lo + P.groups_per_chunk);
  // sums of 8 rows (one group) are added to the chunk's running sums with compensation (Kahan): the error of a gradient
  // stays that of an 8-term sum, whatever the chunk length
  float acc[4][4] = {}, cmp[4][4] = {}, dbs[4] = {}, dbc[4] = {};
  const bool sum_b = tl.k0 == 0 && tx == 0;
  for (long long g0 = g_lo; g0 < g_hi; g0 += RM_DW_ROWS / RM_ROWS) {
    for (int e = threadIdx.x; e < RM_DW_ROWS * 64; e += 256) {  // 4 groups x 64 features x 8 rows
      const int q = e >> 9, f = (e >> 3) & 63, r = e & 7;
      const long long grp = g0 + q;
      float gv = 0.0f, xv = 0.0f;
      if (grp < g_hi) {
        if (f < jn) gv = __ldg(P.delta + ((size_t)grp * P.delta_floats + P.goff[tl.op] + tl.j0 + f) * RM_ROWS + r);
        if (f < kn) xv = __ldg(P.tape + ((size_t)grp * P.tape_floats + P.tape_src[tl.op] + tl.k0 + f) * RM_ROWS + r);
      }
      Gs[(q * RM_ROWS + r) * RM_DW_LD + f] = gv;
      Xs[(q * RM_ROWS + r) * RM_DW_LD + f] = xv;
    }
    __syncthreads();
#pragma unroll 1
    for (int q = 0; q < RM_DW_ROWS / RM_ROWS; ++q) {
      float blk[4][4] = {}, bb[4] = {};
#pragma unroll
      for (int r = q * RM_ROWS; r < (q + 1) * RM_ROWS; ++r) {
        float gj[4], xk[4];
#pragma unroll
        for (int a = 0; a < 4; ++a) {
          gj[a] = Gs[r * RM_DW_LD + ty + 16 * a];
          xk[a] = Xs[r * RM_DW_LD + tx + 16 * a];
        }
#pragma unroll
        for (int a = 0; a < 4; ++a) {
#pragma unroll
          for (int c = 0; c < 4; ++c) blk[a][c] = fmaf(gj[a], xk[c], blk[a][c]);
          bb[a] += gj[a];
        }
      }
#pragma unroll
      for (int a = 0; a < 4; ++a) {
#pragma unroll
        for (int c = 0; c < 4; ++c) kahan_add(acc[a][c], cmp[a][c], blk[a][c]);
        if (sum_b) kahan_add(dbs[a], dbc[a], bb[a]);
      }
    }
    __syncthreads();
  }
  float* out = P.workspace + (size_t)blockIdx.y * P.pack_floats + op.w_off;  // torch layout: W (out, in), then b
#pragma unroll
  for (int a = 0; a < 4; ++a) {
    const int j = ty + 16 * a;
    if (j >= jn) continue;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int k = tx + 16 * c;
      if (k < kn) out[(size_t)(tl.j0 + j) * op.in_dim + tl.k0 + k] = acc[a][c];
    }
    if (sum_b) out[(size_t)op.out_dim * op.in_dim + tl.j0 + j] = dbs[a];
  }
}

__global__ void __launch_bounds__(256) k_row_mlp_dw_sum(const float* __restrict__ ws, long long pack_floats, int chunks,
                                                        float* __restrict__ grads) {
  for (long long p = blockIdx.x * 256ll + threadIdx.x; p < pack_floats; p += (long long)gridDim.x * 256) {
    float s = 0.0f, comp = 0.0f;
    for (int c = 0; c < chunks; ++c) kahan_add(s, comp, ws[(size_t)c * pack_floats + p]);
    grads[p] = s;
  }
}

// ---- host side -------------------------------------------------------------------------------------------------------------
static int validate_program(const mmf_mlp_op* ops, int n_ops, int scratch, const char* what) {
  MMF_REQUIRE(n_ops >= 1 && n_ops <= MMF_MLP_MAX_OPS, "%s: %d ops outside 1..%d", what, n_ops, MMF_MLP_MAX_OPS);
  MMF_REQUIRE(scratch >= 1 && scratch <= 1536, "%s: scratch of %d floats per row outside 1..1536", what, scratch);
  MMF_REQUIRE(ops != nullptr, "%s: NULL program", what);
  auto inside = [&](int slot, int dim) { return slot >= 0 && dim >= 1 && slot + dim <= scratch; };
  for (int o = 0; o < n_ops; ++o) {
    const mmf_mlp_op& op = ops[o];
    MMF_REQUIRE(op.in_dim >= 1 && op.out_dim >= 1 && op.out_dim <= RM_MAX_OUT && op.w_off >= 0,
                "%s: op %d has bad dimensions (%d -> %d)", what, o, op.in_dim, op.out_dim);
    MMF_REQUIRE(inside(op.src, op.in_dim) && inside(op.dst, op.out_dim) && (op.res < 0 || inside(op.res, op.out_dim)),
                "%s: op %d addresses scratch outside [0, %d)", what, o, scratch);
    MMF_REQUIRE(op.dst + op.out_dim <= op.src || op.src + op.in_dim <= op.dst, "%s: op %d: dst overlaps src", what, o);
    MMF_REQUIRE(op.res < 0 || op.dst + op.out_dim <= op.res || op.res + op.out_dim <= op.dst,
                "%s: op %d: dst overlaps the residual", what, o);
    MMF_REQUIRE(op.act >= MMF_MLP_NONE && op.act <= MMF_MLP_SIGMOID, "%s: op %d: unknown activation %d", what, o, op.act);
  }
  return MMF_OK;
}

// Warps per CTA from the shared-memory budget and the grid: the per-row scratch lives in shared memory, which therefore
// decides how many warps an SM holds: take the better of one CTA per SM (whole window) and two CTAs per SM (half of it
// each); every CTA carries its own two weight tiles.
template <typename Kernel>
static int rm_geometry(Kernel kernel, int& configured_dev, size_t& window, long long rows, int scratch, const char* what,
                       int* warps_out, long long* grid_out, size_t* smem_out) {
  const size_t wtiles = 2 * (size_t)RM_TILE * sizeof(float);
  const size_t per_warp = (size_t)RM_ROWS * scratch * sizeof(float);
  int dev = 0, sms = 148;
  MMF_CUDA(cudaGetDevice(&dev));
  if (configured_dev != dev) {
    int rc = opt_in_shared_memory(kernel, &window);
    if (rc) return rc;
    configured_dev = dev;
  }
  auto fit = [&](size_t budget) {
    const long long w = budget > wtiles + 1024 ? (long long)((budget - wtiles - 1024) / per_warp) : 0;
    return (int)(w > RM_WARPS ? RM_WARPS : w);
  };
  const int w1 = fit(window), w2 = fit(window / 2);
  const int per_sm = 2 * w2 >= w1 ? 2 : 1;
  const int warps = per_sm == 2 ? w2 : w1;
  MMF_REQUIRE(warps >= 1, "%s: a scratch of %d floats per row does not fit shared memory (window %zu B)", what, scratch, window);
  MMF_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const long long cta_rows = (long long)warps * RM_ROWS;
  long long grid = (rows + cta_rows - 1) / cta_rows;
  const long long cap = (long long)sms * per_sm;
  if (grid > cap) grid = cap;
  *warps_out = warps;
  *grid_out = grid;
  *smem_out = wtiles + (size_t)warps * per_warp;
  return MMF_OK;
}

static int fill_forward(RowMlpParams& P, long long rows, const mmf_mlp_op* ops, int n_ops, const float* weights,
                        const float* const* inputs, const int32_t* in_dims, const int32_t* in_slots, int n_inputs,
                        float* const* outputs, const int32_t* out_dims, const int32_t* out_slots, int n_outputs, int scratch) {
  int rc = validate_program(ops, n_ops, scratch, "row_mlp");
  if (rc) return rc;
  MMF_REQUIRE(n_inputs >= 1 && n_inputs <= MMF_MLP_MAX_IO && n_outputs >= 1 && n_outputs <= MMF_MLP_MAX_IO,
              "row_mlp: %d inputs / %d outputs outside 1..%d", n_inputs, n_outputs, MMF_MLP_MAX_IO);
  MMF_REQUIRE(weights != nullptr, "row_mlp: NULL weights");
  P.n_ops = n_ops; P.n_inputs = n_inputs; P.n_outputs = n_outputs; P.scratch = scratch; P.rows = rows;
  P.weights = weights;
  P.tape = nullptr;
  P.tape_floats = 0;
  auto inside = [&](int slot, int dim) { return slot >= 0 && dim >= 1 && slot + dim <= scratch; };
  for (int o = 0; o < n_ops; ++o) P.ops[o] = ops[o];
  for (int i = 0; i < n_inputs; ++i) {
    MMF_REQUIRE(inputs[i] != nullptr && inside(in_slots[i], in_dims[i]), "row_mlp: input %d is NULL or outside the scratch", i);
    P.inputs[i] = inputs[i]; P.in_dims[i] = in_dims[i]; P.in_slots[i] = in_slots[i];
  }
  for (int i = 0; i < n_outputs; ++i) {
    MMF_REQUIRE(outputs[i] != nullptr && inside(out_slots[i], out_dims[i]), "row_mlp: output %d is NULL or outside the scratch", i);
    P.outputs[i] = outputs[i]; P.out_dims[i] = out_dims[i]; P.out_slots[i] = out_slots[i];
  }
  return MMF_OK;
}

int launch_row_mlp(long long rows, const mmf_mlp_op* ops, int n_ops, const float* weights, const float* const* inputs,
                   const int32_t* in_dims, const int32_t* in_slots, int n_inputs, float* const* outputs,
                   const int32_t* out_dims, const int32_t* out_slots, int n_outputs, int scratch, float* tape,
                   cudaStream_t stream) {
  if (rows == 0) return MMF_OK;
  RowMlpParams P;
  int rc = fill_forward(P, rows, ops, n_ops, weights, inputs, in_dims, in_slots, n_inputs, outputs, out_dims, out_slots,
                        n_outputs, scratch);
  if (rc) return rc;
  int warps;
  long long grid;
  size_t smem;
  if (tape == nullptr) {
    static thread_local int configured_dev = -1;
    static thread_local size_t window = 0;
    rc = rm_geometry(k_row_mlp, configured_dev, window, rows, scratch, "row_mlp", &warps, &grid, &smem);
    if (rc) return rc;
    k_row_mlp<<<(unsigned)grid, warps * 32, smem, stream>>>(P);
    MMF_LAUNCH_CHECK("k_row_mlp");
    return MMF_OK;
  }
  MMF_REQUIRE(((uintptr_t)tape & 15) == 0, "row_mlp_train: the tape must be 16-byte aligned");
  for (int o = 0; o < n_ops; ++o) P.tape_floats += ops[o].in_dim + ops[o].out_dim;
  P.tape = tape;
  static thread_local int configured_dev = -1;
  static thread_local size_t window = 0;
  rc = rm_geometry(k_row_mlp_train, configured_dev, window, rows, scratch, "row_mlp_train", &warps, &grid, &smem);
  if (rc) return rc;
  k_row_mlp_train<<<(unsigned)grid, warps * 32, smem, stream>>>(P);
  MMF_LAUNCH_CHECK("k_row_mlp_train");
  return MMF_OK;
}

static long long rm_groups(long long rows) { return (rows + RM_ROWS - 1) / RM_ROWS; }

static int rm_tiles(const mmf_mlp_op* ops, int n_ops, RmTile* tiles) {
  int n = 0;
  for (int o = 0; o < n_ops; ++o)
    for (int j0 = 0; j0 < ops[o].out_dim; j0 += 64)
      for (int k0 = 0; k0 < ops[o].in_dim; k0 += 64) {
        if (tiles && n < RM_MAX_TILES) tiles[n] = RmTile{o, j0, k0, 0};
        ++n;
      }
  return n;
}

// Row chunks of the weight-gradient reduction: about four CTAs per SM of a 148-SM B200 over all tiles, fixed by the shape
// alone (not by the device) so that the sums, and the workspace size, are the same everywhere.
static int rm_chunks(long long rows, int tiles) {
  const long long groups = rm_groups(rows);
  long long chunks = (4 * 148 + tiles - 1) / tiles;
  if (chunks > groups) chunks = groups;
  if (chunks > 1024) chunks = 1024;
  return (int)(chunks < 1 ? 1 : chunks);
}

int row_mlp_train_sizes(long long rows, const mmf_mlp_op* ops, int n_ops, long long* tape_floats, long long* delta_floats,
                        size_t* workspace_bytes) {
  MMF_REQUIRE(rows >= 0 && ops && n_ops >= 1 && n_ops <= MMF_MLP_MAX_OPS, "row_mlp_train_sizes: bad arguments");
  long long tf = 0, gf = 0, pack = 0;
  for (int o = 0; o < n_ops; ++o) {
    tf += ops[o].in_dim + ops[o].out_dim;
    gf += ops[o].out_dim;
    const long long end = ops[o].w_off + (long long)ops[o].out_dim * (ops[o].in_dim + 1);
    pack = end > pack ? end : pack;
  }
  const long long padded = rm_groups(rows) * RM_ROWS;
  if (tape_floats) *tape_floats = padded * tf;
  if (delta_floats) *delta_floats = padded * gf;
  if (workspace_bytes) *workspace_bytes = rows == 0 ? 0 : (size_t)rm_chunks(rows, rm_tiles(ops, n_ops, nullptr)) * pack * sizeof(float);
  return MMF_OK;
}

int launch_row_mlp_bwd(long long rows, const mmf_mlp_op* ops, int n_ops, const float* weights_t, const float* tape,
                       const mmf_mlp_bwd_op* bops, int n_bops, const float* const* d_outputs, const int32_t* out_dims,
                       const int32_t* dout_slots, int n_outputs, float* const* d_inputs, const int32_t* din_dims,
                       const int32_t* din_slots, int n_dinputs, int scratch, float* delta, cudaStream_t stream) {
  if (rows == 0) return MMF_OK;
  MMF_REQUIRE(n_ops >= 1 && n_ops <= MMF_MLP_MAX_OPS && ops != nullptr, "row_mlp_bwd: %d ops outside 1..%d", n_ops, MMF_MLP_MAX_OPS);
  MMF_REQUIRE(scratch >= 1 && scratch <= 1536, "row_mlp_bwd: delta scratch of %d floats per row outside 1..1536", scratch);
  MMF_REQUIRE(n_bops >= 1 && n_bops <= MMF_MLP_MAX_OPS && bops != nullptr, "row_mlp_bwd: %d reverse ops outside 1..%d", n_bops,
              MMF_MLP_MAX_OPS);
  MMF_REQUIRE(n_outputs >= 1 && n_outputs <= MMF_MLP_MAX_IO && n_dinputs >= 0 && n_dinputs <= MMF_MLP_MAX_IO,
              "row_mlp_bwd: %d outputs / %d input gradients outside the limits", n_outputs, n_dinputs);
  MMF_REQUIRE(weights_t && tape && delta, "row_mlp_bwd: NULL weights, tape or delta planes");
  MMF_REQUIRE((((uintptr_t)tape | (uintptr_t)delta) & 15) == 0, "row_mlp_bwd: tape and delta planes must be 16-byte aligned");
  RowMlpBwdParams P;
  auto inside = [&](int slot, int dim) { return slot >= 0 && dim >= 1 && slot + dim <= scratch; };
  int tf = 0, gf = 0;
  for (int o = 0; o < n_ops; ++o) {
    const mmf_mlp_op& op = ops[o];
    // any input width: delta_src is rm_op's output, which it tiles by 64 features (bounded by the delta scratch)
    MMF_REQUIRE(op.in_dim >= 1 && op.out_dim >= 1 && op.out_dim <= RM_MAX_OUT && op.w_off >= 0,
                "row_mlp_bwd: op %d has bad dimensions (%d -> %d)", o, op.in_dim, op.out_dim);
    MMF_REQUIRE(op.act >= MMF_MLP_NONE && op.act <= MMF_MLP_SIGMOID, "row_mlp_bwd: op %d: unknown activation %d", o, op.act);
    P.ops[o] = op;
    P.tape_dst[o] = tf + op.in_dim;
    P.goff[o] = gf;
    tf += op.in_dim + op.out_dim;
    gf += op.out_dim;
  }
  for (int q = 0; q < n_bops; ++q) {
    const mmf_mlp_bwd_op& b = bops[q];
    MMF_REQUIRE(b.op >= 0 && b.op < n_ops, "row_mlp_bwd: reverse op %d names forward op %d", q, b.op);
    const mmf_mlp_op& op = ops[b.op];
    MMF_REQUIRE(inside(b.g, op.out_dim) && (b.dsrc < 0 || inside(b.dsrc, op.in_dim)) && (b.dres < 0 || inside(b.dres, op.out_dim)),
                "row_mlp_bwd: reverse op %d addresses the delta scratch outside [0, %d)", q, scratch);
    MMF_REQUIRE(b.dsrc < 0 || b.g + op.out_dim <= b.dsrc || b.dsrc + op.in_dim <= b.g, "row_mlp_bwd: reverse op %d: g overlaps delta_src", q);
    MMF_REQUIRE(b.dres < 0 || b.g + op.out_dim <= b.dres || b.dres + op.out_dim <= b.g, "row_mlp_bwd: reverse op %d: g overlaps delta_res", q);
    P.bops[q] = b;
  }
  for (int i = 0; i < n_outputs; ++i) {
    MMF_REQUIRE(d_outputs[i] != nullptr && inside(dout_slots[i], out_dims[i]), "row_mlp_bwd: d output %d is NULL or outside the scratch", i);
    P.d_outputs[i] = d_outputs[i]; P.out_dims[i] = out_dims[i]; P.dout_slots[i] = dout_slots[i];
  }
  for (int i = 0; i < n_dinputs; ++i) {
    MMF_REQUIRE(d_inputs[i] != nullptr && inside(din_slots[i], din_dims[i]), "row_mlp_bwd: d input %d is NULL or outside the scratch", i);
    P.d_inputs[i] = d_inputs[i]; P.din_dims[i] = din_dims[i]; P.din_slots[i] = din_slots[i];
  }
  P.n_bops = n_bops; P.n_outputs = n_outputs; P.n_dinputs = n_dinputs; P.scratch = scratch;
  P.tape_floats = tf; P.delta_floats = gf; P.rows = rows;
  P.weights_t = weights_t; P.tape = tape; P.delta = delta;
  static thread_local int configured_dev = -1;
  static thread_local size_t window = 0;
  int warps;
  long long grid;
  size_t smem;
  const int rc = rm_geometry(k_row_mlp_bwd, configured_dev, window, rows, scratch, "row_mlp_bwd", &warps, &grid, &smem);
  if (rc) return rc;
  k_row_mlp_bwd<<<(unsigned)grid, warps * 32, smem, stream>>>(P);
  MMF_LAUNCH_CHECK("k_row_mlp_bwd");
  return MMF_OK;
}

int launch_row_mlp_dw(long long rows, const mmf_mlp_op* ops, int n_ops, const float* tape, const float* delta, float* grads,
                      void* workspace, cudaStream_t stream) {
  MMF_REQUIRE(ops && n_ops >= 1 && n_ops <= MMF_MLP_MAX_OPS, "row_mlp_weight_grads: %d ops outside 1..%d", n_ops, MMF_MLP_MAX_OPS);
  MMF_REQUIRE(grads != nullptr, "row_mlp_weight_grads: NULL gradient pack");
  RowMlpDwParams P;
  int tf = 0, gf = 0;
  long long pack = 0;
  for (int o = 0; o < n_ops; ++o) {
    const mmf_mlp_op& op = ops[o];
    MMF_REQUIRE(op.in_dim >= 1 && op.out_dim >= 1 && op.out_dim <= RM_MAX_OUT && op.w_off >= 0,
                "row_mlp_weight_grads: op %d has bad dimensions (%d -> %d)", o, op.in_dim, op.out_dim);
    P.ops[o] = op;
    P.tape_src[o] = tf;
    P.goff[o] = gf;
    tf += op.in_dim + op.out_dim;
    gf += op.out_dim;
    const long long end = op.w_off + (long long)op.out_dim * (op.in_dim + 1);
    pack = end > pack ? end : pack;
  }
  const int n_tiles = rm_tiles(ops, n_ops, P.tiles);
  MMF_REQUIRE(n_tiles <= RM_MAX_TILES, "row_mlp_weight_grads: %d weight tiles exceed %d", n_tiles, RM_MAX_TILES);
  if (rows == 0) {
    MMF_CUDA(cudaMemsetAsync(grads, 0, (size_t)pack * sizeof(float), stream));
    return MMF_OK;
  }
  MMF_REQUIRE(tape && delta && workspace, "row_mlp_weight_grads: NULL tape, delta planes or workspace");
  const int chunks = rm_chunks(rows, n_tiles);
  P.tape_floats = tf; P.delta_floats = gf;
  P.groups = rm_groups(rows);
  P.groups_per_chunk = (int)((P.groups + chunks - 1) / chunks);
  P.pack_floats = pack;
  P.tape = tape; P.delta = delta; P.workspace = static_cast<float*>(workspace);
  k_row_mlp_dw<<<dim3(n_tiles, chunks), 256, 0, stream>>>(P);
  MMF_LAUNCH_CHECK("k_row_mlp_dw");
  long long blocks = (pack + 255) / 256;
  if (blocks > 4096) blocks = 4096;
  k_row_mlp_dw_sum<<<(unsigned)blocks, 256, 0, stream>>>(P.workspace, pack, chunks, grads);
  MMF_LAUNCH_CHECK("k_row_mlp_dw_sum");
  return MMF_OK;
}

}  // namespace mmf
