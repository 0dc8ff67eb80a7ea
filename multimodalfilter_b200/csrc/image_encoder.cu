// image_encoder.cu -- the convolutional trunk of the image observation encoder (SURVEY.md section 8(f)-1):
//   Conv2d(1,32,5,p=2) ReLU | resblock Conv2d(32,k=3) | Conv2d(32,16,3,p=1) ReLU | Conv2d(16,8,3,p=1)
// (ref: crossmodal/push_models/layers.py:93-104, crossmodal/door_models/layers.py:43-63), 32x32 images.
// The encoders are state independent, so the host runs them once over all T*N images of a sequence
// (fused.batched_over_time); at BASELINE config C3 that is 409,600 images = 21 TFLOP of fp32 convolution, which
// dominates the end-to-end forward_loop time when left to the library's fp32 path.
//
// Here every 3x3 convolution is an implicit GEMM on the tensor cores with fp32-grade accuracy:
//   * activations live in HBM as bf16 hi/lo PLANES: map[image][channel chunk of 8][hi|lo][position][8 ch], a
//     position being y * 34 + x (row pitch 34 = 32 pixels + 2 zero pad columns) behind a 64-position zero guard,
//     so the neighbour (dy, dx) of position p is simply position p + 34 dy + dx and the zero padding of the
//     convolution is data, not control flow;
//   * a tile is 128 consecutive positions (9 tiles per image); its input window (208 positions per plane) is
//     brought into shared memory by bulk async copies (TMA), and the A operand of tap (dy, dx) is that same
//     shared memory addressed through a no-swizzle K-major UMMA descriptor whose start address is shifted by
//     34 dy + dx positions: no im2col, no gather instructions at all;
//   * D[128 positions x Cout] += A_tap[128 x Cin] * W_tap[Cin x Cout] for the 9 taps with split operands
//     (hi*hi + hi*lo + lo*hi).  The MMAs read A from shared memory and are bound by that traffic, so W_hi and W_lo
//     are stacked along N: ONE MMA A_hi x [W_hi | W_lo] (N = 2 Cout) yields both products from one pass over A_hi,
//     a second A_lo x W_hi adds the third; the epilogue sums the two column halves.  fp32 accumulation in TMEM;
//   * warp-specialised pipeline: warp 0 = TMA producer, warp 1 = MMA issuer, warps 4-11 = two epilogue groups
//     (bias, residual, ReLU, bf16 split, coalesced 16-byte plane stores), 4 stages of shared memory / TMEM.
// The 5x5 stem (one input channel, 1.6 MFLOP per image) runs on the CUDA cores and emits the first map.
#include "tc_common.cuh"

namespace mmf {

constexpr int ENC_PITCH = 34;                 // positions per image row (32 pixels + 2 zero pads)
constexpr int ENC_NPOS = 32 * ENC_PITCH;      // 1088 positions hold an image
constexpr int ENC_TILES = 9;                  // 9 x 128 = 1152 >= 1088
constexpr int ENC_GUARD = 64;                 // zero positions in front of position 0
constexpr int ENC_PLANE_POS = ENC_GUARD + ENC_TILES * 128 + 64;  // 1280
constexpr int ENC_PLANE_B = ENC_PLANE_POS * 16;                  // bytes of one (chunk, hi|lo) plane
constexpr int ENC_HALO = 40;                  // >= 35 = pitch + 1, multiple of 8
constexpr int ENC_WIN_POS = 128 + 2 * ENC_HALO;  // 208 positions per plane in a stage
constexpr int ENC_WIN_B = ENC_WIN_POS * 16;      // 3328 B
constexpr int ENC_STAGES = 4;
constexpr int ENC_THREADS = 384;
constexpr int ENC_DCOLS = 64;                 // TMEM columns per stage: [hi*hi + lo*hi | hi*lo] halves of up to 32 channels

__host__ __device__ inline size_t enc_map_bytes(int channels) { return (size_t)(channels / 8) * 2 * ENC_PLANE_B; }

// no-swizzle K-major shared-memory matrix descriptor: rows of 16 bytes, 8 consecutive rows = one core matrix,
// SBO = distance between 8-row groups, LBO = distance between the two 16-byte K chunks of one K = 16 step.
__device__ __forceinline__ uint64_t make_desc_interleave(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return (uint64_t)((smem_addr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) |
         ((uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32) | (1ull << 46);
}
__device__ __forceinline__ void mma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(acc)
      : "memory");
}

// bf16 hi/lo split of 8 channels -> two 16-byte plane elements: hi = rn_bf16(v), lo = rn_bf16(v - hi) (v - hi is
// exact), so hi + lo carries v to 2^-18 relative; the remainder uses the mixed-precision FMA like store_a_chunk
__device__ __forceinline__ void split8(const float (&v)[8], uint4& hi4, uint4& lo4) {
  uint32_t hi[4], lo[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(hi[j]) : "f"(v[2 * j + 1]), "f"(v[2 * j]));
    float rx, ry;
    asm("{\n\t"
        ".reg .b16 l, h, m1;\n\t"
        "mov.b32 {l, h}, %2;\n\t"
        "mov.b16 m1, 0xBF80;\n\t"
        "fma.rn.f32.bf16 %0, l, m1, %3;\n\t"
        "fma.rn.f32.bf16 %1, h, m1, %4;\n\t"
        "}"
        : "=f"(rx), "=f"(ry)
        : "r"(hi[j]), "f"(v[2 * j]), "f"(v[2 * j + 1]));
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(lo[j]) : "f"(ry), "f"(rx));
  }
  hi4 = make_uint4(hi[0], hi[1], hi[2], hi[3]);
  lo4 = make_uint4(lo[0], lo[1], lo[2], lo[3]);
}
__device__ __forceinline__ void unpack8(const uint4& hi4, const uint4& lo4, float (&v)[8]) {
  const uint32_t h[4] = {hi4.x, hi4.y, hi4.z, hi4.w}, l[4] = {lo4.x, lo4.y, lo4.z, lo4.w};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    v[2 * j] = __uint_as_float(h[j] << 16) + __uint_as_float(l[j] << 16);
    v[2 * j + 1] = __uint_as_float(h[j] & 0xffff0000u) + __uint_as_float(l[j] & 0xffff0000u);
  }
}
__device__ __forceinline__ bool enc_valid(int pos) { return pos < ENC_NPOS && (pos % ENC_PITCH) < 32; }

// this thread's accumulator row: columns [0, NPAD) hold hi*hi + lo*hi, [NPAD, 2 NPAD) hold hi*lo -> their sum
template <int NPAD>
__device__ __forceinline__ void load_accumulator(uint32_t taddr, uint32_t (&d)[NPAD]) {
  uint32_t e[NPAD];
#pragma unroll
  for (int c = 0; c < NPAD; c += 16) {
    tmem_ld16(taddr + c, reinterpret_cast<uint32_t(&)[16]>(d[c]));
    tmem_ld16(taddr + NPAD + c, reinterpret_cast<uint32_t(&)[16]>(e[c]));
  }
  tc_wait_ld();
#pragma unroll
  for (int c = 0; c < NPAD; ++c) d[c] = __float_as_uint(__uint_as_float(d[c]) + __uint_as_float(e[c]));
}

template <int CIN, int NPAD>
__device__ __forceinline__ void issue_conv(uint32_t st_addr, uint32_t w_addr, uint32_t d) {
  constexpr int KC = CIN / 8;
  constexpr uint32_t IDESC2 = make_idesc(2 * NPAD, 128);  // A_hi x [W_hi | W_lo]
  constexpr uint32_t IDESC1 = make_idesc(NPAD, 128);      // A_lo x W_hi
  uint32_t acc = 0;
#pragma unroll
  for (int tap = 0; tap < 9; ++tap) {
    const int shift = ENC_HALO + (tap / 3 - 1) * ENC_PITCH + (tap % 3 - 1);
#pragma unroll
    for (int ks = 0; ks < CIN / 16; ++ks) {
      // A: plane (chunk 2 ks, hi|lo) at the shifted position; the second K chunk is the next chunk's plane
      const uint32_t a_hi = st_addr + (uint32_t)((2 * ks) * 2) * ENC_WIN_B + (uint32_t)shift * 16;
      const uint32_t a_lo = a_hi + ENC_WIN_B;
      const uint64_t da_hi = make_desc_interleave(a_hi, 2 * ENC_WIN_B, 128);
      const uint64_t da_lo = make_desc_interleave(a_lo, 2 * ENC_WIN_B, 128);
      // B: [tap][chunk][2 NPAD rows][8]; rows [0, NPAD) = W_hi, [NPAD, 2 NPAD) = W_lo
      const uint32_t b = w_addr + (uint32_t)((tap * KC + 2 * ks) * 2 * NPAD) * 16;
      const uint64_t db = make_desc_interleave(b, 2 * NPAD * 16, 128);
      mma_ss(d, da_hi, db, IDESC2, acc);  // columns [0, NPAD) += hi*hi, [NPAD, 2 NPAD) += hi*lo
      mma_ss(d, da_lo, db, IDESC1, 1);    // columns [0, NPAD) += lo*hi
      acc = 1;
    }
  }
}

// ---- fused trunk: all five layers of one image by one CTA, activation maps in L2-resident scratch ---------------
// A persistent CTA carries an image through stem -> block1 -> block2(+x) -> 32->16 -> 16->8 by itself: its four
// scratch maps (640 KB: x double-buffered, t/z, y) are private, so 148 CTAs keep 95 MB hot in the 126 MB L2 and HBM only
// sees the raw image and the final (8, 32, 32) activations.  Work items = (layer, tile) in order; tile t of layer l+1 only needs tiles
// t-1..t+1 of layer l, tracked by one mbarrier per (layer, tile), so the TMA -> MMA -> epilogue ring never drains
// between layers.  Epilogue warps write the maps with generic stores and publish them to the async proxy
// (fence.proxy.async.global + mbarrier release) before the producer's bulk copies read them.
constexpr int TR_LAYERS = 5;                    // 0 = stem (CUDA cores), 1..4 = 3x3 convolutions
constexpr int TR_CONV_ITEMS = 4 * ENC_TILES;    // per image
constexpr int TR_STAGE_B = 8 * ENC_WIN_B;       // a stage holds the widest window (32 channels)
constexpr int TR_W2_B = 2 * 9 * 4 * 32 * 16 + 128;   // 32->32: operand image + bias
constexpr int TR_W3_B = 2 * 9 * 4 * 16 * 16 + 64;    // 32->16
constexpr int TR_W4_B = 2 * 9 * 2 * 16 * 16 + 64;    // 16->(<=16)
constexpr int TR_WSTEM_B = (25 * 32 + 32) * 4;
constexpr int TR_W_B = 2 * TR_W2_B + TR_W3_B + TR_W4_B + TR_WSTEM_B;
constexpr int TR_SCRATCH_MAPS = 4;            // x (two buffers), t / z, y

struct TrunkParams {
  const float* images;      // (n, 32, 32)
  const uint8_t* weights;   // [W block1 | W block2 | W 32->16 | W 16->8 | stem fp32], layouts in mmf_b200.h
  uint8_t* scratch;         // gridDim.x * TR_SCRATCH_MAPS * enc_map_bytes(32), zero-initialised once
  float* out_nchw;          // (n, cout, 32, 32)
  int n_images, cout;
};

__device__ __forceinline__ void publish_tile(uint64_t* bar) {
  asm volatile("fence.proxy.async.global;" ::: "memory");
  __syncwarp();
  if ((threadIdx.x & 31) == 0) mbar_arrive(bar);
}

// accumulator row -> bias (+ residual) (+ ReLU) -> planes in `out_map` or NCHW fp32
template <int NPAD>
__device__ __forceinline__ void epilogue_conv(const uint32_t (&d)[32], const float* bias_s, const uint8_t* res_map,
                                              bool relu, bool valid, int pos, uint8_t* out_map, float* out_img, int cout) {
  const size_t plane_off = (size_t)(ENC_GUARD + pos) * 16;
#pragma unroll
  for (int kc = 0; kc < NPAD / 8; ++kc) {
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = __uint_as_float(d[kc * 8 + j]) + bias_s[kc * 8 + j];
    if (res_map != nullptr) {
      const uint8_t* rp = res_map + (size_t)(kc * 2) * ENC_PLANE_B + plane_off;
      float x[8];
      unpack8(*reinterpret_cast<const uint4*>(rp), *reinterpret_cast<const uint4*>(rp + ENC_PLANE_B), x);
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] += x[j];
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (relu) v[j] = fmaxf(v[j], 0.0f);
      if (!valid) v[j] = 0.0f;
    }
    if (out_map != nullptr) {
      uint4 hi4, lo4;
      split8(v, hi4, lo4);
      uint8_t* op = out_map + (size_t)(kc * 2) * ENC_PLANE_B + plane_off;
      *reinterpret_cast<uint4*>(op) = hi4;
      *reinterpret_cast<uint4*>(op + ENC_PLANE_B) = lo4;
    }
    if (out_img != nullptr && valid) {
      const int y = pos / ENC_PITCH, x = pos % ENC_PITCH;
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (kc * 8 + j < cout) out_img[((size_t)(kc * 8 + j) * 32 + y) * 32 + x] = v[j];
    }
  }
}

__global__ void __launch_bounds__(ENC_THREADS, 1) k_enc_trunk(const __grid_constant__ TrunkParams P) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* w_s = smem;
  uint8_t* stage0 = smem + ((TR_W_B + 127) & ~127);
  uint64_t* bars = reinterpret_cast<uint64_t*>(stage0 + ENC_STAGES * TR_STAGE_B);
  uint64_t* full = bars;
  uint64_t* mma_done = bars + ENC_STAGES;
  uint64_t* stage_free = bars + 2 * ENC_STAGES;
  uint64_t* tmem_free = bars + 3 * ENC_STAGES;
  uint64_t* wbar = bars + 4 * ENC_STAGES;
  uint64_t* stem_done = wbar + 1;                  // [x buffer 0|1][tile]: stem output of an image is written and published
  uint64_t* tile_done = stem_done + 2 * ENC_TILES;  // [layer 1..3][tile]: that tile of the layer's OUTPUT map
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tile_done + 3 * ENC_TILES);

  const int tid = threadIdx.x;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  if (tid == 0) {
    for (int s = 0; s < ENC_STAGES; ++s) {
      mbar_init(full + s, 1);
      mbar_init(mma_done + s, 1);
      mbar_init(stage_free + s, 1);
      mbar_init(tmem_free + s, 4);
    }
    for (int i = 0; i < 5 * ENC_TILES; ++i) mbar_init(stem_done + i, 4);
    mbar_init(wbar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"(ENC_STAGES * ENC_DCOLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const size_t map32 = enc_map_bytes(32);
  // x is double-buffered: the stem of image k+1 is computed in the shadow of image k's convolutions
  uint8_t* sx0 = P.scratch + (size_t)blockIdx.x * TR_SCRATCH_MAPS * map32;
  uint8_t* st = sx0 + 2 * map32;                              // block1 output, later the 16-channel map z
  uint8_t* sy = st + map32;                                   // resblock output
  // shared-memory offsets of the per-layer weights
  constexpr int OFF_W[5] = {2 * TR_W2_B + TR_W3_B + TR_W4_B, 0, TR_W2_B, 2 * TR_W2_B, 2 * TR_W2_B + TR_W3_B};

  if (warp == 0) {
    // ------------------------------------------------------------------------------------------ TMA producer
    if (elect_one_sync()) {
      mbar_expect_tx(wbar, TR_W_B);
      for (uint32_t off = 0; off < (uint32_t)TR_W_B; off += 32768) {
        const uint32_t n = (uint32_t)TR_W_B - off < 32768 ? (uint32_t)TR_W_B - off : 32768;
        bulk_g2s(w_s + off, P.weights + off, n, wbar);
      }
      long long c = 0;
      int k = 0;
      for (long long image = blockIdx.x; image < P.n_images; image += gridDim.x, ++k) {
        const uint32_t ipar = (uint32_t)(k & 1);
        for (int layer = 1; layer <= 4; ++layer) {
          const uint8_t* in = layer == 1 ? sx0 + (size_t)(k & 1) * map32 : layer == 2 ? st : layer == 3 ? sy : st;
          const int planes = layer == 4 ? 4 : 8;
          for (int tile = 0; tile < ENC_TILES; ++tile, ++c) {
            const int s = (int)(c % ENC_STAGES);
            const uint32_t par = (uint32_t)((c / ENC_STAGES) & 1);
            mbar_wait(stage_free + s, par ^ 1u);
            // the window reaches into the neighbouring tiles of the producing layer
            // layer 1 reads the stem output in x[k & 1] (completed once every second image), the others layer - 1
            uint64_t* dep = layer == 1 ? stem_done + (k & 1) * ENC_TILES : tile_done + (layer - 2) * ENC_TILES;
            const uint32_t dpar = layer == 1 ? (uint32_t)((k >> 1) & 1) : ipar;
            if (tile > 0) mbar_wait(dep + tile - 1, dpar);
            mbar_wait(dep + tile, dpar);
            if (tile + 1 < ENC_TILES) mbar_wait(dep + tile + 1, dpar);
            asm volatile("fence.proxy.async.global;" ::: "memory");
            const uint8_t* src = in + (size_t)(ENC_GUARD + tile * 128 - ENC_HALO) * 16;
            mbar_expect_tx(full + s, (uint32_t)planes * ENC_WIN_B);
            for (int pl = 0; pl < planes; ++pl)
              bulk_g2s(stage0 + s * TR_STAGE_B + pl * ENC_WIN_B, src + (size_t)pl * ENC_PLANE_B, ENC_WIN_B, full + s);
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // -------------------------------------------------------------------------------------------- MMA issuer
    mbar_wait(wbar, 0);
    if (elect_one_sync()) {
      const uint32_t w_addr = smem_u32(w_s);
      long long c = 0;
      for (long long image = blockIdx.x; image < P.n_images; image += gridDim.x) {
        for (int layer = 1; layer <= 4; ++layer) {
          for (int tile = 0; tile < ENC_TILES; ++tile, ++c) {
            const int s = (int)(c % ENC_STAGES);
            const uint32_t par = (uint32_t)((c / ENC_STAGES) & 1);
            mbar_wait(tmem_free + s, par ^ 1u);
            mbar_wait(full + s, par);
            tc_fence_after();
            const uint32_t st_addr = smem_u32(stage0 + s * TR_STAGE_B);
            const uint32_t d = tmem_base + s * ENC_DCOLS;
            if (layer <= 2) issue_conv<32, 32>(st_addr, w_addr + OFF_W[layer], d);
            else if (layer == 3) issue_conv<32, 16>(st_addr, w_addr + OFF_W[3], d);
            else issue_conv<16, 16>(st_addr, w_addr + OFF_W[4], d);
            tc_commit(mma_done + s);
            tc_commit(stage_free + s);
          }
        }
      }
    }
    __syncwarp();
  } else if (warp >= 4) {
    // ------------------------------------------------------------ epilogue groups (and the stem on the CUDA cores)
    const int eg = (warp - 4) >> 2;
    const int quad = warp & 3;
    const int r = quad * 32 + (tid & 31);
    mbar_wait(wbar, 0);
    const float* wstem = reinterpret_cast<const float*>(w_s + OFF_W[0]);
    // stem tile `tile` of image `img` (the kk-th image of this CTA) -> x[kk & 1]
    auto stem_tile = [&](long long img, int kk, int tile) {
      const float* im = P.images + (size_t)img * 1024;
      uint8_t* sx = sx0 + (size_t)(kk & 1) * map32;
      const int pos = tile * 128 + r;
      const bool valid = enc_valid(pos);
      float acc[32];
#pragma unroll
      for (int ch = 0; ch < 32; ++ch) acc[ch] = wstem[25 * 32 + ch];
      if (valid) {
        const int y = pos / ENC_PITCH, x = pos % ENC_PITCH;
        for (int ky = 0; ky < 5; ++ky) {
          const int yy = y + ky - 2;
#pragma unroll
          for (int kx = 0; kx < 5; ++kx) {
            const int xx = x + kx - 2;
            const float p = (yy >= 0 && yy < 32 && xx >= 0 && xx < 32) ? __ldg(im + yy * 32 + xx) : 0.0f;
            const float4* w4 = reinterpret_cast<const float4*>(wstem + (ky * 5 + kx) * 32);
#pragma unroll
            for (int q = 0; q < 8; ++q) {
              const float4 t = w4[q];
              acc[4 * q] = fmaf(t.x, p, acc[4 * q]);
              acc[4 * q + 1] = fmaf(t.y, p, acc[4 * q + 1]);
              acc[4 * q + 2] = fmaf(t.z, p, acc[4 * q + 2]);
              acc[4 * q + 3] = fmaf(t.w, p, acc[4 * q + 3]);
            }
          }
        }
      }
#pragma unroll
      for (int kc = 0; kc < 4; ++kc) {
        float v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = valid ? fmaxf(acc[kc * 8 + j], 0.0f) : 0.0f;
        uint4 hi4, lo4;
        split8(v, hi4, lo4);
        uint8_t* plane = sx + (size_t)(kc * 2) * ENC_PLANE_B + (size_t)(ENC_GUARD + pos) * 16;
        *reinterpret_cast<uint4*>(plane) = hi4;
        *reinterpret_cast<uint4*>(plane + ENC_PLANE_B) = lo4;
      }
      publish_tile(stem_done + (kk & 1) * ENC_TILES + tile);
    };
    // the first image's stem up front; afterwards the stem of image k+1 rides along with the convolution items of
    // image k (one stem tile every fourth item), where the epilogue warps would otherwise wait for the tensor pipe
    if ((long long)blockIdx.x < P.n_images)
      for (int tile = 0; tile < ENC_TILES; ++tile)
        if ((tile & 1) == eg) stem_tile(blockIdx.x, 0, tile);
    long long c = 0;
    int k = 0;
    for (long long image = blockIdx.x; image < P.n_images; image += gridDim.x, ++k) {
      const long long next = image + gridDim.x;
      const uint8_t* sx = sx0 + (size_t)(k & 1) * map32;
      int j = 0;
      for (int layer = 1; layer <= 4; ++layer) {
        for (int tile = 0; tile < ENC_TILES; ++tile, ++c, ++j) {
          if ((j & 3) == 0 && (j >> 2) < ENC_TILES && next < P.n_images && (((j >> 2) & 1) == eg)) stem_tile(next, k + 1, j >> 2);
          if ((int)(c & 1) != eg) continue;
          const int pos = tile * 128 + r;
          const bool valid = enc_valid(pos);
          const int s = (int)(c % ENC_STAGES);
          const uint32_t par = (uint32_t)((c / ENC_STAGES) & 1);
          mbar_wait(mma_done + s, par);
          tc_fence_after();
          uint32_t d[32];
          const uint32_t taddr = tmem_base + s * ENC_DCOLS + ((uint32_t)(quad * 32) << 16);
          if (layer <= 2) load_accumulator<32>(taddr, d);
          else load_accumulator<16>(taddr, reinterpret_cast<uint32_t(&)[16]>(d[0]));
          tc_fence_before();
          __syncwarp();
          if ((tid & 31) == 0) mbar_arrive(tmem_free + s);
          const float* bias_s = reinterpret_cast<const float*>(
              w_s + OFF_W[layer] + (layer <= 2 ? TR_W2_B - 128 : layer == 3 ? TR_W3_B - 64 : TR_W4_B - 64));
          if (layer == 1) epilogue_conv<32>(d, bias_s, nullptr, true, valid, pos, st, nullptr, 0);
          else if (layer == 2) epilogue_conv<32>(d, bias_s, sx, true, valid, pos, sy, nullptr, 0);
          else if (layer == 3) epilogue_conv<16>(d, bias_s, nullptr, true, valid, pos, st, nullptr, 0);
          else epilogue_conv<16>(d, bias_s, nullptr, false, valid, pos, nullptr, P.out_nchw + (size_t)image * P.cout * 1024, P.cout);
          if (layer < 4) publish_tile(tile_done + (layer - 1) * ENC_TILES + tile);
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(ENC_STAGES * ENC_DCOLS) : "memory");
  }
}

static int trunk_grid(int* grid_out) {
  int dev = 0, sms = 148;
  MMF_CUDA(cudaGetDevice(&dev));
  MMF_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  *grid_out = sms;
  return MMF_OK;
}

size_t enc_trunk_weight_bytes() { return TR_W_B; }

size_t enc_trunk_scratch_bytes() {
  int grid = 148;
  trunk_grid(&grid);
  return (size_t)grid * TR_SCRATCH_MAPS * enc_map_bytes(32);
}

int launch_enc_trunk(int n_images, int cout, const float* images, const void* weights, void* scratch, float* out_nchw,
                     cudaStream_t stream) {
  if (n_images == 0) return MMF_OK;
  TrunkParams P;
  P.images = images;
  P.weights = static_cast<const uint8_t*>(weights);
  P.scratch = static_cast<uint8_t*>(scratch);
  P.out_nchw = out_nchw;
  P.n_images = n_images;
  P.cout = cout;
  const size_t smem = ((TR_W_B + 127) & ~127) + (size_t)ENC_STAGES * TR_STAGE_B + 1024 + 8192;
  static thread_local int configured_dev = -1;
  static thread_local size_t window = 0;
  int dev = 0, grid = 148;
  MMF_CUDA(cudaGetDevice(&dev));
  int rc = trunk_grid(&grid);
  if (rc) return rc;
  if (configured_dev != dev) {
    rc = opt_in_shared_memory(k_enc_trunk, &window);
    if (rc) return rc;
    configured_dev = dev;
  }
  MMF_REQUIRE(smem <= window, "encoder trunk needs %zu B of shared memory (window %zu B)", smem, window);
  if (grid > n_images) grid = n_images;
  k_enc_trunk<<<grid, ENC_THREADS, smem, stream>>>(P);
  MMF_LAUNCH_CHECK("k_enc_trunk");
  return MMF_OK;
}

}  // namespace mmf
