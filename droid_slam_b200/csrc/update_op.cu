// The update operator of DROID-SLAM (SURVEY section 8a row A6) as hand-written sm_100a kernels:
//   UpdateModule.forward   reference droid_slam/droid_net.py:111-143  (encoders :83-93, heads :95-106)
//   ConvGRU.forward        reference droid_slam/modules/gru.py:19-32
//   GraphAgg.forward       reference droid_slam/droid_net.py:59-75
//
// Every convolution is an implicit GEMM on the 5th-generation tensor cores -- no im2col buffer, no library call:
//   * activations live channels-last ([image, y, x, C], f16), so a tile of 128 pixels x 64 channels is a K-major operand
//     with 128-byte rows; a 3x3 tap (dy,dx) is the same tile shifted by one pixel, which TMA delivers with the zero padding
//     for free (cp.async.bulk.tensor.4d with out-of-bounds fill at negative / beyond-the-edge coordinates);
//   * per (64-channel block, dx) ONE halo tile of (rows + 2) image rows is loaded and the three dy taps are the same
//     shared-memory buffer at +dy*TW*128 bytes (a multiple of the 1024-byte swizzle atom), so a 3x3 convolution reads its
//     input 3x (not 9x) from L2;
//   * weights are pre-packed [tap][N][K] f16 (K contiguous) and stream through a second TMA ring;
//   * tcgen05.mma.cta_group::1.kind::f16, M = 128 (x MT tiles sharing every weight stage), N up to 384, fp32 accumulators in
//     TMEM; persistent CTAs (one per SM) with a static tile schedule: warp 0 = TMA producer (runs ahead across tiles),
//     warp 1 = MMA issuer, warps 2..9 = epilogue (tcgen05.ld 32 lanes x 32 columns, thread = one output pixel);
//     accumulators are double-buffered in TMEM whenever MT*N <= 256 so the epilogue of tile i overlaps the MMAs of tile i+1;
//   * the epilogues fuse everything elementwise: bias, ReLU, the GRU gates (z, r*h, tanh, (1-z)h + zq), the gated global
//     context sum, sigmoid / softplus of the heads and the NCHW layout of the upsampling mask.
// Segment mean (GraphAgg's scatter_mean), the 7x7 flow encoder's im2col (4 input channels: 49 taps x 4 = one 196-wide K),
// the global-context mat-vec and the NCHW -> channels-last transposes are small SIMT kernels around it.
#include "common.cuh"
#include "tcgen05.cuh"
#include <cuda.h>
#include <string.h>

namespace dba {

enum { EPI_STORE = 0, EPI_GATE = 1, EPI_ZR = 2, EPI_Q = 3, EPI_F32 = 4, EPI_NCHW = 5 };

constexpr int kUpThreads = 320;   // warp 0 TMA, warp 1 MMA, warps 2..9 epilogue

struct ConvParams {
  int E, HT, WD;                    // images (edges or frames), image height / width
  int TW, RM, MT;                   // tile width in pixels, image rows per 128-pixel M tile (RM * TW = 128), M tiles per CTA tile
  int tiles_x, tiles_y, n_ntiles;   // CTA tiles per image, N tiles (output-channel blocks)
  int KS;                           // kernel size 1 or 3
  int nk0, nk1;                     // 64-channel K blocks taken from source 0 / source 1
  int N;                            // accumulator columns per M tile
  int w_rows;                       // rows per tap of the packed weight tensor (0: n_ntiles * N); larger when only the first N rows are used
  int boxn;                         // weight rows per TMA box
  int a_stages, b_stages, a_bytes, b_bytes;
  int nbuf;                         // TMEM accumulator buffers (2 when MT * N <= 256)
  const float* bias;                // [n_ntiles * N]
  int relu;
  __half* out; int out_stride;      // EPI_STORE / EPI_Q: channels-last f16, out[pix * out_stride + n]
  const __half* h; int h_stride;    // hidden state, channels-last (EPI_GATE, EPI_ZR, EPI_Q)
  const float* glo;                 // [E][384] global-context terms: z | r | q
  __half* z; __half* rh;            // EPI_ZR outputs [pix][128]; EPI_Q reads z
  float* partial; int slots;        // EPI_GATE: [E][slots][128] column sums of sigmoid(.) * h over 32-pixel groups
  float* f32a; int f32_cols, f32_stride;      // EPI_F32: f32 out[pix * f32_stride + n] for n < f32_cols (per-tap partial sums of the narrow heads)
  __half* nchw; int nchw_C;         // EPI_NCHW: out[(img * nchw_C + n) * HT*WD + pixel]
};

__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
               ::"r"(smem_u32(smem_dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void tma_load_3d_w(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
               ::"r"(smem_u32(smem_dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
// instruction descriptor: D = f32, A = B = f16, both K-major
__device__ __forceinline__ uint32_t umma_idesc_f16_kk(int M, int N) {
  return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_f16_ss(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ float tanh_fast(float x) { float y; asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float sigmoid_fast(float x) { return fmaf(0.5f, tanh_fast(0.5f * x), 0.5f); }
__device__ __forceinline__ uint32_t pack2(float a, float b) {
  const __half2 t = __floats2half2_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&t);
}
__device__ __forceinline__ float2 unpack2(uint32_t u) { return __half22float2(*reinterpret_cast<const __half2*>(&u)); }

// 32 consecutive f16 (64 bytes) of one pixel row
__device__ __forceinline__ void load32h(const __half* p, float (&f)[32]) {
  const uint4* q = reinterpret_cast<const uint4*>(p);
#pragma unroll
  for (int i = 0; i < 4; i++) {
    const uint4 u = __ldg(q + i);
    float2 a = unpack2(u.x), b = unpack2(u.y), c = unpack2(u.z), d = unpack2(u.w);
    f[8 * i + 0] = a.x; f[8 * i + 1] = a.y; f[8 * i + 2] = b.x; f[8 * i + 3] = b.y;
    f[8 * i + 4] = c.x; f[8 * i + 5] = c.y; f[8 * i + 6] = d.x; f[8 * i + 7] = d.y;
  }
}
__device__ __forceinline__ void store32h(__half* p, const float (&f)[32]) {
  uint4* q = reinterpret_cast<uint4*>(p);
#pragma unroll
  for (int i = 0; i < 4; i++)
    q[i] = make_uint4(pack2(f[8 * i], f[8 * i + 1]), pack2(f[8 * i + 2], f[8 * i + 3]), pack2(f[8 * i + 4], f[8 * i + 5]), pack2(f[8 * i + 6], f[8 * i + 7]));
}

// column sums over the 32 lanes of a warp: on return lane l holds sum_lanes v[l] (31 shuffles instead of 160)
__device__ __forceinline__ float warp_column_sums(float (&v)[32], int lane) {
#pragma unroll
  for (int j = 0; j < 16; j++) {
    const bool up = lane & 16;
    const float send = up ? v[j] : v[j + 16];
    const float keep = up ? v[j + 16] : v[j];
    v[j] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
  }
#pragma unroll
  for (int j = 0; j < 8; j++) {
    const bool up = lane & 8;
    const float send = up ? v[j] : v[j + 8];
    const float keep = up ? v[j + 8] : v[j];
    v[j] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
  }
#pragma unroll
  for (int j = 0; j < 4; j++) {
    const bool up = lane & 4;
    const float send = up ? v[j] : v[j + 4];
    const float keep = up ? v[j + 4] : v[j];
    v[j] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
  }
#pragma unroll
  for (int j = 0; j < 2; j++) {
    const bool up = lane & 2;
    const float send = up ? v[j] : v[j + 2];
    const float keep = up ? v[j + 2] : v[j];
    v[j] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
  }
  {
    const bool up = lane & 1;
    const float send = up ? v[0] : v[1];
    const float keep = up ? v[1] : v[0];
    v[0] = keep + __shfl_xor_sync(0xffffffffu, send, 1);
  }
  return v[0];
}

// epilogue of one CTA tile (MT x 128 pixels x this warp's column range) out of the TMEM accumulator buffer `buf`
template <int EPI>
__device__ __forceinline__ void conv_epilogue_tile(const ConvParams& p, uint32_t tmem_base, uint32_t buf, int q, int lane, int c_begin, int c_end, int my, int mx,
                                                   int nt, int e, int ty, int tx) {
  for (int t = 0; t < p.MT; t++) {
    const int y = ty * (p.MT * p.RM) + t * p.RM + my, x = tx * p.TW + mx;
    const bool valid = y < p.HT && x < p.WD;
    const size_t pix = ((size_t)e * p.HT + (valid ? y : 0)) * p.WD + (valid ? x : 0);
    for (int c0 = c_begin; c0 < c_end; c0 += 32) {
      uint32_t raw[32];
      tmem_ld32(tmem_base + buf * 256 + t * p.N + c0 + ((uint32_t)(q * 32) << 16), raw);
      asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
      float v[32];
      const float* bias = p.bias + nt * p.N + c0;
#pragma unroll
      for (int j = 0; j < 32; j++) v[j] = __uint_as_float(raw[j]) + __ldg(bias + j);

      if (EPI == EPI_STORE) {
        if (p.relu) {
#pragma unroll
          for (int j = 0; j < 32; j++) v[j] = fmaxf(v[j], 0.f);
        }
        if (valid) store32h(p.out + pix * p.out_stride + c0, v);
      } else if (EPI == EPI_GATE) {
        float hh[32];
        if (valid) load32h(p.h + pix * p.h_stride + c0, hh);
#pragma unroll
        for (int j = 0; j < 32; j++) v[j] = valid ? sigmoid_fast(v[j]) * hh[j] : 0.f;
        const float s = warp_column_sums(v, lane);
        const int slot = ((ty * p.tiles_x + tx) * p.MT + t) * 4 + q;
        p.partial[((size_t)e * p.slots + slot) * 128 + c0 + lane] = s;
      } else if (EPI == EPI_ZR) {
        const float* g = p.glo + (size_t)e * 384 + c0;
#pragma unroll
        for (int j = 0; j < 32; j++) v[j] = sigmoid_fast(v[j] + __ldg(g + j));
        if (c0 < 128) {
          if (valid) store32h(p.z + pix * 128 + c0, v);
        } else {
          float hh[32];
          if (valid) {
            load32h(p.h + pix * p.h_stride + (c0 - 128), hh);
#pragma unroll
            for (int j = 0; j < 32; j++) v[j] *= hh[j];
            store32h(p.rh + pix * 128 + (c0 - 128), v);
          }
        }
      } else if (EPI == EPI_Q) {
        const float* g = p.glo + (size_t)e * 384 + 256 + c0;
        if (valid) {
          float hh[32], zz[32];
          load32h(p.h + pix * p.h_stride + c0, hh);
          load32h(p.z + pix * 128 + c0, zz);
#pragma unroll
          for (int j = 0; j < 32; j++) {
            const float qq = tanh_fast(v[j] + __ldg(g + j));
            v[j] = (1.f - zz[j]) * hh[j] + zz[j] * qq;
          }
          store32h(p.out + pix * p.out_stride + c0, v);
        }
      } else if (EPI == EPI_F32) {
        if (valid) {
          float* o = p.f32a + pix * p.f32_stride + c0;
#pragma unroll
          for (int j = 0; j < 32; j += 4)
            if (c0 + j < p.f32_cols) *reinterpret_cast<float4*>(o + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);     // f32_cols, f32_stride: multiples of 4
        }
      } else if (EPI == EPI_NCHW) {
        if (valid) {
          const size_t HW = (size_t)p.HT * p.WD;
          __half* o = p.nchw + ((size_t)e * p.nchw_C + nt * p.N + c0) * HW + (size_t)y * p.WD + x;
#pragma unroll
          for (int j = 0; j < 32; j++) o[j * HW] = __float2half_rn(v[j]);
        }
      }
    }
  }
}

template <int EPI>
__global__ void __launch_bounds__(kUpThreads, 1) conv_tc_kernel(const __grid_constant__ CUtensorMap tmA0, const __grid_constant__ CUtensorMap tmA1,
                                                               const __grid_constant__ CUtensorMap tmW, const ConvParams p) {
  extern __shared__ uint8_t up_smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(up_smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sA = smem;
  uint8_t* sB = smem + p.a_stages * p.a_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sB + p.b_stages * p.b_bytes);
  uint64_t* a_full = bars;              // [4]
  uint64_t* a_empty = bars + 4;         // [4]
  uint64_t* b_full = bars + 8;          // [8]
  uint64_t* b_empty = bars + 16;        // [8]
  uint64_t* tmem_full = bars + 24;      // [2]
  uint64_t* tmem_empty = bars + 26;     // [2]
  uint32_t* tmem_base_smem = reinterpret_cast<uint32_t*>(bars + 28);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tiles_per_img = p.tiles_x * p.tiles_y;
  const int total_tiles = p.n_ntiles * p.E * tiles_per_img;
  const int nk = p.nk0 + p.nk1;
  const int pad = p.KS >> 1;

  if (threadIdx.x == 0) {
    for (int s = 0; s < p.a_stages; s++) { mbar_init(a_full + s, 1); mbar_init(a_empty + s, 1); }
    for (int s = 0; s < p.b_stages; s++) { mbar_init(b_full + s, 1); mbar_init(b_empty + s, 1); }
    for (int s = 0; s < 2; s++) { mbar_init(tmem_full + s, 1); mbar_init(tmem_empty + s, 8); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_base_smem)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_base_smem;

  if (warp == 0) {
    // ================= TMA producer (one thread) =================
    if (lane == 0) {
      uint32_t ac = 0, bc = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const int nt = tile / (p.E * tiles_per_img);
        const int r0 = tile - nt * (p.E * tiles_per_img);
        const int e = r0 / tiles_per_img;
        const int r1 = r0 - e * tiles_per_img;
        const int ty = r1 / p.tiles_x, tx = r1 - ty * p.tiles_x;
        const int y0 = ty * (p.MT * p.RM), x0 = tx * p.TW;
        for (int kb = 0; kb < nk; kb++) {
          const CUtensorMap* am = kb < p.nk0 ? &tmA0 : &tmA1;
          const int ch = (kb < p.nk0 ? kb : kb - p.nk0) * 64;
          for (int dx = 0; dx < p.KS; dx++) {
            const int as = ac % p.a_stages;
            mbar_wait(a_empty + as, ((ac / p.a_stages) & 1) ^ 1);
            mbar_expect_tx(a_full + as, p.a_bytes);
            tma_load_4d(sA + as * p.a_bytes, am, a_full + as, ch, x0 + dx - pad, y0 - pad, e);
            ac++;
            for (int dy = 0; dy < p.KS; dy++) {
              const int bs = bc % p.b_stages;
              mbar_wait(b_empty + bs, ((bc / p.b_stages) & 1) ^ 1);
              mbar_expect_tx(b_full + bs, p.b_bytes);
              for (int n = 0; n < p.N; n += p.boxn)
                tma_load_3d_w(sB + bs * p.b_bytes + n * 128, &tmW, b_full + bs, kb * 64, nt * p.N + n, dy * p.KS + dx);
              bc++;
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer =================
    const int n_c0 = p.N > 256 ? 256 : p.N, n_c1 = p.N - n_c0;
    const uint32_t idesc0 = umma_idesc_f16_kk(128, n_c0);
    const uint32_t idesc1 = n_c1 ? umma_idesc_f16_kk(128, n_c1) : 0u;
    const uint32_t sA_u = smem_u32(sA), sB_u = smem_u32(sB);
    uint32_t ac = 0, bc = 0, it = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, it++) {
      const uint32_t buf = it % p.nbuf;
      mbar_wait(tmem_empty + buf, ((it / p.nbuf) & 1) ^ 1);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t tcol = tmem_base + buf * 256;
      bool first = true;
      for (int kb = 0; kb < nk; kb++) {
        for (int dx = 0; dx < p.KS; dx++) {
          const int as = ac % p.a_stages;
          mbar_wait(a_full + as, (ac / p.a_stages) & 1);
          for (int dy = 0; dy < p.KS; dy++) {
            const int bs = bc % p.b_stages;
            mbar_wait(b_full + bs, (bc / p.b_stages) & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            if (lane == 0) {
              const uint32_t b_base = sB_u + bs * p.b_bytes;
              for (int t = 0; t < p.MT; t++) {
                const uint32_t a_base = sA_u + as * p.a_bytes + (uint32_t)((t * p.RM + dy) * p.TW) * 128u;
#pragma unroll
                for (int k = 0; k < 4; k++) {
                  const uint32_t acc = (first && k == 0) ? 0u : 1u;
                  const uint64_t ad = umma_desc_k_sw128(a_base + k * 32, 1024);
                  umma_f16_ss(tcol + t * p.N, ad, umma_desc_k_sw128(b_base + k * 32, 1024), idesc0, acc);
                  if (n_c1) umma_f16_ss(tcol + t * p.N + 256, ad, umma_desc_k_sw128(b_base + 256 * 128 + k * 32, 1024), idesc1, acc);
                }
              }
              umma_commit(b_empty + bs);
            }
            __syncwarp();
            first = false;
            bc++;
          }
          if (lane == 0) umma_commit(a_empty + as);
          __syncwarp();
          ac++;
        }
      }
      if (lane == 0) umma_commit(tmem_full + buf);
      __syncwarp();
    }
  } else {
    // ================= epilogue: warps 2..9; TMEM lane quarter q = warp % 4, the two warps of a quarter split the columns =================
    const int q = warp & 3;
    const int half = (warp - 2) >> 2;
    const int cols_per_half = p.N >= 64 ? p.N / 2 : p.N;
    const int c_begin = half * cols_per_half;
    const int c_end = (p.N >= 64 || half == 0) ? c_begin + cols_per_half : c_begin;
    const int m = q * 32 + lane;
    const int my = m / p.TW, mx = m - my * p.TW;
    uint32_t it = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, it++) {
      const int nt = tile / (p.E * tiles_per_img);
      const int r0 = tile - nt * (p.E * tiles_per_img);
      const int e = r0 / tiles_per_img;
      const int r1 = r0 - e * tiles_per_img;
      const int ty = r1 / p.tiles_x, tx = r1 - ty * p.tiles_x;
      const uint32_t buf = it % p.nbuf;
      mbar_wait(tmem_full + buf, (it / p.nbuf) & 1);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      conv_epilogue_tile<EPI>(p, tmem_base, buf, q, lane, c_begin, c_end, my, mx, nt, e, ty, tx);
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) mbar_arrive(tmem_empty + buf);
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
}

// ---------------------------------------------------------------------------------------------------------------------------
// small SIMT kernels around the tensor-core convolutions
// ---------------------------------------------------------------------------------------------------------------------------

// [E][C][HW] (f16 or f32) -> channels-last f16 dst[(e*HW + p) * dst_stride + c] for c < cwrite (channels C..cwrite-1 are zeros).
// 64 channels x 64 pixels per CTA; a thread loads a 2 x 2 (channel pair x pixel pair) patch, transposes it in registers and parks
// the two channel-pair words in shared memory, so that both the global loads (pixel pairs of one channel row) and the global stores
// (channel pairs of one pixel) are 4-byte lanes of 128-byte rows.
template <typename T> struct Load2;
template <> struct Load2<__half> {
  static __device__ __forceinline__ float2 ld(const __half* p, bool ok0, bool ok1, bool aligned) {
    if (ok1 && aligned) return __half22float2(*reinterpret_cast<const __half2*>(p));
    return make_float2(ok0 ? __half2float(p[0]) : 0.f, ok1 ? __half2float(p[1]) : 0.f);
  }
};
template <> struct Load2<float> {
  static __device__ __forceinline__ float2 ld(const float* p, bool ok0, bool ok1, bool aligned) {
    if (ok1 && aligned) return *reinterpret_cast<const float2*>(p);
    return make_float2(ok0 ? p[0] : 0.f, ok1 ? p[1] : 0.f);
  }
};
template <typename T>
__global__ void __launch_bounds__(256) nchw_to_nhwc_kernel(const T* __restrict__ src, __half* __restrict__ dst, int C, int HW, int dst_stride, int cwrite) {
  __shared__ uint32_t tile[2][64][33];                      // [channel block][pixel][channel pair]
  // a CTA moves TWO 64-channel blocks of a 64-pixel tile: 16 loads per thread are in flight before the first use, and a pixel's
  // output row is one 256-byte run
  const int e = blockIdx.z, p0 = blockIdx.x * 64;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const bool even = (HW & 1) == 0;                           // pixel pairs are 4 / 8-byte aligned when HW is even
  float2 va[2][4], vb[2][4];
#pragma unroll
  for (int cbk = 0; cbk < 2; cbk++) {
    const int c0 = (blockIdx.y * 2 + cbk) * 64;
#pragma unroll
    for (int k = 0; k < 4; k++) {
      const int cp = w + 8 * k;                              // channel pair 0..31
      const int c = c0 + 2 * cp, pp = p0 + 2 * lane;
      va[cbk][k] = make_float2(0.f, 0.f); vb[cbk][k] = make_float2(0.f, 0.f);
      if (c < C && pp < HW) va[cbk][k] = Load2<T>::ld(src + ((size_t)e * C + c) * HW + pp, true, pp + 1 < HW, even);
      if (c + 1 < C && pp < HW) vb[cbk][k] = Load2<T>::ld(src + ((size_t)e * C + c + 1) * HW + pp, true, pp + 1 < HW, even);
    }
  }
#pragma unroll
  for (int cbk = 0; cbk < 2; cbk++)
#pragma unroll
    for (int k = 0; k < 4; k++) {
      const int cp = w + 8 * k;
      tile[cbk][2 * lane][cp] = pack2(va[cbk][k].x, vb[cbk][k].x);
      tile[cbk][2 * lane + 1][cp] = pack2(va[cbk][k].y, vb[cbk][k].y);
    }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < 8; k++) {
    const int px = w + 8 * k, pp = p0 + px;
#pragma unroll
    for (int cbk = 0; cbk < 2; cbk++) {
      const int c = (blockIdx.y * 2 + cbk) * 64 + 2 * lane;
      if (pp < HW && c < cwrite) *reinterpret_cast<uint32_t*>(dst + ((size_t)e * HW + pp) * dst_stride + c) = tile[cbk][px][lane];   // cwrite and strides are even
    }
  }
}

// 7x7 / 4-channel flow encoder input as one 196-wide K: dst[(e*HW + p) * 200 + (dy*7+dx)*4 + c] = flow[e][c][y+dy-3][x+dx-3] (0 outside;
// slot 49 = the 4 zero padding channels).  CTA = 64 pixels of one image row: the 4 x 7 x 70 halo goes through shared memory
// (coalesced row loads), the 64 x 400-byte output rows leave as consecutive 8-byte lanes.
__global__ void __launch_bounds__(256) flow_im2col_kernel(const float* __restrict__ flow, __half* __restrict__ dst, int HT, int WD) {
  __shared__ float halo[4][7][72];
  const int e = blockIdx.z, y = blockIdx.y, x0 = blockIdx.x * 64;
  const int HW = HT * WD;
  for (int i = threadIdx.x; i < 4 * 7 * 70; i += 256) {
    const int c = i / 490, r = (i - c * 490) / 70, col = i - c * 490 - r * 70;
    const int yy = y + r - 3, xx = x0 + col - 3;
    float v = 0.f;
    if (flow && yy >= 0 && yy < HT && xx >= 0 && xx < WD) v = __ldg(flow + ((size_t)e * 4 + c) * HW + (size_t)yy * WD + xx);
    halo[c][r][col] = v;
  }
  __syncthreads();
  const int npx = min(64, WD - x0);
  __half* out = dst + ((size_t)e * HW + (size_t)y * WD + x0) * 200;
  for (int i = threadIdx.x; i < npx * 50; i += 256) {
    const int px = i / 50, slot = i - px * 50;
    uint2 o = make_uint2(0u, 0u);
    if (slot < 49) {
      const int dy = slot / 7, dx = slot - dy * 7;
      o = make_uint2(pack2(halo[0][dy][px + dx], halo[1][dy][px + dx]), pack2(halo[2][dy][px + dx], halo[3][dy][px + dx]));
    }
    *reinterpret_cast<uint2*>(out + (size_t)i * 4) = o;
  }
}

// The 3x3 convolutions with 1-2 output channels (delta.2, weight.2, agg.eta.0) are computed as ONE 1x1 convolution that produces, per
// pixel, the 9 per-tap partial sums of every output (Y[p][t*no + o] = sum_c act[p][c] w[t][o][c]; on the tensor cores, the input is read
// once instead of three times), followed by this gather: out[p][o] = bias[o] + sum_t Y[p + shift_t][t*no + o] (zero outside the image).
// mode 0: no = 4 -> delta (o = 0,1) and sigmoid weight (o = 2,3), [img,ht,wd,2] each;  mode 1: no = 1 -> eta = 0.01 * softplus
__global__ void __launch_bounds__(256) head_gather_kernel(const float* __restrict__ Y, int ystride, int no, const float* __restrict__ bias, int mode,
                                                          float* __restrict__ out_a, float* __restrict__ out_b, int n_img, int HT, int WD) {
  const long long total = (long long)n_img * HT * WD;
  const long long id = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= total) return;
  const int HW = HT * WD;
  const int pin = (int)(id % HW);
  const long long img = id / HW;
  const int y = pin / WD, x = pin - y * WD;
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int t = 0; t < 9; t++) {
    const int yy = y + t / 3 - 1, xx = x + t % 3 - 1;
    if (yy < 0 || yy >= HT || xx < 0 || xx >= WD) continue;
    const float* q = Y + ((size_t)img * HW + (size_t)yy * WD + xx) * ystride + t * no;
    if (no == 4) { const float4 v = __ldg(reinterpret_cast<const float4*>(q)); acc[0] += v.x; acc[1] += v.y; acc[2] += v.z; acc[3] += v.w; }
    else acc[0] += __ldg(q);
  }
  if (mode == 0) {
    *reinterpret_cast<float2*>(out_a + (size_t)id * 2) = make_float2(acc[0] + bias[0], acc[1] + bias[1]);
    *reinterpret_cast<float2*>(out_b + (size_t)id * 2) = make_float2(1.f / (1.f + __expf(-(acc[2] + bias[2]))), 1.f / (1.f + __expf(-(acc[3] + bias[3]))));
  } else {
    const float xx = acc[0] + bias[0];
    out_a[id] = 0.01f * (xx > 20.f ? xx : log1pf(__expf(xx)));     // torch Softplus(beta = 1, threshold = 20)
  }
}

// global context (gru.py:25-30): g = mean over pixels of sigmoid(w(h)) * h (from the EPI_GATE partial sums), then the three 1x1
// convolutions on g as one [384 x 128] mat-vec per edge -> glo[e][384] = z | r | q terms
__global__ void __launch_bounds__(384) glo_kernel(const float* __restrict__ partial, int slots, float inv_hw, const float* __restrict__ wg /*[384][128]*/,
                                                  const float* __restrict__ bg, float* __restrict__ glo) {
  __shared__ float g[128];
  const int e = blockIdx.x;
  if (threadIdx.x < 128) {
    float s = 0.f;
    for (int k = 0; k < slots; k++) s += partial[((size_t)e * slots + k) * 128 + threadIdx.x];
    g[threadIdx.x] = s * inv_hw;
  }
  __syncthreads();
  const float* w = wg + (size_t)threadIdx.x * 128;
  float acc = bg[threadIdx.x];
#pragma unroll 8
  for (int k = 0; k < 128; k++) acc = fmaf(__ldg(w + k), g[k], acc);
  glo[(size_t)e * 384 + threadIdx.x] = acc;
}

// CSR of the edges by aggregation segment (segment = rank of the source frame among the distinct sources, ascending), edge order kept
__global__ void seg_csr_kernel(const int64_t* __restrict__ ix, int E, int n_seg, int* __restrict__ seg_ptr, int* __restrict__ seg_edges) {
  extern __shared__ int cnt[];
  for (int s = threadIdx.x; s < n_seg; s += blockDim.x) {
    int c = 0;
    for (int e = 0; e < E; e++) c += ((int)ix[e] == s);
    cnt[s] = c;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int a = 0;
    for (int s = 0; s < n_seg; s++) { seg_ptr[s] = a; a += cnt[s]; }
    seg_ptr[n_seg] = a;
  }
  __syncthreads();
  for (int s = threadIdx.x; s < n_seg; s += blockDim.x) {
    int o = seg_ptr[s];
    for (int e = 0; e < E; e++) if ((int)ix[e] == s) seg_edges[o++] = e;
  }
}

// scatter_mean over edges with equal source frame (droid_net.py:63-67): src channels-last with stride src_stride, dst [n_seg][HW][128]
__global__ void __launch_bounds__(256) segment_mean_kernel(const __half* __restrict__ src, int src_stride, const int* __restrict__ seg_ptr,
                                                           const int* __restrict__ seg_edges, __half* __restrict__ dst, int HW) {
  const int s = blockIdx.y;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;     // (pixel, 8-channel group)
  if (i >= HW * 16) return;
  const int pp = i >> 4, cg = (i & 15) * 8;
  const int b = seg_ptr[s], en = seg_ptr[s + 1];
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (int k = b; k < en; k++) {
    const int e = seg_edges[k];
    const uint4 u = __ldg(reinterpret_cast<const uint4*>(src + ((size_t)e * HW + pp) * src_stride + cg));
    float2 a = unpack2(u.x), bb = unpack2(u.y), c = unpack2(u.z), d = unpack2(u.w);
    acc[0] += a.x; acc[1] += a.y; acc[2] += bb.x; acc[3] += bb.y; acc[4] += c.x; acc[5] += c.y; acc[6] += d.x; acc[7] += d.y;
  }
  const float inv = en > b ? 1.f / (float)(en - b) : 0.f;
  *reinterpret_cast<uint4*>(dst + ((size_t)s * HW + pp) * 128 + cg) =
      make_uint4(pack2(acc[0] * inv, acc[1] * inv), pack2(acc[2] * inv, acc[3] * inv), pack2(acc[4] * inv, acc[5] * inv), pack2(acc[6] * inv, acc[7] * inv));
}

// ---------------------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------------------
// activation map: channels-last f16 [E][HT][WD][stride], channels [0, C) of the slice starting at `base`
static int make_act_map(CUtensorMap* map, const void* base, int C, int stride, int WD, int HT, int E, int TW, int box_rows) {
  EncodeTiledFn enc = tensor_map_encoder();
  if (!enc) { set_error("cuTensorMapEncodeTiled entry point not available"); return DBA_ERR_CUDA; }
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)WD, (cuuint64_t)HT, (cuuint64_t)E};
  cuuint64_t strides[3] = {(cuuint64_t)stride * 2, (cuuint64_t)WD * stride * 2, (cuuint64_t)HT * WD * stride * 2};
  cuuint32_t box[4] = {64, (cuuint32_t)TW, (cuuint32_t)box_rows, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled (activation, C=%d stride=%d %dx%d E=%d box %dx%d) failed with CUresult %d", C, stride, HT, WD, E, TW, box_rows, (int)r); return DBA_ERR_CUDA; }
  return DBA_OK;
}
// weight map: [taps][Ntot][Kpad] f16
static int make_weight_map(CUtensorMap* map, const void* base, int Kpad, int Ntot, int taps, int boxn) {
  EncodeTiledFn enc = tensor_map_encoder();
  if (!enc) { set_error("cuTensorMapEncodeTiled entry point not available"); return DBA_ERR_CUDA; }
  cuuint64_t dims[3] = {(cuuint64_t)Kpad, (cuuint64_t)Ntot, (cuuint64_t)taps};
  cuuint64_t strides[2] = {(cuuint64_t)Kpad * 2, (cuuint64_t)Ntot * Kpad * 2};
  cuuint32_t box[3] = {64, (cuuint32_t)boxn, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled (weights K=%d N=%d taps=%d) failed with CUresult %d", Kpad, Ntot, taps, (int)r); return DBA_ERR_CUDA; }
  return DBA_OK;
}

struct ConvSrc { const void* base; int C; int stride; };

// one convolution launch.  src0 (+ optional src1) = channels-last sources concatenated along K; wpk = packed weights
// [KS*KS][n_ntiles*N][Kpad] with Kpad = 64 * (kblocks(src0) + kblocks(src1)).
template <int EPI>
static int launch_conv(ConvParams p, ConvSrc s0, ConvSrc s1, const void* wpk, cudaStream_t st, int* slots_out = nullptr) {
  DeviceInfo dev;
  int rc = device_info(&dev); if (rc) return rc;
  p.TW = (p.WD % 64 == 0) ? 64 : 32;
  p.RM = 128 / p.TW;
  // M tiles per CTA tile: every weight stage is shared by MT tiles (and every halo row by 3 taps), so larger is better for the
  // L2 -> SM traffic per MAC; bounded by TMEM (MT * N <= 512 columns) and by the image height
  p.MT = (p.N <= 256 && p.HT >= 2 * p.RM) ? 2 : 1;
  // N <= 128 with a long K loop (the q convolution): 4 tiles per weight stage beat the overlapped epilogue of 2 (measured:
  // profiles/r2_conv_pipeline_experiments.txt); short K loops keep the double-buffered accumulators
  if (p.N <= 128 && p.HT >= 4 * p.RM && (s0.C + 63) / 64 + (s1.base ? (s1.C + 63) / 64 : 0) >= 4 && p.KS == 3) p.MT = 4;
  p.tiles_x = (p.WD + p.TW - 1) / p.TW;
  p.tiles_y = (p.HT + p.MT * p.RM - 1) / (p.MT * p.RM);
  p.nk0 = (s0.C + 63) / 64;
  p.nk1 = s1.base ? (s1.C + 63) / 64 : 0;
  p.boxn = p.N <= 256 ? p.N : 128;
  p.nbuf = (p.MT * p.N <= 256) ? 2 : 1;
  const int box_rows = p.MT * p.RM + p.KS - 1;
  p.a_bytes = box_rows * p.TW * 128;
  p.b_bytes = p.N * 128;
  // shared memory: at least 2 halo stages and 3 weight stages; what is left goes to more halo stages (up to 4: with narrow N the
  // MMAs of a stage are short and the TMA latency of the next halo tile is what the pipeline has to cover), then weight stages
  const int budget = 227 * 1024 - 2048;
  p.a_stages = 2;
  while (p.a_stages < 4 && (p.a_stages + 1) * p.a_bytes + 4 * p.b_bytes <= budget) p.a_stages++;
  p.b_stages = (budget - p.a_stages * p.a_bytes) / p.b_bytes;
  if (p.b_stages > 8) p.b_stages = 8;
  if (p.b_stages < 2) { set_error("update operator: tile does not fit shared memory"); return DBA_ERR_INVALID; }
  p.slots = p.tiles_x * p.tiles_y * p.MT * 4;
  if (slots_out) *slots_out = p.slots;
  const int smem = p.a_stages * p.a_bytes + p.b_stages * p.b_bytes + 1024 + 256;
  CUtensorMap tA0, tA1, tW;
  rc = make_act_map(&tA0, s0.base, s0.C, s0.stride, p.WD, p.HT, p.E, p.TW, box_rows); if (rc) return rc;
  if (s1.base) { rc = make_act_map(&tA1, s1.base, s1.C, s1.stride, p.WD, p.HT, p.E, p.TW, box_rows); if (rc) return rc; }
  else tA1 = tA0;
  rc = make_weight_map(&tW, wpk, 64 * (p.nk0 + p.nk1), p.w_rows > 0 ? p.w_rows : p.n_ntiles * p.N, p.KS * p.KS, p.boxn); if (rc) return rc;
  rc = kernel_setup((const void*)conv_tc_kernel<EPI>, 227 * 1024); if (rc) return rc;
  const long long total = (long long)p.n_ntiles * p.E * p.tiles_x * p.tiles_y;
  if (total <= 0) return DBA_OK;
  const int grid = (int)(total < dev.num_sms ? total : dev.num_sms);
  conv_tc_kernel<EPI><<<grid, kUpThreads, smem, st>>>(tA0, tA1, tW, p);
  DBA_CHECK_LAUNCH("conv_tc_kernel");
  return DBA_OK;
}

static size_t al256(size_t x) { return (x + 255) & ~(size_t)255; }

struct UpWs {
  size_t hin, x320, cc, f0, c1, f1, z, rh, s, partial, glo, am, b2, segptr, segedges, total;
};
static UpWs up_layout(int E, int n_src, int ht, int wd) {
  UpWs w;
  const size_t px = (size_t)E * ht * wd, spx = (size_t)(n_src > 0 ? n_src : 1) * ht * wd;
  const int tw = (wd % 64 == 0) ? 64 : 32, rm = 128 / tw;
  const size_t slots = (size_t)((wd + tw - 1) / tw) * ((ht + rm - 1) / rm) * 4 * 2;   // upper bound over MT
  size_t o = 0;
  w.hin = o; o += al256(px * 128 * 2);
  w.x320 = o; o += al256(px * 320 * 2);
  w.cc = o; o += al256(px * 200 * 2);
  w.f0 = o; o += al256(px * 200 * 2);
  w.c1 = o; o += al256(px * 128 * 2);
  w.f1 = o; o += al256(px * 128 * 2);
  w.z = o; o += al256(px * 128 * 2);
  w.rh = o; o += al256(px * 128 * 2);
  w.s = o; o += al256(px * 384 * 2);
  w.partial = o; o += al256((size_t)E * slots * 128 * 4);
  w.glo = o; o += al256((size_t)E * 384 * 4);
  w.am = o; o += al256(spx * 128 * 2);
  w.b2 = o; o += al256(spx * 128 * 2);
  w.segptr = o; o += al256((size_t)(n_src + 2) * 4);
  w.segedges = o; o += al256((size_t)(E + 1) * 4);
  w.total = o;
  return w;
}

}  // namespace dba
using namespace dba;

extern "C" size_t dba_update_workspace_bytes(int n_edges, int n_src, int ht, int wd) {
  if (n_edges <= 0 || ht <= 0 || wd <= 0) return 0;
  return up_layout(n_edges, n_src, ht, wd).total;
}

extern "C" int dba_update_forward(const dba_update_args* a) {
  DBA_CHECK_ARG(a, "null args");
  const int E = a->n_edges, ht = a->ht, wd = a->wd, n_src = a->n_src;
  DBA_CHECK_ARG(E >= 0 && ht > 0 && wd > 0 && n_src >= 0, "bad extents");
  if (E == 0) return DBA_OK;
  DBA_CHECK_ARG(a->net && a->inp && a->corr && a->net_out && a->delta && a->weight && a->weights && a->workspace, "null pointer");
  DBA_CHECK_ARG(n_src == 0 || (a->seg && a->eta && a->upmask), "aggregation outputs / segment ids missing");
  DBA_CHECK_ARG(wd % 8 == 0, "update operator: image width must be a multiple of 8");
  const UpWs L = up_layout(E, n_src, ht, wd);
  DBA_CHECK_ARG(a->workspace_bytes >= L.total, "workspace too small (dba_update_workspace_bytes)");
  DBA_CHECK_ARG(((uintptr_t)a->workspace & 255) == 0 && ((uintptr_t)a->net_out & 15) == 0 && ((uintptr_t)a->net & 15) == 0, "pointers must be 16-byte aligned (workspace 256)");
  cudaStream_t st = (cudaStream_t)a->stream;
  uint8_t* ws = (uint8_t*)a->workspace;
  const dba_update_weights* W = a->weights;
  const int HW = ht * wd;
  __half* X = (__half*)(ws + L.x320);
  __half* Cc = (__half*)(ws + L.cc);
  __half* F0 = (__half*)(ws + L.f0);
  __half* C1 = (__half*)(ws + L.c1);
  __half* F1 = (__half*)(ws + L.f1);
  __half* Z = (__half*)(ws + L.z);
  __half* RH = (__half*)(ws + L.rh);
  __half* S = (__half*)(ws + L.s);
  float* partial = (float*)(ws + L.partial);
  float* glo = (float*)(ws + L.glo);
  __half* Am = (__half*)(ws + L.am);
  __half* B2 = (__half*)(ws + L.b2);
  int* seg_ptr = (int*)(ws + L.segptr);
  int* seg_edges = (int*)(ws + L.segedges);

  // ---- layout changes into channels-last f16 --------------------------------------------------------------------------
  const dim3 tgrid128((HW + 63) / 64, 1, E);
  const __half* H;      // hidden state, channels-last [E][HW][128]
  if (a->net_layout == 1) H = (const __half*)a->net;
  else {
    __half* hin = (__half*)(ws + L.hin);
    if (a->net_dtype == DBA_F16) nchw_to_nhwc_kernel<__half><<<tgrid128, 256, 0, st>>>((const __half*)a->net, hin, 128, HW, 128, 128);
    else if (a->net_dtype == DBA_F32) nchw_to_nhwc_kernel<float><<<tgrid128, 256, 0, st>>>((const float*)a->net, hin, 128, HW, 128, 128);
    else { set_error("invalid argument: net dtype must be f16 or f32"); return DBA_ERR_INVALID; }
    H = hin;
  }
  // inp -> X[:, 0:128] (X = inp | corr features | flow features, 320 channels)
  if (a->inp_dtype == DBA_F16) nchw_to_nhwc_kernel<__half><<<tgrid128, 256, 0, st>>>((const __half*)a->inp, X, 128, HW, 320, 128);
  else if (a->inp_dtype == DBA_F32) nchw_to_nhwc_kernel<float><<<tgrid128, 256, 0, st>>>((const float*)a->inp, X, 128, HW, 320, 128);
  else { set_error("invalid argument: inp dtype must be f16 or f32"); return DBA_ERR_INVALID; }
  {
    const dim3 g((HW + 63) / 64, 2, E);
    if (a->corr_dtype == DBA_F16) nchw_to_nhwc_kernel<__half><<<g, 256, 0, st>>>((const __half*)a->corr, Cc, 196, HW, 200, 200);
    else if (a->corr_dtype == DBA_F32) nchw_to_nhwc_kernel<float><<<g, 256, 0, st>>>((const float*)a->corr, Cc, 196, HW, 200, 200);
    else { set_error("invalid argument: corr dtype must be f16 or f32"); return DBA_ERR_INVALID; }
  }
  flow_im2col_kernel<<<dim3((wd + 63) / 64, ht, E), 256, 0, st>>>(a->flow, F0, ht, wd);
  DBA_CHECK_LAUNCH("update layout kernels");

  ConvParams base;
  memset(&base, 0, sizeof(base));
  base.E = E; base.HT = ht; base.WD = wd; base.n_ntiles = 1;
  const ConvSrc none = {nullptr, 0, 0};
  int rc;
  // ---- corr_encoder: 1x1 196->128 + ReLU, 3x3 128->128 + ReLU -> X[:, 128:256]   (droid_net.py:83-87)
  { ConvParams p = base; p.KS = 1; p.N = 128; p.bias = W->b_corr0; p.relu = 1; p.out = C1; p.out_stride = 128;
    rc = launch_conv<EPI_STORE>(p, ConvSrc{Cc, 196, 200}, none, W->w_corr0, st); if (rc) return rc; }
  { ConvParams p = base; p.KS = 3; p.N = 128; p.bias = W->b_corr2; p.relu = 1; p.out = X + 128; p.out_stride = 320;
    rc = launch_conv<EPI_STORE>(p, ConvSrc{C1, 128, 128}, none, W->w_corr2, st); if (rc) return rc; }
  // ---- flow_encoder: 7x7 4->128 + ReLU (as a 196-wide 1x1 over the im2col rows), 3x3 128->64 + ReLU -> X[:, 256:320]   (:89-93)
  { ConvParams p = base; p.KS = 1; p.N = 128; p.bias = W->b_flow0; p.relu = 1; p.out = F1; p.out_stride = 128;
    rc = launch_conv<EPI_STORE>(p, ConvSrc{F0, 196, 200}, none, W->w_flow0, st); if (rc) return rc; }
  { ConvParams p = base; p.KS = 3; p.N = 64; p.bias = W->b_flow2; p.relu = 1; p.out = X + 256; p.out_stride = 320;
    rc = launch_conv<EPI_STORE>(p, ConvSrc{F1, 128, 128}, none, W->w_flow2, st); if (rc) return rc; }
  // ---- ConvGRU (gru.py:19-32): global context
  int slots = 0;
  { ConvParams p = base; p.KS = 1; p.N = 128; p.bias = W->b_gate; p.h = H; p.h_stride = 128; p.partial = partial;
    rc = launch_conv<EPI_GATE>(p, ConvSrc{H, 128, 128}, none, W->w_gate, st, &slots); if (rc) return rc; }
  glo_kernel<<<E, 384, 0, st>>>(partial, slots, 1.f / (float)HW, W->w_glo, W->b_glo, glo);
  DBA_CHECK_LAUNCH("glo_kernel");
  // z, r = sigmoid(conv3x3(h | x) + glo): one 256-output convolution; epilogue writes z and r*h
  { ConvParams p = base; p.KS = 3; p.N = 256; p.bias = W->b_zr; p.h = H; p.h_stride = 128; p.glo = glo; p.z = Z; p.rh = RH;
    rc = launch_conv<EPI_ZR>(p, ConvSrc{H, 128, 128}, ConvSrc{X, 320, 320}, W->w_zr, st); if (rc) return rc; }
  // q = tanh(conv3x3(r*h | x) + glo); h' = (1-z) h + z q
  { ConvParams p = base; p.KS = 3; p.N = 128; p.bias = W->b_q; p.h = H; p.h_stride = 128; p.glo = glo; p.z = Z;
    p.out = (__half*)a->net_out; p.out_stride = 128;
    rc = launch_conv<EPI_Q>(p, ConvSrc{RH, 128, 128}, ConvSrc{X, 320, 320}, W->w_q, st); if (rc) return rc; }
  // ---- heads: stems delta.0 | weight.0 | agg.conv1 as one 384-output convolution + ReLU (droid_net.py:95-106, :60)
  const int stemN = n_src > 0 ? 384 : 256;
  { ConvParams p = base; p.KS = 3; p.N = stemN; p.w_rows = 384; p.bias = W->b_stem; p.relu = 1; p.out = S; p.out_stride = 384;
    rc = launch_conv<EPI_STORE>(p, ConvSrc{a->net_out, 128, 128}, none, W->w_stem, st); if (rc) return rc; }
  // delta.2 and weight.2 (3x3 128->2 each): per-tap partial sums by one 1x1 convolution 256 -> 36 (block-diagonal weights), then the
  // 9-tap gather with bias / sigmoid
  float* Yh = (float*)(ws + L.cc);                        // [E,HW,36] f32 on the (dead) corr staging buffer
  { ConvParams p = base; p.KS = 1; p.N = 64; p.bias = W->b_zero; p.f32a = Yh; p.f32_cols = 36; p.f32_stride = 36;
    rc = launch_conv<EPI_F32>(p, ConvSrc{S, 256, 384}, none, W->w_heads, st); if (rc) return rc; }
  head_gather_kernel<<<(unsigned)(((size_t)E * HW + 255) / 256), 256, 0, st>>>(Yh, 36, 4, W->b_heads, 0, a->delta, a->weight, E, ht, wd);
  DBA_CHECK_LAUNCH("head_gather_kernel");
  if (n_src > 0) {
    // ---- GraphAgg (droid_net.py:59-75): segment mean over edges with equal source frame, conv2, eta, upmask
    seg_csr_kernel<<<1, 256, (size_t)n_src * sizeof(int), st>>>(a->seg, E, n_src, seg_ptr, seg_edges);
    segment_mean_kernel<<<dim3((HW * 16 + 255) / 256, n_src), 256, 0, st>>>(S + 256, 384, seg_ptr, seg_edges, Am, HW);
    DBA_CHECK_LAUNCH("segment mean");
    ConvParams fb = base; fb.E = n_src;
    { ConvParams p = fb; p.KS = 3; p.N = 128; p.bias = W->b_agg2; p.relu = 1; p.out = B2; p.out_stride = 128;
      rc = launch_conv<EPI_STORE>(p, ConvSrc{Am, 128, 128}, none, W->w_agg2, st); if (rc) return rc; }
    float* Ye = (float*)(ws + L.f0);                      // [n_src,HW,12] f32 (9 used) on the (dead) flow im2col buffer
    { ConvParams p = fb; p.KS = 1; p.N = 32; p.bias = W->b_zero; p.f32a = Ye; p.f32_cols = 12; p.f32_stride = 12;
      rc = launch_conv<EPI_F32>(p, ConvSrc{B2, 128, 128}, none, W->w_eta, st); if (rc) return rc; }
    head_gather_kernel<<<(unsigned)(((size_t)n_src * HW + 255) / 256), 256, 0, st>>>(Ye, 12, 1, W->b_eta, 1, a->eta, nullptr, n_src, ht, wd);
    DBA_CHECK_LAUNCH("head_gather_kernel(eta)");
    { ConvParams p = fb; p.KS = 1; p.N = 192; p.n_ntiles = 3; p.bias = W->b_upmask; p.nchw = (__half*)a->upmask; p.nchw_C = 576;
      rc = launch_conv<EPI_NCHW>(p, ConvSrc{B2, 128, 128}, none, W->w_upmask, st); if (rc) return rc; }
  }
  return DBA_OK;
}

// channels-last tensor-core convolution building block (the kernel behind every layer of dba_update_forward), exported for
// tests and for callers that keep activations channels-last: out[e,y,x,n] = act(bias[n] + sum_{tap,k} src[e,y+dy,x+dx,k] w[tap][n][k])
extern "C" int dba_conv_nhwc(const void* src0, int c0, int stride0, const void* src1, int c1, int stride1, const void* wpk, const float* bias,
                             void* out, int out_stride, int n_images, int ht, int wd, int ksize, int n_out, int relu, dba_stream_t stream) {
  DBA_CHECK_ARG(src0 && wpk && bias && out, "null pointer");
  DBA_CHECK_ARG(n_images >= 0 && ht > 0 && wd > 0, "bad extents");
  DBA_CHECK_ARG(ksize == 1 || ksize == 3, "kernel size must be 1 or 3");
  DBA_CHECK_ARG(n_out >= 32 && n_out <= 384 && (n_out <= 256 ? n_out % 32 == 0 : n_out == 384), "n_out must be 32..256 (multiple of 32) or 384");
  DBA_CHECK_ARG(c0 > 0 && stride0 % 8 == 0 && stride0 >= c0 && (!src1 || (c1 > 0 && stride1 % 8 == 0 && stride1 >= c1)), "row pitches must be multiples of 8 elements and hold the channels");
  DBA_CHECK_ARG(!src1 || c0 % 64 == 0, "with two sources the first must hold a multiple of 64 channels");
  DBA_CHECK_ARG(out_stride % 8 == 0 && out_stride >= n_out, "bad output stride");
  if (n_images == 0) return DBA_OK;
  ConvParams p;
  memset(&p, 0, sizeof(p));
  p.E = n_images; p.HT = ht; p.WD = wd; p.n_ntiles = 1; p.KS = ksize; p.N = n_out; p.bias = bias; p.relu = relu;
  p.out = (__half*)out; p.out_stride = out_stride;
  return launch_conv<EPI_STORE>(p, ConvSrc{src0, c0, stride0}, ConvSrc{src1, c1, stride1}, wpk, (cudaStream_t)stream);
}
