// All-pairs correlation volume + 4-level pooled pyramid in ONE pass on the 5th-gen tensor cores (tcgen05 + TMEM + TMA).
//
// Replaces CorrBlock.__init__ / CorrBlock.corr (reference droid_slam/modules/corr.py:24-38, 63-71): a cuBLAS batched GEMM
// writing the [E,HW,HW] level-0 volume followed by three avg_pool2d passes that re-read it.  Here, per edge e:
//     L0[m][n]  = fp16( (1/16) * sum_c f1[ii[e]][c][m] * f2[jj[e]][c][n] )           (fp32 accumulation in TMEM)
//     L1..L3    = 2x2 average pooling over n = (y2,x2) (ATen rounds every level to fp16 before pooling the next; here the
//                 cascade runs in fp32 on the accumulator and each level is rounded once -- closer to exact, within fp16 ulp)
// are produced by one kernel: the GEMM is write bound (2*HW^2*128 flop vs 1.33*HW^2*2 bytes per edge, ~150 flop/B, far
// below the B200 ridge), so the pyramid is computed in the epilogue from the accumulator while it is still on chip and the
// volume is written exactly once (25.1 MB/edge at 48x64 instead of ~50 MB of traffic for GEMM + 3 pooling passes).
//
// CTA = (edge, 128 source pixels m).  Warp 0: TMA producer (cp.async.bulk.tensor, 128B swizzle) -- the A tile
// [128 ch x 128 px] once, then B chunks [128 ch x 256 px] (= 4 image rows of frame j), double buffered.  Warp 1: MMA issuer,
// tcgen05.mma.cta_group::1.kind::f16, M=128, N=256, K=16 x 8, both operands MN-major straight from the [C,H,W] feature
// layout (no transposes anywhere), two 256-column fp32 accumulators in TMEM so the MMA of chunk c+1 overlaps the epilogue of
// chunk c.  Warps 2-9: epilogue, tcgen05.ld 32 lanes x 32 columns, thread = one source pixel row m x half an image row, which
// makes every pooling window thread-local (registers only); outputs leave as 256-bit stores.
#include "common.cuh"
#include "tcgen05.cuh"
#include <cuda.h>

namespace dba {

constexpr int kCvThreads = 320;          // warp 0 TMA, warp 1 MMA, warps 2..9 epilogue (two per TMEM lane quarter)
constexpr int kCvM = 128;                // source pixels per CTA
constexpr int kCvN = 256;                // target pixels per chunk (4 image rows at wd = 64)
constexpr int kCvK = 128;                // channels
constexpr int kBoxBytes = 64 * kCvK * 2; // one TMA box: 64 pixels x 128 channels fp16 = 16 KB
constexpr int kSmemA = 2 * kBoxBytes;    // 32 KB
constexpr int kSmemB = 4 * kBoxBytes;    // 64 KB per stage
constexpr int kCvSmem = kSmemA + 2 * kSmemB + 1024 /*alignment slack*/ + 256 /*barriers*/;

__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
               ::"r"(smem_u32(smem_dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}

// shared-memory matrix descriptor, MN-major, SWIZZLE_128B (cute::UMMA::SmemDescriptor): start>>4 | LBO>>4 <<16 | SBO>>4 <<32 |
// version 1 <<46 | layout_type 2 <<61.  LBO = byte distance between 64-element MN atoms, SBO = between 8-row K groups.
__device__ __forceinline__ uint64_t umma_desc_mn_sw128(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

// instruction descriptor (cute::UMMA::InstrDescriptor): c=f32, a=b=f16, both MN-major, N>>3 at bit 17, M>>4 at bit 24
__device__ __forceinline__ uint32_t umma_idesc_f16(int M, int N) {
  uint32_t d = 0;
  d |= 1u << 4;                 // c_format = F32
  d |= 1u << 15;                // a_major = MN
  d |= 1u << 16;                // b_major = MN
  d |= (uint32_t)(N >> 3) << 17;
  d |= (uint32_t)(M >> 4) << 24;
  return d;
}

__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
struct CvParams {
  const int64_t* ii; const int64_t* jj;
  __half* out0; __half* out1; __half* out2; __half* out3;
  int HW, wd, n_chunks;
  int tiled;     // levels 0 and 1 in 4x8-element tiles ([h/4][w/8][4][8], one 64-byte DRAM atom per tile) for corr_lookup_pyramid
};

__device__ __forceinline__ uint32_t pack_h2(float lo, float hi) {
  const __half2 t = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&t);
}
// 256-bit global store (sm_100: st.global.v8.b32): one full 32-byte sector per thread per instruction
__device__ __forceinline__ void st_v8(__half* dst, const uint32_t* w) {
  asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(dst), "r"(w[0]), "r"(w[1]), "r"(w[2]), "r"(w[3]), "r"(w[4]), "r"(w[5]),
               "r"(w[6]), "r"(w[7]) : "memory");
}

__global__ void __launch_bounds__(kCvThreads, 1) corr_volume_pyramid_kernel(const __grid_constant__ CUtensorMap tmA,
                                                                           const __grid_constant__ CUtensorMap tmB, CvParams p) {
  extern __shared__ uint8_t cv_smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(cv_smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sA = smem;
  uint8_t* sB = smem + kSmemA;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kSmemA + 2 * kSmemB);
  uint64_t* bar_a = bars + 0;
  uint64_t* full_b = bars + 1;       // [2]
  uint64_t* empty_b = bars + 3;      // [2]
  uint64_t* tmem_full = bars + 5;    // [2]
  uint64_t* tmem_empty = bars + 7;   // [2]
  uint32_t* tmem_base_smem = reinterpret_cast<uint32_t*>(bars + 10);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int e = blockIdx.y;
  const int m0 = blockIdx.x * kCvM;
  const int fi = (int)p.ii[e], fj = (int)p.jj[e];

  if (threadIdx.x == 0) {
    mbar_init(bar_a, 1);
    for (int s = 0; s < 2; s++) { mbar_init(full_b + s, 1); mbar_init(empty_b + s, 1); mbar_init(tmem_full + s, 1); mbar_init(tmem_empty + s, 8); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {   // TMEM: 512 columns = two 128x256 fp32 accumulators
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_base_smem)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_base_smem;

  if (warp == 0) {
    // ================= TMA producer =================
    if (lane == 0) {
      mbar_expect_tx(bar_a, kSmemA);
      tma_load_3d(sA, &tmA, bar_a, m0, 0, fi);
      tma_load_3d(sA + kBoxBytes, &tmA, bar_a, m0 + 64, 0, fi);
      for (int c = 0; c < p.n_chunks; c++) {
        const int s = c & 1;
        if (c >= 2) mbar_wait(empty_b + s, ((c >> 1) - 1) & 1);
        mbar_expect_tx(full_b + s, kSmemB);
        for (int b = 0; b < 4; b++) tma_load_3d(sB + s * kSmemB + b * kBoxBytes, &tmB, full_b + s, c * kCvN + 64 * b, 0, fj);
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer =================
    const uint32_t idesc = umma_idesc_f16(kCvM, kCvN);
    mbar_wait(bar_a, 0);
    for (int c = 0; c < p.n_chunks; c++) {
      const int s = c & 1;
      mbar_wait(full_b + s, (c >> 1) & 1);
      if (c >= 2) mbar_wait(tmem_empty + s, ((c >> 1) - 1) & 1);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      if (lane == 0) {
        const uint32_t a0 = smem_u32(sA), b0 = smem_u32(sB + s * kSmemB);
#pragma unroll
        for (int k = 0; k < kCvK / 16; k++) {
          const uint64_t ad = umma_desc_mn_sw128(a0 + k * 2048, kBoxBytes, 1024);
          const uint64_t bd = umma_desc_mn_sw128(b0 + k * 2048, kBoxBytes, 1024);
          umma_f16(tmem_base + s * kCvN, ad, bd, idesc, k > 0 ? 1u : 0u);
        }
        umma_commit(empty_b + s);     // smem stage may be refilled when these MMAs have read it
        umma_commit(tmem_full + s);   // accumulator ready for the epilogue
      }
      __syncwarp();
    }
  } else {
    // ================= epilogue: warps 2..9.  TMEM lane quarter q = warp % 4 (hardware rule); the two warps of a quarter
    // split every image row of frame j into its left / right 32 columns, so all 2x2 / 4x4 / 8x8 pooling windows stay
    // thread-local.  Pooling runs in fp32 on the accumulator values and is rounded once per level. =================
    const int q = warp & 3;
    const int half = (warp - 2) >> 2;                                  // 0: columns 0..31, 1: columns 32..63 of each image row
    const int m = m0 + q * 32 + lane;                                  // this thread's source pixel
    const int wd = p.wd;                                               // 64
    __half* o0 = p.out0 + ((size_t)e * p.HW + m) * (size_t)p.HW + half * 32;
    __half* o1 = p.out1 + ((size_t)e * p.HW + m) * (size_t)(p.HW / 4) + half * 16;
    __half* o2 = p.out2 + ((size_t)e * p.HW + m) * (size_t)(p.HW / 16) + half * 8;
    __half* o3 = p.out3 + ((size_t)e * p.HW + m) * (size_t)(p.HW / 64) + half * 4;
    const float sc = 0.0625f;                                          // (f1/4).(f2/4)
    float l2prev[8];
    for (int c = 0; c < p.n_chunks; c++) {
      const int s = c & 1;
      mbar_wait(tmem_full + s, (c >> 1) & 1);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t tbase = tmem_base + s * kCvN + ((uint32_t)(q * 32) << 16) + half * 32;
      float l1f[2][16];
#pragma unroll
      for (int rp = 0; rp < 2; rp++) {                                 // image rows 4c + 2rp, 4c + 2rp + 1
        uint32_t ra[32], rb[32];
        tmem_ld32(tbase + (2 * rp) * 64, ra);
        tmem_ld32(tbase + (2 * rp + 1) * 64, rb);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        uint32_t wa[16], wb[16];
#pragma unroll
        for (int k = 0; k < 16; k++) {
          wa[k] = pack_h2(__uint_as_float(ra[2 * k]) * sc, __uint_as_float(ra[2 * k + 1]) * sc);
          wb[k] = pack_h2(__uint_as_float(rb[2 * k]) * sc, __uint_as_float(rb[2 * k + 1]) * sc);
          l1f[rp][k] = ((__uint_as_float(ra[2 * k]) + __uint_as_float(ra[2 * k + 1])) + (__uint_as_float(rb[2 * k]) + __uint_as_float(rb[2 * k + 1]))) * (0.25f * sc);
        }
        if (!p.tiled) {
          // level 0: 32 halves = 64 contiguous bytes per image row, as 256-bit stores (one full 32-byte sector each)
          st_v8(o0 + (size_t)c * kCvN + (2 * rp) * 64, wa);      st_v8(o0 + (size_t)c * kCvN + (2 * rp) * 64 + 16, wa + 8);
          st_v8(o0 + (size_t)c * kCvN + (2 * rp + 1) * 64, wb);  st_v8(o0 + (size_t)c * kCvN + (2 * rp + 1) * 64 + 16, wb + 8);
          // level 1 row 2c + rp: 16 halves = 32 bytes
          uint32_t w1[8];
#pragma unroll
          for (int k = 0; k < 8; k++) w1[k] = pack_h2(l1f[rp][2 * k], l1f[rp][2 * k + 1]);
          st_v8(o1 + (size_t)(2 * c + rp) * (wd / 2), w1);
        } else {
          // tiled level 0: chunk c = tile row c; this thread's 32 columns = tiles 4*half .. 4*half+3; rows 2rp, 2rp+1 of a tile are
          // adjacent 16-byte pieces -> one 32-byte sector per tile
          __half* t0 = p.out0 + ((size_t)e * p.HW + m) * (size_t)p.HW + ((size_t)c * 8 + 4 * half) * 32 + (2 * rp) * 8;
#pragma unroll
          for (int t = 0; t < 4; t++) {
            const uint32_t w8[8] = {wa[4 * t], wa[4 * t + 1], wa[4 * t + 2], wa[4 * t + 3], wb[4 * t], wb[4 * t + 1], wb[4 * t + 2], wb[4 * t + 3]};
            st_v8(t0 + t * 32, w8);
          }
          // tiled level 1 (24 x 32 plane, 4 tiles per tile row): row 2c+rp -> tile row c/2, row 2(c&1)+rp inside; tiles 2*half, 2*half+1
          __half* t1 = p.out1 + ((size_t)e * p.HW + m) * (size_t)(p.HW / 4) + ((size_t)(c >> 1) * 4 + 2 * half) * 32 + (2 * (c & 1) + rp) * 8;
#pragma unroll
          for (int t = 0; t < 2; t++)
            *reinterpret_cast<uint4*>(t1 + t * 32) = make_uint4(pack_h2(l1f[rp][8 * t], l1f[rp][8 * t + 1]), pack_h2(l1f[rp][8 * t + 2], l1f[rp][8 * t + 3]),
                                                               pack_h2(l1f[rp][8 * t + 4], l1f[rp][8 * t + 5]), pack_h2(l1f[rp][8 * t + 6], l1f[rp][8 * t + 7]));
        }
      }
      // accumulator drained: hand the TMEM stage back to the MMA warp
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) mbar_arrive(tmem_empty + s);
      // level 2 row c: 8 halves = 16 bytes
      float l2f[8];
#pragma unroll
      for (int k = 0; k < 8; k++) l2f[k] = ((l1f[0][2 * k] + l1f[0][2 * k + 1]) + (l1f[1][2 * k] + l1f[1][2 * k + 1])) * 0.25f;
      *reinterpret_cast<uint4*>(o2 + (size_t)c * (wd / 4)) =
          make_uint4(pack_h2(l2f[0], l2f[1]), pack_h2(l2f[2], l2f[3]), pack_h2(l2f[4], l2f[5]), pack_h2(l2f[6], l2f[7]));
      if (c & 1) {   // level 3 row c/2: 4 halves = 8 bytes
        float l3f[4];
#pragma unroll
        for (int k = 0; k < 4; k++) l3f[k] = ((l2prev[2 * k] + l2prev[2 * k + 1]) + (l2f[2 * k] + l2f[2 * k + 1])) * 0.25f;
        *reinterpret_cast<uint2*>(o3 + (size_t)(c >> 1) * (wd / 8)) = make_uint2(pack_h2(l3f[0], l3f[1]), pack_h2(l3f[2], l3f[3]));
      } else {
#pragma unroll
        for (int k = 0; k < 8; k++) l2prev[k] = l2f[k];
      }
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
}

// ---- host -------------------------------------------------------------------------------------------------------------
static int make_fmap_tensor_map(CUtensorMap* map, const void* base, int n_frames, int C, int HW) {
  EncodeTiledFn enc = tensor_map_encoder();
  if (!enc) { set_error("cuTensorMapEncodeTiled entry point not available"); return DBA_ERR_CUDA; }
  cuuint64_t dims[3] = {(cuuint64_t)HW, (cuuint64_t)C, (cuuint64_t)n_frames};
  cuuint64_t strides[2] = {(cuuint64_t)HW * 2, (cuuint64_t)HW * C * 2};       // bytes, dims 1..2
  cuuint32_t box[3] = {64, (cuuint32_t)C, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed with CUresult %d", (int)r); return DBA_ERR_CUDA; }
  return DBA_OK;
}

}  // namespace dba
using namespace dba;

extern "C" int dba_corr_volume_supported(int channels, int ht, int wd, int dtype) {
  return (dtype == DBA_F16 && channels == 128 && wd == 64 && ht > 0 && ht % 8 == 0) ? 1 : 0;
}

static int corr_volume_launch(const void* fmap1, const void* fmap2, const int64_t* ii, const int64_t* jj, void* out0, void* out1,
                              void* out2, void* out3, int n_edges, int n_frames1, int n_frames2, int channels, int ht, int wd,
                              int dtype, int tiled, dba_stream_t stream) {
  DBA_CHECK_ARG(n_edges >= 0 && n_frames1 > 0 && n_frames2 > 0, "bad extents");
  DBA_CHECK_ARG(dtype == DBA_F16, "corr_volume_pyramid: only f16 features (the live system's autocast dtype) are implemented");
  DBA_CHECK_ARG(channels == 128, "corr_volume_pyramid: 128 feature channels expected (reference fnet)");
  DBA_CHECK_ARG(wd == 64 && ht % 8 == 0 && ht > 0, "corr_volume_pyramid: implemented for wd = 64, ht % 8 == 0 (512-wide inputs at 1/8 resolution)");
  if (n_edges == 0) return DBA_OK;
  DBA_CHECK_ARG(fmap1 && fmap2 && ii && jj && out0 && out1 && out2 && out3, "null pointer");
  DBA_CHECK_ARG((((uintptr_t)fmap1 | (uintptr_t)fmap2 | (uintptr_t)out0 | (uintptr_t)out1 | (uintptr_t)out2 | (uintptr_t)out3) & 15) == 0, "pointers must be 16-byte aligned");
  DBA_CHECK_ARG(n_edges <= 65535, "more than 65535 edges per call");
  const int HW = ht * wd;
  CUtensorMap tmA, tmB;
  int rc = make_fmap_tensor_map(&tmA, fmap1, n_frames1, channels, HW); if (rc) return rc;
  rc = make_fmap_tensor_map(&tmB, fmap2, n_frames2, channels, HW); if (rc) return rc;
  rc = kernel_setup((const void*)corr_volume_pyramid_kernel, kCvSmem); if (rc) return rc;
  CvParams p;
  p.ii = ii; p.jj = jj; p.out0 = (__half*)out0; p.out1 = (__half*)out1; p.out2 = (__half*)out2; p.out3 = (__half*)out3;
  p.HW = HW; p.wd = wd; p.n_chunks = HW / kCvN; p.tiled = tiled;
  dim3 grid(HW / kCvM, n_edges);
  corr_volume_pyramid_kernel<<<grid, kCvThreads, kCvSmem, (cudaStream_t)stream>>>(tmA, tmB, p);
  DBA_CHECK_LAUNCH("corr_volume_pyramid");
  return DBA_OK;
}

extern "C" int dba_corr_volume_pyramid(const void* fmap1, const void* fmap2, const int64_t* ii, const int64_t* jj, void* out0, void* out1,
                                       void* out2, void* out3, int n_edges, int n_frames1, int n_frames2, int channels, int ht, int wd,
                                       int dtype, dba_stream_t stream) {
  return corr_volume_launch(fmap1, fmap2, ii, jj, out0, out1, out2, out3, n_edges, n_frames1, n_frames2, channels, ht, wd, dtype, 0, stream);
}

// same volumes, levels 0 and 1 stored as 4x8-element tiles per plane (private layout of dba_corr_lookup_pyramid with tiled_mask = 3;
// levels 2 and 3 keep the reference layout).  The tensors keep their [E,ht,wd,h2,w2] shapes and sizes; only the order inside a plane differs.
extern "C" int dba_corr_volume_pyramid_tiled(const void* fmap1, const void* fmap2, const int64_t* ii, const int64_t* jj, void* out0, void* out1,
                                             void* out2, void* out3, int n_edges, int n_frames1, int n_frames2, int channels, int ht, int wd,
                                             int dtype, dba_stream_t stream) {
  return corr_volume_launch(fmap1, fmap2, ii, jj, out0, out1, out2, out3, n_edges, n_frames1, n_frames2, channels, ht, wd, dtype, 1, stream);
}

