// Shared device helpers for the sm_100a kernels of the dense-BA update path.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include "../../include/droid_b200.h"

namespace dba {

void set_error(const char* fmt, ...);

// ---- per-device host setup (common.cu), keyed by the current device and safe to call from several threads --------------
struct DeviceInfo {
  int num_sms;
  int smem_optin;       // cudaDevAttrMaxSharedMemoryPerBlockOptin
  int chol_cluster;     // largest cluster (16 or 8 CTAs) chol_cluster_kernel can be launched with
};
// facts of the current device, gathered on its first use
int device_info(DeviceInfo* out);
// opts `kernel` into `smem_bytes` of dynamic shared memory (and into non-portable cluster sizes) on the current device; the
// attribute is applied on the first call per device, so a kernel must always be passed the same values
int kernel_setup(const void* kernel, int smem_bytes, bool nonportable_cluster = false);
// cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time dependency on libcuda); nullptr if unavailable
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn tensor_map_encoder();

// chol.cu: damped SPD solve (fp64, one thread-block cluster)
size_t chol_workspace_bytes(int n);
int chol_cluster_probe();     // for device_info(): the cluster-size probe of chol_cluster_kernel on the current device
struct CholPeers {            // fused peer-to-peer reduction (world > 1): H/b are summed over peer copies in rank order
  int world;
  const double* sys[8];       // peer-mapped pointers to each rank's [n*n + n] system for this epoch
  const unsigned long long* flags;   // this rank's flag array [world], flag[p] >= epoch when rank p has published
  unsigned long long epoch;
  const unsigned long long* epoch_dev;   // when set, the awaited value is read from this rank-local device counter (CUDA-graph replay)
};
int chol_solve_launch(const double* H, const double* b, int n, double lm, double ep, void* workspace, int* fail, float* x, cudaStream_t st,
                      const CholPeers* peers = nullptr);
int cuda_fail(cudaError_t e, const char* what);

#define DBA_CHECK_ARG(cond, msg)                                   \
  do { if (!(cond)) { dba::set_error("invalid argument: %s", msg); return DBA_ERR_INVALID; } } while (0)
#define DBA_CHECK_LAUNCH(what)                                     \
  do { cudaError_t e__ = cudaGetLastError(); if (e__ != cudaSuccess) return dba::cuda_fail(e__, what); } while (0)
#define DBA_CHECK_CUDA(expr, what)                                 \
  do { cudaError_t e__ = (expr); if (e__ != cudaSuccess) return dba::cuda_fail(e__, what); } while (0)

constexpr float kMinDepth = 0.25f;   // reference MIN_DEPTH, src/droid_kernels.cu:35

__device__ __forceinline__ int floor_to_int_sat(float f) {
  // static_cast<int>(floor(f)) as the GPU evaluates it: saturating, NaN -> 0; then kept away from INT limits
  int i = __float2int_rd(f);
  return max(-(1 << 30), min(1 << 30, i));
}

// ---- 128-bit streaming loads / stores -----------------------------------------------------------------
__device__ __forceinline__ uint4 ldg_nc_v4(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}

// ---- SE3 helpers, same arithmetic as the reference device functions ---------------------------------------
// (reference src/droid_kernels.cu:67-116; double-literal `2.0 *` there promotes to fp64 and rounds once, which
//  is the same value as the fp32 product because multiplying by 2 is exact)
__device__ __forceinline__ void act_so3(const float* q, const float* X, float* Y) {
  float uv0 = 2.0f * (q[1] * X[2] - q[2] * X[1]);
  float uv1 = 2.0f * (q[2] * X[0] - q[0] * X[2]);
  float uv2 = 2.0f * (q[0] * X[1] - q[1] * X[0]);
  Y[0] = X[0] + q[3] * uv0 + (q[1] * uv2 - q[2] * uv1);
  Y[1] = X[1] + q[3] * uv1 + (q[2] * uv0 - q[0] * uv2);
  Y[2] = X[2] + q[3] * uv2 + (q[0] * uv1 - q[1] * uv0);
}

__device__ __forceinline__ void act_se3(const float* t, const float* q, const float* X, float* Y) {
  act_so3(q, X, Y);
  Y[3] = X[3];
  Y[0] += X[3] * t[0];
  Y[1] += X[3] * t[1];
  Y[2] += X[3] * t[2];
}

__device__ __forceinline__ void rel_se3(const float* ti, const float* qi, const float* tj, const float* qj,
                                        float* tij, float* qij) {
  qij[0] = -qj[3] * qi[0] + qj[0] * qi[3] - qj[1] * qi[2] + qj[2] * qi[1];
  qij[1] = -qj[3] * qi[1] + qj[1] * qi[3] - qj[2] * qi[0] + qj[0] * qi[2];
  qij[2] = -qj[3] * qi[2] + qj[2] * qi[3] - qj[0] * qi[1] + qj[1] * qi[0];
  qij[3] = qj[3] * qi[3] + qj[0] * qi[0] + qj[1] * qi[1] + qj[2] * qi[2];
  act_so3(qij, ti, tij);
  tij[0] = tj[0] - tij[0];
  tij[1] = tj[1] - tij[1];
  tij[2] = tj[2] - tij[2];
}

// relative transform of an edge; stereo edges (ix==jx) get the fixed baseline when `stereo_quirk`
__device__ __forceinline__ void edge_transform(const float* __restrict__ poses, int ix, int jx, bool stereo_quirk,
                                               float* tij, float* qij) {
  if (stereo_quirk && ix == jx) {
    tij[0] = -0.1f; tij[1] = 0.f; tij[2] = 0.f;
    qij[0] = 0.f; qij[1] = 0.f; qij[2] = 0.f; qij[3] = 1.f;
    return;
  }
  float ti[3], tj[3], qi[4], qj[4];
#pragma unroll
  for (int k = 0; k < 3; k++) { ti[k] = __ldg(poses + 7 * (size_t)ix + k); tj[k] = __ldg(poses + 7 * (size_t)jx + k); }
#pragma unroll
  for (int k = 0; k < 4; k++) { qi[k] = __ldg(poses + 7 * (size_t)ix + 3 + k); qj[k] = __ldg(poses + 7 * (size_t)jx + 3 + k); }
  rel_se3(ti, qi, tj, qj, tij, qij);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

}  // namespace dba
