#include "common.cuh"
#include <stdarg.h>
#include <string.h>
#include <map>
#include <mutex>
#include <set>
#include <utility>

namespace dba {
static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
  va_list ap; va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
int cuda_fail(cudaError_t e, const char* what) {
  set_error("CUDA error in %s: %s", what, cudaGetErrorString(e));
  return DBA_ERR_CUDA;
}

// cudaFuncSetAttribute and the device facts belong to one device: a process that drives several GPUs needs them per device.
// Recursive, because the Cholesky probe inside device_info() sets up its kernel through kernel_setup().
static std::recursive_mutex g_dev_mu;
static std::map<int, DeviceInfo> g_dev_info;
static std::set<std::pair<int, const void*>> g_kernels_set_up;

int device_info(DeviceInfo* out) {
  int dev = 0;
  DBA_CHECK_CUDA(cudaGetDevice(&dev), "cudaGetDevice");
  std::lock_guard<std::recursive_mutex> lock(g_dev_mu);
  auto it = g_dev_info.find(dev);
  if (it == g_dev_info.end()) {
    DeviceInfo d;
    DBA_CHECK_CUDA(cudaDeviceGetAttribute(&d.num_sms, cudaDevAttrMultiProcessorCount, dev), "cudaDeviceGetAttribute(SM count)");
    DBA_CHECK_CUDA(cudaDeviceGetAttribute(&d.smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev), "cudaDeviceGetAttribute(shared memory)");
    d.chol_cluster = chol_cluster_probe();
    it = g_dev_info.emplace(dev, d).first;
  }
  *out = it->second;
  return DBA_OK;
}

int kernel_setup(const void* kernel, int smem_bytes, bool nonportable_cluster) {
  int dev = 0;
  DBA_CHECK_CUDA(cudaGetDevice(&dev), "cudaGetDevice");
  std::lock_guard<std::recursive_mutex> lock(g_dev_mu);
  if (g_kernels_set_up.count({dev, kernel})) return DBA_OK;
  if (nonportable_cluster)
    DBA_CHECK_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1), "cudaFuncSetAttribute(non-portable cluster)");
  DBA_CHECK_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes), "cudaFuncSetAttribute(dynamic shared memory)");
  g_kernels_set_up.insert({dev, kernel});
  return DBA_OK;
}

// a driver entry point is the same for every device: one lookup per process
EncodeTiledFn tensor_map_encoder() {
  static const EncodeTiledFn fn = [] {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) != cudaSuccess || qres != cudaDriverEntryPointSuccess) return (EncodeTiledFn) nullptr;
    return reinterpret_cast<EncodeTiledFn>(ptr);
  }();
  return fn;
}
}  // namespace dba

extern "C" const char* dba_last_error(void) { return dba::g_err; }
extern "C" int dba_version(void) { return 100; }

// L2 fetch granularity (cudaLimitMaxL2FetchGranularity: 32, 64 or 128 bytes; device-wide hint).  The corr_index gather
// touches 16-32 byte runs at arbitrary alignment; with the default 64-byte granularity every touched 32-byte sector drags
// its neighbour out of HBM (measured: 5.4x read amplification at pyramid level 0, see profiles/).  Callers that own the
// device may lower it to 32.
extern "C" int dba_set_l2_fetch_granularity(int bytes) {
  if (bytes != 32 && bytes != 64 && bytes != 128) { dba::set_error("invalid argument: granularity must be 32, 64 or 128"); return DBA_ERR_INVALID; }
  cudaError_t e = cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, (size_t)bytes);
  if (e != cudaSuccess) return dba::cuda_fail(e, "cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity)");
  return DBA_OK;
}
extern "C" int dba_get_l2_fetch_granularity(void) {
  size_t v = 0;
  if (cudaDeviceGetLimit(&v, cudaLimitMaxL2FetchGranularity) != cudaSuccess) { cudaGetLastError(); return -1; }
  return (int)v;
}
