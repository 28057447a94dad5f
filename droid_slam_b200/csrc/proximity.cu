// Row F1 (SURVEY section 8f): proximity edge selection of the factor graph on the device.
//
// Replaces everything between `video.distance(...)` and `add_factors(...)` in the reference's FactorGraph.add_proximity_factors
// (droid_slam/factor_graph.py:346-412): a Python / NumPy triple loop over a CPU copy of the distance matrix, entered on every frontend
// step behind a device->host copy.  Same result, order included (the edge list feeds add_factors, whose order the graph keeps).
//
//   prox_keys_kernel     one thread per pair (i, j): masked distance (factor_graph.py:359-360) -> 64-bit key (orderable value | flat index)
//   cub radix sort       by (value, index): the order torch.argsort(d) visits distinct values in; ties by index (see oracle/proximity.py)
//   prox_select_kernel   one CTA: "still alive" bitmap of the pairs in shared memory (one bit per pair), suppression by the edges the graph
//                        already has (:362-373), temporal-neighbour edges (:375-384, including the unchecked index of the reference),
//                        then ONE warp walks the sorted pairs and does the greedy selection + non-maximum suppression (:386-409):
//                        inherently serial, ~30 cycles per candidate with the bitmap on chip.
// The reference re-reads d[k] when it visits k; here "d[k] was set to inf" is the bitmap.  NaN distances are not > thresh, so they are
// taken (after everything else: they sort last) -- kept.
#include "common.cuh"
#include <cub/device/device_radix_sort.cuh>

namespace dba {

constexpr int kProxThreads = 1024;
enum { PROX_OVERFLOW = 1, PROX_INDEX = 2 };

__device__ __forceinline__ float prox_masked(const float* d, long idx, int n_j, int t0, int t1, int rad) {
  const int i = t0 + (int)(idx / n_j), j = t1 + (int)(idx % n_j);
  float v = d[idx];
  if (i - rad < j) v = INFINITY;
  if (v > 100.f) v = INFINITY;
  return v;
}
// float -> unsigned with the same order; every NaN maps to the largest value (argsort puts NaNs last)
__device__ __forceinline__ unsigned prox_orderable(float v) {
  if (v != v) return 0xFFFFFFFFu;
  const unsigned b = __float_as_uint(v);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

__global__ void prox_keys_kernel(const float* __restrict__ d, long n, int n_j, int t0, int t1, int rad, unsigned long long* __restrict__ keys, int* hdr) {
  const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n) return;
  const float v = prox_masked(d, idx, n_j, t0, t1, rad);
  if (v != v) atomicAdd(hdr + 2, 1);                        // number of NaN pairs: they form the tail of the sorted keys
  keys[idx] = ((unsigned long long)prox_orderable(v) << 32) | (unsigned long long)(unsigned)idx;
}

struct ProxParams {
  const float* d;
  const unsigned long long* sorted;
  const long long* ii_known; const long long* jj_known; int n_known;
  int t0, t1, t, rad, nms, max_factors, stereo;
  float thresh;
  long long* es; int cap;
  int* hdr;                    // [0] number of (i, j) rows written, [1] status bits, [2] NaN count
  unsigned* bitmap_global;     // used when the bitmap does not fit in shared memory
  int bitmap_in_smem;
};

__device__ __forceinline__ void prox_kill(unsigned* bm, long idx) { atomicOr(bm + (idx >> 5), 1u << (idx & 31)); }
__device__ __forceinline__ bool prox_dead(const unsigned* bm, long idx) { return (bm[idx >> 5] >> (idx & 31)) & 1u; }

// the |di| + |dj| <= min(|i-j| - 2, nms) diamond around (i, j) (factor_graph.py:365-373 / :401-409); `worker` of `nworkers` threads share it
__device__ __forceinline__ void prox_suppress(unsigned* bm, int i, int j, int t0, int t1, int t, int nms, int worker, int nworkers) {
  const int w = max(min(abs(i - j) - 2, nms), 0);
  const int side = 2 * nms + 1;
  for (int o = worker; o < side * side; o += nworkers) {
    const int di = o / side - nms, dj = o % side - nms;
    if (abs(di) + abs(dj) <= w) {
      const int i1 = i + di, j1 = j + dj;
      if (i1 >= t0 && i1 < t && j1 >= t1 && j1 < t) prox_kill(bm, (long)(i1 - t0) * (t - t1) + (j1 - t1));
    }
  }
}

__global__ void __launch_bounds__(kProxThreads, 1) prox_select_kernel(ProxParams p) {
  extern __shared__ unsigned s_bitmap[];
  unsigned* bm = p.bitmap_in_smem ? s_bitmap : p.bitmap_global;
  const int tid = threadIdx.x;
  const int n_i = p.t - p.t0, n_j = p.t - p.t1;
  const long n = (long)n_i * n_j;
  const long words = (n + 31) / 32;
  // ---- alive bitmap: a pair is dead from the start if its masked distance is > thresh (what the walk below would skip anyway)
  for (long w = tid; w < words; w += kProxThreads) {
    unsigned bits = 0;
    for (int b = 0; b < 32; b++) {
      const long idx = w * 32 + b;
      if (idx < n) {
        const float v = prox_masked(p.d, idx, n_j, p.t0, p.t1, p.rad);
        if (v > p.thresh) bits |= 1u << b;
      }
    }
    bm[w] = bits;
  }
  __syncthreads();
  // ---- edges the graph already has
  for (int e = tid; e < p.n_known; e += kProxThreads) prox_suppress(bm, (int)p.ii_known[e], (int)p.jj_known[e], p.t0, p.t1, p.t, p.nms, 0, 1);
  // ---- temporal neighbours: frame i emits [(i,i) if stereo] then (i,j), (j,i) for j = max(i-rad-1, 0) .. i-1; its rows start at a closed-form offset
  __shared__ int s_nbase;
  if (tid == 0) {
    long tot = 0;
    for (int i = p.t0; i < p.t; i++) tot += (p.stereo ? 1 : 0) + 2 * (i - max(i - p.rad - 1, 0));
    s_nbase = tot > p.cap ? -1 : (int)tot;
  }
  __syncthreads();
  if (s_nbase < 0) { if (tid == 0) { atomicOr(p.hdr + 1, PROX_OVERFLOW); p.hdr[0] = 0; } return; }
  for (int i = p.t0 + tid; i < p.t; i += kProxThreads) {
    long off = 0;
    for (int q = p.t0; q < i; q++) off += (p.stereo ? 1 : 0) + 2 * (q - max(q - p.rad - 1, 0));
    auto mask = [&](int jj) {                                // d[(i - t0) * (t - t1) + (jj - t1)] = inf with the reference's unchecked index
      long idx = (long)(i - p.t0) * n_j + (jj - p.t1);
      if (idx < 0) idx += n;                                 // Python / torch negative index
      if (idx < 0 || idx >= n) atomicOr(p.hdr + 1, PROX_INDEX);   // the reference raises IndexError here
      else prox_kill(bm, idx);
    };
    if (p.stereo) { p.es[2 * off] = i; p.es[2 * off + 1] = i; off++; mask(i); }
    for (int j = max(i - p.rad - 1, 0); j < i; j++) {
      p.es[2 * off] = i; p.es[2 * off + 1] = j; off++;
      p.es[2 * off] = j; p.es[2 * off + 1] = i; off++;
      mask(j);
    }
  }
  __syncthreads();
  if (tid >= 32) return;
  // ---- greedy walk in sorted order, one warp; lanes share the suppression diamond
  const int lane = tid;
  int len = s_nbase;
  const unsigned th = prox_orderable(p.thresh);
  const long n_nan = p.hdr[2];
  bool stop = false;
  for (int seg = 0; seg < 2 && !stop; seg++) {               // segment 0: values <= thresh from the front; segment 1: the NaN tail
    long pos = seg == 0 ? 0 : n - n_nan;
    const long end = seg == 0 ? n - n_nan : n;
    while (pos < end && !stop) {
      const long mine = pos + lane;
      const unsigned long long key = mine < end ? p.sorted[mine] : ~0ull;
      for (int l = 0; l < 32 && pos + l < end; l++) {
        const unsigned long long k = __shfl_sync(0xffffffffu, key, l);
        const unsigned hi = (unsigned)(k >> 32);
        const long idx = (long)(unsigned)(k & 0xffffffffu);
        if (seg == 0 && hi > th) { pos = end; break; }        // everything from here on is > thresh (until the NaN tail)
        __syncwarp();
        if (prox_dead(bm, idx)) continue;
        if (p.max_factors > 0 && len > p.max_factors) { stop = true; break; }
        if (len + 2 > p.cap) { if (lane == 0) atomicOr(p.hdr + 1, PROX_OVERFLOW); stop = true; break; }
        const int i = p.t0 + (int)(idx / n_j), j = p.t1 + (int)(idx % n_j);
        if (lane == 0) { p.es[2 * len] = i; p.es[2 * len + 1] = j; p.es[2 * len + 2] = j; p.es[2 * len + 3] = i; }
        len += 2;
        prox_suppress(bm, i, j, p.t0, p.t1, p.t, p.nms, lane, 32);
        __syncwarp();
      }
      if (pos < end) pos += 32;
    }
  }
  if (lane == 0) p.hdr[0] = len;
}

static size_t prox_sort_temp_bytes(long n) {
  size_t tb = 0;
  cub::DeviceRadixSort::SortKeys(nullptr, tb, (const unsigned long long*)nullptr, (unsigned long long*)nullptr, (int)n);
  return tb;
}

}  // namespace dba

extern "C" size_t dba_proximity_workspace_bytes(int t0, int t1, int t) {
  if (t <= t0 || t <= t1 || t0 < 0 || t1 < 0) return 256;
  const long n = (long)(t - t0) * (t - t1);
  return 256 + 2 * (size_t)n * 8 + dba::prox_sort_temp_bytes(n) + 256 + ((size_t)(n + 31) / 32) * 4 + 256;
}

extern "C" int dba_proximity_edges(const float* d, int t0, int t1, int t, const int64_t* ii_known, const int64_t* jj_known, int n_known, int rad, int nms,
                                   float thresh, int max_factors, int stereo, int64_t* es, int cap, int* n_out_status, void* workspace, size_t workspace_bytes,
                                   dba_stream_t stream) {
  using namespace dba;
  DBA_CHECK_ARG(t0 >= 0 && t1 >= 0 && rad >= 0 && nms >= 0 && cap >= 0 && n_known >= 0, "negative argument");
  DBA_CHECK_ARG(n_out_status && workspace, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  DBA_CHECK_CUDA(cudaMemsetAsync(n_out_status, 0, 2 * sizeof(int), st), "proximity header");
  if (t <= t0 || t <= t1) return DBA_OK;                     // empty grid: no frames to connect (the reference's loops do not run)
  DBA_CHECK_ARG(d && es, "null pointer");
  DBA_CHECK_ARG(n_known == 0 || (ii_known && jj_known), "known edges missing");
  const long n = (long)(t - t0) * (t - t1);
  DBA_CHECK_ARG(n < (1l << 31), "more than 2^31 pairs");
  if (workspace_bytes < dba_proximity_workspace_bytes(t0, t1, t)) { set_error("proximity workspace too small"); return DBA_ERR_WORKSPACE; }
  char* w = reinterpret_cast<char*>(workspace);
  int* hdr = reinterpret_cast<int*>(w);                      // [0] rows, [1] status, [2] NaN count
  unsigned long long* keys_in = reinterpret_cast<unsigned long long*>(w + 256);
  unsigned long long* keys_out = keys_in + n;
  size_t temp_bytes = prox_sort_temp_bytes(n);
  char* temp = reinterpret_cast<char*>(keys_out + n);
  unsigned* bitmap = reinterpret_cast<unsigned*>(temp + ((temp_bytes + 255) / 256) * 256);
  DBA_CHECK_CUDA(cudaMemsetAsync(hdr, 0, 3 * sizeof(int), st), "proximity header");
  prox_keys_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d, n, t - t1, t0, t1, rad, keys_in, hdr);
  DBA_CHECK_LAUNCH("prox_keys");
  DBA_CHECK_CUDA(cub::DeviceRadixSort::SortKeys(temp, temp_bytes, keys_in, keys_out, (int)n, 0, 64, st), "proximity sort");
  ProxParams p;
  p.d = d; p.sorted = keys_out; p.ii_known = reinterpret_cast<const long long*>(ii_known); p.jj_known = reinterpret_cast<const long long*>(jj_known); p.n_known = n_known;
  p.t0 = t0; p.t1 = t1; p.t = t; p.rad = rad; p.nms = nms; p.max_factors = max_factors; p.stereo = stereo; p.thresh = thresh;
  p.es = reinterpret_cast<long long*>(es); p.cap = cap; p.hdr = hdr; p.bitmap_global = bitmap;
  const size_t bm_bytes = ((size_t)(n + 31) / 32) * 4;
  DeviceInfo dev;
  int rc = device_info(&dev); if (rc) return rc;
  const int max_smem = dev.smem_optin - 1024;
  rc = kernel_setup((const void*)prox_select_kernel, max_smem); if (rc) return rc;
  p.bitmap_in_smem = bm_bytes <= (size_t)max_smem ? 1 : 0;
  prox_select_kernel<<<1, kProxThreads, p.bitmap_in_smem ? bm_bytes : 0, st>>>(p);
  DBA_CHECK_LAUNCH("prox_select");
  DBA_CHECK_CUDA(cudaMemcpyAsync(n_out_status, hdr, 2 * sizeof(int), cudaMemcpyDeviceToDevice, st), "proximity result header");
  return DBA_OK;
}
