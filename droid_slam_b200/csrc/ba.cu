// Dense bundle adjustment (Gauss-Newton, Schur complement over per-pixel inverse depth) for sm_100a.
//
// Replaces reference src/droid_kernels.cu:185-433 (K1), :863-1124 (accum / retraction / Schur kernels),
// :1126-1320 (CPU SparseBlock + schur_block) and the driver :1323-1443.  Same maths, different machine mapping:
//
//   * everything stays on the device and on one stream: no .to(kCPU), no argsort/CSR on the host, no Eigen;
//   * edges are grouped by SOURCE frame (CSR built once per call by two small kernels).  One CTA owns
//     (depth frame k, pixel chunk): it walks the out-edges of k, so the depth-block sums C_k, w_k, Ei_k are plain
//     register accumulations (no atomics, no segmented-sum kernels, deterministic);
//   * only Hjj (21 unique) and vj (6) are accumulated per pixel.  Ji = -Adj^T(G_ij) Jj is linear in Jj, hence
//     Hii = A Hjj A^T, Hij = -A Hjj, vi = -A vj are formed once per edge from the reduced fp64 sums
//     (the reference accumulates all 78+12 sums per pixel and does 90 serial block reductions);
//   * reductions: fp32 per thread over its pixels -> warp shuffles -> fp64 across warps -> fp64 atomics into the
//     dense reduced system Hsys [6P x 6P] / bsys [6P] (this is the buffer an edge-sharded multi-GPU run all-reduces);
//   * the Schur complement S = sum_k E_k Q_k E_k^T is a per-frame SYRK over the (1+deg_k) rows of frame k with the
//     6x6 block pairs register-tiled per thread (the reference enumerates (i,j,k) triples on the CPU, O(P^2 deg^2));
//   * solve: damping (diag += ep + lm*diag) and a tiled fp64 Cholesky on the device; a non-positive pivot gives
//     dx = 0 like the reference's `solver.info() != Success` branch;
//   * back-substitution dz = Q (w - E^T dx) keeps the reference quirk Q9 (rows whose pose index is <= 0 are skipped,
//     src/droid_kernels.cu:1114), then retraction of poses (left-multiplicative Exp, no renormalisation) and disps.
#include "common.cuh"
#include "tcgen05.cuh"
#include <math.h>
#include <algorithm>

namespace dba {

constexpr int kBuildThreads = 256;
constexpr int kEdgeBatch = 16;     // edges whose transforms / partial sums live in shared memory at once

struct Layout {
  size_t off_hdr, off_frame2k, off_kx, off_rowptr, off_edgeidx, off_big, off_sys, off_L, off_dx, off_Eij, off_C, off_w, off_Ei, total;
  int P, n;
};

__host__ inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

__host__ inline Layout make_layout(int N, int E, int ht, int wd, int t0, int t1) {
  Layout L;
  const size_t HW = (size_t)ht * wd;
  L.P = t1 - t0 > 0 ? t1 - t0 : 0;
  L.n = 6 * L.P;
  size_t o = 0;
  L.off_hdr = o;      o = align_up(o + 64 * sizeof(int), 256);
  L.off_frame2k = o;  o = align_up(o + (size_t)(N + 1) * sizeof(int), 256);
  L.off_kx = o;       o = align_up(o + (size_t)(N + 1) * sizeof(int), 256);
  L.off_rowptr = o;   o = align_up(o + (size_t)(N + 2) * sizeof(int), 256);
  L.off_edgeidx = o;  o = align_up(o + (size_t)(E + 1) * sizeof(int), 256);
  L.off_big = o;      o = align_up(o + (size_t)(N + 1) * sizeof(int), 256);     // depth frames with more than 21 possible rows (pair-mode Schur)
  L.off_sys = o;      o = align_up(o + ((size_t)L.n * L.n + L.n) * sizeof(double), 256);
  L.off_L = o;        o = align_up(o + chol_workspace_bytes(L.n), 256);
  L.off_dx = o;       o = align_up(o + (size_t)(L.n + 6) * sizeof(float), 256);
  L.off_Eij = o;      o = align_up(o + (size_t)E * 6 * HW * sizeof(float), 256);
  const size_t Mmax = (size_t)N;   // at most one depth frame per buffer frame
  L.off_C = o;        o = align_up(o + Mmax * HW * sizeof(float), 256);
  L.off_w = o;        o = align_up(o + Mmax * HW * sizeof(float), 256);
  L.off_Ei = o;       o = align_up(o + Mmax * 6 * HW * sizeof(float), 256);
  L.total = o;
  return L;
}

// header words
enum { HDR_STATUS = 0, HDR_M = 1, HDR_CHOL_FAIL = 2, HDR_NBIG = 3 };
enum { ST_BAD_INDEX = 1, ST_ETA_ROWS = 2, ST_CHOL_FAIL = 4, ST_DEGREE = 8 };

// ---------------------------------------------------------------------------------------------------------
// prepare: kx = sorted unique(ii U [t0,t1)), frame2k, CSR of edges by source frame (stable in edge order)
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) ba_prepare_kernel(const int64_t* __restrict__ ii, const int64_t* __restrict__ jj, int E, int N,
                                                          int t0, int t1, int eta_rows, int* __restrict__ hdr,
                                                          int* __restrict__ frame2k, int* __restrict__ kx, int* __restrict__ rowptr, int* __restrict__ big) {
  __shared__ int s_scan[1024];
  __shared__ int s_carry;
  const int tid = threadIdx.x;
  if (tid == 0) { hdr[HDR_STATUS] = 0; hdr[HDR_CHOL_FAIL] = 0; }
  for (int f = tid; f < N; f += blockDim.x) { frame2k[f] = (f >= t0 && f < t1) ? 1 : 0; rowptr[f] = 0; }
  if (tid == 0) { rowptr[N] = 0; rowptr[N + 1] = 0; }
  __syncthreads();
  for (int e = tid; e < E; e += blockDim.x) {
    const long long i = ii[e], j = jj[e];
    if (i < 0 || i >= N || j < 0 || j >= N) { atomicOr(&hdr[HDR_STATUS], ST_BAD_INDEX); continue; }
    frame2k[i] = 1;
  }
  __syncthreads();
  // exclusive scan of the presence flags -> dense index
  if (tid == 0) s_carry = 0;
  __syncthreads();
  for (int base = 0; base < N; base += blockDim.x) {
    const int f = base + tid;
    const int flag = (f < N) ? frame2k[f] : 0;
    s_scan[tid] = flag;
    __syncthreads();
    for (int off = 1; off < (int)blockDim.x; off <<= 1) {
      int v = (tid >= off) ? s_scan[tid - off] : 0;
      __syncthreads();
      s_scan[tid] += v;
      __syncthreads();
    }
    const int incl = s_scan[tid];
    const int idx = s_carry + incl - flag;
    if (f < N) {
      frame2k[f] = flag ? idx : -1;
      if (flag) kx[idx] = f;
    }
    __syncthreads();
    if (tid == blockDim.x - 1) s_carry += incl;
    __syncthreads();
  }
  const int M = s_carry;
  if (tid == 0) {
    hdr[HDR_M] = M;
    if (eta_rows != M && eta_rows != 1) atomicOr(&hdr[HDR_STATUS], ST_ETA_ROWS);
  }
  // out-degree per depth frame -> rowptr (exclusive scan, serial per chunk is fine: M <= N small)
  for (int e = tid; e < E; e += blockDim.x) {
    const long long i = ii[e], j = jj[e];
    if (i < 0 || i >= N || j < 0 || j >= N) continue;
    atomicAdd(&rowptr[frame2k[i] + 1], 1);
  }
  __syncthreads();
  if (tid == 0) s_carry = 0;
  __syncthreads();
  for (int base = 0; base <= M; base += blockDim.x) {
    const int m = base + tid;
    const int cnt = (m <= M) ? rowptr[m] : 0;     // rowptr[m] currently holds deg(m-1), rowptr[0] = 0
    s_scan[tid] = cnt;
    __syncthreads();
    for (int off = 1; off < (int)blockDim.x; off <<= 1) {
      int v = (tid >= off) ? s_scan[tid - off] : 0;
      __syncthreads();
      s_scan[tid] += v;
      __syncthreads();
    }
    if (m <= M) rowptr[m] = s_carry + s_scan[tid];
    __syncthreads();
    if (tid == blockDim.x - 1) s_carry += s_scan[tid];
    __syncthreads();
  }
  // depth frames that can have more than kTcRowsMax (21) rows = out-degree + 1: the pair-mode Schur launch only visits these
  // (ascending order; there are at most E / 21 of them, which is what sizes that launch's grid)
  if (tid == 0) s_carry = 0;
  __syncthreads();
  for (int base = 0; base < M; base += blockDim.x) {
    const int m = base + tid;
    const int flag = (m < M && rowptr[m + 1] - rowptr[m] + 1 > 21) ? 1 : 0;
    s_scan[tid] = flag;
    __syncthreads();
    for (int off = 1; off < (int)blockDim.x; off <<= 1) {
      int v = (tid >= off) ? s_scan[tid - off] : 0;
      __syncthreads();
      s_scan[tid] += v;
      __syncthreads();
    }
    if (flag) big[s_carry + s_scan[tid] - 1] = m;
    __syncthreads();
    if (tid == blockDim.x - 1) s_carry += s_scan[tid];
    __syncthreads();
  }
  if (tid == 0) hdr[HDR_NBIG] = s_carry;
}

// stable placement of every edge inside its source frame's segment: rank = #earlier edges with the same source.
// One warp per edge, lanes stride over the earlier edges (E^2/2 compares spread over E warps).
__global__ void __launch_bounds__(256) ba_fill_csr_kernel(const int64_t* __restrict__ ii, const int64_t* __restrict__ jj, int E, int N,
                                                          const int* __restrict__ frame2k, const int* __restrict__ rowptr,
                                                          int* __restrict__ edgeidx) {
  const int e = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (e >= E) return;
  const long long i = ii[e], j = jj[e];
  if (i < 0 || i >= N || j < 0 || j >= N) return;
  int rank = 0;
  for (int f = lane; f < e; f += 32) {
    const long long i2 = ii[f], j2 = jj[f];
    rank += (i2 == i && j2 >= 0 && j2 < N) ? 1 : 0;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) rank += __shfl_xor_sync(0xffffffffu, rank, o);
  if (lane == 0) edgeidx[rowptr[frame2k[i]] + rank] = e;
}

// ---------------------------------------------------------------------------------------------------------
// build: per (depth frame, pixel chunk): geometry of all out-edges, depth-block sums, per-edge pose blocks
// ---------------------------------------------------------------------------------------------------------
// total of value i ends up in lane i  (v[0] on return), 31 shuffles
__device__ __forceinline__ float transpose_reduce32(float (&v)[32], int lane) {
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) {
    const bool up = (lane & off) != 0;
#pragma unroll
    for (int i = 0; i < off; i++) {
      const float send = up ? v[i] : v[i + off];
      const float keep = up ? v[i + off] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
    }
  }
  return v[0];
}

struct EdgeSm {
  float t[3], q[4];      // G_ij
  float A[36];           // Ji = -A Jj   (A = transposed adjoint, applied with the reference's adjSE3 arithmetic)
  int e, jx, stereo;
};

// Y = adjSE3(t,q,X)  (reference src/droid_kernels.cu:88-103)
__device__ __forceinline__ void adj_se3(const float* t, const float* q, const float* X, float* Y) {
  float qinv[4] = {-q[0], -q[1], -q[2], q[3]};
  act_so3(qinv, X, Y);
  act_so3(qinv, X + 3, Y + 3);
  float u[3], v[3];
  u[0] = t[2] * X[1] - t[1] * X[2];
  u[1] = t[0] * X[2] - t[2] * X[0];
  u[2] = t[1] * X[0] - t[0] * X[1];
  act_so3(qinv, u, v);
  Y[3] += v[0]; Y[4] += v[1]; Y[5] += v[2];
}

template <int kPPT>   // pixels per thread: 4 when many frames fill the GPU, fewer when a rank owns only a few source frames
__global__ void __launch_bounds__(kBuildThreads, 2) ba_build_kernel(
    const float* __restrict__ poses, const float* __restrict__ disps, const float* __restrict__ intr,
    const float* __restrict__ disps_sens, const float* __restrict__ targets, const float* __restrict__ weights,
    const float* __restrict__ eta, int eta_rows, int eta_by_frame, const int64_t* __restrict__ jj,
    const int* __restrict__ hdr, const int* __restrict__ kx, const int* __restrict__ rowptr, const int* __restrict__ edgeidx,
    int HW, int wd, int t0, int P, int motion_only,
    double* __restrict__ Hsys, double* __restrict__ bsys, float* __restrict__ Eij, float* __restrict__ Cout, float* __restrict__ wout,
    float* __restrict__ Eiout) {
  const int m = blockIdx.y;
  if (m >= hdr[HDR_M]) return;
  const int ix = kx[m];
  const int e_begin = rowptr[m], e_end = rowptr[m + 1];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int NW = kBuildThreads / 32;

  __shared__ EdgeSm s_edge[kEdgeBatch];
  __shared__ float s_part[NW][kEdgeBatch][27];
  __shared__ double s_sum[kEdgeBatch][27];

  const float fx = __ldg(intr), fy = __ldg(intr + 1), cx = __ldg(intr + 2), cy = __ldg(intr + 3);
  const int n = 6 * P;

  // this thread's pixels
  int pix[kPPT];
  float Xi0[kPPT], Xi1[kPPT], dsp[kPPT];
  float Cacc[kPPT], wacc[kPPT], Eiacc[kPPT][6];
#pragma unroll
  for (int s = 0; s < kPPT; s++) {
    const int p = blockIdx.x * (kPPT * kBuildThreads) + s * kBuildThreads + tid;
    pix[s] = p;
    const bool ok = p < HW;
    const int i = ok ? p / wd : 0, j = ok ? p - i * wd : 0;
    Xi0[s] = ((float)j - cx) / fx;
    Xi1[s] = ((float)i - cy) / fy;
    dsp[s] = ok ? __ldg(disps + (size_t)ix * HW + p) : 1.f;
    Cacc[s] = 0.f; wacc[s] = 0.f;
#pragma unroll
    for (int c = 0; c < 6; c++) Eiacc[s][c] = 0.f;
  }

  for (int eb = e_begin; eb < e_end; eb += kEdgeBatch) {
    const int nb = min(kEdgeBatch, e_end - eb);
    __syncthreads();   // previous batch fully consumed
    // ---- edge transforms + adjoint matrices for the batch
    if (tid < nb) {
      EdgeSm& S = s_edge[tid];
      const int e = edgeidx[eb + tid];
      S.e = e; S.jx = (int)jj[e]; S.stereo = (S.jx == ix);
      edge_transform(poses, ix, S.jx, /*stereo_quirk=*/true, S.t, S.q);
    }
    __syncthreads();
    if (tid < nb * 6) {
      const int b = tid / 6, c = tid - b * 6;
      float X[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, Y[6];
      X[c] = 1.f;
      adj_se3(s_edge[b].t, s_edge[b].q, X, Y);
#pragma unroll
      for (int r = 0; r < 6; r++) s_edge[b].A[r * 6 + c] = Y[r];
    }
    __syncthreads();

    // software pipeline: the four target/weight loads of edge b+1 are in flight while edge b is computed
    float nw_u[kPPT], nw_v[kPPT], nt_u[kPPT], nt_v[kPPT];
    {
      const int e0 = s_edge[0].e;
#pragma unroll
      for (int s = 0; s < kPPT; s++) {
        const int p = pix[s];
        const bool okp = p < HW;
        nw_u[s] = okp ? __ldg(weights + ((size_t)e0 * 2 + 0) * HW + p) : 0.f;
        nw_v[s] = okp ? __ldg(weights + ((size_t)e0 * 2 + 1) * HW + p) : 0.f;
        nt_u[s] = okp ? __ldg(targets + ((size_t)e0 * 2 + 0) * HW + p) : 0.f;
        nt_v[s] = okp ? __ldg(targets + ((size_t)e0 * 2 + 1) * HW + p) : 0.f;
      }
    }
    for (int b = 0; b < nb; b++) {
      const EdgeSm& S = s_edge[b];
      const float t0_ = S.t[0], t1_ = S.t[1], t2_ = S.t[2];
      const int e = S.e;
      float cw_u[kPPT], cw_v[kPPT], ct_u[kPPT], ct_v[kPPT];
#pragma unroll
      for (int s = 0; s < kPPT; s++) { cw_u[s] = nw_u[s]; cw_v[s] = nw_v[s]; ct_u[s] = nt_u[s]; ct_v[s] = nt_v[s]; }
      if (b + 1 < nb) {
        const int e1 = s_edge[b + 1].e;
#pragma unroll
        for (int s = 0; s < kPPT; s++) {
          const int p = pix[s];
          if (p < HW) {
            nw_u[s] = __ldg(weights + ((size_t)e1 * 2 + 0) * HW + p);
            nw_v[s] = __ldg(weights + ((size_t)e1 * 2 + 1) * HW + p);
            nt_u[s] = __ldg(targets + ((size_t)e1 * 2 + 0) * HW + p);
            nt_v[s] = __ldg(targets + ((size_t)e1 * 2 + 1) * HW + p);
          }
        }
      }
      const bool stereo = S.stereo != 0;
      float Hjj[21], vj[6];
#pragma unroll
      for (int k = 0; k < 21; k++) Hjj[k] = 0.f;
#pragma unroll
      for (int k = 0; k < 6; k++) vj[k] = 0.f;

#pragma unroll
      for (int s = 0; s < kPPT; s++) {
        const int p = pix[s];
        if (p < HW) {
          float Xi[4] = {Xi0[s], Xi1[s], 1.f, dsp[s]}, Xj[4];
          act_se3(S.t, S.q, Xi, Xj);
          const float x = Xj[0], y = Xj[1], h = Xj[3];
          const bool close = (double)Xj[2] < 0.25;   // MIN_DEPTH is a double literal in the reference
          const float d = close ? 0.f : 1.0f / Xj[2];
          const float d2 = d * d;
          // `.001 * weight`: fp64 product rounded to fp32 (reference :314-315)
          float wu = close ? 0.f : (float)(.001 * (double)cw_u[s]);
          float wv = close ? 0.f : (float)(.001 * (double)cw_v[s]);
          const float ru = ct_u[s] - (fx * d * x + cx);
          const float rv = ct_v[s] - (fy * d * y + cy);
          float Ju[6], Jv[6];
          Ju[0] = fx * (h * d); Ju[1] = fx * 0; Ju[2] = fx * (-x * h * d2);
          Ju[3] = fx * (-x * y * d2); Ju[4] = fx * (1 + x * x * d2); Ju[5] = fx * (-y * d);
          Jv[0] = fy * 0; Jv[1] = fy * (h * d); Jv[2] = fy * (-y * h * d2);
          Jv[3] = fy * (-1 - y * y * d2); Jv[4] = fy * (x * y * d2); Jv[5] = fy * (x * d);
          const float Jzu = fx * (t0_ * d - t2_ * (x * d2));
          const float Jzv = fy * (t1_ * d - t2_ * (y * d2));
          Cacc[s] += wu * Jzu * Jzu + wv * Jzv * Jzv;
          wacc[s] += wu * ru * Jzu + wv * rv * Jzv;
          if (stereo) { wu = 0.f; wv = 0.f; }       // pose weights vanish AFTER the depth terms (Q1)
          const float au = wu * Jzu, av = wv * Jzv;
          float Ej[6];
#pragma unroll
          for (int c = 0; c < 6; c++) Ej[c] = au * Ju[c] + av * Jv[c];
          if (!motion_only) {
#pragma unroll
            for (int c = 0; c < 6; c++) Eij[((size_t)e * 6 + c) * HW + p] = Ej[c];
            // Eii = -A Eij, accumulated over the out-edges of this frame
#pragma unroll
            for (int r = 0; r < 6; r++) {
              float acc = 0.f;
#pragma unroll
              for (int c = 0; c < 6; c++) acc += S.A[r * 6 + c] * Ej[c];
              Eiacc[s][r] -= acc;
            }
          }
          const float wru = wu * ru, wrv = wv * rv;
          int l = 0;
#pragma unroll
          for (int a = 0; a < 6; a++) {
            vj[a] += wru * Ju[a] + wrv * Jv[a];
            const float wa_u = wu * Ju[a], wa_v = wv * Jv[a];
#pragma unroll
            for (int c = 0; c <= a; c++) { Hjj[l] += wa_u * Ju[c] + wa_v * Jv[c]; l++; }
          }
        }
      }
      // warp reduction of the 27 sums (padded to 32): transpose-reduction, 31 shuffles; lane k ends with the total of value k
      {
        float v32[32];
#pragma unroll
        for (int k = 0; k < 21; k++) v32[k] = Hjj[k];
#pragma unroll
        for (int k = 0; k < 6; k++) v32[21 + k] = vj[k];
#pragma unroll
        for (int k = 27; k < 32; k++) v32[k] = 0.f;
        const float tot = transpose_reduce32(v32, lane);
        if (lane < 27) s_part[warp][b][lane] = tot;
      }
    }
    __syncthreads();
    // ---- cross-warp sums in fp64
    for (int k = tid; k < nb * 27; k += kBuildThreads) {
      const int b = k / 27, c = k - b * 27;
      double s = 0.0;
#pragma unroll
      for (int w = 0; w < NW; w++) s += (double)s_part[w][b][c];
      s_sum[b][c] = s;
    }
    __syncthreads();
    // ---- per edge: Hii = A Hjj A^T, Hij = -A Hjj, Hji = Hij^T, vi = -A vj ; scatter into the reduced system
    // 156 outputs per edge: 144 matrix entries (4 blocks x 36) + 12 vector entries
    for (int k = tid; k < nb * 156; k += kBuildThreads) {
      const int b = k / 156, o = k - b * 156;
      const EdgeSm& S = s_edge[b];
      if (S.stereo) continue;                           // all-zero blocks
      const int pi = ix - t0, pj = S.jx - t0;
      const double* hs = s_sum[b];
      auto H = [&](int a, int c) -> double { return (a >= c) ? hs[a * (a + 1) / 2 + c] : hs[c * (c + 1) / 2 + a]; };
      if (o < 144) {
        const int blk = o / 36, rc = o - blk * 36, r = rc / 6, c = rc - r * 6;
        int prow, pcol; double val = 0.0;
        if (blk == 0) {          // Hii[r][c] = sum_ab A[r][a] Hjj[a][b] A[c][b]
          prow = pi; pcol = pi;
          for (int a = 0; a < 6; a++) { double t = 0.0; for (int b2 = 0; b2 < 6; b2++) t += H(a, b2) * (double)S.A[c * 6 + b2]; val += (double)S.A[r * 6 + a] * t; }
        } else if (blk == 1) {   // Hij[r][c] = -sum_a A[r][a] Hjj[a][c]
          prow = pi; pcol = pj;
          for (int a = 0; a < 6; a++) val -= (double)S.A[r * 6 + a] * H(a, c);
        } else if (blk == 2) {   // Hji[r][c] = Hij[c][r]
          prow = pj; pcol = pi;
          for (int a = 0; a < 6; a++) val -= (double)S.A[c * 6 + a] * H(a, r);
        } else {
          prow = pj; pcol = pj; val = H(r, c);
        }
        if (prow >= 0 && prow < P && pcol >= 0 && pcol < P) atomicAdd(&Hsys[(size_t)(prow * 6 + r) * n + pcol * 6 + c], val);
      } else {
        const int v = o - 144, blk = v / 6, r = v - blk * 6;
        double val = 0.0; int prow;
        if (blk == 0) { prow = pi; for (int a = 0; a < 6; a++) val -= (double)S.A[r * 6 + a] * hs[21 + a]; }
        else { prow = pj; val = hs[21 + r]; }
        if (prow >= 0 && prow < P) atomicAdd(&bsys[prow * 6 + r], val);
      }
    }
  }

  if (!motion_only) {
    // depth block:  C = sum Cii + m*alpha + (1-m)*eta ;  w = sum bz - m*alpha*(d - d_sens)   (reference :1405-1408)
    const float alpha = 0.05f;
    const int erow = (eta_rows == 1) ? 0 : min(eta_by_frame ? ix : m, eta_rows - 1);
#pragma unroll
    for (int s = 0; s < kPPT; s++) {
      const int p = pix[s];
      if (p < HW) {
        const float dsn = __ldg(disps_sens + (size_t)ix * HW + p);
        const float mk = (dsn > 0.f) ? 1.f : 0.f;
        const float C = Cacc[s] + mk * alpha + (1 - mk) * __ldg(eta + (size_t)erow * HW + p);
        const float w = wacc[s] - mk * alpha * (dsp[s] - dsn);
        Cout[(size_t)m * HW + p] = C;
        wout[(size_t)m * HW + p] = w;
#pragma unroll
        for (int c = 0; c < 6; c++) Eiout[((size_t)m * 6 + c) * HW + p] = Eiacc[s][c];
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------------
// Schur complement:  Hsys -= sum_k E_k Q_k E_k^T ,  bsys -= sum_k E_k Q_k w_k       (reference K9/K10 + schur_block)
// rows of frame k: (pose k, Ei_k) if k is in [t0,t1), then (pose jj[e], Eij[e]) for the out-edges e of k; rows whose pose
// is outside [t0,t1) are dropped (they contribute nothing, reference :1155,:1257).
// Two kernels share the work: ba_schur_small_kernel (frames with <= 16 rows, the usual case) and ba_schur_gemm_kernel (more rows:
// dense graphs, edge-sharded ranks).  Both keep 6x6 block pairs in registers over a whole pixel chunk, accumulate in fp32 like the
// reference and flush once with fp64 atomics into the LOWER triangle of the reduced system.
// ---------------------------------------------------------------------------------------------------------
// Q = 1/C of the eliminated depth block.  C <= 0 only for a pixel with eta = 0 and no weight on any edge; the reference divides
// anyway (inf -> NaN system -> zero pose update and NaN depths at that pixel).  All Schur kernels and the back-substitution here
// drop such a pixel instead (Q = 0, dz = 0): one rule on every path, documented in INTEGRATION.md.
__device__ __forceinline__ float safe_rcp(float c) { return c > 0.f ? 1.0f / c : 0.f; }

constexpr int kSchurMaxRows = 255;   // rows per frame (out-degree + 1); larger frames raise ST_DEGREE

// Row list of a depth frame: (pose ix, Ei) first when ix is inside the window, then (pose jj[e], Eij[e]) for its out-edges in CSR
// order whose target pose is inside the window.  Built by the whole CTA: thread a handles out-edge a, an order-preserving
// ballot compaction keeps the reference's row order.  Ends with a __syncthreads().
template <int kThreads>
__device__ __forceinline__ void build_row_list(const int64_t* __restrict__ jj, int* __restrict__ hdr, const int* __restrict__ edgeidx,
                                               int e_begin, int deg, int ix, int m, int HW, int t0, int P, const float* __restrict__ Eij,
                                               const float* __restrict__ Eiin, int* s_pose, const float** s_ptr, int* s_nrows, int* s_wcount) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const bool self = (ix >= t0 && ix < t0 + P);
  int pj = -1, e = -1;
  if (tid < deg && tid < kSchurMaxRows - 1) { e = edgeidx[e_begin + tid]; pj = (int)jj[e] - t0; }
  const bool keep = (pj >= 0 && pj < P);
  const unsigned bal = __ballot_sync(0xffffffffu, keep);
  if (lane == 0) s_wcount[warp] = __popc(bal);
  __syncthreads();
  int base = self ? 1 : 0;
  for (int w = 0; w < warp; w++) base += s_wcount[w];
  if (keep) {
    const int pos = base + __popc(bal & ((1u << lane) - 1u));
    s_pose[pos] = pj; s_ptr[pos] = Eij + (size_t)e * 6 * HW;
  }
  if (tid == 0) {
    if (self) { s_pose[0] = ix - t0; s_ptr[0] = Eiin + (size_t)m * 6 * HW; }
    int tot = self ? 1 : 0;
    for (int w = 0; w < kThreads / 32; w++) tot += s_wcount[w];
    *s_nrows = tot;
    if (deg > kSchurMaxRows - 1) atomicOr(&hdr[HDR_STATUS], ST_DEGREE);
  }
  __syncthreads();
}

// ---------------------------------------------------------------------------------------------------------
// Schur complement for frames with many rows (dense graphs / edge-sharded ranks: out-degree >> 12): SGEMM-style kernel.
// C = A diag(Q) A^T with A = [6R x pixels].  A CTA computes one 16-row x 16-row tile pair (96 x 96 scalars) for a pixel
// chunk: thread (ty,tx) owns the 6x6 block pair (row 16*ti+ty, row 16*tj+tx) in registers for the WHOLE chunk (no per-tile
// reductions), the K loop walks 64-pixel shared-memory tiles stored pixel-major so that a thread reads its 6+6 operands as
// three 64-bit broadcasts each: 36 FMA per 6 LDS.64.  Tile pairs (ti >= tj) go over blockIdx.z.
// ---------------------------------------------------------------------------------------------------------
constexpr int kSgRows = 16;                 // rows per tile
constexpr int kSgK = 64;                    // pixels per shared-memory tile
constexpr int kSgStride = kSgRows * 6 + 2;  // 98 floats per pixel line (even -> 8-byte aligned LDS.64)
constexpr int kSgThreads = 256;

__global__ void __launch_bounds__(kSgThreads) ba_schur_gemm_kernel(
    const int64_t* __restrict__ jj, int* __restrict__ hdr, const int* __restrict__ kx, const int* __restrict__ rowptr,
    const int* __restrict__ edgeidx, int HW, int t0, int P, int px_per_cta, int min_rows,
    const float* __restrict__ Eij, const float* __restrict__ Cin, const float* __restrict__ win, const float* __restrict__ Eiin,
    double* __restrict__ Hsys, double* __restrict__ bsys) {
  const int m = blockIdx.y;
  if (m >= hdr[HDR_M]) return;
  const int ix = kx[m];
  const int e_begin = rowptr[m];
  const int deg = rowptr[m + 1] - e_begin;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int ty = tid >> 4, tx = tid & 15;
  const int n = 6 * P;

  __shared__ int s_pose[kSchurMaxRows + 1];
  __shared__ const float* s_ptr[kSchurMaxRows + 1];
  __shared__ int s_nrows;
  __shared__ int s_wcount[kSgThreads / 32];
  extern __shared__ float sg_dyn[];
  float* sA = sg_dyn;
  float* sB = sg_dyn + kSgK * kSgStride;
  __shared__ float sQw[kSgK];
  __shared__ float sQ[kSgK];

  if (deg + 1 <= min_rows) return;                     // at most deg + 1 rows: not this kernel's frame (skips the row-list build)
  build_row_list<kSgThreads>(jj, hdr, edgeidx, e_begin, deg, ix, m, HW, t0, P, Eij, Eiin, s_pose, s_ptr, &s_nrows, s_wcount);
  const int nrows = s_nrows;
  if (nrows <= min_rows) return;                       // smaller frames belong to ba_schur_tc_kernel / ba_schur_small_kernel
  const int nT = (nrows + kSgRows - 1) / kSgRows;
  const int npairs = nT * (nT + 1) / 2;
  const int px_begin = blockIdx.x * px_per_cta;
  const int px_end = min(HW, px_begin + px_per_cta);
  if (px_begin >= px_end) return;

  for (int pr = blockIdx.z; pr < npairs; pr += gridDim.z) {
    int ti = (int)((sqrtf(8.f * (float)pr + 1.f) - 1.f) * 0.5f);
    while (ti * (ti + 1) / 2 > pr) ti--;
    while ((ti + 1) * (ti + 2) / 2 <= pr) ti++;
    const int tj = pr - ti * (ti + 1) / 2;             // ti >= tj
    const int ra = min(kSgRows, nrows - ti * kSgRows), rb = min(kSgRows, nrows - tj * kSgRows);
    const bool diag_tile = (ti == tj);
    const bool active = (ty < ra) && (tx < rb) && (!diag_tile || ty >= tx);
    const bool diag_pair = diag_tile && (ty == tx);
    float acc[36], bacc[6];
#pragma unroll
    for (int k = 0; k < 36; k++) acc[k] = 0.f;
#pragma unroll
    for (int k = 0; k < 6; k++) bacc[k] = 0.f;

    for (int p0 = px_begin; p0 < px_end; p0 += kSgK) {
      const int np = min(kSgK, px_end - p0);
      __syncthreads();
      // ---- stage: A tile scaled by Q, B tile raw; one warp per (row, component) line of 64 pixels, transposed into [px][row*6+c]
      for (int px = tid; px < kSgK; px += kSgThreads) {
        const bool okp = px < np;
        const float q = okp ? safe_rcp(__ldg(Cin + (size_t)m * HW + p0 + px)) : 0.f;
        sQ[px] = q;
        sQw[px] = okp ? __ldg(win + (size_t)m * HW + p0 + px) : 0.f;
      }
      __syncthreads();
      for (int ln = warp; ln < (ra + (diag_tile ? 0 : rb)) * 6; ln += kSgThreads / 32) {
        const int rowl = ln / 6, c = ln - rowl * 6;
        const bool second = rowl >= ra;
        const int row = second ? (tj * kSgRows + rowl - ra) : (ti * kSgRows + rowl);
        const float* src = s_ptr[row] + (size_t)c * HW + p0;
        float* dst = (second ? sB : sA) + (second ? rowl - ra : rowl) * 6 + c;
#pragma unroll
        for (int h = 0; h < kSgK / 32; h++) {
          const int px = h * 32 + lane;
          float v = (px < np) ? __ldg(src + px) : 0.f;
          if (!second) {
            // A operand carries Q = 1/C (reference K9: ei = E*q); diagonal tiles keep the unscaled copy in sB
            if (diag_tile) sB[px * kSgStride + rowl * 6 + c] = v;
            v *= sQ[px];
          }
          dst[px * kSgStride] = v;
        }
      }
      __syncthreads();
      if (active) {
        const float* pa = sA + ty * 6;
        const float* pb = sB + tx * 6;
#pragma unroll 4
        for (int px = 0; px < kSgK; px++) {
          const float2 a01 = *reinterpret_cast<const float2*>(pa + px * kSgStride);
          const float2 a23 = *reinterpret_cast<const float2*>(pa + px * kSgStride + 2);
          const float2 a45 = *reinterpret_cast<const float2*>(pa + px * kSgStride + 4);
          const float2 b01 = *reinterpret_cast<const float2*>(pb + px * kSgStride);
          const float2 b23 = *reinterpret_cast<const float2*>(pb + px * kSgStride + 2);
          const float2 b45 = *reinterpret_cast<const float2*>(pb + px * kSgStride + 4);
          const float ea[6] = {a01.x, a01.y, a23.x, a23.y, a45.x, a45.y};
          const float eb[6] = {b01.x, b01.y, b23.x, b23.y, b45.x, b45.y};
#pragma unroll
          for (int a = 0; a < 6; a++)
#pragma unroll
            for (int c = 0; c < 6; c++) acc[a * 6 + c] += ea[a] * eb[c];
          if (diag_pair) {
            const float w = sQw[px];          // (Q E) w = Q w E
#pragma unroll
            for (int c = 0; c < 6; c++) bacc[c] += w * ea[c];
          }
        }
      }
    }
    // ---- flush this thread's block pair into the lower triangle
    if (active) {
      const int pa_ = s_pose[ti * kSgRows + ty], pb_ = s_pose[tj * kSgRows + tx];
#pragma unroll
      for (int a = 0; a < 6; a++) {
#pragma unroll
        for (int c = 0; c < 6; c++) {
          const double v = -(double)acc[a * 6 + c];
          const int gr = pa_ * 6 + a, gc = pb_ * 6 + c;
          if (diag_pair) {
            if (gr >= gc) atomicAdd(&Hsys[(size_t)gr * n + gc], v);
          } else {
            if (gr >= gc) atomicAdd(&Hsys[(size_t)gr * n + gc], v);
            if (gc >= gr) atomicAdd(&Hsys[(size_t)gc * n + gr], v);
          }
        }
      }
      if (diag_pair) {
#pragma unroll
        for (int a = 0; a < 6; a++) atomicAdd(&bsys[pa_ * 6 + a], -(double)bacc[a]);
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------------
// Schur complement for frames with at most 16 rows (the usual case: out-degree + 1): the same register-resident 6x6 block pairs
// as the SGEMM-style kernel, but the T = R(R+1)/2 pairs of a frame do not fill a CTA, so the 256 threads form G = 256/T groups
// that split the pixels of every 64-pixel tile (a K split); the groups' partial blocks meet once in shared memory at the end and
// the CTA flushes T x 42 values with fp64 atomics.  The next tile travels global -> registers while the current one is being
// multiplied (36 FMA per 6 LDS.64 per pixel and thread).
// ---------------------------------------------------------------------------------------------------------
constexpr int kSsLines = (kSgRows * 6) / (kSgThreads / 32);     // (row, component) lines per warp: 12

__global__ void __launch_bounds__(kSgThreads, 2) ba_schur_small_kernel(
    const int64_t* __restrict__ jj, int* __restrict__ hdr, const int* __restrict__ kx, const int* __restrict__ rowptr,
    const int* __restrict__ edgeidx, int HW, int t0, int P, int px_per_cta,
    const float* __restrict__ Eij, const float* __restrict__ Cin, const float* __restrict__ win, const float* __restrict__ Eiin,
    double* __restrict__ Hsys, double* __restrict__ bsys) {
  const int m = blockIdx.y;
  if (m >= hdr[HDR_M]) return;
  const int ix = kx[m];
  const int e_begin = rowptr[m];
  const int deg = rowptr[m + 1] - e_begin;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n = 6 * P;

  __shared__ int s_pose[kSchurMaxRows + 1];
  __shared__ const float* s_ptr[kSchurMaxRows + 1];
  __shared__ int s_nrows;
  __shared__ int s_wcount[kSgThreads / 32];
  extern __shared__ float sg_dyn[];
  float* sA = sg_dyn;                                  // [64 px][98]: rows scaled by Q = 1/C
  float* sB = sg_dyn + kSgK * kSgStride;               // raw rows
  __shared__ float sQw[kSgK];

  build_row_list<kSgThreads>(jj, hdr, edgeidx, e_begin, deg, ix, m, HW, t0, P, Eij, Eiin, s_pose, s_ptr, &s_nrows, s_wcount);
  const int nrows = s_nrows;
  if (nrows == 0 || nrows > kSgRows) return;           // larger frames belong to ba_schur_gemm_kernel
  const int px_begin = blockIdx.x * px_per_cta;
  const int px_end = min(HW, px_begin + px_per_cta);
  if (px_begin >= px_end) return;

  const int T = nrows * (nrows + 1) / 2;
  const int G = kSgThreads / T;                        // T <= 136 -> G >= 1
  const int g = tid / T;
  const int pr = tid - g * T;
  const bool active = g < G;
  int ty = (int)((sqrtf(8.f * (float)pr + 1.f) - 1.f) * 0.5f);       // pr -> (ty >= tx)
  while (ty * (ty + 1) / 2 > pr) ty--;
  while ((ty + 1) * (ty + 2) / 2 <= pr) ty++;
  const int tx = pr - ty * (ty + 1) / 2;
  const bool diag_pair = (ty == tx);
  const int nlines = nrows * 6;

  float acc[36], bacc[6];
#pragma unroll
  for (int k = 0; k < 36; k++) acc[k] = 0.f;
#pragma unroll
  for (int k = 0; k < 6; k++) bacc[k] = 0.f;

  float pre[kSsLines][2], q0, q1, w0, w1;
  auto load_tile = [&](int p0) {
    const int np = min(kSgK, px_end - p0);
    const bool ok0 = lane < np, ok1 = lane + 32 < np;
    const size_t base = (size_t)m * HW + p0;
    q0 = ok0 ? safe_rcp(__ldg(Cin + base + lane)) : 0.f;
    q1 = ok1 ? safe_rcp(__ldg(Cin + base + lane + 32)) : 0.f;
    w0 = ok0 ? __ldg(win + base + lane) : 0.f;
    w1 = ok1 ? __ldg(win + base + lane + 32) : 0.f;
#pragma unroll
    for (int i = 0; i < kSsLines; i++) {
      const int ln = warp + (kSgThreads / 32) * i;
      pre[i][0] = 0.f; pre[i][1] = 0.f;
      if (ln < nlines) {
        const int rowl = ln / 6, c = ln - rowl * 6;
        const float* src = s_ptr[rowl] + (size_t)c * HW + p0;
        if (ok0) pre[i][0] = __ldg(src + lane);
        if (ok1) pre[i][1] = __ldg(src + lane + 32);
      }
    }
  };

  load_tile(px_begin);
  for (int p0 = px_begin; p0 < px_end; p0 += kSgK) {
    __syncthreads();                                   // the previous tile has been consumed
#pragma unroll
    for (int i = 0; i < kSsLines; i++) {
      const int ln = warp + (kSgThreads / 32) * i;
      if (ln < nlines) {
        const int o = ln;                              // = row * 6 + component
        sB[lane * kSgStride + o] = pre[i][0];
        sB[(lane + 32) * kSgStride + o] = pre[i][1];
        sA[lane * kSgStride + o] = pre[i][0] * q0;     // ei = E*q   (reference K9)
        sA[(lane + 32) * kSgStride + o] = pre[i][1] * q1;
      }
    }
    if (warp == 0) { sQw[lane] = w0; sQw[lane + 32] = w1; }
    __syncthreads();
    if (p0 + kSgK < px_end) load_tile(p0 + kSgK);      // in flight while this tile is multiplied
    if (active) {
      const float* pa = sA + ty * 6;
      const float* pb = sB + tx * 6;
#pragma unroll 2
      for (int px = g; px < kSgK; px += G) {
        const float2 a01 = *reinterpret_cast<const float2*>(pa + px * kSgStride);
        const float2 a23 = *reinterpret_cast<const float2*>(pa + px * kSgStride + 2);
        const float2 a45 = *reinterpret_cast<const float2*>(pa + px * kSgStride + 4);
        const float2 b01 = *reinterpret_cast<const float2*>(pb + px * kSgStride);
        const float2 b23 = *reinterpret_cast<const float2*>(pb + px * kSgStride + 2);
        const float2 b45 = *reinterpret_cast<const float2*>(pb + px * kSgStride + 4);
        const float ea[6] = {a01.x, a01.y, a23.x, a23.y, a45.x, a45.y};
        const float eb[6] = {b01.x, b01.y, b23.x, b23.y, b45.x, b45.y};
#pragma unroll
        for (int a = 0; a < 6; a++)
#pragma unroll
          for (int c = 0; c < 6; c++) acc[a * 6 + c] += ea[a] * eb[c];
        if (diag_pair) {
          const float w = sQw[px];                     // (Q E) w = Q w E
#pragma unroll
          for (int c = 0; c < 6; c++) bacc[c] += w * ea[c];
        }
      }
    }
  }
  // ---- the G pixel groups meet in shared memory (the staging area is free now), then one flush into the lower triangle
  __syncthreads();
  float* red = sg_dyn;                                 // [G][T][42]
  if (active) {
    float* dst = red + (size_t)(g * T + pr) * 42;
#pragma unroll
    for (int k = 0; k < 36; k++) dst[k] = acc[k];
#pragma unroll
    for (int k = 0; k < 6; k++) dst[36 + k] = bacc[k];
  }
  __syncthreads();
  for (int k = tid; k < T * 42; k += kSgThreads) {
    const int q = k / 42, o = k - q * 42;
    int r2 = (int)((sqrtf(8.f * (float)q + 1.f) - 1.f) * 0.5f);
    while (r2 * (r2 + 1) / 2 > q) r2--;
    while ((r2 + 1) * (r2 + 2) / 2 <= q) r2++;
    const int r = q - r2 * (r2 + 1) / 2;
    const bool same_row = (r == r2);
    if (o >= 36 && !same_row) continue;
    float sum = 0.f;
    for (int gg = 0; gg < G; gg++) sum += red[(size_t)(gg * T + q) * 42 + o];
    const double v = -(double)sum;
    const int pa_ = s_pose[r2], pb_ = s_pose[r];       // block S(pa_, pb_)[a][c]; its transpose sits at (pb_, pa_)[c][a]
    if (o < 36) {
      const int a = o / 6, c = o - a * 6;
      const int gr = pa_ * 6 + a, gc = pb_ * 6 + c;
      if (same_row) {
        if (gr >= gc) atomicAdd(&Hsys[(size_t)gr * n + gc], v);
      } else {
        if (gr >= gc) atomicAdd(&Hsys[(size_t)gr * n + gc], v);
        if (gc >= gr) atomicAdd(&Hsys[(size_t)gc * n + gr], v);
      }
    } else {
      atomicAdd(&bsys[pa_ * 6 + (o - 36)], v);
    }
  }
}

// ---------------------------------------------------------------------------------------------------------
// Schur complement on the tensor cores (frames with at most 21 rows, i.e. every frame of a sliding-window graph):
//   S = X X^T  with  X = [ E_r / sqrt(C) ; w / sqrt(C) ]  (6R + 1 rows x pixels),  so that S[:6R,:6R] = sum E q E^T and
//   S[:6R, 6R] = sum E q w  -- one symmetric rank-K update per frame, K = pixels.
// fp32 accuracy on the tf32 pipe by operand splitting (3xTF32): x = hi + lo with hi = tf32(x), lo = x - hi (exact), and
//   S = hi hi^T + G + G^T,  G = hi lo^T   (the dropped lo lo^T term is ~2^-22 relative),
// i.e. TWO tcgen05.mma per 8-pixel K step: G is accumulated once and symmetrised in the epilogue.
// The tensor core truncates every addend to the accumulator's exponent, so a long accumulation chain drifts (measured: one
// accumulator over the whole pixel range -> 1e-4 on the depths).  hi hi^T therefore gets a fresh TMEM accumulator per chunk
// (three 128-column slots in rotation) which the producer warps drain into fp32 registers two chunks later; G is 2^-11 smaller
// and keeps one accumulator for the whole range.
// CTA = (frame, pixel range), 288 threads.  Warps 0-7: cp.async their own raw rows of a chunk into a 4-deep warp-private raw ring,
// split them into the two K-major SWIZZLE_128B operand tiles [128 rows x 32 px] of a 4-deep operand ring (generic-proxy stores +
// fence.proxy.async), drain accumulators, and finally add the lower triangle into the reduced system with fp64 atomics.
// Warp 8: one thread issues the MMAs (M = 128, both operands described from the SAME tile) and commits to the mbarriers.
// Frames with 6R + 2 <= 64 (R <= 10) run "packed": the two halves of a 64-pixel chunk sit in operand rows 0..63 and 64..127,
// one M = N = 128 MMA then yields both halves' products on the diagonal blocks (the MMA cost is set by the 128 operand rows
// it streams whether they are live or not), and the epilogue adds the two blocks.
// ---------------------------------------------------------------------------------------------------------
constexpr int kTcRowsMax = 21;
constexpr int kPairTileRows = 10;               // pair mode: row tiles of 10 frame rows (60 lines + the w line <= 64 operand rows)
constexpr int kPairRowsMax = 100;               // pair mode handles 22..100 rows (up to 45 tile pairs over gridDim.z); more rows: SIMT kernel
constexpr int kPairGridZ = 45;
constexpr int kTcThreads = 288;
constexpr int kTcProducers = 256;
constexpr int kTcRawStages = 4;
constexpr int kTcRawBytes = 128 * 128;          // up to 128 lines (6R rows, w, C; two halves when packed) x 128 bytes
constexpr int kTcOpBytes = 128 * 128;           // one operand tile (hi or lo)
constexpr int kTcOpStages = 4;
constexpr int kTcAccSlots = 3;                  // rotating TMEM accumulators (128 columns each) for hi hi^T; G lives in columns 384..511
constexpr int kTcCxStride = 129;                // floats per row of the G staging matrix (conflict-free transposed reads)
constexpr int kTcSmem = kTcRawStages * kTcRawBytes + kTcOpStages * 2 * kTcOpBytes + 1024 /*alignment*/ + 256 /*barriers*/;
static_assert(128 * kTcCxStride * 4 <= kTcOpStages * 2 * kTcOpBytes, "G staging matrix must fit the operand ring");

__device__ __forceinline__ void cp_async16_zfill(uint32_t dst, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ float lds_f32(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void sts_f32(uint32_t addr, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory"); }

// PAIR mode (frames with 22..100 rows: dense graphs, edge-sharded ranks): the rows are cut into tiles of 10; CTA (frame, pair z) stacks
// tile a in operand rows 0..63 and tile b in rows 64..127 over the SAME 32 pixels (the packed layout with a zero pixel offset for the
// second half), so the one M = N = 128 product holds S_ba in its lower-left block and S_aa / S_bb on the diagonal (emitted only by
// the designated pair (t, t+1)); G + G^T symmetrisation unchanged.  Off-diagonal-block entries go to (max, min) of the global
// indices and count twice where two different rows share a pose.
template <bool PAIR>
__global__ void __launch_bounds__(kTcThreads, 1) ba_schur_tc_kernel(
    const int64_t* __restrict__ jj, int* __restrict__ hdr, const int* __restrict__ kx, const int* __restrict__ rowptr,
    const int* __restrict__ edgeidx, int HW, int t0, int P, int px_per_cta,
    const float* __restrict__ Eij, const float* __restrict__ Cin, const float* __restrict__ win, const float* __restrict__ Eiin,
    double* __restrict__ Hsys, double* __restrict__ bsys, const int* __restrict__ big) {
  if (PAIR && (int)blockIdx.y >= hdr[HDR_NBIG]) return;          // PAIR: blockIdx.y runs over the list of high-degree depth frames
  const int m = PAIR ? big[blockIdx.y] : blockIdx.y;
  if (m >= hdr[HDR_M]) return;
  const int ix = kx[m];
  const int e_begin = rowptr[m];
  const int deg = rowptr[m + 1] - e_begin;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n = 6 * P;

  __shared__ int s_pose[kSchurMaxRows + 1];
  __shared__ const float* s_ptr[kSchurMaxRows + 1];
  __shared__ int s_nrows;
  __shared__ int s_wcount[kTcThreads / 32];
  __shared__ int s_gidx[128];                     // operand row / column -> index in the reduced system (-1: rhs, -2: padding)
  extern __shared__ uint8_t tc_smem_raw[];

  if (deg == 0) return;                           // no out-edge (e.g. a frame another rank owns): E_k = 0, nothing to subtract
  if (PAIR) {                                     // cheap exits before the row-list build: at most deg + 1 rows
    if (deg + 1 <= kTcRowsMax) return;
    const int tmax = (min(deg + 1, kPairRowsMax) + kPairTileRows - 1) / kPairTileRows;
    if ((int)blockIdx.z >= tmax * (tmax - 1) / 2) return;
  }
  build_row_list<kTcThreads>(jj, hdr, edgeidx, e_begin, deg, ix, m, HW, t0, P, Eij, Eiin, s_pose, s_ptr, &s_nrows, s_wcount);
  const int nrows = s_nrows;
  if (!PAIR && (nrows == 0 || nrows > kTcRowsMax)) return;            // larger frames belong to the pair-mode launch / ba_schur_gemm_kernel
  if (PAIR && (nrows <= kTcRowsMax || nrows > kPairRowsMax)) return;
  int ta = 0, tb = 0;                                    // PAIR: the two row tiles of this CTA (ta < tb)
  bool emit_a = true, emit_b = true;
  if (PAIR) {
    const int T = (nrows + kPairTileRows - 1) / kPairTileRows;         // >= 3
    const int pr = blockIdx.z;
    if (pr >= T * (T - 1) / 2) return;
    tb = (int)((sqrtf(8.f * (float)pr + 1.f) + 1.f) * 0.5f);
    while (tb * (tb - 1) / 2 > pr) tb--;
    while ((tb + 1) * tb / 2 <= pr) tb++;
    ta = pr - tb * (tb - 1) / 2;
    emit_a = (tb == ta + 1);                             // S_tt of tile t < T-1 comes from pair (t, t+1), of tile T-1 from pair (T-2, T-1)
    emit_b = (tb == T - 1 && ta == T - 2);
  }
  const int px_begin = blockIdx.x * px_per_cta;
  const int px_end = min(HW, px_begin + px_per_cta);
  if (px_begin >= px_end) return;
  const int R6a = PAIR ? 6 * min(kPairTileRows, nrows - kPairTileRows * ta) : 6 * nrows;
  const int R6b = PAIR ? 6 * min(kPairTileRows, nrows - kPairTileRows * tb) : 6 * nrows;
  const int R6 = R6a;                                    // operand rows 0..R6-1: E rows, row R6: w  (PAIR: of the half, see R6h)
  const bool packed = !PAIR && (R6 + 2 <= 64);          // two PIXEL halves of a 64-pixel chunk in operand rows 0..63 / 64..127
  const bool two_halves = PAIR || packed;                // operand rows 64..127 carry a second set of lines
  const int nhalf = packed ? 2 : 1;
  const int cpx = 32 * nhalf;                            // pixels per chunk
  const int nchunks = (px_end - px_begin + cpx - 1) / cpx;
  const int N = two_halves ? 128 : ((R6 + 1 + 15) & ~15);    // MMA N

  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(tc_smem_raw) + 1023) & ~(uintptr_t)1023);
  const uint32_t op_base = smem_u32(smem);               // [stage][hi|lo][128 rows][128 B], 1024-byte aligned tiles
  const uint32_t raw_base = op_base + kTcOpStages * 2 * kTcOpBytes;   // [stage][row][128 B]
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kTcOpStages * 2 * kTcOpBytes + kTcRawStages * kTcRawBytes);
  uint64_t* full = bars;                                 // [4] operand stage written (8 producer warps arrive)
  uint64_t* empty = bars + kTcOpStages;                  // [4] operand stage consumed (tcgen05.commit)
  uint64_t* acc_full = bars + 2 * kTcOpStages;           // [3] accumulator slot holds one chunk's hi hi^T (tcgen05.commit)
  uint64_t* acc_empty = acc_full + kTcAccSlots;          // [3] slot drained into registers (8 warps arrive)
  uint64_t* done = acc_empty + kTcAccSlots;              // every MMA has completed
  uint32_t* tmem_base_smem = reinterpret_cast<uint32_t*>(done + 2);

  if (tid < 128) {
    if (PAIR) {                                          // operand row -> index in the reduced system, per half
      const int hfx = tid >> 6, ln = tid & 63, R6x = hfx ? R6b : R6a, row0 = kPairTileRows * (hfx ? tb : ta);
      s_gidx[tid] = (ln < R6x) ? s_pose[row0 + ln / 6] * 6 + (ln % 6) : (ln == R6x ? -1 : -2);
    } else s_gidx[tid] = (tid < R6) ? s_pose[tid / 6] * 6 + (tid % 6) : (tid == R6 ? -1 : -2);
  }
  if (tid == 0) {
    for (int s = 0; s < kTcOpStages; s++) { mbar_init(full + s, kTcProducers / 32); mbar_init(empty + s, 1); }
    for (int s = 0; s < kTcAccSlots; s++) { mbar_init(acc_full + s, 1); mbar_init(acc_empty + s, kTcProducers / 32); }
    mbar_init(done, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 8) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_base_smem)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  } else {
    // operand tiles start as zeros: rows that carry no line are never written again
    uint4* z = reinterpret_cast<uint4*>(smem);
    for (int k = tid; k < kTcOpStages * 2 * kTcOpBytes / 16; k += kTcProducers) z[k] = make_uint4(0u, 0u, 0u, 0u);
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_base_smem;

  if (warp == 8) {
    // ================= MMA issuer =================
    if (lane == 0) {
      const uint32_t idesc = umma_idesc_tf32(128, N);
      const uint32_t d_g = tmem_base + 3 * 128;
      for (int c = 0; c < nchunks; c++) {
        const int os = c % kTcOpStages, slot = c % kTcAccSlots;
        mbar_wait(full + os, (c / kTcOpStages) & 1);
        if (c >= kTcAccSlots) mbar_wait(acc_empty + slot, ((c / kTcAccSlots) - 1) & 1);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t hi0 = op_base + (uint32_t)os * 2 * kTcOpBytes, lo0 = hi0 + kTcOpBytes;
        const uint32_t d = tmem_base + (uint32_t)(slot * 128);
#pragma unroll
        for (int k = 0; k < 4; k++) {
          const uint64_t dh = umma_desc_k_sw128(hi0 + k * 32, 1024), dl = umma_desc_k_sw128(lo0 + k * 32, 1024);
          umma_tf32(d, dh, dh, idesc, k > 0 ? 1u : 0u);
          umma_tf32(d_g, dh, dl, idesc, (c > 0 || k > 0) ? 1u : 0u);
        }
        umma_commit(empty + os);          // the operand stage may be overwritten once these MMAs have read it
        umma_commit(acc_full + slot);     // ... and the chunk's hi hi^T is ready to be drained
      }
      umma_commit(done);
    }
    __syncwarp();
  } else {
    // ================= producers: raw rows -> split operands =================
    // Every warp stages and splits its OWN lines (line = warp + 8 i), so the only CTA-wide coupling is through the mbarriers.
    // Warp-private raw slab: 16 rows x 128 B per stage; slab row li = i (not packed) or hf * 8 + i (packed: half hf of the chunk).
    // A thread owns four (slab row, 16-byte piece) copy slots: li = 4 s + lane / 8, piece = lane % 8.
    const float* src[4];
    uint32_t dst[4];
    int pxo[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
      const int li = 4 * i + (lane >> 3), piece = lane & 7;
      const int hf = two_halves ? (li >> 3) : 0, line = warp + 8 * (two_halves ? (li & 7) : li);
      const int R6x = PAIR ? (hf ? R6b : R6a) : R6, row0 = PAIR ? kPairTileRows * (hf ? tb : ta) : 0;
      // slots without a line copy zero bytes (cp.async zero-fills) into their unused slab row: no branch in the copy loop
      src[i] = Cin; pxo[i] = 1 << 30;
      dst[i] = raw_base + warp * 2048 + li * 128 + piece * 16;
      if (line <= R6x) {
        const float* base = (line < R6x) ? s_ptr[row0 + line / 6] + (size_t)(line % 6) * HW : win + (size_t)m * HW;
        pxo[i] = (packed ? hf * 32 : 0) + piece * 4;
        src[i] = base + pxo[i];
      }
    }
    const float* Cm = Cin + (size_t)m * HW;
    // this thread's share of S: operand row q*32 + lane; column blocks of 32: packed -> the one block of its own half,
    // otherwise half_w*32 and 64 + half_w*32
    const int q = warp & 3, half_w = warp >> 2;
    const int row = q * 32 + lane;
    const int lrow = packed ? (row & 63) : row;                     // line of this row
    const int lq = two_halves ? (q & 1) : q;                        // 32-row group inside the half
    const int ncb = packed ? 1 : 2;
    const int cb0 = packed ? ((q >> 1) * 64 + half_w * 32) : half_w * 32;
    const int R6q = PAIR ? ((q >> 1) ? R6b : R6a) : R6;             // lines of this row's half
    // PAIR: which of this thread's two column blocks are wanted: rows of tile a only need S_aa (block 0, if this CTA emits it);
    // rows of tile b need S_ba (block 0) and S_bb (block 1, if emitted)
    const bool need0 = !PAIR || ((q >> 1) ? true : emit_a);
    const bool need1 = !PAIR || ((q >> 1) ? emit_b : false);
    float acc[2][32];
#pragma unroll
    for (int h = 0; h < 2; h++)
#pragma unroll
      for (int j = 0; j < 32; j++) acc[h][j] = 0.f;
    auto drain = [&](int cd) {
      const int slot = cd % kTcAccSlots;
      mbar_wait(acc_full + slot, (cd / kTcAccSlots) & 1);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
      for (int h = 0; h < 2; h++) {
        const int cb = cb0 + h * 64;
        if (h < ncb && cb < N && lq * 32 < R6q && (h ? need1 : need0)) {     // warp-uniform: groups without live rows skip the TMEM read
          uint32_t r[32];
          tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(slot * 128 + cb), r);
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
          for (int j = 0; j < 32; j++) acc[h][j] += __uint_as_float(r[j]);
        }
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncwarp();
      if (lane == 0) mbar_arrive(acc_empty + slot);
    };
    auto issue = [&](int c) {
      if (c < nchunks) {
        const int p0 = px_begin + c * cpx;
        const uint32_t stage_off = (uint32_t)(c % kTcRawStages) * kTcRawBytes;
#pragma unroll
        for (int i = 0; i < 4; i++) {
          const bool ok = p0 + pxo[i] < px_end;            // false for slots without a line (pxo = 2^30)
          cp_async16_zfill(dst[i] + stage_off, ok ? (const void*)(src[i] + p0) : (const void*)Cin, ok ? 16u : 0u);
        }
      }
      asm volatile("cp.async.commit_group;" ::: "memory");
    };
#pragma unroll
    for (int s = 0; s < kTcRawStages - 1; s++) issue(s);

    // A thread splits exactly the 16-byte pieces it copied (slot i: slab row 4 i + lane / 8, pixels 4 (lane % 8) .. + 3): one
    // 128-bit shared load, four scale / round / subtract chains, two 128-bit swizzled stores per slot.  A 16-byte piece stays
    // contiguous under the 128-byte swizzle (chunk index ^ row % 8).
    const int piece = lane & 7;
    uint32_t op_off[4];                                      // byte offset of the slot's piece inside an operand tile
    bool live[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
      const int li = 4 * i + (lane >> 3);
      const int hf = two_halves ? (li >> 3) : 0, line = warp + 8 * (two_halves ? (li & 7) : li);
      const uint32_t rr = (uint32_t)(hf * 64 + line);
      live[i] = line <= (PAIR ? (hf ? R6b : R6a) : R6);
      op_off[i] = rr * 128 + (((uint32_t)piece ^ (rr & 7u)) << 4);
    }
    auto load_c4 = [&](int c, int hf) -> float4 {          // C of this thread's four pixels in half hf of chunk c (0 beyond the range)
      const int px = px_begin + c * cpx + hf * 32 + 4 * piece;
      return (c < nchunks && px < px_end) ? __ldg(reinterpret_cast<const float4*>(Cm + px)) : make_float4(0.f, 0.f, 0.f, 0.f);
    };
    auto rsq4 = [](float4 v) -> float4 {                     // sqrt(Q); pixels beyond the range stay zero
      return make_float4(v.x > 0.f ? rsqrtf(v.x) : 0.f, v.y > 0.f ? rsqrtf(v.y) : 0.f, v.z > 0.f ? rsqrtf(v.z) : 0.f, v.w > 0.f ? rsqrtf(v.w) : 0.f);
    };
    float4 Cn0 = load_c4(0, 0), Cn1 = packed ? load_c4(0, 1) : make_float4(0.f, 0.f, 0.f, 0.f);
    for (int c = 0; c < nchunks; c++) {
      asm volatile("cp.async.wait_group %0;" ::"n"(kTcRawStages - 2) : "memory");
      __syncwarp();                                          // this warp's copies of chunk c have landed
      const int os = c % kTcOpStages;
      if (c >= kTcOpStages) mbar_wait(empty + os, ((c / kTcOpStages) - 1) & 1);
      const uint32_t raw = raw_base + (uint32_t)(c % kTcRawStages) * kTcRawBytes + (uint32_t)warp * 2048 + (uint32_t)(lane >> 3) * 128 +
                           (uint32_t)piece * 16;
      const uint32_t ophi = op_base + (uint32_t)os * 2 * kTcOpBytes;
      const float4 sq0 = rsq4(Cn0), sq1 = rsq4(Cn1);
      Cn0 = load_c4(c + 1, 0); Cn1 = packed ? load_c4(c + 1, 1) : Cn1;      // one chunk ahead
      float4 xv[4];
#pragma unroll
      for (int i = 0; i < 4; i++)
        asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(xv[i].x), "=f"(xv[i].y), "=f"(xv[i].z), "=f"(xv[i].w) : "r"(raw + (uint32_t)i * 512) : "memory");
#pragma unroll
      for (int i = 0; i < 4; i++) {
        const float4 q = (packed && i >= 2) ? sq1 : sq0;
        const float x[4] = {xv[i].x * q.x, xv[i].y * q.y, xv[i].z * q.z, xv[i].w * q.w};
        float hi[4], lo[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {                        // tf32 round-to-nearest (ties away), as cvt.rna.tf32.f32 for finite x
          hi[k] = __uint_as_float((__float_as_uint(x[k]) + 0x1000u) & 0xffffe000u);
          lo[k] = x[k] - hi[k];
        }
        if (live[i]) {
          asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(ophi + op_off[i]), "f"(hi[0]), "f"(hi[1]), "f"(hi[2]), "f"(hi[3]) : "memory");
          asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(ophi + kTcOpBytes + op_off[i]), "f"(lo[0]), "f"(lo[1]), "f"(lo[2]), "f"(lo[3]) : "memory");
        }
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");         // generic-proxy stores -> visible to the tensor core
      __syncwarp();
      if (lane == 0) mbar_arrive(full + os);
      issue(c + kTcRawStages - 1);
      if (c >= 2) drain(c - 2);
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    if (nchunks >= 2) drain(nchunks - 2);
    drain(nchunks - 1);

    // ================= G = hi lo^T: through shared memory (the operand ring is idle now) so that G + G^T can be formed
    mbar_wait(done, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
    for (int h = 0; h < 2; h++) {
      const int cb = cb0 + h * 64;
      if (h < ncb && cb < N && lq * 32 <= R6q) {                     // PAIR: all four blocks of G (the lower-left block needs G^T from the upper right)
        uint32_t r[32];
        tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(3 * 128 + cb), r);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int j = 0; j < 32; j++) sts_f32(op_base + (uint32_t)(row * kTcCxStride + cb + j) * 4, __uint_as_float(r[j]));
      }
    }
    asm volatile("bar.sync 1, %0;" ::"n"(kTcProducers) : "memory");

    // ================= epilogue: lower triangle of S (and the rhs column) into the reduced system =================
    const int gr = PAIR ? s_gidx[row] : ((lrow < R6) ? s_gidx[lrow] : -2);
    if (gr >= 0) {
      const int cofs = packed ? (row & 64) : 0;                     // first operand column of this row's half
#pragma unroll
      for (int h = 0; h < 2; h++) {
        const int cb = cb0 + h * 64;
        if (h < ncb && cb < N && (h ? need1 : need0)) {
          const bool cross = PAIR && ((row >> 6) != (cb >> 6));     // lower-left block S_ba: every unordered row pair appears once
#pragma unroll
          for (int j = 0; j < 32; j++) {
            const int col = cb + j;
            const int gc = s_gidx[col - cofs];
            if (gc == -2) continue;
            const float g = lds_f32(op_base + (uint32_t)(row * kTcCxStride + col) * 4) + lds_f32(op_base + (uint32_t)(col * kTcCxStride + row) * 4);
            const double v = -(double)(acc[h][j] + g);
            if (cross) {
              if (gc < 0) continue;                                 // the rhs comes from the diagonal blocks
              if (gr > gc) atomicAdd(&Hsys[(size_t)gr * n + gc], v);
              else if (gr < gc) atomicAdd(&Hsys[(size_t)gc * n + gr], v);
              else atomicAdd(&Hsys[(size_t)gr * n + gr], 2.0 * v);  // two different rows with the same pose: (r,c) and (c,r) land on one entry
            } else if (gc >= 0) {
              if (gr >= gc) atomicAdd(&Hsys[(size_t)gr * n + gc], v);
            } else {
              atomicAdd(&bsys[gr], v);
            }
          }
        }
      }
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 8) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
}

// ---------------------------------------------------------------------------------------------------------
// back substitution + retractions
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void exp_so3(const float* phi, float* q) {
  const float theta_sq = phi[0] * phi[0] + phi[1] * phi[1] + phi[2] * phi[2];
  const float theta_p4 = theta_sq * theta_sq;
  const float theta = sqrtf(theta_sq);
  float imag, real;
  if ((double)theta_sq < 1e-8) {        // double literal comparison in the reference (:128)
    imag = (float)(0.5 - (1.0 / 48.0) * (double)theta_sq + (1.0 / 3840.0) * (double)theta_p4);
    real = (float)(1.0 - (1.0 / 8.0) * (double)theta_sq + (1.0 / 384.0) * (double)theta_p4);
  } else {
    imag = (float)((double)sinf((float)(0.5 * (double)theta)) / (double)theta);
    real = cosf((float)(0.5 * (double)theta));
  }
  q[0] = imag * phi[0]; q[1] = imag * phi[1]; q[2] = imag * phi[2]; q[3] = real;
}

__device__ __forceinline__ void cross_inplace(const float* a, float* b) {
  const float x0 = a[1] * b[2] - a[2] * b[1], x1 = a[2] * b[0] - a[0] * b[2], x2 = a[0] * b[1] - a[1] * b[0];
  b[0] = x0; b[1] = x1; b[2] = x2;
}

__device__ __forceinline__ void exp_se3(const float* xi, float* t, float* q) {
  exp_so3(xi + 3, q);
  float tau[3] = {xi[0], xi[1], xi[2]};
  const float phi[3] = {xi[3], xi[4], xi[5]};
  const float theta_sq = phi[0] * phi[0] + phi[1] * phi[1] + phi[2] * phi[2];
  const float theta = sqrtf(theta_sq);
  t[0] = tau[0]; t[1] = tau[1]; t[2] = tau[2];
  if ((double)theta > 1e-4) {
    const float a = (1 - cosf(theta)) / theta_sq;
    cross_inplace(phi, tau);
    t[0] += a * tau[0]; t[1] += a * tau[1]; t[2] += a * tau[2];
    const float b = (theta - sinf(theta)) / (theta * theta_sq);
    cross_inplace(phi, tau);
    t[0] += b * tau[0]; t[1] += b * tau[1]; t[2] += b * tau[2];
  }
}

__global__ void __launch_bounds__(256) ba_backsub_kernel(
    const int64_t* __restrict__ jj, const int* __restrict__ hdr, const int* __restrict__ kx, const int* __restrict__ rowptr,
    const int* __restrict__ edgeidx, int HW, int t0, int P,
    const float* __restrict__ Eij, const float* __restrict__ Cin, const float* __restrict__ win, const float* __restrict__ Eiin,
    const float* __restrict__ dx, float* __restrict__ disps, float* __restrict__ dz_out, int own_lo, int own_hi) {
  const int m = blockIdx.y;
  if (m >= hdr[HDR_M]) return;
  const int ix = kx[m];
  const bool owned = ix >= own_lo && ix < own_hi;   // edge-sharded runs: other ranks hold the out-edges of the other frames
  const int e_begin = rowptr[m], e_end = rowptr[m + 1];
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= HW) return;
  // dw = sum over rows of frame m of  E[row,:,p] . dx[pose]   with the Q9 guard 0 < pose < P   (reference :1114)
  float dw = 0.f;
  {
    const int ps = ix - t0;
    if (ps > 0 && ps < P) {
      float s = 0.f;
#pragma unroll
      for (int c = 0; c < 6; c++) s += __ldg(Eiin + ((size_t)m * 6 + c) * HW + p) * __ldg(dx + ps * 6 + c);
      dw += s;
    }
  }
  for (int a = e_begin; a < e_end; a++) {
    const int e = edgeidx[a];
    const int pj = (int)jj[e] - t0;
    if (pj > 0 && pj < P) {
      float s = 0.f;
#pragma unroll
      for (int c = 0; c < 6; c++) s += __ldg(Eij + ((size_t)e * 6 + c) * HW + p) * __ldg(dx + pj * 6 + c);
      dw += s;
    }
  }
  const float q = safe_rcp(__ldg(Cin + (size_t)m * HW + p));
  const float dz = q * (__ldg(win + (size_t)m * HW + p) - dw);
  dz_out[(size_t)m * HW + p] = owned ? dz : 0.f;
  if (owned) disps[(size_t)ix * HW + p] += dz;       // K8 (:942-955)
}

__global__ void ba_pose_retr_kernel(float* __restrict__ poses, const float* __restrict__ dx, int t0, int P, float* __restrict__ dx_out,
                                    int* __restrict__ hdr) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k == 0 && hdr[HDR_CHOL_FAIL]) atomicOr(&hdr[HDR_STATUS], ST_CHOL_FAIL);   // sticky: some iteration was not SPD (its dx is 0)
  if (k >= P) return;
  float xi[6], t[3], q[4], dt[3] = {0, 0, 0}, dq[4] = {0, 0, 0, 1}, t1[3], q1[4];
  float* ps = poses + 7 * (size_t)(t0 + k);
#pragma unroll
  for (int c = 0; c < 6; c++) { xi[c] = dx[k * 6 + c]; if (dx_out) dx_out[k * 6 + c] = xi[c]; }
  t[0] = ps[0]; t[1] = ps[1]; t[2] = ps[2];
  q[0] = ps[3]; q[1] = ps[4]; q[2] = ps[5]; q[3] = ps[6];
  exp_se3(xi, dt, dq);
  q1[0] = dq[3] * q[0] + dq[0] * q[3] + dq[1] * q[2] - dq[2] * q[1];
  q1[1] = dq[3] * q[1] + dq[1] * q[3] + dq[2] * q[0] - dq[0] * q[2];
  q1[2] = dq[3] * q[2] + dq[2] * q[3] + dq[0] * q[1] - dq[1] * q[0];
  q1[3] = dq[3] * q[3] - dq[0] * q[0] - dq[1] * q[1] - dq[2] * q[2];
  act_so3(dq, t, t1);
  ps[0] = t1[0] + dt[0]; ps[1] = t1[1] + dt[1]; ps[2] = t1[2] + dt[2];
  ps[3] = q1[0]; ps[4] = q1[1]; ps[5] = q1[2]; ps[6] = q1[3];
}

}  // namespace dba
using namespace dba;

// ---------------------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------------------
extern "C" size_t dba_ba_workspace_bytes(int n_frames, int n_edges, int ht, int wd, int t0, int t1) {
  return make_layout(n_frames, n_edges, ht, wd, t0, t1).total;
}
extern "C" size_t dba_ba_system_offset(int n_frames, int n_edges, int ht, int wd, int t0, int t1) {
  return make_layout(n_frames, n_edges, ht, wd, t0, t1).off_sys;
}
extern "C" size_t dba_ba_system_bytes(int t0, int t1) {
  const size_t n = 6 * (size_t)(t1 - t0 > 0 ? t1 - t0 : 0);
  return (n * n + n) * sizeof(double);
}

static int check_ba_args(const dba_ba_args* a, Layout& L) {
  DBA_CHECK_ARG(a != nullptr, "null args");
  DBA_CHECK_ARG(a->n_frames > 0 && a->n_edges >= 0 && a->ht > 0 && a->wd > 0, "bad extents");
  DBA_CHECK_ARG(a->t0 >= 0 && a->t1 >= a->t0 && a->t1 <= a->n_frames, "bad window [t0,t1)");
  DBA_CHECK_ARG(a->poses && a->disps && a->intrinsics && a->disps_sens, "null state pointer");
  DBA_CHECK_ARG(a->n_edges == 0 || (a->targets && a->weights && a->ii && a->jj), "null edge pointer");
  DBA_CHECK_ARG(a->motion_only || (a->eta && a->eta_rows >= 1), "eta missing");
  DBA_CHECK_ARG(a->motion_only || !a->eta_by_frame || a->eta_rows >= a->n_frames, "eta_by_frame needs one eta row per frame");
  DBA_CHECK_ARG(a->own_lo >= 0 && a->own_hi >= a->own_lo, "bad ownership range");
  DBA_CHECK_ARG(a->p2p_world <= 8 && (a->p2p_world <= 1 || (a->p2p_rank >= 0 && a->p2p_rank < a->p2p_world)), "bad p2p rank/world");
  DBA_CHECK_ARG(a->workspace != nullptr, "null workspace");
  DBA_CHECK_ARG(a->n_frames <= 65535, "more than 65535 frames");
  L = make_layout(a->n_frames, a->n_edges, a->ht, a->wd, a->t0, a->t1);
  if (a->workspace_bytes < L.total) { dba::set_error("workspace too small: %zu < %zu", a->workspace_bytes, L.total); return DBA_ERR_WORKSPACE; }
  return DBA_OK;
}

#define WS(T, off) reinterpret_cast<T*>(reinterpret_cast<char*>(a->workspace) + (off))

// where the reduced pose system of this Gauss-Newton iteration is accumulated: the private workspace, or -- for the fused
// peer-to-peer reduction -- slot (epoch & 1) of this rank's peer-visible buffer
static double* system_ptr(const dba_ba_args* a, const Layout& L) {
  if (a->p2p_world > 1) return reinterpret_cast<double*>(a->p2p_system[a->p2p_rank]) + (size_t)(a->p2p_epoch & 1ull) * ((size_t)L.n * L.n + L.n);
  return reinterpret_cast<double*>(reinterpret_cast<char*>(a->workspace) + L.off_sys);
}

extern "C" int dba_ba_prepare(const dba_ba_args* a) {
  Layout L; int rc = check_ba_args(a, L); if (rc) return rc;
  cudaStream_t st = (cudaStream_t)a->stream;
  ba_prepare_kernel<<<1, 1024, 0, st>>>(a->ii, a->jj, a->n_edges, a->n_frames, a->t0, a->t1, (a->motion_only || a->eta_by_frame) ? 1 : a->eta_rows,
                                        WS(int, L.off_hdr), WS(int, L.off_frame2k), WS(int, L.off_kx), WS(int, L.off_rowptr), WS(int, L.off_big));
  DBA_CHECK_LAUNCH("ba_prepare");
  if (a->n_edges > 0) {
    ba_fill_csr_kernel<<<(a->n_edges + 7) / 8, 256, 0, st>>>(a->ii, a->jj, a->n_edges, a->n_frames, WS(int, L.off_frame2k),
                                                                  WS(int, L.off_rowptr), WS(int, L.off_edgeidx));
    DBA_CHECK_LAUNCH("ba_fill_csr");
  }
  return DBA_OK;
}

extern "C" int dba_ba_build(const dba_ba_args* a) {
  Layout L; int rc = check_ba_args(a, L); if (rc) return rc;
  cudaStream_t st = (cudaStream_t)a->stream;
  const int HW = a->ht * a->wd;
  double* Hsys = system_ptr(a, L);
  double* bsys = Hsys + (size_t)L.n * L.n;
  DBA_CHECK_CUDA(cudaMemsetAsync(Hsys, 0, ((size_t)L.n * L.n + L.n) * sizeof(double), st), "ba_build memset");
  DBA_CHECK_CUDA(cudaMemsetAsync(WS(int, L.off_hdr) + HDR_CHOL_FAIL, 0, sizeof(int), st), "ba_build memset");
  if (L.P == 0) return DBA_OK;
  // frames that can own edges on this rank (edge-sharded runs own a sub-range): size the pixel chunks so the grid fills the GPU
  const int eff_frames = std::max(1, std::min(a->n_frames, a->own_hi - a->own_lo));
  const int ppt = (eff_frames * ((HW + 4 * kBuildThreads - 1) / (4 * kBuildThreads)) >= 148) ? 4
                : (eff_frames * ((HW + 2 * kBuildThreads - 1) / (2 * kBuildThreads)) >= 148) ? 2 : 1;
#define LAUNCH_BUILD(PPT)                                                                                                               \
  ba_build_kernel<PPT><<<dim3((HW + PPT * kBuildThreads - 1) / (PPT * kBuildThreads), a->n_frames), kBuildThreads, 0, st>>>(             \
      a->poses, a->disps, a->intrinsics, a->disps_sens, a->targets, a->weights, a->eta, a->eta_rows, a->eta_by_frame, a->jj, WS(int, L.off_hdr),  \
      WS(int, L.off_kx), WS(int, L.off_rowptr), WS(int, L.off_edgeidx), HW, a->wd, a->t0, L.P, a->motion_only, Hsys, bsys,               \
      WS(float, L.off_Eij), WS(float, L.off_C), WS(float, L.off_w), WS(float, L.off_Ei))
  if (ppt == 4) LAUNCH_BUILD(4); else if (ppt == 2) LAUNCH_BUILD(2); else LAUNCH_BUILD(1);
#undef LAUNCH_BUILD
  DBA_CHECK_LAUNCH("ba_build");
  if (!a->motion_only) {
    const size_t smem2 = (size_t)2 * kSgK * kSgStride * sizeof(float);
    // small frames: about 2.5 CTAs per SM worth of (frame, chunk) work items of whole 64-pixel tiles
    const int tiles1 = (HW + kSgK - 1) / kSgK;
    const int chunks1 = std::max(1, std::min(tiles1, (5 * 148 / 2 + eff_frames - 1) / eff_frames));
    const int px_per_cta1 = ((tiles1 + chunks1 - 1) / chunks1) * kSgK;
    const int gx1 = (HW + px_per_cta1 - 1) / px_per_cta1;
    // the SGEMM-style kernel keeps its accumulators in registers over the whole pixel chunk: few long chunks, tile pairs over z
    const int px_per_cta2 = ((HW + 2) / 3 + kSgK - 1) / kSgK * kSgK;
    const int gx2 = (HW + px_per_cta2 - 1) / px_per_cta2;
    const int zsplit2 = std::max(1, std::min(32, (6 * 148 + eff_frames * gx2 - 1) / (eff_frames * gx2)));
    if ((rc = kernel_setup((const void*)ba_schur_gemm_kernel, (int)smem2))) return rc;
    if ((rc = kernel_setup((const void*)ba_schur_small_kernel, (int)smem2))) return rc;
    if ((rc = kernel_setup((const void*)ba_schur_tc_kernel<false>, (int)kTcSmem))) return rc;
    if ((rc = kernel_setup((const void*)ba_schur_tc_kernel<true>, (int)kTcSmem))) return rc;
    // frames with at most 21 rows go to the tensor cores (needs 16-byte aligned pixel rows)
    const bool use_tc = HW % 4 == 0;
    if (use_tc) {
      const int tiles64 = (HW + 63) / 64;
      const int chunks_tc = std::max(1, std::min(tiles64, (148 + eff_frames / 2) / eff_frames));     // one CTA per SM
      const int px_per_cta_tc = ((tiles64 + chunks_tc - 1) / chunks_tc) * 64;
      const int gx_tc = (HW + px_per_cta_tc - 1) / px_per_cta_tc;
      ba_schur_tc_kernel<false><<<dim3(gx_tc, a->n_frames, 1), kTcThreads, kTcSmem, st>>>(a->jj, WS(int, L.off_hdr), WS(int, L.off_kx), WS(int, L.off_rowptr),
                                                           WS(int, L.off_edgeidx), HW, a->t0, L.P, px_per_cta_tc, WS(float, L.off_Eij),
                                                           WS(float, L.off_C), WS(float, L.off_w), WS(float, L.off_Ei), Hsys, bsys, WS(int, L.off_big));
      // frames with 22..100 rows (dense graphs, edge-sharded ranks): tile pairs over gridDim.z, whole pixel range per CTA; CTAs of
      // frames outside that range (and pair indices beyond a frame's count) exit after the row-list build
      const int max_big = std::min(a->n_frames, a->n_edges / kTcRowsMax);     // a frame with 22+ rows has 21+ out-edges
      if (max_big > 0)
        ba_schur_tc_kernel<true><<<dim3(1, max_big, kPairGridZ), kTcThreads, kTcSmem, st>>>(a->jj, WS(int, L.off_hdr), WS(int, L.off_kx), WS(int, L.off_rowptr),
                                                           WS(int, L.off_edgeidx), HW, a->t0, L.P, ((HW + 31) / 32) * 32, WS(float, L.off_Eij),
                                                           WS(float, L.off_C), WS(float, L.off_w), WS(float, L.off_Ei), Hsys, bsys, WS(int, L.off_big));
    } else {
      ba_schur_small_kernel<<<dim3(gx1, a->n_frames, 1), kSgThreads, smem2, st>>>(a->jj, WS(int, L.off_hdr), WS(int, L.off_kx), WS(int, L.off_rowptr),
                                                           WS(int, L.off_edgeidx), HW, a->t0, L.P, px_per_cta1, WS(float, L.off_Eij),
                                                           WS(float, L.off_C), WS(float, L.off_w), WS(float, L.off_Ei), Hsys, bsys);
    }
    DBA_CHECK_LAUNCH("ba_schur<single>");
    ba_schur_gemm_kernel<<<dim3(gx2, a->n_frames, zsplit2), kSgThreads, smem2, st>>>(a->jj, WS(int, L.off_hdr), WS(int, L.off_kx), WS(int, L.off_rowptr),
                                                                         WS(int, L.off_edgeidx), HW, a->t0, L.P, px_per_cta2, use_tc ? kPairRowsMax : kSgRows, WS(float, L.off_Eij),
                                                                         WS(float, L.off_C), WS(float, L.off_w), WS(float, L.off_Ei), Hsys, bsys);
    DBA_CHECK_LAUNCH("ba_schur<multi>");
  }
  return DBA_OK;
}

extern "C" int dba_ba_solve(const dba_ba_args* a) {
  Layout L; int rc = check_ba_args(a, L); if (rc) return rc;
  if (L.P == 0) return DBA_OK;
  cudaStream_t st = (cudaStream_t)a->stream;
  const int HW = a->ht * a->wd;
  double* Hsys = system_ptr(a, L);
  double* bsys = Hsys + (size_t)L.n * L.n;
  float* dx = WS(float, L.off_dx);
  {
    CholPeers peers; peers.world = 0;
    if (a->p2p_world > 1) {
      const size_t nd = (size_t)L.n * L.n + L.n;
      peers.world = a->p2p_world; peers.epoch = a->p2p_epoch; peers.epoch_dev = a->p2p_epoch_dev;
      for (int k = 0; k < a->p2p_world; k++) peers.sys[k] = reinterpret_cast<const double*>(a->p2p_system[k]) + (size_t)(a->p2p_epoch & 1ull) * nd;
      peers.flags = reinterpret_cast<const unsigned long long*>(reinterpret_cast<const double*>(a->p2p_system[a->p2p_rank]) + 2 * nd);
    }
    int rc2 = chol_solve_launch(Hsys, bsys, L.n, (double)a->lm, (double)a->ep, WS(void, L.off_L), WS(int, L.off_hdr) + HDR_CHOL_FAIL, dx, st,
                                a->p2p_world > 1 ? &peers : nullptr);
    if (rc2) return rc2;
  }
  if (!a->motion_only) {
    DBA_CHECK_ARG(a->dz_out != nullptr, "dz_out missing");
    dim3 grid((HW + 255) / 256, a->n_frames);
    ba_backsub_kernel<<<grid, 256, 0, st>>>(a->jj, WS(int, L.off_hdr), WS(int, L.off_kx), WS(int, L.off_rowptr), WS(int, L.off_edgeidx),
                                            HW, a->t0, L.P, WS(float, L.off_Eij), WS(float, L.off_C), WS(float, L.off_w),
                                            WS(float, L.off_Ei), dx, a->disps, a->dz_out, a->own_lo, a->own_hi);
    DBA_CHECK_LAUNCH("ba_backsub");
  }
  ba_pose_retr_kernel<<<(L.P + 127) / 128, 128, 0, st>>>(a->poses, dx, a->t0, L.P, a->dx_out, WS(int, L.off_hdr));
  DBA_CHECK_LAUNCH("ba_pose_retr");
  return DBA_OK;
}

// publish this rank's partial system to every peer: release stores of the epoch into flags[rank] of each peer's buffer
namespace dba {
struct P2PSignal { unsigned long long* flag[8]; int world; unsigned long long epoch; unsigned long long* epoch_dev; };
__global__ void ba_p2p_signal_kernel2(P2PSignal s) {
  __threadfence_system();
  const int lane = threadIdx.x;
  unsigned long long e = s.epoch;
  if (s.epoch_dev) {                     // device-resident epoch: advance it here so a captured graph publishes a fresh value per replay
    if (lane == 0) { e = *s.epoch_dev + 1ull; *s.epoch_dev = e; }
    e = __shfl_sync(0xffffffffu, e, 0);
  }
  if (lane < s.world) asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(s.flag[lane]), "l"(e) : "memory");
}
}  // namespace dba

extern "C" int dba_ba_p2p_signal(const dba_ba_args* a) {
  Layout L; int rc = check_ba_args(a, L); if (rc) return rc;
  if (a->p2p_world <= 1) return DBA_OK;
  const size_t nd = (size_t)L.n * L.n + L.n;
  dba::P2PSignal s; s.world = a->p2p_world; s.epoch = a->p2p_epoch; s.epoch_dev = a->p2p_epoch_dev;
  for (int k = 0; k < a->p2p_world; k++)
    s.flag[k] = reinterpret_cast<unsigned long long*>(reinterpret_cast<double*>(a->p2p_system[k]) + 2 * nd) + a->p2p_rank;
  dba::ba_p2p_signal_kernel2<<<1, 32, 0, (cudaStream_t)a->stream>>>(s);
  DBA_CHECK_LAUNCH("ba_p2p_signal");
  return DBA_OK;
}

extern "C" int dba_ba(const dba_ba_args* a, int iterations) {
  int rc = dba_ba_prepare(a);
  if (rc) return rc;
  for (int it = 0; it < iterations; it++) {
    rc = dba_ba_build(a); if (rc) return rc;
    rc = dba_ba_solve(a); if (rc) return rc;
  }
  return DBA_OK;
}

extern "C" int dba_ba_read_info(const dba_ba_args* a, int* n_depth_frames, int* device_status) {
  Layout L; int rc = check_ba_args(a, L); if (rc) return rc;
  int h[4] = {0, 0, 0, 0};
  DBA_CHECK_CUDA(cudaMemcpyAsync(h, WS(int, L.off_hdr), sizeof(h), cudaMemcpyDeviceToHost, (cudaStream_t)a->stream), "read_info copy");
  DBA_CHECK_CUDA(cudaStreamSynchronize((cudaStream_t)a->stream), "read_info sync");
  if (n_depth_frames) *n_depth_frames = h[HDR_M];
  if (device_status) *device_status = h[HDR_STATUS];
  return DBA_OK;
}
