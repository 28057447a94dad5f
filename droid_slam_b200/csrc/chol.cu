// Damped SPD solve of the reduced pose system on the device, fp64:  (H + diag(ep + lm*diag(H))) x = b.
//
// Replaces the reference's host-side SparseBlock::solve (src/droid_kernels.cu:1201-1222: Eigen::SimplicialLLT in
// fp64 on the CPU behind two PCIe round trips).  Same contract: fp64 arithmetic, a non-positive pivot means
// "not SPD" and yields x = 0.  Two kernels, both one thread-block CLUSTER of up to 16 CTAs (16 SMs of one GPC), 32x32 fp64 tiles:
//
//  * chol_resident_kernel (n <= 448, i.e. <= 14 tile rows: frontend windows, the 72-keyframe metric window) -- every tile has one owner
//    warp for the whole factorisation and lives in its registers; tiles are handed over through global memory (L2) WITHOUT flags, fences
//    or barriers: every output location is pre-filled with a NaN bit pattern no arithmetic produces and a consumer re-reads a tile until no
//    element is that sentinel.  See the comment block above the kernel and DESIGN.md 4.4 for the measurements that led there (every
//    acquire ends in CCTL.IVALL and makes the next global loads ~10x slower; the unrolled potrf was bound by instruction delivery).
//  * chol_cluster_kernel (larger systems) -- right-looking tiled Cholesky with the tiles in global memory (L2 resident).  Per panel k:
//     TRSM of the column-k tiles (one warp per tile, lane = row, forward substitution against L_kk in shared memory)
//       -- cluster barrier --
//     trailing update A_ij -= L_ik L_jk^T: one warp per tile with an 8x4 register block per lane (operands staged in the
//     warp's padded shared-memory slabs, coalesced global I/O).  The NEXT diagonal tile is on the critical path, so CTA 0
//     updates it with all 256 threads and its warp 0 factors it immediately (rows in registers, the pivot column is
//     broadcast through shared memory) while every other warp of the cluster works on the remaining tiles; a spare
//     warp inverts L_kk for the backward pass
//       -- cluster barrier --
//    The barriers are acquire-free (cluster_sync_light: relaxed mbarrier arrivals over distributed shared memory behind a release
//    store per thread), all exchanged data is st.cg / ld.cg.
// ENVELOPE (chol_cluster_kernel): the reduced pose system of a sliding-window / proximity factor graph is block banded (pose a couples to
// pose b only through a common source frame), and a Cholesky factor never fills in left of a row's first nonzero.  The load phase
// records, per 32-row tile row, the first structurally nonzero tile column (`first`); TRSM, trailing updates and the backward
// substitution then skip every tile outside that envelope: the global-BA configs (6P = 2394 ... 5994, half bandwidth ~150) drop from
// O(n^3) to O(n b^2) -- what Eigen's sparse LLT does for the reference.
// The right-hand side rides along as an extra tile row, so L^-1 b comes out of the factorisation for free; the
// backward substitution uses the inverted diagonal tiles and runs in CTA 0.
// (B200 note, measured: a dependent fp64 op costs ~9 cycles, the fp64 pipe issues one warp instruction per ~2.3 cycles per SM
//  sub-partition, and a 64-bit warp shuffle pair is slower than a shared-memory broadcast, which is why the pivot column goes through
//  shared memory and the pivot uses an fp32 rsqrt seed + one Newton step -- 3e-14 relative, far below the fp32 rounding of the result.)
#include "common.cuh"
#include <cooperative_groups.h>
#include <math.h>
#include <stdint.h>

namespace cg = cooperative_groups;

namespace dba {

constexpr int kT = 32;                 // tile edge
constexpr int kTP = kT + 1;            // padded row length in shared memory
constexpr int kCholThreads = 256;      // 8 warps per CTA
constexpr int kCholWarps = kCholThreads / 32;

__device__ __forceinline__ double ldcg(const double* p) { return __ldcg(p); }
__device__ __forceinline__ void stcg(double* p, double v) { __stcg(p, v); }

// 1/sqrt(d): MUFU.RSQ64H seed (~2^-22) + one third-order correction r += r t (1/2 + 3/8 t), t = 1 - d r^2 (error ~ t^3: full fp64).
// Deliberately branch-free: a branch here splits warp_potrf into basic blocks and stops ptxas from scheduling the rank-1 update
// under the latency of this chain.  d <= 0 yields NaN/inf, which the caller flags through its pivot test.
__device__ __forceinline__ double fast_rsqrt(double d) {
  double r;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(d));
  const double t = fma(-d, r * r, 1.0);
  return fma(fma(0.375, t, 0.5), r * t, r);
}

// Cholesky of a 32x32 tile, one row per lane in registers; the pivot column is broadcast through `col` (2 x 32 doubles
// of shared memory private to the warp).  rdiag_out receives 1/L[k][k] (lane k's value).  Returns false on a
// non-positive pivot.
__device__ __forceinline__ bool warp_potrf(double (&a)[kT], int lane, double* col, double& rdiag_out) {
  bool ok = true;
  rdiag_out = 0.0;
  // software-pipelined: the pivot of column k+1 only needs a[k+1] after the rank-1 update of column k, so that element is updated
  // first and its shuffle + rsqrt chain (the latency that bounds this routine) runs under the remaining 30 updates of column k
  double d = __shfl_sync(0xffffffffu, a[0], 0);
  double r = fast_rsqrt(d);
#pragma unroll
  for (int k = 0; k < kT; k++) {
    if (!(d > 0.0)) ok = false;
    const double l = (lane == k) ? d * r : a[k] * r;
    if (lane == k) rdiag_out = r;
    a[k] = l;
    double* cb = col + (k & 1) * kT;
    cb[lane] = l;
    __syncwarp();
    if (k + 1 < kT) {
      a[k + 1] -= l * cb[k + 1];
      d = __shfl_sync(0xffffffffu, a[k + 1], k + 1);
      r = fast_rsqrt(d);
    }
#pragma unroll
    for (int j = k + 2; j < kT; j++) a[j] -= l * cb[j];   // only rows >= j are meaningful
  }
  return ok;
}

// Cholesky of a 32x32 tile, one row per lane, in ~300 instructions instead of the ~1800 straight-line ones of warp_potrf.  ncu on the
// resident kernel (profiles/r2_chol_resident_stalls.txt): 40 % of the samples inside the unrolled potrf are "no instruction" -- the code is
// executed once per SM and its delivery from the GPC-level instruction cache, not its dependent chain, sets the pace (2.9 us on an idle
// GPC, 5.3 us while the other 15 SMs fetch code of their own).  Here the row is shifted down one register per column, so a[0] is always
// the pivot column and all register indices are static inside a rolled loop; four loops of eight columns with widths 32/24/16/8 keep
// the extra arithmetic at 608 instead of 496 DFMAs.  The pivot column is published twice (offset by one double) so that the operands
// of the rank-1 update can be fetched with aligned 16-byte loads whatever the parity of the column.  Per element the operations and
// their order are those of warp_potrf: identical bits.  out[lane][k] receives L (zeros above the diagonal).
template <int W>
__device__ __forceinline__ void potrf_phase(double (&a)[kT], int lane, int k0, double* cx, double* cy, double (*out)[kTP], double& d, double& r, bool& ok,
                                            double& rdiag_out) {
#pragma unroll 1
  for (int k = k0; k < k0 + 8; k++) {
    if (!(d > 0.0)) ok = false;
    const double l = (lane == k) ? d * r : a[0] * r;
    if (lane == k) rdiag_out = r;
    out[lane][k] = (lane >= k) ? l : 0.0;
    double* bx = cx + (k & 1) * (2 * kT + 2);               // double-buffered over k: no second barrier per column
    double* by = cy + (k & 1) * (2 * kT + 2);
    bx[lane] = l;                                            // bx[t]     = l of row t
    by[lane + 1] = l;                                        // by[t + 1] = l of row t
    __syncwarp();
    const double* ck = ((k + 1) & 1) ? (by + k + 2) : (bx + k + 1);   // ck[m] = l of row k+1+m, 16-byte aligned either way
    const double2 c01 = *reinterpret_cast<const double2*>(ck);
    const double a0 = a[1] - l * c01.x;
    d = __shfl_sync(0xffffffffu, a0, (k + 1) & 31);
    r = fast_rsqrt(d);
    if (W > 2) a[1] = a[2] - l * c01.y;
#pragma unroll
    for (int m = 2; m + 1 < W - 1; m += 2) {
      const double2 c = *reinterpret_cast<const double2*>(ck + m);
      a[m] = a[m + 1] - l * c.x;
      a[m + 1] = a[m + 2] - l * c.y;
    }
    if (((W - 1) & 1) && W > 3) a[W - 2] = a[W - 1] - l * ck[W - 2];   // odd count: one element left (W - 1 updates in total)
    a[0] = a0;
  }
}

__device__ __forceinline__ bool warp_potrf_compact(double (&a)[kT], int lane, double* cbuf, double (*out)[kTP], double& rdiag_out) {
  bool ok = true;
  rdiag_out = 0.0;
  double* cx = cbuf;                                         // 2 x (2*kT + 2) doubles
  double* cy = cbuf + 2 * (2 * kT + 2);                      // 2 x (2*kT + 2) doubles; both 16-byte aligned
  double d = __shfl_sync(0xffffffffu, a[0], 0);
  double r = fast_rsqrt(d);
  potrf_phase<32>(a, lane, 0, cx, cy, out, d, r, ok, rdiag_out);
  potrf_phase<24>(a, lane, 8, cx, cy, out, d, r, ok, rdiag_out);
  potrf_phase<16>(a, lane, 16, cx, cy, out, d, r, ok, rdiag_out);
  potrf_phase<8>(a, lane, 24, cx, cy, out, d, r, ok, rdiag_out);
  return ok;
}

struct CholParams {
  const double* H;   // [n][n] fp64, lower triangle valid
  const double* b;   // [n]
  double* L;         // [(nt+1)*32][nt*32] row-major working matrix (tile row nt carries b^T in its row 0)
  double* Linv;      // [nt][32][32] inverses of the diagonal tiles
  double* rdiag;     // [nt*32] reciprocals of diag(L)
  int* first;        // [nt+2] envelope: first nonzero tile column of each tile row (rhs row nt: 0); [nt+1]: spare word
  double* Cs;                          // resident-tile kernel: [nt][32][32] tiles (j+1, j) BEFORE the substitution
  unsigned char map_i[128], map_j[128];   // resident-tile kernel: tile (i, j) of warp slot cta*8 + warp; 0xFF = none
  int* fail;         // sticky flag: non-positive pivot
  float* x;          // [n] result (fp32 like the reference's dx)
  int n, nt;
  double lm, ep;
  CholPeers peers;              // world <= 1: plain local system
};

// one warp: C (32x32 at Ct) -= A (at At) * B^T (at Bt); lane (rg = lane>>3, cg = lane&7) owns rows 8rg..8rg+7, cols 4cg..4cg+3
__device__ __forceinline__ void warp_tile_update(const double* At, const double* Bt, double* Ct, int ld, int lane,
                                                 double (*sA)[kTP], double (*sB)[kTP]) {
  const int rg = lane >> 3, cgp = lane & 7;
  double acc[8][4];
  // the C tile's loads go out first and return under the operand staging (one L2 round trip instead of two)
#pragma unroll
  for (int i = 0; i < 8; i++) {
    const double2 c01 = __ldcg(reinterpret_cast<const double2*>(Ct + (size_t)(8 * rg + i) * ld + 4 * cgp));
    const double2 c23 = __ldcg(reinterpret_cast<const double2*>(Ct + (size_t)(8 * rg + i) * ld + 4 * cgp + 2));
    acc[i][0] = c01.x; acc[i][1] = c01.y; acc[i][2] = c23.x; acc[i][3] = c23.y;
  }
#pragma unroll 16
  for (int r = 0; r < kT; r++) { sA[r][lane] = ldcg(At + (size_t)r * ld + lane); sB[r][lane] = ldcg(Bt + (size_t)r * ld + lane); }
  __syncwarp();
#pragma unroll 4
  for (int q = 0; q < kT; q++) {
    double av[8], bv[4];
#pragma unroll
    for (int i = 0; i < 8; i++) av[i] = sA[8 * rg + i][q];
#pragma unroll
    for (int jx = 0; jx < 4; jx++) bv[jx] = sB[4 * cgp + jx][q];
#pragma unroll
    for (int i = 0; i < 8; i++)
#pragma unroll
      for (int jx = 0; jx < 4; jx++) acc[i][jx] -= av[i] * bv[jx];
  }
#pragma unroll
  for (int i = 0; i < 8; i++) {
    __stcg(reinterpret_cast<double2*>(Ct + (size_t)(8 * rg + i) * ld + 4 * cgp), make_double2(acc[i][0], acc[i][1]));
    __stcg(reinterpret_cast<double2*>(Ct + (size_t)(8 * rg + i) * ld + 4 * cgp + 2), make_double2(acc[i][2], acc[i][3]));
  }
  __syncwarp();
}

// Cluster-wide barrier WITHOUT the acquire side of barrier.cluster.wait.  Measured on B200 (this kernel, in-kernel timer stamps): every acquire --
// barrier.cluster.wait, ld.acquire, fence -- ends in CCTL.IVALL, and the first global loads a warp issues after it take ~3 us instead of
// ~0.3.  All data exchanged through this barrier is written with st.global.cg and read with ld.global.cg (L2 on both sides), so no L1
// line ever has to be invalidated: every thread drains its own stores to L2 with a release store (MEMBAR.ALL.GPU, no CCTL), the CTA
// meets at bar.sync, ncta of its threads arrive (relaxed) on the ncta per-CTA mbarriers through distributed shared memory, and everyone
// waits (relaxed) on the local one.
__device__ __forceinline__ void cluster_sync_light(unsigned mbar, unsigned& phase, int ncta, int tid, unsigned* drain) {
  asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(drain), "r"(0u) : "memory");
  __syncthreads();
  if (tid < ncta) {
    unsigned remote;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(mbar), "r"((unsigned)tid));
    asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(remote) : "memory");
  }
  unsigned done = 0;
  while (!done) {
    asm volatile("{ .reg .pred q; mbarrier.try_wait.parity.relaxed.cluster.shared::cta.b64 q, [%1], %2; selp.u32 %0, 1, 0, q; }"
                 : "=r"(done) : "r"(mbar), "r"(phase) : "memory");
  }
  phase ^= 1u;
}

__global__ void __launch_bounds__(kCholThreads, 1) chol_cluster_kernel(CholParams p) {
  cg::cluster_group cluster = cg::this_cluster();
  const int ncta = (int)cluster.num_blocks();
  const int cta = (int)cluster.block_rank();
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int gw = cta * kCholWarps + warp;          // warp id within the cluster
  const int nwarps = ncta * kCholWarps;
  const int nt = p.nt, n = p.n;
  const int ld = nt * kT;                          // leading dimension of L
  double* __restrict__ L = p.L;

  __shared__ double s_Lkk[kT][kTP];
  __shared__ double s_rdiag[kT];
  __shared__ double s_vec[kT];
  __shared__ __align__(16) double s_col[4 * (2 * kT + 2)];
  __shared__ int s_act[kCholThreads];                // tile rows with a nonzero tile in panel k (ascending; the rhs row nt is always last)
  __shared__ int s_wc[kCholWarps];
  __shared__ int s_nact;
  extern __shared__ double s_dyn[];                  // per-warp slabs + two CTA-wide tiles, rows padded to 33 doubles
  double (*s_A)[kT][kTP] = reinterpret_cast<double (*)[kT][kTP]>(s_dyn);
  double (*s_B)[kT][kTP] = reinterpret_cast<double (*)[kT][kTP]>(s_dyn + (size_t)kCholWarps * kT * kTP);
  double (*s_D)[kTP] = reinterpret_cast<double (*)[kTP]>(s_dyn + (size_t)2 * kCholWarps * kT * kTP);
  double (*s_T)[kTP] = reinterpret_cast<double (*)[kTP]>(s_dyn + (size_t)2 * kCholWarps * kT * kTP + kT * kTP);

  // ---- fused peer-to-peer reduction: wait until every rank has published its partial system for this epoch ------------
  const int world = p.peers.world;
  if (world > 1) {
    __shared__ int s_timeout;
    if (tid == 0) {
      int bad = 0;
      const unsigned long long want = p.peers.epoch_dev ? *p.peers.epoch_dev : p.peers.epoch;
      for (int r = 0; r < world; r++) {
        unsigned long long v = 0;
        long long spins = 0;
        do {
          asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p.peers.flags + r) : "memory");
        } while (v < want && ++spins < (1ll << 24));
        if (v < want) bad = 1;
      }
      s_timeout = bad;
    }
    __syncthreads();
    if (cta == 0 && tid == 0) *p.fail = s_timeout ? 2 : 0;   // a peer never arrived: give up loudly (dx = 0), never hang
  } else if (cta == 0 && tid == 0) *p.fail = 0;
  // ---- envelope: first[i] starts at the diagonal, the load below lowers it to the first nonzero tile of the row
  const bool envelope = nt < kCholThreads;             // one thread per tile row in the per-panel scan below
  for (int i = cta * kCholThreads + tid; i <= nt; i += ncta * kCholThreads) p.first[i] = (i < nt && envelope) ? i : 0;
  __shared__ unsigned long long s_mbar;
  const unsigned mbar = (unsigned)__cvta_generic_to_shared(&s_mbar);
  unsigned mphase = 0;
  unsigned* drain = reinterpret_cast<unsigned*>(p.first + nt + 1);   // spare word: target of the store-draining release stores
  if (tid == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mbar), "r"((unsigned)ncta) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  cluster.sync();
  // ---- load: lower tiles of H with damping (reference :1205-1206), identity padding, rhs row ------------------
  {
    const size_t total = (size_t)(nt + 1) * kT * ld;
    const size_t nn = (size_t)n * n;
    const size_t stride = (size_t)ncta * kCholThreads;
    constexpr int kU = 4;                               // elements per thread in flight: with peers, kU x world NVLink loads overlap their ~2 us round trips
    for (size_t base = (size_t)cta * kCholThreads + tid; base < total; base += kU * stride) {
      size_t srcs[kU];
      double vals[kU];
      double t[kU][8];
#pragma unroll
      for (int u = 0; u < kU; u++) {
        const size_t idx = base + u * stride;
        srcs[u] = (size_t)-1; vals[u] = 0.0;
        if (idx < total) {
          const int r = (int)(idx / ld), c = (int)(idx - (size_t)r * ld);
          if (r < nt * kT) {
            if (r < n && c < n) {
              if (c <= r) srcs[u] = (size_t)r * n + c;
              else if ((r >> 5) == (c >> 5)) srcs[u] = (size_t)c * n + r;     // diagonal tiles are kept fully symmetric
            } else if (r == c) vals[u] = 1.0;
          } else if (r == nt * kT && c < n) srcs[u] = nn + c;
        }
        if (srcs[u] != (size_t)-1) {                      // element of the [n*n | n] system feeding this entry
          if (world > 1) {
#pragma unroll
            for (int q = 0; q < 8; q++) {
              t[u][q] = 0.0;
              if (q < world) asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(t[u][q]) : "l"(p.peers.sys[q] + srcs[u]) : "memory");
            }
          } else t[u][0] = (srcs[u] < nn) ? p.H[srcs[u]] : p.b[srcs[u] - nn];
        }
      }
#pragma unroll
      for (int u = 0; u < kU; u++) {
        const size_t idx = base + u * stride;
        if (idx >= total) continue;
        double v = vals[u];
        if (srcs[u] != (size_t)-1) {
          // all peer loads were issued before the first add, then summed in fixed rank order: every rank computes the identical sum
          if (world > 1) {
#pragma unroll
            for (int q = 0; q < 8; q++)
              if (q < world) v += t[u][q];
          } else v = t[u][0];
          const int r = (int)(idx / ld), c = (int)(idx - (size_t)r * ld);
          if (srcs[u] < nn && r == c) v += p.ep + p.lm * v;
          if (envelope && v != 0.0 && r < nt * kT) {
            const int tr = r >> 5, tc = c >> 5;
            if (tc < tr && tc < *reinterpret_cast<volatile int*>(p.first + tr)) atomicMin(p.first + tr, tc);
          }
        }
        stcg(L + idx, v);
      }
    }
  }
  cluster.sync();

  // ---- potrf of tile (0,0) --------------------------------------------------------------------------------------
  if (gw == 0) {
    double a[kT], rd;
#pragma unroll
    for (int c = 0; c < kT; c++) a[c] = ldcg(L + (size_t)lane * ld + c);
    if (!warp_potrf(a, lane, s_col, rd) && lane == 0) *p.fail = 1;
#pragma unroll
    for (int c = 0; c < kT; c++) stcg(L + (size_t)lane * ld + c, (c <= lane) ? a[c] : 0.0);
    stcg(p.rdiag + lane, rd);
  }
  cluster_sync_light(mbar, mphase, ncta, tid, drain);

  for (int k = 0; k < nt; k++) {
    // ---- every CTA: L_kk and its reciprocal diagonal into shared memory
    for (int e = tid; e < kT * kT; e += kCholThreads) {
      const int r = e >> 5, c = e & 31;
      s_Lkk[r][c] = ldcg(L + (size_t)(k * kT + r) * ld + k * kT + c);
    }
    if (tid < kT) s_rdiag[tid] = ldcg(p.rdiag + k * kT + tid);
    // active tile rows of panel k (inside the envelope), in ascending order -- every CTA builds the identical list
    {
      const int i_row = k + 1 + tid;
      const bool act = envelope ? (i_row <= nt && (i_row == nt || __ldcg(p.first + i_row) <= k)) : false;
      const unsigned bal = __ballot_sync(0xffffffffu, act);
      if (lane == 0) s_wc[warp] = __popc(bal);
      __syncthreads();
      int base = 0;
      for (int w = 0; w < warp; w++) base += s_wc[w];
      if (act) s_act[base + __popc(bal & ((1u << lane) - 1u))] = i_row;
      if (tid == 0) { int tot = 0; for (int w = 0; w < kCholWarps; w++) tot += s_wc[w]; s_nact = tot; }
    }
    __syncthreads();
    const int nact = envelope ? s_nact : (nt - k);       // >= 1: the rhs row
    // ---- TRSM: tiles (i,k) of the active rows (tile row nt is the right-hand side)
    for (int ta = gw; ta < nact; ta += nwarps) {
      const int i = envelope ? s_act[ta] : k + 1 + ta;
      double a[kT];
      double* tile = L + (size_t)(i * kT) * ld + k * kT;
#pragma unroll
      for (int r = 0; r < kT; r++) s_A[warp][r][lane] = ldcg(tile + (size_t)r * ld + lane);     // coalesced rows, all 32 loads in flight
      __syncwarp();
#pragma unroll
      for (int c = 0; c < kT; c++) a[c] = s_A[warp][lane][c];                                   // lane = row
#pragma unroll
      for (int c = 0; c < kT; c++) {
        const double xv = a[c] * s_rdiag[c];
        a[c] = xv;
#pragma unroll
        for (int j = c + 1; j < kT; j++) a[j] -= xv * s_Lkk[j][c];
        asm volatile("" ::: "memory");
      }
      __syncwarp();
#pragma unroll
      for (int c = 0; c < kT; c++) s_A[warp][lane][c] = a[c];
      __syncwarp();
#pragma unroll 8
      for (int r = 0; r < kT; r++) stcg(tile + (size_t)r * ld + lane, s_A[warp][r][lane]);
      __syncwarp();
    }
    cluster_sync_light(mbar, mphase, ncta, tid, drain);
    // ---- trailing update with panel k
    const int rem = nt - k - 1;                       // remaining tile columns
    const int m1 = nact - 1;                          // active rows without the rhs row
    const int ntri = m1 * (m1 + 1) / 2;
    const int ntasks = ntri + m1;                     // tiles (i,j) of active rows, j <= i < nt, plus the rhs row tiles (nt,j)
    // task 0 = tile (k+1,k+1) when row k+1 is active: CTA 0 updates + factors it below; otherwise that tile needs no update (CTA 0 still
    // factors it) and task 0 is an ordinary tile of the workers
    const bool diag_active = envelope ? (m1 >= 1 && s_act[0] == k + 1) : (rem >= 1);
    if (cta == 0 && rem >= 1) {
      // next diagonal tile (task 0): all 256 threads update it, warp 0 factors it
      const double* At = L + (size_t)((k + 1) * kT) * ld + k * kT;
      double* Ct = L + (size_t)((k + 1) * kT) * ld + (k + 1) * kT;
      for (int e = tid; e < kT * kT; e += kCholThreads) {
        const int r = e >> 5, c = e & 31;
        s_D[r][c] = ldcg(At + (size_t)r * ld + c);
        s_T[r][c] = ldcg(Ct + (size_t)r * ld + c);
      }
      __syncthreads();
      {
        const int r = tid >> 3, c0 = (tid & 7) * 4;
        double acc[4] = {s_T[r][c0], s_T[r][c0 + 1], s_T[r][c0 + 2], s_T[r][c0 + 3]};
#pragma unroll 8
        for (int q = 0; q < kT; q++) {
          const double ar = s_D[r][q];
#pragma unroll
          for (int jx = 0; jx < 4; jx++) acc[jx] -= ar * s_D[c0 + jx][q];
        }
        __syncthreads();
#pragma unroll
        for (int jx = 0; jx < 4; jx++) s_T[r][c0 + jx] = acc[jx];
      }
      __syncthreads();
      if (warp == 0) {
        double a[kT], rd;
#pragma unroll
        for (int c = 0; c < kT; c++) a[c] = s_T[lane][c];
        __syncwarp();
        if (!warp_potrf_compact(a, lane, s_col, s_T, rd) && lane == 0) *p.fail = 1;   // writes L into s_T
        __syncwarp();
#pragma unroll 8
        for (int r = 0; r < kT; r++) stcg(Ct + (size_t)r * ld + lane, s_T[r][lane]);
        stcg(p.rdiag + (k + 1) * kT + lane, rd);
      }
    }
    // remaining tiles: every warp of the cluster except the factoring one
    if (gw != 0) {
      for (int t = (diag_active ? 1 : 0) + gw - 1; t < ntasks; t += nwarps - 1) {
        int i, j;
        if (t < ntri) {
          int bi = (int)((sqrtf(8.f * (float)t + 1.f) - 1.f) * 0.5f);
          while (bi * (bi + 1) / 2 > t) bi--;
          while ((bi + 1) * (bi + 2) / 2 <= t) bi++;
          const int bj = t - bi * (bi + 1) / 2;
          i = envelope ? s_act[bi] : k + 1 + bi; j = envelope ? s_act[bj] : k + 1 + bj;
        } else { i = nt; j = envelope ? s_act[t - ntri] : k + 1 + (t - ntri); }
        warp_tile_update(L + (size_t)(i * kT) * ld + k * kT, L + (size_t)(j * kT) * ld + k * kT, L + (size_t)(i * kT) * ld + j * kT, ld, lane,
                         s_A[warp], s_B[warp]);
      }
    }
    // inverse of L_kk (for the backward substitution) by the last warp of the cluster: lane j owns column j
    if (gw == nwarps - 1) {
      double xcol[kT];
#pragma unroll
      for (int i = 0; i < kT; i++) {
        double s = 0.0;
#pragma unroll
        for (int m = 0; m < i; m++) s += (m >= lane) ? s_Lkk[i][m] * xcol[m] : 0.0;
        xcol[i] = (i == lane) ? s_rdiag[i] : ((i > lane) ? -s * s_rdiag[i] : 0.0);
      }
#pragma unroll
      for (int i = 0; i < kT; i++) stcg(p.Linv + ((size_t)k * kT + i) * kT + lane, xcol[i]);
    }
    cluster_sync_light(mbar, mphase, ncta, tid, drain);
  }

  if (cta != 0) return;
  // ---- backward substitution  L^T x = y  in CTA 0;  y^T = row 0 of tile row nt -------------------------------------
  double* y = L + (size_t)(nt * kT) * ld;            // [ld], overwritten by x
  for (int k = nt - 1; k >= 0; k--) {
    if (warp == 0) {
      // x_k = Linv_kk^T y_k : lane c computes sum_r Linv[r][c] * y[r]
      const double yk = ldcg(y + k * kT + lane);
      double s = 0.0;
#pragma unroll
      for (int r = 0; r < kT; r++) s += ldcg(p.Linv + ((size_t)k * kT + r) * kT + lane) * __shfl_sync(0xffffffffu, yk, r);
      stcg(y + k * kT + lane, s);
      s_vec[lane] = s;
    }
    __syncthreads();
    // y_i -= L_ki^T x_k  for first[k] <= i < k (tiles left of the envelope are zero): lane = column of tile (k,i)
    for (int i = __ldcg(p.first + k) + warp; i < k; i += kCholWarps) {
      double s = 0.0;
#pragma unroll 8
      for (int r = 0; r < kT; r++) s += ldcg(L + (size_t)(k * kT + r) * ld + i * kT + lane) * s_vec[r];
      stcg(y + i * kT + lane, ldcg(y + i * kT + lane) - s);
    }
    __syncthreads();
  }
  const bool failed = (*reinterpret_cast<volatile int*>(p.fail)) != 0;
  for (int i = tid; i < n; i += kCholThreads) {
    const double v = ldcg(y + i);
    p.x[i] = (failed || !isfinite(v)) ? 0.f : (float)v;      // reference: solver.info() != Success -> zeros
  }
}


// =====================================================================================================================================
// Resident-tile dataflow variant for nt <= 14 (n <= 448: every frontend window, the 72-keyframe metric window).
//
// The barrier version above spends a panel on  L_kk reload -> TRSM -> cluster barrier -> trailing update -> cluster barrier.  Measured
// (in-kernel timer stamps): the arithmetic is ~3 us of that; the rest is synchronisation -- in particular every acquire (cluster barrier,
// ld.acquire, fence) ends in CCTL.IVALL, after which the next global loads of the warp take ~3 us instead of ~0.3.
// Here every lower tile (i,j) and every 32-entry piece of the right-hand side has ONE owner warp for the whole factorisation (105 + 14
// tiles <= 128 warps of the 16-CTA cluster) and lives in that warp's registers.  An owner applies  C -= L_ik L_jk^T  for k = 0..j-1 as
// soon as the two operand tiles exist, then finalises its tile (potrf on the diagonal, a substitution against L_jj below it) and writes it
// to global memory once.  There are no flags, fences or barriers inside the factorisation: the data validates itself.  Every output
// location is filled with a NaN bit pattern that no arithmetic produces before the (single) cluster barrier of the prologue, a double
// is written with one 8-byte store, and a consumer simply re-reads a tile from L2 (ld.global.cg) until no element is the sentinel --
// the scheme of NCCL's low-latency protocol, without spending bits on a flag.  The only serial path left is the true one,
// potrf(k) -> tile (k+1,k) -> last update of (k+1,k+1) -> potrf(k+1), with one L2 round trip per hand-over.
// Waits are bounded; a wait that expires marks the solve failed (dx = 0) instead of hanging.
constexpr int kResMaxNt = 14;
constexpr unsigned long long kSentinel = 0xFFF7DEADBEEF5A5Aull;
constexpr unsigned kSleepUrgent = 300;    // ns between the polls of a warp on the critical path
constexpr unsigned kSleepIdle = 4000;     // ... and of a warp off it


__device__ __forceinline__ bool is_sentinel(double v) { return __double2hiint(v) == (int)(kSentinel >> 32); }   // arithmetic NaNs are canonical
__device__ __forceinline__ double sentinel() { return __longlong_as_double((long long)kSentinel); }

// wait until the 32x32 tile at src is completely written, then stage it in the warp's padded slab.  false on time-out.
// `urgent` (the consumer sits on the critical path): no probe stage, short back-off; otherwise a one-row probe with a long back-off so
// that the ~100 waiting warps take neither issue slots nor L2 bandwidth from the working ones.
__device__ __forceinline__ bool tile_fetch(const double* src, int ld, int lane, double (*slab)[kTP], unsigned sleep_ns, unsigned sleep_retry) {
  int tries = 0;
  while (true) {                                             // cheap probe: the row that is stored last
    const double v = __ldcg(src + (size_t)(kT - 1) * ld + lane);
    if (!__any_sync(0xffffffffu, is_sentinel(v))) break;
    if (++tries > (1 << 19)) return false;
    __nanosleep(sleep_ns);
  }
  for (tries = 0; tries < (1 << 19); tries++) {
    double t[kT];
#pragma unroll
    for (int r = 0; r < kT; r++) t[r] = __ldcg(src + (size_t)r * ld + lane);
    bool bad = false;
#pragma unroll
    for (int r = 0; r < kT; r++) bad |= is_sentinel(t[r]);
    if (!__any_sync(0xffffffffu, bad)) {
#pragma unroll
      for (int r = 0; r < kT; r++) slab[r][lane] = t[r];
      __syncwarp();
      return true;
    }
    __nanosleep(sleep_retry);
  }
  return false;
}
// the same for a 32-entry vector (a piece of y, the reciprocal diagonal of a tile): lane c receives entry c
__device__ __forceinline__ bool vec_fetch(const double* src, int lane, double& out, unsigned sleep_ns) {
  for (int tries = 0; tries < (1 << 20); tries++) {
    const double v = __ldcg(src + lane);
    if (!__any_sync(0xffffffffu, is_sentinel(v))) { out = v; return true; }
    __nanosleep(sleep_ns);
  }
  out = 0.0;
  return false;
}

// acc (8x4 per lane: rows 8rg+i, cols 4cg+jx) -= A * B^T with A, B 32x32 tiles already staged in the warp's padded slabs
__device__ __forceinline__ void slab_mac(double (&acc)[8][4], const double (*sA)[kTP], const double (*sB)[kTP], int lane) {
  const int rg = lane >> 3, cgp = lane & 7;
#pragma unroll 4
  for (int q = 0; q < kT; q++) {
    double av[8], bv[4];
#pragma unroll
    for (int i = 0; i < 8; i++) av[i] = sA[8 * rg + i][q];
#pragma unroll
    for (int jx = 0; jx < 4; jx++) bv[jx] = sB[4 * cgp + jx][q];
#pragma unroll
    for (int i = 0; i < 8; i++)
#pragma unroll
      for (int jx = 0; jx < 4; jx++) acc[i][jx] -= av[i] * bv[jx];
  }
}

// one entry of the damped, padded working matrix straight from H / b (or from the peers' partial systems, summed in rank order)
__device__ __forceinline__ size_t sys_index(int r, int c, int n, bool diag_tile) {
  if (r < n && c < n) {
    if (c <= r) return (size_t)r * n + c;
    if (diag_tile) return (size_t)c * n + r;
  }
  return (size_t)-1;
}

template <bool PEERS>
__global__ void __launch_bounds__(kCholThreads, 1) chol_resident_kernel(CholParams p) {
  cg::cluster_group cluster = cg::this_cluster();
  const int ncta = (int)cluster.num_blocks();
  const int cta = (int)cluster.block_rank();
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nt = p.nt, n = p.n;
  const int ld = nt * kT;
  double* __restrict__ L = p.L;
  double* yrow = L + (size_t)(nt * kT) * ld;
  const int world = PEERS ? p.peers.world : 0;
  const size_t nn = (size_t)n * n;

  __shared__ double s_rd[kCholWarps][kT];
  __shared__ __align__(16) double s_colb[kCholWarps][4 * (2 * kT + 2)];
  __shared__ double s_vec[kT];
  extern __shared__ double s_dyn[];
  double (*s_A)[kT][kTP] = reinterpret_cast<double (*)[kT][kTP]>(s_dyn);
  double (*s_B)[kT][kTP] = reinterpret_cast<double (*)[kT][kTP]>(s_dyn + (size_t)kCholWarps * kT * kTP);

  // ---- prologue: wait for the peers' systems (multi-GPU), dense envelope for the backward pass
  for (int i = cta * kCholThreads + tid; i <= nt; i += ncta * kCholThreads) p.first[i] = 0;
  if (PEERS) {
    __shared__ int s_timeout;
    if (tid == 0) {
      int bad = 0;
      const unsigned long long want = p.peers.epoch_dev ? *p.peers.epoch_dev : p.peers.epoch;
      for (int r = 0; r < world; r++) {
        unsigned long long v = 0;
        long long spins = 0;
        do {
          asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p.peers.flags + r) : "memory");
        } while (v < want && ++spins < (1ll << 24));
        if (v < want) bad = 1;
      }
      s_timeout = bad;
    }
    __syncthreads();
    if (cta == 0 && tid == 0) *p.fail = s_timeout ? 2 : 0;
  } else if (cta == 0 && tid == 0) *p.fail = 0;

  // ---- tile of this warp: placed by the host (resident_tile_map below) so that a potrf never shares its SM with a working warp
  const int slot = cta * kCholWarps + warp;
  const bool has_tile = p.map_i[slot] != 0xFF;
  const int i = has_tile ? (int)p.map_i[slot] : 0, j = has_tile ? (int)p.map_j[slot] : 0;
  const int rg = lane >> 3, cgp = lane & 7;
  double acc[8][4];
  double y = 0.0;
  if (has_tile && i < nt) {
    // own tile from H (damping, identity padding, diagonal tiles kept fully symmetric) -- issued before the barrier below
    double t[8];
#pragma unroll
    for (int a = 0; a < 8; a++) {
#pragma unroll
      for (int jx = 0; jx < 4; jx++) {
        const int r = i * kT + 8 * rg + a, c = j * kT + 4 * cgp + jx;
        const size_t src = sys_index(r, c, n, i == j);
        double v = (src == (size_t)-1 && r == c) ? 1.0 : 0.0;
        if (src != (size_t)-1) {
          if (PEERS) {
#pragma unroll
            for (int q = 0; q < 8; q++) {
              t[q] = 0.0;
              if (q < world) asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(t[q]) : "l"(p.peers.sys[q] + src) : "memory");
            }
#pragma unroll
            for (int q = 0; q < 8; q++)
              if (q < world) v += t[q];
          } else v = p.H[src];
          if (r == c) v += p.ep + p.lm * v;
        }
        acc[a][jx] = v;
      }
    }
    // sentinel over everything this warp will publish
    double* tile = L + (size_t)(i * kT) * ld + j * kT;
#pragma unroll 8
    for (int r = 0; r < kT; r++) stcg(tile + (size_t)r * ld + lane, sentinel());
    if (i == j + 1) {
#pragma unroll 8
      for (int r = 0; r < kT; r++) stcg(p.Cs + ((size_t)j * kT + r) * kT + lane, sentinel());
    }
    if (i == j) {
      stcg(p.rdiag + j * kT + lane, sentinel());
#pragma unroll 8
      for (int r = 0; r < kT; r++) stcg(p.Linv + ((size_t)j * kT + r) * kT + lane, sentinel());
    }
  } else if (has_tile) {
    const int c0 = j * kT + lane;
    if (c0 < n) {
      if (PEERS) {
        for (int q = 0; q < world; q++) {
          double v;
          asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(v) : "l"(p.peers.sys[q] + nn + c0) : "memory");
          y += v;
        }
      } else y = p.b[c0];
    }
    stcg(yrow + c0, sentinel());
  }
  __threadfence();
  cluster.sync();

  if (has_tile) {
    double (*sA)[kTP] = s_A[warp];
    double (*sB)[kTP] = s_B[warp];
    bool alive = true;

    if (i < nt) {
      // ---------------- matrix tile (i, j): updates with the finished columns k < j
      for (int k = 0; k < j && alive; k++) {
        const bool last = (i == j && k == j - 1);
        if (last) {
          // the diagonal owner does not wait for tile (j, j-1) to come back from its owner; it takes that tile as it was BEFORE
          // the substitution (published early, off the critical path), substitutes against L_{j-1,j-1} itself and updates: one hand-over
          // per column instead of two.  The owner of (j, j-1) does the same substitution for everybody else.
          alive = tile_fetch(p.Cs + (size_t)(j - 1) * kT * kT, kT, lane, sA, kSleepUrgent, kSleepUrgent);
          alive = tile_fetch(L + (size_t)((j - 1) * kT) * ld + (j - 1) * kT, ld, lane, sB, kSleepUrgent, kSleepUrgent) && alive;
          double rdl;
          alive = vec_fetch(p.rdiag + (j - 1) * kT, lane, rdl, kSleepUrgent) && alive;
          s_rd[warp][lane] = rdl;
          __syncwarp();
          double x[kT];
#pragma unroll
          for (int c = 0; c < kT; c++) x[c] = sA[lane][c];
          __syncwarp();
#pragma unroll
          for (int c = 0; c < kT; c++) {
            const double xv = x[c] * s_rd[warp][c];
            x[c] = xv;
#pragma unroll
            for (int jj = c + 1; jj < kT; jj++) x[jj] -= xv * sB[jj][c];
            asm volatile("" ::: "memory");
          }
#pragma unroll
          for (int c = 0; c < kT; c++) sA[lane][c] = x[c];
          __syncwarp();
          slab_mac(acc, sA, sA, lane);
          __syncwarp();
          continue;
        }
        const bool urgent = (i <= j + 1) && (k >= j - 2);     // the tile is (about to be) on the critical path
        const unsigned slp = urgent ? kSleepUrgent : kSleepIdle;
        alive = tile_fetch(L + (size_t)(i * kT) * ld + k * kT, ld, lane, sA, slp, kSleepUrgent);
        if (i != j) {
          alive = tile_fetch(L + (size_t)(j * kT) * ld + k * kT, ld, lane, sB, slp, kSleepUrgent) && alive;
          slab_mac(acc, sA, sB, lane);
        } else {
          slab_mac(acc, sA, sA, lane);
        }
        __syncwarp();
      }
      // ---------------- finalise
      double* tile = L + (size_t)(i * kT) * ld + j * kT;
#pragma unroll
      for (int a = 0; a < 8; a++)
#pragma unroll
        for (int jx = 0; jx < 4; jx++) sA[8 * rg + a][4 * cgp + jx] = acc[a][jx];
      __syncwarp();
      double a[kT];
#pragma unroll
      for (int c = 0; c < kT; c++) a[c] = sA[lane][c];                 // lane = row
      __syncwarp();
      if (i == j) {
        double rd;
        if (!warp_potrf_compact(a, lane, s_colb[warp], sA, rd) && lane == 0) *p.fail = 1;
        s_rd[warp][lane] = rd;
        __syncwarp();
        stcg(p.rdiag + j * kT + lane, rd);
#pragma unroll 8
        for (int r = 0; r < kT; r++) stcg(tile + (size_t)r * ld + lane, sA[r][lane]);
        // inverse of L_jj for the backward pass (off the critical path), rolled: lane c owns column c of X = L^-1, kept in the warp's
        // second slab;  X[r][c] = (delta_rc - sum_{m<r} L[r][m] X[m][c]) / L[r][r]  (entries above the diagonal come out as zeros)
#pragma unroll 1
        for (int r = 0; r < kT; r++) {
          double s0 = 0.0, s1 = 0.0;
          int m = 0;
#pragma unroll 1
          for (; m + 1 < r; m += 2) { s0 += sA[r][m] * sB[m][lane]; s1 += sA[r][m + 1] * sB[m + 1][lane]; }
          if (m < r) s0 += sA[r][m] * sB[m][lane];
          sB[r][lane] = (((r == lane) ? 1.0 : 0.0) - (s0 + s1)) * s_rd[warp][r];
        }
#pragma unroll 4
        for (int r = 0; r < kT; r++) stcg(p.Linv + ((size_t)j * kT + r) * kT + lane, sB[r][lane]);
      } else {
        const bool sub = (i == j + 1);
        if (sub) {
#pragma unroll 8
          for (int r = 0; r < kT; r++) stcg(p.Cs + ((size_t)j * kT + r) * kT + lane, sA[r][lane]);
        }
        double rdl;
        const unsigned slp = sub ? kSleepUrgent : kSleepIdle;
        alive = tile_fetch(L + (size_t)(j * kT) * ld + j * kT, ld, lane, sB, slp, kSleepUrgent) && alive;
        alive = vec_fetch(p.rdiag + j * kT, lane, rdl, kSleepUrgent) && alive;
        s_rd[warp][lane] = rdl;
        __syncwarp();
#pragma unroll
        for (int c = 0; c < kT; c++) {
          const double xv = a[c] * s_rd[warp][c];
          a[c] = xv;
#pragma unroll
          for (int jj = c + 1; jj < kT; jj++) a[jj] -= xv * sB[jj][c];
          asm volatile("" ::: "memory");
        }
#pragma unroll
        for (int c = 0; c < kT; c++) sA[lane][c] = a[c];
        __syncwarp();
#pragma unroll 8
        for (int r = 0; r < kT; r++) stcg(tile + (size_t)r * ld + lane, sA[r][lane]);
      }
    } else {
      // ---------------- right-hand side piece j: lane c holds entry 32 j + c;  y_j = L_jj^-1 (b_j - sum_k L_jk y_k)
      for (int k = 0; k < j && alive; k++) {
        double yk;
        alive = vec_fetch(yrow + k * kT, lane, yk, kSleepIdle);
        alive = tile_fetch(L + (size_t)(j * kT) * ld + k * kT, ld, lane, sA, kSleepIdle, kSleepUrgent) && alive;
        double s0 = 0.0, s1 = 0.0;
#pragma unroll
        for (int c = 0; c < kT; c += 2) {
          s0 += sA[lane][c] * __shfl_sync(0xffffffffu, yk, c);
          s1 += sA[lane][c + 1] * __shfl_sync(0xffffffffu, yk, c + 1);
        }
        y -= s0 + s1;
        __syncwarp();
      }
      double rdl;
      alive = tile_fetch(L + (size_t)(j * kT) * ld + j * kT, ld, lane, sB, j == nt - 1 ? kSleepUrgent : kSleepIdle, kSleepUrgent) && alive;
      alive = vec_fetch(p.rdiag + j * kT, lane, rdl, kSleepUrgent) && alive;
#pragma unroll
      for (int c = 0; c < kT; c++) {
        const double yc = __shfl_sync(0xffffffffu, y, c) * __shfl_sync(0xffffffffu, rdl, c);
        if (lane == c) y = yc;
        else if (lane > c) y -= sB[lane][c] * yc;
      }
      stcg(yrow + j * kT + lane, y);
    }
    if (!alive && lane == 0) *p.fail = 4;                    // a producer never arrived: give up loudly, never hang
  }
  if (cta != 0) return;
  // ---- backward substitution  L^T x = y  in CTA 0.  No barrier with the other CTAs: every load below validates itself against the
  //      sentinel (the last things to appear are y_{nt-1} and the inverse of the last diagonal tile).  y lives in shared memory, the
  //      operands of step k-1 (inverse diagonal tile for warp 0, up to two tiles (k-1, i) per warp) are fetched during step k.
  __shared__ double s_y[kResMaxNt * kT];
  auto ld_valid = [&](const double* q) -> double {
    double v = __ldcg(q);
    for (int tries = 0; is_sentinel(v) && tries < (1 << 20); tries++) { __nanosleep(100); v = __ldcg(q); }
    return v;
  };
  {                                                          // the last piece of y is the last thing the forward pass produces
    const double* ylast = yrow + (nt - 1) * kT;
    for (int tries = 0; tries < (1 << 20); tries++) {
      const double v = __ldcg(ylast + lane);
      if (!__any_sync(0xffffffffu, is_sentinel(v))) break;
      __nanosleep(250);
    }
  }
  for (int q = tid; q < nt * kT; q += kCholThreads) s_y[q] = ld_valid(yrow + q);
  // warp 0 turns y_k into x_k (inverse diagonal tile prefetched one step ahead); warps 1..7 subtract L_ki^T x_k from the y_i above it,
  // their tiles (k, i) -- at most two per warp -- fetched into registers before x_k exists.  Named barrier 1: "x_k is in s_vec",
  // named barrier 2: "step k is folded into s_y".
  if (warp == 0) {
    double inv_c[kT], inv_n[kT];
#pragma unroll
    for (int r = 0; r < kT; r++) inv_c[r] = __ldcg(p.Linv + ((size_t)(nt - 1) * kT + r) * kT + lane);
    __syncthreads();
    for (int k = nt - 1; k >= 0; k--) {
      const double* invp = p.Linv + (size_t)k * kT * kT + lane;
      if (k > 0) {
#pragma unroll
        for (int r = 0; r < kT; r++) inv_n[r] = __ldcg(invp - kT * kT + r * kT);
      }
      // x_k = Linv_kk^T y_k : lane c computes sum_r Linv[r][c] * y[r].  A sentinel (a NaN) in an operand shows in the result: only then are
      // the operands re-read until they are all there -- no per-element test on the fast path
      const double yk = s_y[k * kT + lane];
      double xk;
      for (int tries = 0;; tries++) {
        double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
#pragma unroll
        for (int r = 0; r < kT; r += 4) {
          s0 += inv_c[r] * __shfl_sync(0xffffffffu, yk, r);
          s1 += inv_c[r + 1] * __shfl_sync(0xffffffffu, yk, r + 1);
          s2 += inv_c[r + 2] * __shfl_sync(0xffffffffu, yk, r + 2);
          s3 += inv_c[r + 3] * __shfl_sync(0xffffffffu, yk, r + 3);
        }
        xk = (s0 + s1) + (s2 + s3);
        if (!__any_sync(0xffffffffu, xk != xk)) break;
        bool bad = false;
#pragma unroll
        for (int r = 0; r < kT; r++) bad |= is_sentinel(inv_c[r]);
        if (!__any_sync(0xffffffffu, bad) || tries > (1 << 18)) break;     // a genuine NaN (failed factorisation), or time-out
        __nanosleep(100);
#pragma unroll
        for (int r = 0; r < kT; r++) inv_c[r] = __ldcg(invp + r * kT);
      }
      s_vec[lane] = xk;
      s_y[k * kT + lane] = xk;
      asm volatile("bar.sync 1, %0;" ::"n"(kCholThreads) : "memory");
      asm volatile("bar.sync 2, %0;" ::"n"(kCholThreads) : "memory");
#pragma unroll
      for (int r = 0; r < kT; r++) inv_c[r] = inv_n[r];
    }
  } else {
    double tl[2][kT];
    auto fetch_tile = [&](int k, int sl) {
      const int ii = (warp - 1) + (kCholWarps - 1) * sl;
      if (ii < k) {
        const double* tp = L + (size_t)(k * kT) * ld + ii * kT + lane;
#pragma unroll
        for (int r = 0; r < kT; r++) tl[sl][r] = __ldcg(tp + (size_t)r * ld);
      }
    };
    __syncthreads();
    fetch_tile(nt - 1, 0);
    fetch_tile(nt - 1, 1);
    for (int k = nt - 1; k >= 0; k--) {
      asm volatile("bar.sync 1, %0;" ::"n"(kCholThreads) : "memory");
      // y_i -= L_ki^T x_k : lane = column of tile (k,i)
#pragma unroll
      for (int sl = 0; sl < 2; sl++) {
        const int ii = (warp - 1) + (kCholWarps - 1) * sl;
        if (ii < k) {
          double sum;
          for (int tries = 0;; tries++) {
            double s0 = 0.0, s1 = 0.0;
#pragma unroll
            for (int r = 0; r < kT; r += 2) { s0 += tl[sl][r] * s_vec[r]; s1 += tl[sl][r + 1] * s_vec[r + 1]; }
            sum = s0 + s1;
            if (!__any_sync(0xffffffffu, sum != sum)) break;
            bool bad = false;
#pragma unroll
            for (int r = 0; r < kT; r++) bad |= is_sentinel(tl[sl][r]);
            if (!__any_sync(0xffffffffu, bad) || tries > (1 << 18)) break;
            __nanosleep(100);
            fetch_tile(k, sl);
          }
          s_y[ii * kT + lane] -= sum;
        }
      }
      if (k > 0) { fetch_tile(k - 1, 0); fetch_tile(k - 1, 1); }
      asm volatile("bar.sync 2, %0;" ::"n"(kCholThreads) : "memory");
    }
  }
  __syncthreads();
  const bool failed = (*reinterpret_cast<volatile int*>(p.fail)) != 0;
  for (int q = tid; q < n; q += kCholThreads) {
    const double v = s_y[q];
    p.x[q] = (failed || !isfinite(v)) ? 0.f : (float)v;      // a failed factorisation leaves NaNs (or sentinels) everywhere: zeros, like the reference
  }
}

// Placement of the resident kernel's tiles on the cluster's warp slots.  The fp64 pipe of an SM is narrow (64 lanes/clk, measured) and the
// potrf of a diagonal tile is a chain of ~8 dependent fp64 operations per column: measured, it takes 5.3 us while other warps of the
// SM stream the DFMAs of their trailing updates and 2.9 us alone.  A tile of column c works until column c is finished, and potrf(s)
// runs when column s-1 is finished, so diagonal tile s gets CTA s to itself *in time*: a column-c tile may only share that SM if c < s
// (finished before), if the SM has no diagonal tile (s >= nt), or if s == 0 (potrf(0) runs before anything else has operands).
// Tiles of one column substitute at the same time and are spread over different SMs where possible.  Returns false if ncta is too small.
static bool resident_tile_map(int nt, int ncta, unsigned char* map_i, unsigned char* map_j) {
  int nfree[16], used[16][kCholWarps];
  unsigned colmask[16];
  for (int s = 0; s < 16; s++) { nfree[s] = kCholWarps; colmask[s] = 0; for (int w = 0; w < kCholWarps; w++) used[s][w] = 0; }
  for (int q = 0; q < 128; q++) map_i[q] = map_j[q] = 0xFF;
  if (ncta > 16 || ncta < nt) return false;
  auto place = [&](int s, int i, int j) {
    for (int w = 0; w < kCholWarps; w++)
      if (!used[s][w]) { used[s][w] = 1; nfree[s]--; map_i[s * kCholWarps + w] = (unsigned char)i; map_j[s * kCholWarps + w] = (unsigned char)j; return; }
  };
  for (int j = 0; j < nt; j++) place(j, j, j);
  for (int c = nt - 1; c >= 0; c--) {
    for (int i = c + 1; i <= nt; i++) {                      // i == nt: the right-hand side piece of column c
      int best = -1, best_key = 1 << 30;
      for (int pass = 0; pass < 2 && best < 0; pass++) {
        for (int s = 0; s < ncta; s++) {
          if (nfree[s] == 0) continue;
          const bool eligible = (s > c) || (s >= nt) || (s == 0);
          if (pass == 0 && !eligible) continue;
          const int key = (((colmask[s] >> c) & 1u) ? 4096 : 0) + ((s > c && s < nt) ? 0 : 1024) + (kCholWarps - nfree[s]) * 16 + s;
          if (key < best_key) { best_key = key; best = s; }
        }
      }
      if (best < 0) return false;
      place(best, i, c);
      colmask[best] |= 1u << c;
    }
  }
  return true;
}

// CTAs of the resident kernel's cluster for nt tile rows: every tile needs its own warp and every diagonal tile its own CTA.
// 0: the system is too large for the resident kernel.
static int resident_cluster_size(int nt) {
  if (nt > kResMaxNt) return 0;
  const int tiles = nt * (nt + 1) / 2 + nt;
  int rcs = 1;
  while (rcs * kCholWarps < tiles || rcs < nt) rcs *= 2;
  return rcs;
}

constexpr int kCholDynSmem = (2 * kCholWarps + 2) * kT * kTP * sizeof(double);

// the largest cluster (16 CTAs, else 8) the device can run chol_cluster_kernel with
int chol_cluster_probe() {
  kernel_setup((const void*)chol_cluster_kernel, kCholDynSmem, true);    // a failure here is reported by the launch
  int best = 8;
  for (int cs = 16; cs >= 8; cs -= 8) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(cs); cfg.blockDim = dim3(kCholThreads); cfg.dynamicSmemBytes = kCholDynSmem;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension; at[0].val.clusterDim.x = cs; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    int nclusters = 0;
    if (cudaOccupancyMaxActiveClusters(&nclusters, chol_cluster_kernel, &cfg) == cudaSuccess && nclusters >= 1) { best = cs; break; }
  }
  cudaGetLastError();
  return best;
}

size_t chol_workspace_bytes(int n) {
  const size_t nt = (size_t)(n + kT - 1) / kT;
  const size_t ld = nt * kT;
  return ((nt + 1) * kT * ld + nt * kT * kT + nt * kT) * sizeof(double) + (nt + 2) * sizeof(int) + 256 +
         (size_t)kResMaxNt * kT * kT * sizeof(double) + 256;
}

// H [n][n] fp64, b [n] fp64 -> x [n] fp32; fail flag is a device int
int chol_solve_launch(const double* H, const double* b, int n, double lm, double ep, void* workspace, int* fail, float* x, cudaStream_t st,
                      const CholPeers* peers) {
  if (n <= 0) return DBA_OK;
  CholParams p;
  p.H = H; p.b = b; p.n = n; p.nt = (n + kT - 1) / kT; p.lm = lm; p.ep = ep; p.fail = fail; p.x = x;
  if (peers) p.peers = *peers; else { p.peers.world = 0; p.peers.flags = nullptr; p.peers.epoch = 0; p.peers.epoch_dev = nullptr; for (int k = 0; k < 8; k++) p.peers.sys[k] = nullptr; }
  const size_t ld = (size_t)p.nt * kT;
  p.L = reinterpret_cast<double*>(workspace);
  p.Linv = p.L + (size_t)(p.nt + 1) * kT * ld;
  p.rdiag = p.Linv + (size_t)p.nt * kT * kT;
  p.first = reinterpret_cast<int*>(p.rdiag + (size_t)p.nt * kT);
  p.Cs = reinterpret_cast<double*>((reinterpret_cast<uintptr_t>(p.first + (p.nt + 2)) + 255) & ~(uintptr_t)255);

  int rc;
  if ((rc = kernel_setup((const void*)chol_cluster_kernel, kCholDynSmem, true))) return rc;
  if ((rc = kernel_setup((const void*)chol_resident_kernel<false>, kCholDynSmem, true))) return rc;
  if ((rc = kernel_setup((const void*)chol_resident_kernel<true>, kCholDynSmem, true))) return rc;
  DeviceInfo dev;
  if ((rc = device_info(&dev))) return rc;
  cudaLaunchConfig_t cfg = {};
  cfg.blockDim = dim3(kCholThreads); cfg.dynamicSmemBytes = kCholDynSmem; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  const int rcs = resident_cluster_size(p.nt);
  if (rcs > 0 && rcs <= dev.chol_cluster && resident_tile_map(p.nt, rcs, p.map_i, p.map_j)) {
    cfg.gridDim = dim3(rcs);
    at[0].val.clusterDim.x = rcs;
    if (p.peers.world > 1) DBA_CHECK_CUDA(cudaLaunchKernelEx(&cfg, chol_resident_kernel<true>, p), "chol_resident_kernel launch");
    else DBA_CHECK_CUDA(cudaLaunchKernelEx(&cfg, chol_resident_kernel<false>, p), "chol_resident_kernel launch");
    return DBA_OK;
  }
  // small systems do not need the whole cluster
  int cs = dev.chol_cluster;
  const int tiles_first_panel = p.nt * (p.nt + 1) / 2 + 1;
  while (cs > 1 && (cs / 2) * kCholWarps - 1 >= tiles_first_panel) cs /= 2;
  cfg.gridDim = dim3(cs);
  at[0].val.clusterDim.x = cs;
  DBA_CHECK_CUDA(cudaLaunchKernelEx(&cfg, chol_cluster_kernel, p), "chol_cluster_kernel launch");
  return DBA_OK;
}

}  // namespace dba

// host-side introspection of the resident kernel's tile placement (tests/test_oracle_cpu.py holds its invariants on the CPU):
// map_i / map_j [128] receive the tile of every warp slot (0xFF = none); returns the cluster size, 0 if n is served by the barrier kernel
extern "C" int dba_solve_tile_placement(int n, unsigned char* map_i, unsigned char* map_j) {
  if (n <= 0 || !map_i || !map_j) return 0;
  const int nt = (n + dba::kT - 1) / dba::kT;
  const int rcs = dba::resident_cluster_size(nt);
  if (rcs == 0 || !dba::resident_tile_map(nt, rcs, map_i, map_j)) return 0;
  return rcs;
}

// standalone entry (used by the solver tests and by callers that already hold a reduced system)
extern "C" size_t dba_solve_workspace_bytes(int n) { return dba::chol_workspace_bytes(n) + 64; }

extern "C" int dba_solve_spd(const double* H, const double* b, int n, float lm, float ep, float* x, int* fail_flag_device,
                             void* workspace, size_t workspace_bytes, dba_stream_t stream) {
  DBA_CHECK_ARG(n >= 0, "negative n");
  if (n == 0) return DBA_OK;
  DBA_CHECK_ARG(H && b && x && fail_flag_device && workspace, "null pointer");
  if (workspace_bytes < dba::chol_workspace_bytes(n)) { dba::set_error("solve workspace too small"); return DBA_ERR_WORKSPACE; }
  return dba::chol_solve_launch(H, b, n, (double)lm, (double)ep, workspace, fail_flag_device, x, (cudaStream_t)stream);
}
