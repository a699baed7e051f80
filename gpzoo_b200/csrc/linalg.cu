// K2: batched Cholesky fused with the triangular inverse (gp.py:213,360,55 -> torch.linalg.cholesky; the inverse turns the
// two triangular solves of torch.cholesky_solve, gp.py:218,365, into triangular matrix products), plus the small O(M^2)
// element-wise helpers of the variational parameters (lower-Cholesky transform gp.py:220, KL reductions torch kl.py MVN||MVN).
//
// Right-looking blocked factorisation, panel width NB: for each panel k the NB x NB diagonal block is factored AND inverted
// (leaf_body), then the panel L21 = A21 X11^T and the trailing update A22 -= L21 L21^T; X = Lc^-1 follows by recursive
// doubling, X21 = -X22 (L21 X11).  chol_inv runs it as one cluster kernel per factor (M <= 1536) or as a sweep of GEMM launches;
// chol_inv_hybrid (fp32, large M) runs 256-wide diagonal blocks on the cluster kernel and every larger product on tcgen05, with
// only the look-ahead (next panel block, next diagonal update) on the caller's stream and the rest of each panel, the rest of the
// trailing update and the inverse, one block row at a time (X[k,0:k] = -X[k,k] L[k,0:k] X[0:k,0:k]), on a side stream.
#include <cooperative_groups.h>

#include <mutex>
#include <type_traits>

#include "gemm_simt.cuh"
#include "gpzoo_b200.h"
#include "umma_gemm.h"

namespace gpz {

constexpr int NB = 64;

// ---- leaf: Cholesky + inverse of one 64 x 64 diagonal block -----------------------------------------
// Factor and invert the n x n (n <= 64) diagonal block at (r0, r0) of one factor: W (input, lower), Lm and X (outputs), all with
// row stride ld.  `a`, `x`: two [NB][NB+1] shared-memory tiles.  256 threads; contains block barriers.
//
// The 64 x 64 block is handled as 2 x 2 blocks of 32: each 32 x 32 diagonal block is factored AND inverted by ONE warp entirely
// in registers (lane = row, the pivot column travels by shuffles; no shared memory and no barrier inside the 32 columns), the
// three 32^3 products between them (L21 = A21 X11^T, A22 -= L21 L21^T, X21 = -X22 L21 X11) are spread over all 8 warps.
// This is the serial part of the whole Cholesky (16 leaves at M = 1024), so its latency is what matters, not its flops.
template <typename T> __device__ __forceinline__ T shfl_t(T v, int src) { return __shfl_sync(0xffffffffu, v, src); }

// A 32 x 32 diagonal block is FACTORED by one warp in registers (lane = row) and INVERTED by all eight warps (4 columns each).
// In: a[k] = A[lane][k] (only k <= lane matters).  Rolled loops whose bodies have only compile-time register indices (a fully
// unrolled version is 20 000 instructions of straight-line code that runs once and was bound by instruction fetch):
// the remaining part of the row lives at a[0..31-j]; the update writes entry k into slot k-1, so the active column is always
// slot 0 and the pivot is lane j's slot 0 (slots past the end of the row carry harmless garbage).  After 16 columns the row
// has 16 entries left and a second loop with half the slots takes over.
// Out: column j of L to Ls[lane][j], 1 / L[j][j] to rd[j].
// No division ever sees a zero numerator (an IEEE division resolves 0 / x through FCHK + a slow-path call, which makes the warp
// diverge in the middle of the shuffle sequence; the previous leaf lost 25 % on config 2's mostly-zero Kzz to exactly that).
// Software-pipelined by one column: slot 0 (the next column's entry) is updated first, the next pivot is shuffled out and its
// square root and reciprocal are issued before the other 30 updates, so their latency hides under those shuffles instead of
// starting the next column's dependent chain.
template <typename T>
__device__ __forceinline__ void pivot_sqrt_recip(T d, T& s, T& r) {
  if constexpr (std::is_same<T, float>::value) {
    // one MUFU rsqrt and a Newton step (~1 ulp) instead of sqrt followed by an IEEE division (fp64 keeps the exact path)
    const float y = rsqrtf(d);
    r = y * fmaf(-0.5f * d * y, y, 1.5f);
    s = d * r;
  } else {
    s = Num<T>::sqrt(d);
    r = T(1) / s;
  }
}
template <typename T, int LDS>
__device__ __forceinline__ void warp_chol32(T (&a)[32], T* __restrict__ Ls, T* __restrict__ rd, int lane, int* __restrict__ info_l,
                                            int base) {
  int bad = 0;                                       // first non-positive pivot (uniform)
  T d = shfl_t(a[0], 0), s, r;                       // pivot of the current column, uniform over the warp
  pivot_sqrt_recip(d, s, r);
  auto column = [&](int j, auto nslots) {
    constexpr int NS = decltype(nslots)::value;
    bad = (bad == 0 && !(d > T(0))) ? base + j + 1 : bad;           // not positive definite (also catches NaN)
    const T lij = lane > j ? a[0] * r : (lane == j ? s : T(0));     // L[lane][j]
    Ls[lane * LDS + j] = lij;
    if (lane == 0) rd[j] = r;
    const T lsub = lane > j ? lij : T(0);
    a[0] = fma(-lsub, shfl_t(lij, (j + 1) & 31), a[1]);
    d = shfl_t(a[0], (j + 1) & 31);                  // next pivot (garbage after the last column, never used)
    pivot_sqrt_recip(d, s, r);
#pragma unroll
    for (int k = 2; k < NS; ++k) a[k - 1] = fma(-lsub, shfl_t(lij, (j + k) & 31), a[k]);
  };
#pragma unroll 1
  for (int j = 0; j < 16; ++j) column(j, std::integral_constant<int, 32>{});
#pragma unroll 1
  for (int j = 16; j < 32; ++j) column(j, std::integral_constant<int, 16>{});
  if (bad != 0 && lane == 0 && *info_l == 0) *info_l = bad;
}

// X = L^-1 of the 32 x 32 block by forward substitution on the identity, row-oriented (lane = row): once row j of X is final
// (scaled by 1 / L[j][j]) every later row subtracts L[i][j] times it.  Warp w owns columns 4w .. 4w+3 (rows above them are zero,
// so its sweep starts at j = 4w).  Reads Ls / rd written by warp_chol32, writes Xs[lane][c].
template <typename T, int LDS>
__device__ __forceinline__ void warps_trinv32(const T* __restrict__ Ls, const T* __restrict__ rd, T* __restrict__ Xs, int warp, int lane) {
  const int c0 = warp * 4;
  T v[4];
#pragma unroll
  for (int u = 0; u < 4; ++u) v[u] = (c0 + u == lane) ? T(1) : T(0);
#pragma unroll 2
  for (int j = c0; j < 32; ++j) {
    const T r = rd[j];
    const T lsub = lane > j ? Ls[lane * LDS + j] : T(0);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const T xj = shfl_t(v[u], j) * r;              // X[j][c], final
      v[u] = lane == j ? xj : fma(-lsub, xj, v[u]);
    }
  }
#pragma unroll
  for (int u = 0; u < 4; ++u) Xs[lane * LDS + c0 + u] = (c0 + u <= lane) ? v[u] : T(0);
}

template <typename T>
__device__ void leaf_body(T (*a)[NB + 1], T (*x)[NB + 1], const T* __restrict__ W, T* __restrict__ Lm, T* __restrict__ X, int64_t ld,
                          int r0, int n, int* __restrict__ info_l, int info_off = 0, long long* __restrict__ dbg = nullptr) {
  constexpr int H = 32;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  long long tc0 = clock64();
  auto mark = [&](int slot) { if (dbg != nullptr && tid == 0) { const long long t = clock64(); dbg[slot] = t - tc0; tc0 = t; } };
  // identity padding beyond n keeps the routine free of size tests; the padding never reaches global memory
  // all 16 loads of a thread are issued before the first shared-memory store (one round trip instead of 16 dependent ones)
  T w[NB * NB / 256];
#pragma unroll
  for (int u = 0; u < NB * NB / 256; ++u) {
    const int i = (tid >> 6) + 4 * u, j = tid & (NB - 1);
    w[u] = (i < n && j <= i) ? W[(int64_t)(r0 + i) * ld + r0 + j] : ((i == j && i >= n) ? T(1) : T(0));
  }
#pragma unroll
  for (int u = 0; u < NB * NB / 256; ++u) {
    const int i = (tid >> 6) + 4 * u, j = tid & (NB - 1);
    a[i][j] = w[u];
    x[i][j] = T(0);
  }
  __syncthreads();
  mark(0);
  __shared__ T rdiag[H];
  auto diag_block = [&](int o) {                     // factor (warp 0) + invert (all warps) the 32 x 32 block at (o, o)
    if (warp == 0) {
      T ar[H];
#pragma unroll
      for (int k = 0; k < H; ++k) ar[k] = a[o + lane][o + k];
      warp_chol32<T, NB + 1>(ar, &a[o][o], rdiag, lane, info_l, info_off + r0 + o);
    }
    __syncthreads();
    warps_trinv32<T, NB + 1>(&a[o][o], rdiag, &x[o][o], warp, lane);
    __syncthreads();
  };
  diag_block(0);
  mark(1);
  if (n > H) {
    const int i = H + (tid >> 3), j0 = (tid & 7) * 4;      // 4 outputs (i, j0..j0+3) per thread in every 32^3 product
    T acc[4];
    // L21 = A21 X11^T      (X11 lower: x[j][t] = 0 for t > j)
#pragma unroll
    for (int u = 0; u < 4; ++u) acc[u] = T(0);
#pragma unroll 8
    for (int t = 0; t < H; ++t) {
      const T av = a[i][t];
#pragma unroll
      for (int u = 0; u < 4; ++u) acc[u] = fma(av, x[j0 + u][t], acc[u]);
    }
    __syncthreads();                                       // A21 has been read by everyone: overwrite it with L21
#pragma unroll
    for (int u = 0; u < 4; ++u) a[i][j0 + u] = acc[u];
    __syncthreads();
    // A22 -= L21 L21^T
#pragma unroll
    for (int u = 0; u < 4; ++u) acc[u] = T(0);
#pragma unroll 8
    for (int t = 0; t < H; ++t) {
      const T av = a[i][t];
#pragma unroll
      for (int u = 0; u < 4; ++u) acc[u] = fma(av, a[H + j0 + u][t], acc[u]);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) a[i][H + j0 + u] -= acc[u];
    __syncthreads();
    mark(2);
    diag_block(H);
    mark(3);
    // tmp = L21 X11  (into the still empty X21), then X21 = -X22 tmp
#pragma unroll
    for (int u = 0; u < 4; ++u) acc[u] = T(0);
#pragma unroll 8
    for (int t = 0; t < H; ++t) {
      const T av = a[i][t];
#pragma unroll
      for (int u = 0; u < 4; ++u) acc[u] = fma(av, x[t][j0 + u], acc[u]);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) x[i][j0 + u] = acc[u];
    __syncthreads();
#pragma unroll
    for (int u = 0; u < 4; ++u) acc[u] = T(0);
#pragma unroll 8
    for (int t = 0; t < H; ++t) {
      const T xv = x[i][H + t];                            // X22[i][t] (0 for t > i - 32)
#pragma unroll
      for (int u = 0; u < 4; ++u) acc[u] = fma(xv, x[H + t][j0 + u], acc[u]);
    }
    __syncthreads();                                       // tmp has been read by everyone
#pragma unroll
    for (int u = 0; u < 4; ++u) x[i][j0 + u] = -acc[u];
    __syncthreads();
    mark(4);
  }
#pragma unroll
  for (int u = 0; u < NB * NB / 256; ++u) {
    const int i = (tid >> 6) + 4 * u, j = tid & (NB - 1);
    if (i < n && j < n) {
      Lm[(int64_t)(r0 + i) * ld + r0 + j] = j <= i ? a[i][j] : T(0);
      X[(int64_t)(r0 + i) * ld + r0 + j] = j <= i ? x[i][j] : T(0);
    }
  }
  mark(5);
}

template <typename T>
__global__ void __launch_bounds__(256) chol_inv_leaf_kernel(const T* __restrict__ Wall, T* __restrict__ Lall, T* __restrict__ Xall,
                                                             int M, int r0, int n, int* __restrict__ info) {
  extern __shared__ __align__(16) unsigned char leaf_smem[];
  typedef T Row[NB + 1];
  Row* a = reinterpret_cast<Row*>(leaf_smem);
  Row* x = a + NB;
  const int64_t off = (int64_t)blockIdx.x * M * M;
  leaf_body<T>(a, x, Wall + off, Lall + off, Xall + off, (int64_t)M, r0, n, info + blockIdx.x);
}

// ---- the whole Cholesky + inverse of one factor in ONE kernel: a thread-block cluster of 8 CTAs per factor --------
// Same right-looking algorithm as chol_inv() below, but the ~60 dependent launches become phases separated by
// hardware cluster barriers (barrier.cluster, ~0.2 us): leaf on CTA 0 -> panel row blocks over the 8 CTAs -> trailing
// 64 x 64 tiles over the 8 CTAs, while the inverse grows one block row per step on the CTAs that do not run the leaf.  All tile products are 64 x 64 x 64 from
// shared memory; matrices stay in global memory (L2-resident: 3 x 4 MB per factor).
constexpr int CL = 8;     // CTAs per cluster

constexpr int TLD = NB + 4;     // padded row length of the k-major operand tiles (keeps 16-byte alignment for vector loads)

// k-major operand tile: dst[t][i] = src[(r0+i)*ld + c0+t]  (transpose == false: rows i of a row-major block, reduction index
// t along its columns) or dst[t][i] = src[(r0+t)*ld + c0+i] (transpose == true: reduction index along the rows).
// nr, nc: valid rows / columns of the source block, zero outside.
template <typename T>
__device__ __forceinline__ void load_tile(T (*dst)[TLD], const T* __restrict__ src, int64_t ld, int r0, int c0, int nr, int nc,
                                          bool transpose) {
#pragma unroll 4
  for (int e = threadIdx.x; e < NB * NB; e += 256) {
    const int r = e >> 6, c = e & (NB - 1);           // source row / column inside the block (coalesced along c)
    const T v = (r < nr && c < nc) ? src[(int64_t)(r0 + r) * ld + c0 + c] : T(0);
    if (transpose) dst[r][c] = v; else dst[c][r] = v;
  }
}
__device__ __forceinline__ void ld4(const float* p, float (&o)[4]) {
  const float4 v = *reinterpret_cast<const float4*>(p);
  o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w;
}
__device__ __forceinline__ void ld4(const double* p, double (&o)[4]) {
  const double2 v0 = reinterpret_cast<const double2*>(p)[0], v1 = reinterpret_cast<const double2*>(p)[1];
  o[0] = v0.x; o[1] = v0.y; o[2] = v1.x; o[3] = v1.y;
}
// acc[u][v] += sum_t A[t][ty*4+u] * B[t][tx*4+v]   (both operands k-major in shared memory, two vector loads per 16 FMAs)
template <typename T>
__device__ __forceinline__ void tile_abt(const T (*A)[TLD], const T (*B)[TLD], T (&acc)[4][4]) {
  const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;
#pragma unroll 8
  for (int t = 0; t < NB; ++t) {
    T av[4], bv[4];
    ld4(&A[t][ty * 4], av);
    ld4(&B[t][tx * 4], bv);
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int v = 0; v < 4; ++v) acc[u][v] = fma(av[u], bv[v], acc[u][v]);
  }
}
// dst[(r0+i)*ld + c0+j] = alpha*acc + beta*dst  for i < nr, j < nc
template <typename T>
__device__ __forceinline__ void store_tile(T* __restrict__ dst, int64_t ld, int r0, int c0, int nr, int nc, const T (&acc)[4][4],
                                           T alpha, T beta) {
  const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;
#pragma unroll
  for (int u = 0; u < 4; ++u)
#pragma unroll
    for (int v = 0; v < 4; ++v) {
      const int i = ty * 4 + u, j = tx * 4 + v;
      if (i < nr && j < nc) {
        T* d = dst + (int64_t)(r0 + i) * ld + c0 + j;
        *d = beta == T(0) ? alpha * acc[u][v] : alpha * acc[u][v] + beta * (*d);
      }
    }
}

// One phase of the cluster kernel = a list of tile-product steps (block coordinates gi, gj, gk + first/last flags of the
// output tile), built by thread 0 in shared memory.  run_steps() executes the list with a register-staged pipeline: the 32
// global loads of step s+1 are in flight while step s is multiplied out of shared memory.
//   A operand: MA[gi][gk];  B operand: MB[gj][gk] (b_tr = false) or MB[gk][gj] (b_tr = true);  out: MO[gi][gj] = alpha*acc + beta*MO
constexpr int MAX_STEPS = 192;

template <typename T>
__device__ void run_steps(T (*tA)[TLD], T (*tB)[TLD], const int4* __restrict__ steps, int nsteps, const T* __restrict__ MA,
                          const T* __restrict__ MB, T* __restrict__ MO, bool b_tr, T alpha, T beta, int M, int nsz) {
  // M: row stride of the matrices; nsz: size of the (sub-)matrix the block coordinates refer to
  const int tid = threadIdx.x;
  auto bsz = [&](int b) { return min(NB, nsz - b * NB); };
  T ra[16], rb[16], rc[4][4];
  const int ty = tid >> 4, tx = tid & 15;
  auto fetch = [&](int sidx) {
    const int4 st = steps[sidx];
    if (beta != T(0) && (st.w & 2)) {                  // read-modify-write output tile: its old values ride along with the operands
      const int onr = bsz(st.x), onc = bsz(st.y);
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int v = 0; v < 4; ++v) {
          const int i = ty * 4 + u, j = tx * 4 + v;
          rc[u][v] = (i < onr && j < onc) ? MO[(int64_t)(st.x * NB + i) * M + st.y * NB + j] : T(0);
        }
    }
    const int ar0 = st.x * NB, ac0 = st.z * NB, anr = bsz(st.x), anc = bsz(st.z);
    const int br0 = (b_tr ? st.z : st.y) * NB, bc0 = (b_tr ? st.y : st.z) * NB;
    const int bnr = bsz(b_tr ? st.z : st.y), bnc = bsz(b_tr ? st.y : st.z);
#pragma unroll
    for (int u = 0; u < 16; ++u) {
      const int e = tid + u * 256, r = e >> 6, c = e & (NB - 1);
      ra[u] = (r < anr && c < anc) ? MA[(int64_t)(ar0 + r) * M + ac0 + c] : T(0);
      rb[u] = (r < bnr && c < bnc) ? MB[(int64_t)(br0 + r) * M + bc0 + c] : T(0);
    }
  };
  if (nsteps <= 0) return;
  fetch(0);
  T acc[4][4];
  for (int sidx = 0; sidx < nsteps; ++sidx) {
    const int4 st = steps[sidx];
    __syncthreads();                                   // previous product finished reading the tiles
#pragma unroll
    for (int u = 0; u < 16; ++u) {
      const int e = tid + u * 256, r = e >> 6, c = e & (NB - 1);
      tA[c][r] = ra[u];                               // k-major: [t][i]
      if (b_tr) tB[r][c] = rb[u]; else tB[c][r] = rb[u];
    }
    __syncthreads();
    T oc[4][4];
    if (beta != T(0) && (st.w & 2)) {
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int v = 0; v < 4; ++v) oc[u][v] = rc[u][v];
    }
    if (sidx + 1 < nsteps) fetch(sidx + 1);            // next step's loads overlap this step's FMAs
    if (st.w & 1) {
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int v = 0; v < 4; ++v) acc[u][v] = T(0);
    }
    tile_abt<T>(tA, tB, acc);
    if (st.w & 2) {
      if (beta != T(0)) {
        const int onr = bsz(st.x), onc = bsz(st.y);
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
          for (int v = 0; v < 4; ++v) {
            const int i = ty * 4 + u, j = tx * 4 + v;
            if (i < onr && j < onc) MO[(int64_t)(st.x * NB + i) * M + st.y * NB + j] = alpha * acc[u][v] + beta * oc[u][v];
          }
      } else {
        store_tile<T>(MO, M, st.x * NB, st.y * NB, bsz(st.x), bsz(st.y), acc, alpha, beta);
      }
    }
  }
}

template <typename T>
__global__ void __cluster_dims__(CL, 1, 1) __launch_bounds__(256)
chol_inv_cluster_kernel(T* __restrict__ Wall, T* __restrict__ Lall, T* __restrict__ Xall, T* __restrict__ Tall, int M, int blk0,
                        int nsz, int* __restrict__ info, long long* __restrict__ dbg, float* __restrict__ Xlo_all = nullptr) {
  // factors + inverts the nsz x nsz diagonal block starting at row / column blk0 of every M x M matrix (blk0 = 0, nsz = M: all
  // of it); block coordinates below are relative to that block, M is the row stride.
  // Xlo_all (fp32 only, the hybrid's diagonal blocks): finally write the tf32 lo plane of the X block and zeros above the diagonal
  // of the Lc, X and Xlo blocks, so that nothing has to be zeroed or split before or after this launch.
  namespace cg = cooperative_groups;
  cg::cluster_group cluster = cg::this_cluster();
  extern __shared__ __align__(16) unsigned char cl_smem[];
  typedef T Row[TLD];
  typedef T LeafRow[NB + 1];
  Row* tA = reinterpret_cast<Row*>(cl_smem);
  Row* tB = tA + NB;
  LeafRow* la = reinterpret_cast<LeafRow*>(cl_smem);            // the leaf uses the same memory with its own row length
  LeafRow* lx = la + NB;
  __shared__ int4 steps[MAX_STEPS];
  __shared__ int nsteps_s, q_next_s;
  const int l = blockIdx.x / CL, rank = (int)cluster.block_rank();
  const int64_t off = (int64_t)l * M * M + (int64_t)blk0 * M + blk0;
  T* W = Wall + off; T* Lm = Lall + off; T* X = Xall + off; T* Tm = Tall + off;
  const int nblk = (nsz + NB - 1) / NB;
  auto bsz = [&](int b) { return min(NB, nsz - b * NB); };

  long long t_leaf = 0, t_panel = 0, t_trail = 0, t_inv = 0, t0 = clock64(), t1;
  // ---- factorisation, with look-ahead: while CTAs 1..7 apply the trailing update of step k, CTA 0 updates the next
  //      diagonal tile first and immediately factors / inverts it (the leaf is the serial part of the chain) ----
  if (rank == 0) leaf_body<T>(la, lx, W, Lm, X, (int64_t)M, 0, bsz(0), info + l, blk0, (dbg != nullptr && blockIdx.x == 0) ? dbg + 4 : nullptr);
  cluster.sync();
  t1 = clock64(); t_leaf += t1 - t0; t0 = t1;
  // The inverse is built one block row at a time, X[k][0:k] = -X[k][k] tmp[k][0:k] with tmp[k][0:k] = Lc[k][0:k] X[0:k][0:k]:
  // tmp row k+1 needs nothing of leaf k+1, so CTAs 1..7 compute it while CTA 0 runs that leaf, and block row k joins the panel
  // phase of step k.  Only the last block row is left after the factorisation.
  // Runs one list of tile-product steps; tile q of the list (nq tiles) with `cost(q)` steps goes to CTA `owner(q)`; `emit(q, t,
  // flags)` writes the t-th step of tile q.  The per-CTA list is processed in rounds of at most MAX_STEPS steps.
  auto run_list = [&](int nq, auto owner, auto cost, auto emit, const T* MA, const T* MB, T* MO, bool b_tr, T alpha, T beta) {
    for (int q_start = 0; q_start >= 0;) {
      if (threadIdx.x == 0) {
        int ns = 0, q_next = -1;
        for (int q = q_start; q < nq; ++q) {
          if (owner(q) != rank) continue;
          const int c = cost(q);
          if (ns + c > MAX_STEPS) { q_next = q; break; }
          for (int t = 0; t < c; ++t) steps[ns++] = emit(q, t, (t == 0 ? 1 : 0) | (t == c - 1 ? 2 : 0));
        }
        nsteps_s = ns;
        q_next_s = q_next;
      }
      __syncthreads();
      const int ns = nsteps_s, qn = q_next_s;
      run_steps<T>(tA, tB, steps, ns, MA, MB, MO, b_tr, alpha, beta, M, nsz);
      __syncthreads();
      q_start = qn;
    }
  };
  // X[k][j] = -X[k][k] tmp[k][j], j < k   (one step per tile; owners from the top rank down, the panel's start at rank 0)
  auto inverse_row = [&](int k) {
    run_list(k, [&](int j) { return CL - 1 - j % CL; }, [](int) { return 1; },
             [&](int j, int, int f) { return make_int4(k, j, k, f); }, X, Tm, X, true, T(-1), T(0));
  };
  for (int k = 0; k < nblk - 1; ++k) {
    const int nrb = nblk - k - 1;                       // row blocks below the diagonal block (>= 1 here)
    // panel: L21 = W21 X11^T      (A = W[gi][k], B = X[k][k], out = Lc[gi][k]); block row k of the inverse
    run_list(nrb, [](int rb) { return rb % CL; }, [](int) { return 1; },
             [&](int rb, int, int f) { return make_int4(k + 1 + rb, k, k, f); }, W, X, Lm, false, T(1), T(0));
    inverse_row(k);
    cluster.sync();
    t1 = clock64(); t_panel += t1 - t0; t0 = t1;
    // trailing update of the lower triangle: W[gi][gj] -= Lc[gi][k] Lc[gj][k]^T.
    // Tile 0 (the next diagonal block) belongs to CTA 0, which then runs the next leaf; tiles 1.. go round-robin to CTAs 1..7.
    run_list(nrb * (nrb + 1) / 2, [](int q) { return q == 0 ? 0 : 1 + (q - 1) % (CL - 1); }, [](int) { return 1; },
             [&](int q, int, int f) {
               int bi = 0;
               while ((bi + 1) * (bi + 2) / 2 <= q) ++bi;
               return make_int4(k + 1 + bi, k + 1 + q - bi * (bi + 1) / 2, k, f);
             }, Lm, Lm, W, false, T(-1), T(1));
    if (rank == 0) {
      leaf_body<T>(la, lx, W, Lm, X, (int64_t)M, (k + 1) * NB, bsz(k + 1), info + l, blk0);
    } else {
      // tmp[k+1][j] = sum_{t=j}^{k} Lc[k+1][t] X[t][j]   (k - j + 1 steps; X rows 0..k are final after the panel phase)
      run_list(k + 1, [](int j) { return 1 + j % (CL - 1); }, [&](int j) { return k - j + 1; },
               [&](int j, int t, int f) { return make_int4(k + 1, j, j + t, f); }, Lm, X, Tm, true, T(1), T(0));
    }
    cluster.sync();
    t1 = clock64(); t_trail += t1 - t0; t0 = t1;
  }
  if (nblk > 1) {
    inverse_row(nblk - 1);
    cluster.sync();
  }
  if constexpr (std::is_same<T, float>::value) {
    if (Xlo_all != nullptr) {                              // X is final everywhere after the last cluster barrier
      float* Xlo = Xlo_all + off;
      for (int q = rank; q < nblk * nblk; q += CL) {
        const int bi = q / nblk, bj = q % nblk, nr = bsz(bi), nc = bsz(bj);
        for (int e = threadIdx.x; e < NB * NB; e += 256) {
          const int i = e >> 6, j = e & (NB - 1);
          if (i >= nr || j >= nc) continue;
          const int64_t o = (int64_t)(bi * NB + i) * M + bj * NB + j;
          if (bi >= bj) {
            Xlo[o] = tf32_lo_part(X[o]);
          } else {
            Lm[o] = 0.f; X[o] = 0.f; Xlo[o] = 0.f;
          }
        }
      }
    }
  }
  t1 = clock64(); t_inv = t1 - t0;
  if (dbg != nullptr && blockIdx.x == 0 && threadIdx.x == 0) { dbg[0] = t_leaf; dbg[1] = t_panel; dbg[2] = t_trail; dbg[3] = t_inv; }
}

// profiling hook (tools/prof_chol.py): when set, the first cluster launch of a call writes 10 clock64 counts there, its four phases
// (leaf, panel, trailing update + leaves, inverse) and the six phases of its first leaf
long long* g_chol_dbg = nullptr;
extern "C" void gpz_chol_debug_(long long* p) { g_chol_dbg = p; }

// batched (outer = factor, inner = block pair) GEMM on sub-blocks of L x M x M matrices
template <typename T>
static int gemm_pairs(cudaStream_t st, int m, int n, int k, T alpha, const T* A, const T* B, T beta, T* D, int M, int L, int npairs,
                      int64_t pair_stride, int a_tri, int b_tri) {
  GemmParams<T> p;
  p.A = A; p.B = B; p.D = D; p.m = m; p.n = n; p.k = k; p.lda = p.ldb = p.ldd = M;
  p.sAo = p.sBo = p.sDo = (int64_t)M * M;
  p.sAi = p.sBi = p.sDi = pair_stride;
  p.batch = L * npairs; p.batch_inner = npairs;
  p.alpha = alpha; p.beta = beta; p.a_tri = a_tri; p.b_tri = b_tri; p.d_tri = 0; p.splitk = 1;
  return gemm_launch(p, false, false, st);
}

// W: L x M x M copy of the (jittered) Kzz, destroyed; Lc, X: outputs; tmp: L x M x M scratch.
// Right-looking blocked factorisation (NB = 64): leaf (factor + invert the diagonal block) -> panel L21 = A21 X11^T (GEMM,
// all row blocks in parallel) -> trailing SYRK (GEMM); then X = Lc^-1 by recursive doubling from the 64 x 64 diagonal
// inverses:  X21 = -X22 (L21 X11) for all block pairs of a level at once (log2(M/64) levels, 2 batched GEMMs each).
template <typename T> int chol_inv(T* W, T* Lc, T* X, T* tmp, int M, int L, int* info, cudaStream_t st) {
  const int64_t sL = (int64_t)M * M;
  GPZ_CUDA(cudaMemsetAsync(info, 0, sizeof(int) * L, st));
  GPZ_CUDA(cudaMemsetAsync(Lc, 0, sizeof(T) * sL * L, st));
  GPZ_CUDA(cudaMemsetAsync(X, 0, sizeof(T) * sL * L, st));
  constexpr int smem = (int)(2 * NB * (NB + 1) * sizeof(T));
  // one cluster kernel while the chain is latency-bound (M <= 1536); beyond that the O(M^3) trailing updates dominate and
  // the multi-launch path below, whose GEMMs use the whole GPU, is faster (measured: M = 2048 23.8 vs 26.7 ms/step)
  if (M <= 1536) {
    constexpr int csmem = (int)(2 * NB * TLD * sizeof(T));
    GPZ_CUDA(cudaFuncSetAttribute(chol_inv_cluster_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, csmem));
    chol_inv_cluster_kernel<T><<<L * CL, 256, csmem, st>>>(W, Lc, X, tmp, M, 0, M, info, g_chol_dbg);
    GPZ_CHECK_LAUNCH();
    return GPZ_OK;
  }
  GPZ_CUDA(cudaFuncSetAttribute(chol_inv_leaf_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  for (int k0 = 0; k0 < M; k0 += NB) {
    const int nb = min(NB, M - k0);
    chol_inv_leaf_kernel<T><<<L, 256, smem, st>>>(W, Lc, X, M, k0, nb, info);
    GPZ_CHECK_LAUNCH();
    const int rem = M - k0 - nb;
    if (rem > 0) {
      const int64_t o11 = (int64_t)k0 * M + k0, o21 = (int64_t)(k0 + nb) * M + k0, o22 = (int64_t)(k0 + nb) * M + k0 + nb;
      int rc = gemm<T>(st, false, true, rem, nb, nb, T(1), W + o21, M, sL, X + o11, M, sL, T(0), Lc + o21, M, sL, L, 0, 2, 0);
      if (rc) return rc;
      rc = gemm<T>(st, false, true, rem, rem, nb, T(-1), Lc + o21, M, sL, Lc + o21, M, sL, T(1), W + o22, M, sL, L, 0, 0, 1);
      if (rc) return rc;
    }
  }
  for (int b = NB; b < M; b *= 2) {
    // pairs of blocks [2pb, 2pb+b) (done) and [2pb+b, 2pb+2b) (done): fill the off-diagonal block X21 of the pair
    const int nfull = M / (2 * b);                       // pairs whose second block is complete
    const int64_t pstride = (int64_t)2 * b * M + 2 * b;   // diagonal step from one pair to the next
    if (nfull > 0) {
      // tmp21 = L21 X11 ; X21 = -X22 tmp21      (block offsets inside the first pair)
      int rc = gemm_pairs<T>(st, b, b, b, T(1), Lc + (int64_t)b * M, X, T(0), tmp + (int64_t)b * M, M, L, nfull, pstride, 0, 1);
      if (rc) return rc;
      rc = gemm_pairs<T>(st, b, b, b, T(-1), X + (int64_t)b * M + b, tmp + (int64_t)b * M, T(0), X + (int64_t)b * M, M, L, nfull,
                         pstride, 1, 0);
      if (rc) return rc;
    }
    const int r0 = nfull * 2 * b;                         // a trailing, incomplete pair
    const int m2 = M - r0 - b;
    if (m2 > 0) {
      const int64_t o11 = (int64_t)r0 * M + r0, o21 = (int64_t)(r0 + b) * M + r0, o22 = (int64_t)(r0 + b) * M + r0 + b;
      int rc = gemm<T>(st, false, false, m2, b, b, T(1), Lc + o21, M, sL, X + o11, M, sL, T(0), tmp + o21, M, sL, L, 0, 1, 0);
      if (rc) return rc;
      rc = gemm<T>(st, false, false, m2, b, m2, T(-1), X + o22, M, sL, tmp + o21, M, sL, T(0), X + o21, M, sL, L, 1, 0, 0);
      if (rc) return rc;
    }
  }
  return GPZ_OK;
}

// ---- large M (fp32): right-looking with 256-wide panels; diagonal blocks on the cluster kernel, everything else on tcgen05 -------
// The cluster kernel above is bound by its serial chain of 64 x 64 leaves and by CUDA-core tile products, the sweep by its rank-64
// trailing updates (each a memory-bound read-modify-write of the whole trailing matrix on the CUDA cores: 29 ms at M = 4096, L = 10).
// Here the cluster kernel only factors and inverts the HYB_NB x HYB_NB diagonal blocks (4 leaves each), and every product that
// involves more than one such block is a batched tcgen05 split-TF32 GEMM on sub-blocks in place (row stride M).  The split-TF32
// kernel needs the lo plane (x - tf32(x)) of each operand: Wlo / Llo / Xlo / Tlo shadow W / Lc / X / tmp with the same layout; GEMM
// epilogues write the lo plane of what they produce, the cluster kernel that of its X block.
//
// Only part of the work lies on the path from one diagonal block to the next.  That part runs on the caller's stream (the critical
// stream), everything else on a side stream owned by the library, where it overlaps the next cluster launch.  P = ceil(M / 256)
// panels, block indices in units of 256:
//   critical, k = 0 .. P-1:  [wait T]  cluster(k): (Lc, X, Xlo)[k,k] = chol / inv of W[k,k]
//                                      L[k+1,k] = W[k+1,k] X[k,k]^T                 (look-ahead panel, one 256^3 product)
//                            [record C]  W[k+1,k+1] -= L[k+1,k] L[k+1,k]^T          (look-ahead SYRK)
//   side, first:             zero the upper off-diagonal blocks of Lc and X; Wlo of block column 0; [record T]
//   side, k = 0 .. P-1:      [wait C]  L[k+2:,k] = W[k+2:,k] X[k,k]^T
//                                      W[k+2:,k+1] -= L[k+2:,k] L[k+1,k]^T;  W[k+2:,k+2:] -= L[k+2:,k] L[k+2:,k]^T  (lower)
//                            [record T]  X[k,0:k] = -X[k,k] tmp[k,0:k]               (block row k of the inverse)
//                                      tmp[k+1,0:k+1] = L[k+1,0:k+1] X[0:k+1,0:k+1]  (needs nothing of cluster(k+1))
// The critical stream waits for T(k-1) before its look-ahead of step k (the side's trailing update of k-1 last wrote W[k+1,k] and
// W[k+1,k+1]; one in-order side stream, so one event covers every earlier update), and finally for the side stream's last work.
// So the critical path is P cluster launches, P-1 pairs of 256^3 products and the last block row of the inverse.
// Ownership at step k, which keeps the regions the two streams write disjoint: the critical stream owns the diagonal blocks
// W / Lc / X / Xlo / tmp [k,k] (tmp[k,k] is the cluster kernel's scratch), Lc / Llo [k+1,k] and W [k+1,k+1]; the side stream owns
// Lc / Llo [k+2:,k], W / Wlo [k+2:,k+1:] except the diagonal block [k+1,k+1], X / Xlo [k,0:k], tmp / Tlo [k+1,0:k+1] and the upper
// off-diagonal blocks of Lc and X.  The GEMMs never read above the diagonal of a block (their 256-wide tiles start on block
// boundaries), so those blocks of Llo / Xlo / Tlo are never written.
constexpr int HYB_NB = 256;

// lo plane of a rows x cols block (row stride M) of every factor: blockIdx.z = factor, blockIdx.y = row
__global__ void tf32_lo_block_kernel(const float* __restrict__ x, float* __restrict__ lo, int cols, int M) {
  const int64_t base = (int64_t)blockIdx.z * M * M + (int64_t)blockIdx.y * M;
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < cols; j += gridDim.x * blockDim.x) lo[base + j] = tf32_lo_part(x[base + j]);
}
// zeros in the blocks of Lc and X above the diagonal blocks (the cluster kernel clears the upper part of the diagonal blocks)
__global__ void zero_upper_blocks_kernel(float* __restrict__ Lc, float* __restrict__ X, int M) {
  const int i = blockIdx.x;
  const int64_t row = ((int64_t)blockIdx.y * M + i) * M;
  for (int j = (i / HYB_NB + 1) * HYB_NB + threadIdx.x; j < M; j += blockDim.x) { Lc[row + j] = 0.f; X[row + j] = 0.f; }
}

// the side stream of chol_inv_hybrid and its two events, created once per device and reused by every call
struct HybridStreams {
  cudaStream_t side = nullptr;
  cudaEvent_t crit = nullptr, done = nullptr;      // recorded on the critical / the side stream
};
static int hybrid_streams(HybridStreams** out) {
  constexpr int MAX_DEV = 64;
  static HybridStreams per_dev[MAX_DEV];
  static std::mutex mu;
  int dev = 0;
  GPZ_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= MAX_DEV) return GPZ_ERR_UNSUPPORTED;
  std::lock_guard<std::mutex> lock(mu);
  HybridStreams& h = per_dev[dev];
  if (h.side == nullptr) {
    GPZ_CUDA(cudaStreamCreateWithFlags(&h.side, cudaStreamNonBlocking));
    GPZ_CUDA(cudaEventCreateWithFlags(&h.crit, cudaEventDisableTiming));
    GPZ_CUDA(cudaEventCreateWithFlags(&h.done, cudaEventDisableTiming));
  }
  *out = &h;
  return GPZ_OK;
}

static int chol_inv_hybrid(float* W, float* Lc, float* X, float* tmp, float* lo_ws, int M, int L, int* info, cudaStream_t st) {
  const int64_t sL = (int64_t)M * M, tot = sL * L;
  float* Wlo = lo_ws; float* Llo = lo_ws + tot; float* Xlo = lo_ws + 2 * tot; float* Tlo = lo_ws + 3 * tot;
  HybridStreams* hs = nullptr;
  int rc = hybrid_streams(&hs);
  if (rc) return rc;
  cudaStream_t side = hs->side;
  static int num_sms = 0;
  if (num_sms == 0) {
    int dev = 0;
    GPZ_CUDA(cudaGetDevice(&dev));
    GPZ_CUDA(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev));
  }
  // the side GEMMs are persistent: capped, they leave the SMs for the next cluster launch (L clusters of CL CTAs) free
  const int side_ctas = max(16, num_sms - L * CL);
  const int P = (M + HYB_NB - 1) / HYB_NB;
  auto nb = [&](int k) { return min(HYB_NB, M - k * HYB_NB); };
  auto off = [&](int bi, int bj) { return (int64_t)bi * HYB_NB * M + (int64_t)bj * HYB_NB; };

  GPZ_CUDA(cudaMemsetAsync(info, 0, sizeof(int) * L, st));
  GPZ_CUDA(cudaEventRecord(hs->crit, st));                  // fork: the side stream sees W as the caller left it
  GPZ_CUDA(cudaStreamWaitEvent(side, hs->crit, 0));
  zero_upper_blocks_kernel<<<dim3(M, L), 256, 0, side>>>(Lc, X, M);
  GPZ_CHECK_LAUNCH();
  if (P > 1) {                                              // the first panel product reads W[1:,0] with its lo plane
    tf32_lo_block_kernel<<<dim3(1, M - HYB_NB, L), 256, 0, side>>>(W + off(1, 0), Wlo + off(1, 0), HYB_NB, M);
    GPZ_CHECK_LAUNCH();
  }
  GPZ_CUDA(cudaEventRecord(hs->done, side));

  constexpr int csmem = (int)(2 * NB * TLD * sizeof(float));
  GPZ_CUDA(cudaFuncSetAttribute(chol_inv_cluster_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, csmem));
  for (int k = 0; k < P; ++k) {
    const int n = nb(k);
    // ---- critical stream ----
    chol_inv_cluster_kernel<float><<<L * CL, 256, csmem, st>>>(W, Lc, X, tmp, M, k * HYB_NB, n, info, k == 0 ? g_chol_dbg : nullptr,
                                                                Xlo);
    GPZ_CHECK_LAUNCH();
    if (k + 1 < P) {
      const int n1 = nb(k + 1);
      GPZ_CUDA(cudaStreamWaitEvent(st, hs->done, 0));      // the side's trailing update of k-1 (or its set-up)
      // L[k+1,k] = W[k+1,k] X[k,k]^T      (B = X[k,k] stored n x k: K-major; op(B) = X^T is upper triangular)
      rc = umma_gemm_ex(1, n1, n, n, 1.0f, W + off(k + 1, k), Wlo + off(k + 1, k), M, sL, X + off(k, k), Xlo + off(k, k), M, sL,
                        nullptr, Lc + off(k + 1, k), Llo + off(k + 1, k), M, sL, L, 0, 2, 0, 1, 3, nullptr, (void*)st);
      if (rc) return rc;
      GPZ_CUDA(cudaEventRecord(hs->crit, st));
      // W[k+1,k+1] -= L[k+1,k] L[k+1,k]^T  (lower, in place; its lo plane is never read: the cluster kernel works in fp32)
      rc = umma_gemm_ex(1, n1, n1, n, -1.0f, Lc + off(k + 1, k), Llo + off(k + 1, k), M, sL, Lc + off(k + 1, k), Llo + off(k + 1, k),
                        M, sL, W + off(k + 1, k + 1), W + off(k + 1, k + 1), nullptr, M, sL, L, 0, 0, 1, 1, 3, nullptr, (void*)st);
      if (rc) return rc;
    } else {
      GPZ_CUDA(cudaEventRecord(hs->crit, st));
    }
    // ---- side stream ----
    GPZ_CUDA(cudaStreamWaitEvent(side, hs->crit, 0));
    if (k + 2 < P) {
      const int r2 = (k + 2) * HYB_NB, m2 = M - r2;
      // L[k+2:,k] = W[k+2:,k] X[k,k]^T
      rc = umma_gemm_ex(1, m2, n, n, 1.0f, W + off(k + 2, k), Wlo + off(k + 2, k), M, sL, X + off(k, k), Xlo + off(k, k), M, sL,
                        nullptr, Lc + off(k + 2, k), Llo + off(k + 2, k), M, sL, L, 0, 2, 0, 1, 3, nullptr, (void*)side, side_ctas);
      if (rc) return rc;
      // W[k+2:,k+1] -= L[k+2:,k] L[k+1,k]^T
      rc = umma_gemm_ex(1, m2, HYB_NB, n, -1.0f, Lc + off(k + 2, k), Llo + off(k + 2, k), M, sL, Lc + off(k + 1, k), Llo + off(k + 1, k),
                        M, sL, W + off(k + 2, k + 1), W + off(k + 2, k + 1), Wlo + off(k + 2, k + 1), M, sL, L, 0, 0, 0, 1, 3, nullptr,
                        (void*)side, side_ctas);
      if (rc) return rc;
      // W[k+2:,k+2:] -= L[k+2:,k] L[k+2:,k]^T  (lower)
      rc = umma_gemm_ex(1, m2, m2, n, -1.0f, Lc + off(k + 2, k), Llo + off(k + 2, k), M, sL, Lc + off(k + 2, k), Llo + off(k + 2, k),
                        M, sL, W + off(k + 2, k + 2), W + off(k + 2, k + 2), Wlo + off(k + 2, k + 2), M, sL, L, 0, 0, 1, 1, 3, nullptr,
                        (void*)side, side_ctas);
      if (rc) return rc;
    }
    GPZ_CUDA(cudaEventRecord(hs->done, side));
    if (k > 0) {
      // X[k,0:k] = -X[k,k] tmp[k,0:k]      (X[k,k] lower triangular; the last block row's lo plane is never read)
      rc = umma_gemm_ex(0, n, k * HYB_NB, n, -1.0f, X + off(k, k), Xlo + off(k, k), M, sL, tmp + off(k, 0), Tlo + off(k, 0), M, sL,
                        nullptr, X + off(k, 0), k + 1 < P ? Xlo + off(k, 0) : nullptr, M, sL, L, 1, 0, 0, 1, 3, nullptr, (void*)side,
                        side_ctas);
      if (rc) return rc;
    }
    if (k + 1 < P) {
      // tmp[k+1,0:k+1] = L[k+1,0:k+1] X[0:k+1,0:k+1]      (X lower triangular, stored k x n)
      const int c = (k + 1) * HYB_NB;
      rc = umma_gemm_ex(0, nb(k + 1), c, c, 1.0f, Lc + off(k + 1, 0), Llo + off(k + 1, 0), M, sL, X, Xlo, M, sL, nullptr,
                        tmp + off(k + 1, 0), Tlo + off(k + 1, 0), M, sL, L, 0, 1, 0, 1, 3, nullptr, (void*)side, side_ctas);
      if (rc) return rc;
    }
  }
  GPZ_CUDA(cudaEventRecord(hs->done, side));                // join: everything is final on the caller's stream
  GPZ_CUDA(cudaStreamWaitEvent(st, hs->done, 0));
  return GPZ_OK;
}

// ---- element-wise O(M^2) helpers -------------------------------------------------------------------
// lower-Cholesky transform (torch transforms.py LowerCholeskyTransform._call; gp.py:220):
//   out = tril(raw,-1) + diag(exp(diag raw))
// Row-wise element-wise kernels: blockIdx.x = row i, blockIdx.y = matrix b, threads stride over the columns (no index
// division; consecutive threads touch consecutive addresses).
template <typename T> __global__ void __launch_bounds__(256) lct_fwd_kernel(const T* __restrict__ raw, T* __restrict__ out, int M) {
  const int i = blockIdx.x;
  const int64_t row = ((int64_t)blockIdx.y * M + i) * M;
  for (int j = threadIdx.x; j < M; j += blockDim.x) {
    const T x = j <= i ? raw[row + j] : T(0);
    out[row + j] = j < i ? x : (j == i ? Num<T>::exp(x) : T(0));
  }
}
// graw = tril(g,-1) + diag(g_ii * Lu_ii)
template <typename T>
__global__ void __launch_bounds__(256) lct_bwd_kernel(const T* __restrict__ g, const T* __restrict__ out, T* __restrict__ graw, int M) {
  const int i = blockIdx.x;
  const int64_t row = ((int64_t)blockIdx.y * M + i) * M;
  for (int j = threadIdx.x; j < M; j += blockDim.x) {
    const T x = j <= i ? g[row + j] : T(0);
    graw[row + j] = j < i ? x : (j == i ? x * out[row + j] : T(0));
  }
}
// mode 0: out = tril(in) with halved diagonal (the Phi operator of the Cholesky backward)
// mode 1: out = (in + in^T)/2
// mode 2: out = tril(in)
template <typename T>
__global__ void __launch_bounds__(256) tri_op_kernel(const T* __restrict__ in, T* __restrict__ out, int M, int mode) {
  const int i = blockIdx.x;
  const int64_t mat = (int64_t)blockIdx.y * M * M, row = mat + (int64_t)i * M;
  if (mode == 1) {
    for (int j = threadIdx.x; j < M; j += blockDim.x) out[row + j] = T(0.5) * (in[row + j] + in[mat + (int64_t)j * M + i]);
  } else {
    for (int j = threadIdx.x; j < M; j += blockDim.x) {
      const T x = j <= i ? in[row + j] : T(0);            // the strict upper triangle is never read
      out[row + j] = (mode == 0 && j == i) ? T(0.5) * x : x;
    }
  }
}

// KL(N(mu, Lu Lu^T) || N(0, Lc Lc^T)) per factor from the whitened quantities T = Lc^-1 Lu, q = Lc^-1 mu:
//   kl = sum log diag Lc - sum log diag Lu + 0.5 (|T|_F^2 + |q|^2 - M)         (torch kl.py MVN||MVN)
template <typename T>
__global__ void __launch_bounds__(256) mvn_kl_fwd_kernel(const T* __restrict__ Tm, const T* __restrict__ q, const T* __restrict__ Lc,
                                                          const T* __restrict__ Lu, double* __restrict__ acc_out, int M) {
  __shared__ double red[32];
  const int l = blockIdx.y;
  const int64_t sL = (int64_t)M * M;
  double acc = 0.0;
  // rows are split over blockIdx.x (the full row is read: whitened_KL sums all of Lz like the reference)
  for (int i = blockIdx.x; i < M; i += gridDim.x) {
    const T* row = Tm + l * sL + (int64_t)i * M;
    for (int j = threadIdx.x; j < M; j += blockDim.x) {
      const double t = (double)row[j];
      acc += 0.5 * t * t;
    }
    if (threadIdx.x == 0) {
      const double qq = (double)q[(int64_t)l * M + i];
      acc += 0.5 * qq * qq + ::log((double)Lc[l * sL + (int64_t)i * M + i]) - ::log((double)Lu[l * sL + (int64_t)i * M + i]);
    }
  }
  acc = block_sum<double>(acc, red);
  if (threadIdx.x == 0) atomicAdd(acc_out + l, acc);
}
template <typename T> __global__ void mvn_kl_finish_kernel(const double* __restrict__ acc, T* __restrict__ kl, int M, int L) {
  const int l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l < L) kl[l] = (T)(acc[l] - 0.5 * M);
}
// gT = g*T ; gq = g*q ; gLc = diag(g / Lc_ii) ; gLu = diag(-g / Lu_ii)
template <typename T>
__global__ void mvn_kl_bwd_kernel(const T* __restrict__ g, const T* __restrict__ Tm, const T* __restrict__ q, const T* __restrict__ Lc,
                                  const T* __restrict__ Lu, T* __restrict__ gT, T* __restrict__ gq, T* __restrict__ gLc,
                                  T* __restrict__ gLu, int M, int64_t total) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= total) return;
  const int64_t sL = (int64_t)M * M, l = e / sL, r = e % sL;
  const int i = (int)(r / M), j = (int)(r % M);
  const T gl = g[l];
  gT[e] = gl * Tm[e];
  gLc[e] = i == j ? gl / Lc[e] : T(0);
  gLu[e] = i == j ? -gl / Lu[e] : T(0);
  if (j == 0) gq[l * M + i] = gl * q[l * M + i];
}

}  // namespace gpz

using namespace gpz;
#define ST(s) ((cudaStream_t)(s))

#define GPZ_LINALG_IMPL(SUF, T)                                                                                   \
  extern "C" int gpz_chol_inv_##SUF(T* W, T* Lc, T* X, T* tmp, int M, int L, int* info, void* stream) {          \
    if (M <= 0 || L <= 0) return GPZ_ERR_BADARG;                                                                  \
    return chol_inv<T>(W, Lc, X, tmp, M, L, info, ST(stream));                                                   \
  }                                                                                                               \
  extern "C" int gpz_gemm_##SUF(int ta, int tb, int m, int n, int k, T alpha, const T* A, int64_t lda, int64_t sA, \
                                const T* B, int64_t ldb, int64_t sB, T beta, T* D, int64_t ldd, int64_t sD,      \
                                int batch, int a_tri, int b_tri, int d_tri, int splitk, void* stream) {           \
    return gemm<T>(ST(stream), ta != 0, tb != 0, m, n, k, alpha, A, lda, sA, B, ldb, sB, beta, D, ldd, sD, batch, \
                   a_tri, b_tri, d_tri, splitk);                                                                  \
  }                                                                                                               \
  extern "C" int gpz_lower_cholesky_fwd_##SUF(const T* raw, T* out, int M, int L, void* stream) {                \
    if (M <= 0 || L <= 0) return GPZ_OK;                                                                          \
    lct_fwd_kernel<T><<<dim3(M, L), 256, 0, ST(stream)>>>(raw, out, M);                                          \
    GPZ_CHECK_LAUNCH();                                                                                           \
    return GPZ_OK;                                                                                                \
  }                                                                                                               \
  extern "C" int gpz_lower_cholesky_bwd_##SUF(const T* g, const T* out, T* graw, int M, int L, void* stream) {   \
    if (M <= 0 || L <= 0) return GPZ_OK;                                                                          \
    lct_bwd_kernel<T><<<dim3(M, L), 256, 0, ST(stream)>>>(g, out, graw, M);                                      \
    GPZ_CHECK_LAUNCH();                                                                                           \
    return GPZ_OK;                                                                                                \
  }                                                                                                               \
  extern "C" int gpz_tri_op_##SUF(const T* in, T* out, int M, int L, int mode, void* stream) {                   \
    if (in == out && mode == 1) return GPZ_ERR_BADARG;                                                            \
    if (M <= 0 || L <= 0) return GPZ_OK;                                                                          \
    tri_op_kernel<T><<<dim3(M, L), 256, 0, ST(stream)>>>(in, out, M, mode);                                      \
    GPZ_CHECK_LAUNCH();                                                                                           \
    return GPZ_OK;                                                                                                \
  }                                                                                                               \
  extern "C" int gpz_mvn_kl_fwd_##SUF(const T* Tm, const T* q, const T* Lc, const T* Lu, T* kl, double* ws, int M, \
                                      int L, void* stream) {                                                      \
    GPZ_CUDA(cudaMemsetAsync(ws, 0, sizeof(double) * L, ST(stream)));                                             \
    mvn_kl_fwd_kernel<T><<<dim3((unsigned)min(M, 256), L), 256, 0, ST(stream)>>>(Tm, q, Lc, Lu, ws, M);          \
    GPZ_CHECK_LAUNCH();                                                                                           \
    mvn_kl_finish_kernel<T><<<(unsigned)cdiv(L, 128), 128, 0, ST(stream)>>>(ws, kl, M, L);                       \
    GPZ_CHECK_LAUNCH();                                                                                           \
    return GPZ_OK;                                                                                                \
  }                                                                                                               \
  extern "C" int gpz_mvn_kl_bwd_##SUF(const T* g, const T* Tm, const T* q, const T* Lc, const T* Lu, T* gT,      \
                                      T* gq, T* gLc, T* gLu, int M, int L, void* stream) {                        \
    const int64_t total = (int64_t)M * M * L;                                                                     \
    mvn_kl_bwd_kernel<T><<<(unsigned)cdiv(total, 256), 256, 0, ST(stream)>>>(g, Tm, q, Lc, Lu, gT, gq, gLc, gLu, \
                                                                             M, total);                           \
    GPZ_CHECK_LAUNCH();                                                                                           \
    return GPZ_OK;                                                                                                \
  }

GPZ_LINALG_IMPL(f32, float)
GPZ_LINALG_IMPL(f64, double)

// fp32 Cholesky + inverse for large M with the O(M^3) products on the tensor cores (see chol_inv_hybrid); lo_ws: 4 L M M floats.
// Same outputs and info convention as gpz_chol_inv_f32.  M % 4 == 0.
extern "C" int gpz_chol_inv_tc_f32(float* W, float* Lc, float* X, float* tmp, float* lo_ws, int M, int L, int* info, void* stream) {
  if (M <= 0 || L <= 0) return GPZ_ERR_BADARG;
  if (M % 4) return GPZ_ERR_UNSUPPORTED;
  return chol_inv_hybrid(W, Lc, X, tmp, lo_ws, M, L, info, ST(stream));
}
