// K7: fused Poisson log-likelihood with the factor-loading contraction, forward + backward in one pass.
//
// Reference chain (likelihoods.py:49-53, 80-97, 110-145; utilities.py:611-614; torch poisson.py log_prob):
//   F = mean + eps*sd            (Normal.rsample, E samples)          E x F x B
//   rate = softplus(V) * (softplus(W) @ exp(F))                       E x G x B   (materialised by the reference)
//   ll = mean_e sum_{g,n} [ y log rate - rate (- lgamma(y+1)) ]
// and autograd's backward through all of it.  Here nothing of size G x B is ever written: one pass over
// y (G x B floats, the algorithmic HBM traffic) produces ll and the gradients w.r.t. mean, spread, W, V.
//
// Dense counts: fp32 with F <= 16 runs the contractions on the tensor cores (poisson_prep4 / kernel4 / post4); fp64 and
// F > 16 run poisson_kernel2 on the CUDA cores.  Sparse counts run the K7-CSC kernels at the end of the file.
#include <type_traits>

#include "common.cuh"
#include "gpzoo_b200.h"

namespace gpz {

constexpr int PZ_GCH = 32;

template <typename T> struct PoissonArgs {
  const T* y; int64_t y_ld;           // G x Ntot, row stride
  const int64_t* idx;                  // B or null (minibatch gather y[:, idx], V[idx])
  const T* W; int w_softplus;          // G x F raw loadings; softplus (NSF2/PNMF) or raw (Hybrid_NSF)
  const T* V;                          // Ntot raw
  const T* mean; const T* spread;      // F x B ; spread = variance for f < n_var (clamped at clamp_min), sd otherwise
  const T* eps;                        // E x F x B
  int G, F, B, E, n_var;
  T clamp_min;
  int with_lgamma;
  // outputs
  double* ll_part;                     // gridDim.x * gridDim.y
  T* gW_part;                          // gridDim.x x G x F
  T* gV;                               // B   (d ll / d V[idx[n]])
  T* gmean; T* gspread;                // F x B
  int genes_per_cta;                   // multiple of PZ_GCH
  int atomic_out;                      // gridDim.y > 1
};

// K7-NB: the same call with the negative-binomial likelihood, theta_g = softplus(D_g) per gene (see the NB section below)
template <typename T> struct NegBinArgs : PoissonArgs<T> {
  const T* D;                          // G raw dispersion
  const T* nbg;                        // [G][2] theta, 1 / theta                                          (negbin_tables_kernel)
  const T* tab;                        // [G][64][2] Lambda_g[k] - k log theta (- log k! with_lgamma), Psi_g[k] (negbin_tables_kernel)
  T* gD_part;                          // gridDim.x x G: sum over the CTA's spots and the samples of d log NB / d theta
  T* gD;                               // G output: d ll / d D
};
template <typename T, bool NB> using K7Args = typename std::conditional<NB, NegBinArgs<T>, PoissonArgs<T>>::type;

// ---- negative-binomial helpers ----------------------------------------------------------------------------------------------
// log1p(q) for q >= 0.  fp32: the series to q^5 below 1/32 (truncation < 5e-9 relative; 1 + q would lose q's low bits),
// __log2f(1 + q) above; fp64: the exact function.
__device__ __forceinline__ float nb_log1p(float q) {
  const float s = q * fmaf(q, fmaf(q, fmaf(q, fmaf(q, 0.2f, -0.25f), 0.333333343f), -0.5f), 1.f);
  return q < 0.03125f ? s : __log2f(1.f + q) * 0.69314718055994530942f;
}
__device__ __forceinline__ double nb_log1p(double q) { return ::log1p(q); }

// digamma for x > 0 (CUDA's math library has none): the recurrence psi(x) = psi(x + 1) - 1 / x up to x >= 10, then the asymptotic
// series log x - 1 / (2x) - sum_k B_2k / (2k x^2k) through x^-16 (the next term is below 1e-17 at x = 10).  The recurrence's sum
// is subtracted last: near the root at 1.4616 that order keeps the cancellation to a few ulp of the two sides.
__device__ __forceinline__ double nb_digamma(double x) {
  double acc = 0.0;
  while (x < 10.0) { acc += 1.0 / x; x += 1.0; }
  const double r = 1.0 / x, r2 = r * r;
  const double ser = r2 * (1.0 / 12 - r2 * (1.0 / 120 - r2 * (1.0 / 252 - r2 * (1.0 / 240 - r2 * (1.0 / 132 - r2 * (691.0 / 32760 -
                     r2 * (1.0 / 12 - r2 * (3617.0 / 8160))))))));
  return (::log(x) - 0.5 * r - ser) - acc;
}
// lgamma for x > 0, written like nb_digamma (the library's lgamma is large code: called from the NB kernels' rare path it made them
// spill): the product x (x + 1) ... up to x + n >= 10, then Stirling's series through x^-15 (next term below 1e-17 at x = 10)
__device__ __forceinline__ double nb_lgamma(double x) {
  double prod = 1.0;
  while (x < 10.0) { prod *= x; x += 1.0; }
  const double r = 1.0 / x, r2 = r * r;
  const double ser = r * (1.0 / 12 - r2 * (1.0 / 360 - r2 * (1.0 / 1260 - r2 * (1.0 / 1680 - r2 * (1.0 / 1188 - r2 * (691.0 / 360360 -
                     r2 * (1.0 / 156 - r2 * (3617.0 / 122400))))))));
  return ((x - 0.5) * ::log(x) - x + 0.91893853320467274178 + ser) - ::log(prod);
}

// The table entries for counts >= 64 and non-integer y, in double: lgamma(y + theta) - lgamma(theta) - y log theta
// (- lgamma(y + 1) with_lgamma) and psi(y + theta) - psi(theta).  Rare: the kernels zero these elements' table terms and add this
// afterwards, in a pass of their own, so the call sits where few registers are live.
__device__ __noinline__ double2 nb_slow(double y, double th, int with_lgamma) {
  double l = nb_lgamma(y + th) - nb_lgamma(th) - y * ::log(th);
  if (with_lgamma) l -= nb_lgamma(y + 1.0);
  return make_double2(l, nb_digamma(y + th) - nb_digamma(th));
}

// ---- poisson_kernel2 (fp64, fp32 with F > 16): two spots per thread (256 spots per CTA), sample loop outermost ----------------
// A CTA walks its gene range in chunks of 32.  Phase A (thread = two spots, so y rows are read coalesced): rate, log-lik,
// t = d ll / d zr, d/dF accumulated in registers, t parked in shared memory.  Phase B (lane = gene, warp = a quarter of the spots):
// the gW[g, f] partial sum_n t[g, n] exp(F)[f, n] from shared memory.  Per-CTA gW partials go to a workspace slice and are summed
// by poisson_gw_reduce_kernel (deterministic, no atomics on the G x F output).  The kernel is FMA-issue bound, not HBM bound:
// each softplus(W) row fetched from shared memory serves two spots; per-thread state is only exp(F) and the d/dF
// accumulator of the current sample (the E samples are an outer loop; y is re-read per sample, from L2 when it fits).
constexpr int P2_THREADS = 128, P2_SPOTS = 256;
constexpr int PZ_GRP = 4;        // genes per prefetch group

// NB = true is K7-NB: only the element-wise step, the staging of the per-gene dispersion terms and the d/dD partials differ.
template <typename T, int FMAX, bool NB>
// NB, fp32: two CTAs per SM instead of four, so that the heavier element step and the out-of-line call fit in registers.
__global__ void __launch_bounds__(P2_THREADS, sizeof(T) == 4 ? (NB ? 2 : 4) : 1) poisson_kernel2(const K7Args<T, NB> a) {
  extern __shared__ __align__(16) unsigned char pz_smem[];
  typedef T RowT[P2_SPOTS + 1];
  typedef T RowF[FMAX];
  typedef T AccW[PZ_GCH][FMAX];
  RowT* tS = reinterpret_cast<RowT*>(pz_smem);                         // [PZ_GCH][P2_SPOTS+1]   t = d ll / d zr
  RowF* efS = reinterpret_cast<RowF*>(reinterpret_cast<unsigned char*>(pz_smem) +
                                      ((sizeof(T) * PZ_GCH * (P2_SPOTS + 1) + 15) / 16) * 16);   // [P2_SPOTS][FMAX]
  RowF* sW = efS + P2_SPOTS;                                           // [PZ_GCH][FMAX]
  AccW* sAcc = reinterpret_cast<AccW*>(sW + PZ_GCH);                   // [4][PZ_GCH][FMAX]
  __shared__ double red[32];
  __shared__ T lfact[64];                     // log(y!) for integer counts y < 64 (lgamma(y+1) of torch poisson.py log_prob)
  __shared__ __align__(16) T nbS[NB ? PZ_GCH : 1][2];           // NB: theta, 1 / theta of the chunk's genes
  __shared__ T dS[NB ? P2_THREADS / 32 : 1][PZ_GCH];            // NB: per-warp d ll / d theta of the chunk's genes

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid < 64) lfact[tid] = Num<T>::lgamma(T(tid + 1));
  const int n0 = blockIdx.x * P2_SPOTS;
  int nn[2]; bool act[2]; int64_t col[2]; T spV[2], vraw[2], gVacc[2];
#pragma unroll
  for (int s2 = 0; s2 < 2; ++s2) {
    nn[s2] = n0 + s2 * P2_THREADS + tid;
    act[s2] = nn[s2] < a.B;
    col[s2] = act[s2] ? (a.idx ? a.idx[nn[s2]] : (int64_t)nn[s2]) : 0;
    vraw[s2] = act[s2] ? a.V[col[s2]] : T(0);
    spV[s2] = act[s2] ? softplus(vraw[s2]) : T(0);
    gVacc[s2] = T(0);
  }
  const bool block_full = n0 + P2_SPOTS <= a.B;
  const T invE = T(1) / T(a.E);
  const int g_begin = blockIdx.y * a.genes_per_cta;
  const int g_end = min(a.G, g_begin + a.genes_per_cta);
  double ll = 0.0;

  T ynext[PZ_GRP][2];
  auto prefetch = [&](int gfirst) {
#pragma unroll
    for (int u = 0; u < PZ_GRP; ++u)
#pragma unroll
      for (int s2 = 0; s2 < 2; ++s2)
        ynext[u][s2] = (act[s2] && gfirst + u < g_end) ? __ldcs(a.y + (int64_t)(gfirst + u) * a.y_ld + col[s2]) : T(0);
  };
  prefetch(g_begin);

  for (int e = 0; e < a.E; ++e) {
    T ef[2][FMAX], pg[2][FMAX];
#pragma unroll
    for (int s2 = 0; s2 < 2; ++s2)
#pragma unroll
      for (int f = 0; f < FMAX; ++f) {
        pg[s2][f] = T(0);
        T v = T(0);
        if (f < a.F && act[s2]) {
          const int64_t o = (int64_t)f * a.B + nn[s2];
          const T sp = a.spread[o];
          const T sd = f < a.n_var ? Num<T>::sqrt(sp > a.clamp_min ? sp : a.clamp_min) : sp;
          v = Num<T>::exp(fma(a.eps[((int64_t)e * a.F + f) * a.B + nn[s2]], sd, a.mean[o]));
        }
        ef[s2][f] = v;
      }
    __syncthreads();                               // phase B of the previous sample finished with efS
#pragma unroll
    for (int s2 = 0; s2 < 2; ++s2)
#pragma unroll
      for (int f = 0; f < FMAX; ++f) efS[s2 * P2_THREADS + tid][f] = ef[s2][f];

    for (int g0 = g_begin; g0 < g_end; g0 += PZ_GCH) {
      __syncthreads();                             // previous chunk's phase B / flush finished with sW, tS, sAcc
      for (int i = tid; i < PZ_GCH * FMAX; i += P2_THREADS) {
        const int gi = i / FMAX, f = i % FMAX;
        T w = T(0);
        if (g0 + gi < g_end && f < a.F) {
          w = a.W[(int64_t)(g0 + gi) * a.F + f];
          if (a.w_softplus) w = softplus(w);
        }
        sW[gi][f] = w;
      }
      if constexpr (NB) {
        if (tid < PZ_GCH) {
#pragma unroll
          for (int j = 0; j < 2; ++j) nbS[tid][j] = g0 + tid < g_end ? a.nbg[(int64_t)(g0 + tid) * 2 + j] : T(1);
        }
      }
      __syncthreads();
      // ---- phase A: thread = two spots ----
      T llc = T(0);
#pragma unroll 1
      for (int gb = 0; gb < PZ_GCH; gb += PZ_GRP) {
        T yv[PZ_GRP][2];
#pragma unroll
        for (int u = 0; u < PZ_GRP; ++u) { yv[u][0] = ynext[u][0]; yv[u][1] = ynext[u][1]; }
        {
          int gn = g0 + gb + PZ_GRP;               // first gene of the next group in (sample, chunk, group) order
          if (gb + PZ_GRP == PZ_GCH && g0 + PZ_GCH >= g_end) gn = (e + 1 < a.E) ? g_begin : g_end;
          prefetch(gn);
        }
        T dth[PZ_GRP];                             // NB: d ll / d theta of the group's genes, summed over the thread's two spots
        unsigned slow = 0u;                        // NB: elements (bit 2u + s2) whose table terms nb_slow supplies
        auto body = [&](auto guard, int u) {
          constexpr bool GUARD = decltype(guard)::value;
          const int gi = gb + u;
          T wrow[FMAX];
          load_row<FMAX>(&sW[gi][0], wrow);
          if constexpr (NB) dth[u] = T(0);
#pragma unroll
          for (int s2 = 0; s2 < 2; ++s2) {
            T t = T(0);
            if (!GUARD || (act[s2] && g0 + gi < g_end)) {
              const T y = yv[u][s2];
              T z0 = T(0), z1 = T(0);
#pragma unroll
              for (int f = 0; f < FMAX; f += 2) { z0 = fma(wrow[f], ef[s2][f], z0); z1 = fma(wrow[f + 1], ef[s2][f + 1], z1); }
              const T zr = z0 + z1;
              const T r = spV[s2] * zr;
              if constexpr (NB) {
                const T th = nbS[gi][0], q = r * nbS[gi][1];
                const T l1p = nb_log1p(q);
                const T ud = fast_div(y - r, fma(r, q, r));                 // (y - r) / (r (1 + r / theta)) = d log NB / d r
                const int yi = (int)y;
                T lam = T(0), psi = T(0);                                   // table entries; anything else: the slow pass below
                if (yi >= 0 && yi < 64 && T(yi) == y) {
                  const T* tv = a.tab + ((int64_t)(g0 + gi) * 64 + yi) * 2;
                  lam = tv[0]; psi = tv[1];
                } else {
                  slow |= 1u << (2 * u + s2);
                }
                llc += (y == T(0) ? T(0) : y * fast_log(r)) - (y + th) * l1p + lam;
                t = ud * spV[s2] * invE;
                gVacc[s2] += ud * r;
                dth[u] += psi - l1p - ud * q;
              } else {
                const T ylog = y * fast_log(r);
                T lp = (y == T(0) ? T(0) : ylog) - r;
                if (a.with_lgamma) {
                  const int yi = (int)y;
                  // counts: table lookup (no divergent lgamma call); anything else: the real thing
                  lp -= (yi >= 0 && yi < 64 && T(yi) == y) ? lfact[yi] : Num<T>::lgamma(y + T(1));
                }
                llc += lp;
                t = (fast_div(y, zr) - spV[s2]) * invE;
                gVacc[s2] += y - r;
              }
#pragma unroll
              for (int f = 0; f < FMAX; ++f) pg[s2][f] = fma(wrow[f], t, pg[s2][f]);
            }
            tS[gi][s2 * P2_THREADS + tid] = t;
          }
        };
        if (block_full && g0 + PZ_GCH <= g_end) {
#pragma unroll
          for (int u = 0; u < PZ_GRP; ++u) body(std::false_type{}, u);
        } else {
          if constexpr (NB) {                      // unrolled: dth stays in registers
#pragma unroll
            for (int u = 0; u < PZ_GRP; ++u) body(std::true_type{}, u);
          } else {
#pragma unroll 1
            for (int u = 0; u < PZ_GRP; ++u) body(std::true_type{}, u);
          }
        }
        if constexpr (NB) {
#pragma unroll 1
          while (slow) {                           // one call site, not unrolled: it keeps the call's register cost off the hot path
            const int b = __ffs(slow) - 1, u = b >> 1;
            slow &= slow - 1u;
            T y = T(0);
#pragma unroll
            for (int k = 0; k < 2 * PZ_GRP; ++k) y = k == b ? yv[k >> 1][k & 1] : y;
            const double2 sl = nb_slow((double)y, (double)nbS[gb + u][0], a.with_lgamma);
            llc += (T)sl.x;
#pragma unroll
            for (int k = 0; k < PZ_GRP; ++k) dth[k] += k == u ? (T)sl.y : T(0);
          }
          // sum the four genes' values over the warp's 32 lanes in 6 shuffles (halve, halve, then a plain tree): lane bits 4 and 3
          // end up naming the gene; lanes 0, 8, 16, 24 hold the totals
          const bool hi16 = lane & 16, hi8 = lane & 8;
          T k0 = hi16 ? dth[2] : dth[0], k1 = hi16 ? dth[3] : dth[1];
          k0 += __shfl_xor_sync(0xffffffffu, hi16 ? dth[0] : dth[2], 16);
          k1 += __shfl_xor_sync(0xffffffffu, hi16 ? dth[1] : dth[3], 16);
          T k = hi8 ? k1 : k0;
          k += __shfl_xor_sync(0xffffffffu, hi8 ? k0 : k1, 8);
          k += __shfl_xor_sync(0xffffffffu, k, 4);
          k += __shfl_xor_sync(0xffffffffu, k, 2);
          k += __shfl_xor_sync(0xffffffffu, k, 1);
          if ((lane & 7) == 0) dS[warp][gb + (lane >> 3)] = k;
        }
      }
      ll += (double)(llc * invE);
      __syncthreads();
      // ---- phase B: lane = gene, warp = a quarter (64) of the spots ----
      T acc[FMAX];
#pragma unroll
      for (int f = 0; f < FMAX; ++f) acc[f] = T(0);
      const int nb = warp * 64;
#pragma unroll 4
      for (int k = 0; k < 64; ++k) {
        const T t = tS[lane][nb + k];
        T erow[FMAX];
        load_row<FMAX>(&efS[nb + k][0], erow);
#pragma unroll
        for (int f = 0; f < FMAX; ++f) acc[f] = fma(t, erow[f], acc[f]);
      }
#pragma unroll
      for (int f = 0; f < FMAX; ++f) sAcc[warp][lane][f] = acc[f];
      __syncthreads();
      for (int i = tid; i < PZ_GCH * a.F; i += P2_THREADS) {
        const int gi = i / a.F, f = i % a.F;
        if (g0 + gi < g_end) {
          T* dst = a.gW_part + ((int64_t)blockIdx.x * a.G + g0 + gi) * a.F + f;
          const T v = sAcc[0][gi][f] + sAcc[1][gi][f] + sAcc[2][gi][f] + sAcc[3][gi][f];
          *dst = e == 0 ? v : *dst + v;
        }
      }
      if constexpr (NB) {
        if (tid < PZ_GCH && g0 + tid < g_end) {
          T* dst = a.gD_part + (int64_t)blockIdx.x * a.G + g0 + tid;
          const T v = (dS[0][tid] + dS[1][tid]) + (dS[2][tid] + dS[3][tid]);
          *dst = e == 0 ? v : *dst + v;
        }
      }
    }
    // ---- per-sample epilogue: d ll / d mean, d ll / d spread ----
#pragma unroll
    for (int s2 = 0; s2 < 2; ++s2) {
      if (!act[s2]) continue;
#pragma unroll
      for (int f = 0; f < FMAX; ++f) {
        if (f < a.F) {
          const int64_t o = (int64_t)f * a.B + nn[s2];
          const T gF = ef[s2][f] * pg[s2][f];
          T gsp = gF * a.eps[((int64_t)e * a.F + f) * a.B + nn[s2]];
          if (f < a.n_var) {                       // spread is a variance: d sd / d var = 1 / (2 sd) where not clamped
            const T sp = a.spread[o];
            gsp = sp >= a.clamp_min ? gsp / (T(2) * Num<T>::sqrt(sp)) : T(0);
          }
          if (a.atomic_out) { atomicAdd(a.gmean + o, gF); atomicAdd(a.gspread + o, gsp); }
          else if (e == 0) { a.gmean[o] = gF; a.gspread[o] = gsp; }
          else { a.gmean[o] += gF; a.gspread[o] += gsp; }
        }
      }
    }
  }
#pragma unroll
  for (int s2 = 0; s2 < 2; ++s2) {
    if (act[s2]) {
      const T gv = softplus_grad(vraw[s2]) * gVacc[s2] * invE / spV[s2];
      if (a.atomic_out) atomicAdd(a.gV + nn[s2], gv); else a.gV[nn[s2]] = gv;
    }
  }
  const double tot = block_sum<double>(ll, red);
  if (tid == 0) a.ll_part[blockIdx.y * gridDim.x + blockIdx.x] = tot;
}


// ---- v4 (fp32, F <= 16): the three F-long contractions on the tensor cores ------------------------------------------------
// poisson_kernel2 is bound by instruction issue (3.3 warp instructions per (gene, spot) element, 36 of the 105 thread instructions
// being the FMAs of the contractions); HBM sits at 12 %.  Here the contractions are warp-level MMAs (mma.sync m16n8k16, bf16 operands,
// fp32 accumulation) chained in registers the way a fused attention kernel chains QK^T -> P -> PV:
//   C1[n, g] = EF'^T[n, :] Wm[g, :]^T                      rate tile (16 spots x 8 genes), EF' = softplus(V) exp(F)
//   t'       = (y / C1 - 1) / E,  ll += y log2 C1          element-wise on the accumulator fragment, y read straight into that layout
//   D2[n, l] += t'^T[n, g] Wm[g, l]                        the packed C1 fragments of two gene tiles ARE the A fragment (d ll / d EF')
//   D3[l, g] += EF'[l, n] t'^T[n, g]                       B fragment = movmatrix-transposed packed t' (d ll / d Wm, over the spots)
// Every operand is split x = hi + lo into two bf16 (|x - hi - lo| <= 2^-18 |x|) and a product is hi*hi + hi*lo + lo*hi, so a
// contraction carries ~1e-5 relative error at worst (1e-6 measured on the gradients) - bf16 rather than fp16 because exp(F) and y / r
// have fp32 range.  Three launches:
//   prep  per gene: softplus(W) as bf16 hi / lo planes [G][16] + fp32 column sums per gene range; per spot and sample: EF' as bf16
//         planes [E][B][16]; zeroes the D2 accumulator.  Everything that is per gene or per spot is done ONCE here, not once per CTA.
//   main  grid (256-spot blocks) x (gene ranges).  A warp owns 32 spots (two 16-spot sub-tiles, D2 resident in registers over the
//         CTA's gene range) and walks the range in 16-gene blocks; D3 is summed over the sub-tiles in registers, over the warps through
//         shared memory once per 64-gene chunk, and leaves as per-CTA partials (same workspace layout as kernel2).  D2 leaves by vector
//         atomics into [E][B][16].  ~0.6 warp instructions per element instead of 3.3.
//   post  gW = softplus'(W) * sum of the partials; per spot: gF = EF' D2 -> d/dmean, d/dspread, d/dV, and the terms that never needed
//         the G x B elements: sum_g r = sum_l EF'_l (sum_g Wm_gl), d ll / d V = softplus'(V) / softplus(V) sum_l EF'_l D2_l; the last
//         block to finish adds up the log-likelihood partials.
constexpr int P4_WARPS = 8, P4_THREADS = 32 * P4_WARPS, P4_SUB = 2, P4_SPOTS = P4_WARPS * P4_SUB * 16;
constexpr int P4_GCH = 64;            // genes per staged chunk of loadings (four 16-gene blocks)
constexpr int P4_WLD = 24;            // bf16 per shared-memory row of loadings: 48-byte rows keep ldmatrix conflict-free
constexpr int P4_ALD = 72;            // floats per row of the D3 exchange buffer: float2 stores of a half-warp hit 32 distinct banks

__device__ __forceinline__ uint32_t pack_bf16x2(float e0, float e1) {      // e0 -> bits 0..15, e1 -> bits 16..31
  uint32_t d;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(e1), "f"(e0));
  return d;
}
__device__ __forceinline__ void split_bf16x2(float x0, float x1, uint32_t& hi, uint32_t& lo) {
  hi = pack_bf16x2(x0, x1);
  lo = pack_bf16x2(x0 - __uint_as_float(hi << 16), x1 - __uint_as_float(hi & 0xffff0000u));
}
__device__ __forceinline__ void mma_bf16(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t movmatrix_t(uint32_t a) {              // 8x8 b16 transpose across the warp
  uint32_t d;
  asm volatile("movmatrix.sync.aligned.m8n8.trans.b16 %0, %1;" : "=r"(d) : "r"(a));
  return d;
}
__device__ __forceinline__ void ldmatrix_x4(uint32_t (&d)[4], const void* p) {
  const uint32_t addr = (uint32_t)__cvta_generic_to_shared(p);
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(d[0]), "=r"(d[1]), "=r"(d[2]), "=r"(d[3]) : "r"(addr));
}
__device__ __forceinline__ void ldmatrix_x4_t(uint32_t (&d)[4], const void* p) {
  const uint32_t addr = (uint32_t)__cvta_generic_to_shared(p);
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(d[0]), "=r"(d[1]), "=r"(d[2]), "=r"(d[3]) : "r"(addr));
}

// workspace of the v4 path behind the ll / gW partials
struct Poisson4Ws {
  uint16_t* wh; uint16_t* wl;          // [G][16]   softplus(W), bf16 hi / lo (factors >= F are zero)
  float* wsum;                         // [nby][16] column sums of softplus(W) over the gene range of grid row y
  uint16_t* efh; uint16_t* efl;        // [E][B][16] EF' = softplus(V) exp(mean + eps sd), bf16 hi / lo
  float* d2;                           // [E][B][16] sum_g t'[g, n] Wm[g, l]
  double* rs_part;                     // [post spot blocks] sum over the block's spots of sum_l EF'_l Wsum_l
  unsigned int* ticket;                // last-block-done counter of the post kernel
};

// EF'[l, n] of sample e for the four factors lq .. lq + 3 of spot n (exact fp32; used by prep and by post).  All twelve loads are issued
// before anything is computed (factor indices clamped instead of predicated): one memory latency, not twelve.
__device__ __forceinline__ void poisson_ef4(const PoissonArgs<float>& a, int e, int n, int lq, float spV, float (&ev)[4], float (&epsv)[4],
                                            float (&sdv)[4]) {
  float sp[4], mn[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int f = min(lq + j, a.F - 1);
    const int64_t o = (int64_t)f * a.B + n;
    sp[j] = a.spread[o];
    mn[j] = a.mean[o];
    epsv[j] = a.eps[((int64_t)e * a.F + f) * a.B + n];
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int f = lq + j;
    sdv[j] = f < a.n_var ? sqrtf(sp[j] > a.clamp_min ? sp[j] : a.clamp_min) : sp[j];
    ev[j] = f < a.F ? spV * expf(fmaf(epsv[j], sdv[j], mn[j])) : 0.f;
  }
}

// blocks [0, nby): loadings of one gene range; blocks [nby, ...): 64 spots of one sample each (thread <-> spot tid / 4, factors 4 (tid & 3)..+3)
__global__ void __launch_bounds__(256) poisson_prep4_kernel(const PoissonArgs<float> a, const Poisson4Ws w, int nby, int spot_blocks) {
  __shared__ float part[8][16];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int lq = (tid & 3) * 4;
  if ((int)blockIdx.x < nby) {
    if (blockIdx.x == 0 && tid == 0) *w.ticket = 0u;
    const int g_begin = blockIdx.x * a.genes_per_cta, g_end = min(a.G, g_begin + a.genes_per_cta);
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    for (int g = g_begin + (tid >> 2); g < g_end; g += 64) {
      float wv[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        wv[j] = 0.f;
        if (lq + j < a.F) {
          wv[j] = a.W[(int64_t)g * a.F + lq + j];
          if (a.w_softplus) wv[j] = softplus(wv[j]);
        }
        acc[j] += wv[j];
      }
      uint32_t h0, l0, h1, l1;
      split_bf16x2(wv[0], wv[1], h0, l0);
      split_bf16x2(wv[2], wv[3], h1, l1);
      *reinterpret_cast<uint2*>(w.wh + (int64_t)g * 16 + lq) = make_uint2(h0, h1);
      *reinterpret_cast<uint2*>(w.wl + (int64_t)g * 16 + lq) = make_uint2(l0, l1);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float v = acc[j];
      v += __shfl_xor_sync(0xffffffffu, v, 4);
      v += __shfl_xor_sync(0xffffffffu, v, 8);
      v += __shfl_xor_sync(0xffffffffu, v, 16);
      if (lane < 4) part[warp][lq + j] = v;
    }
    __syncthreads();
    if (tid < 16) {
      float v = 0.f;
#pragma unroll
      for (int w8 = 0; w8 < 8; ++w8) v += part[w8][tid];
      w.wsum[blockIdx.x * 16 + tid] = v;
    }
    return;
  }
  const int sb = blockIdx.x - nby, e = sb / spot_blocks, n = (sb - e * spot_blocks) * 64 + (tid >> 2);
  if (n >= a.B) return;
  const float spV = softplus(a.V[a.idx ? a.idx[n] : (int64_t)n]);
  float ev[4], epsv[4], sdv[4];
  poisson_ef4(a, e, n, lq, spV, ev, epsv, sdv);
  uint32_t h0, l0, h1, l1;
  split_bf16x2(ev[0], ev[1], h0, l0);
  split_bf16x2(ev[2], ev[3], h1, l1);
  const int64_t o = ((int64_t)e * a.B + n) * 16 + lq;
  *reinterpret_cast<uint2*>(w.efh + o) = make_uint2(h0, h1);
  *reinterpret_cast<uint2*>(w.efl + o) = make_uint2(l0, l1);
  *reinterpret_cast<float4*>(w.d2 + o) = make_float4(0.f, 0.f, 0.f, 0.f);
}

// Counts as stored by the caller: fp32 (the reference's format), or uint8 / int16 / int32 (lossless for counts, 4x / 2x less HBM
// traffic and upload).  y_load2 fetches the two neighbouring spots of a fragment row pair with one load.
// Small unsigned integers become floats on the ALU / FMA pipes (2^23 + k has k in its low mantissa bits), not through I2F, which
// shares the quarter-rate XU pipe with the kernel's log2 / reciprocal.
__device__ __forceinline__ float u16_to_float(unsigned k) { return __uint_as_float(0x4B000000u | k) - 8388608.f; }
template <typename YT> __device__ __forceinline__ float y_load1(const YT* p) { return (float)__ldcs(p); }
template <> __device__ __forceinline__ float y_load1<uint8_t>(const uint8_t* p) { return u16_to_float(__ldcs(p)); }
template <> __device__ __forceinline__ float y_load1<int16_t>(const int16_t* p) {
  return u16_to_float(__ldcs(reinterpret_cast<const unsigned short*>(p)));              // counts: non-negative by contract
}
template <typename YT> __device__ __forceinline__ void y_load2(const YT* p, float& a, float& b);
template <> __device__ __forceinline__ void y_load2<float>(const float* p, float& a, float& b) {
  const float2 v = __ldcs(reinterpret_cast<const float2*>(p)); a = v.x; b = v.y;
}
template <> __device__ __forceinline__ void y_load2<uint8_t>(const uint8_t* p, float& a, float& b) {
  const unsigned v = __ldcs(reinterpret_cast<const unsigned short*>(p)); a = u16_to_float(v & 0xffu); b = u16_to_float(v >> 8);
}
template <> __device__ __forceinline__ void y_load2<int16_t>(const int16_t* p, float& a, float& b) {
  const unsigned v = __ldcs(reinterpret_cast<const unsigned*>(p)); a = u16_to_float(v & 0xffffu); b = u16_to_float(v >> 16);
}
template <> __device__ __forceinline__ void y_load2<int32_t>(const int32_t* p, float& a, float& b) {
  const int2 v = __ldcs(reinterpret_cast<const int2*>(p)); a = (float)v.x; b = (float)v.y;
}

__device__ __noinline__ float lfact_slow(float y) { return lgammaf(y + 1.f); }     // counts >= 64 or non-integer y: rare, kept out of line

// NB = true is K7-NB (the NB element step, the per-gene dispersion terms and the d/dD partials).
template <bool HAS_IDX, typename YT, bool NB>
// NB: one CTA per SM.  With two, the NB step needs more than the 128 registers a thread then gets and spills to local memory.
__global__ void __launch_bounds__(P4_THREADS, NB ? 1 : 2) poisson_kernel4(const K7Args<float, NB> a, const Poisson4Ws w) {
  __shared__ __align__(16) uint16_t sWh[P4_GCH][P4_WLD];      // softplus(W) chunk, bf16 hi / lo, [gene][factor]
  __shared__ __align__(16) uint16_t sWl[P4_GCH][P4_WLD];
  __shared__ __align__(16) float sAcc[P4_WARPS][16][P4_ALD];  // per-warp D3[l][gene of the chunk]
  __shared__ double red[32];
  __shared__ float lfact[64];                                 // log(y!) for integer counts y < 64
  __shared__ float2 nbS[NB ? P4_GCH : 1];                     // NB: theta, 1 / theta of the chunk's genes
  __shared__ float dS[NB ? P4_WARPS : 1][P4_GCH];             // NB: per-warp d ll / d theta of the chunk's genes

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int r = lane >> 2, c = lane & 3;                      // fragment coordinates (groupID, threadID_in_group)
  if (a.with_lgamma && tid < 64) lfact[tid] = lgammaf((float)(tid + 1));
  const int nw = blockIdx.x * P4_SPOTS + warp * (16 * P4_SUB);          // first spot of the warp
  const bool block_full = (blockIdx.x + 1) * P4_SPOTS <= a.B;
  // fragment row r (+8) of sub-tile s <-> spot nw + 16 s + 2 r (+1): a thread's two spots of a sub-tile are neighbours, so one 8-byte load
  // per gene row fetches both (the row <-> spot assignment inside a 16-spot tile is free as long as EF' and D2 use the same one)
  const bool fast_cols = !HAS_IDX && block_full && (a.y_ld & 1) == 0 && (reinterpret_cast<uintptr_t>(a.y) & (2 * sizeof(YT) - 1)) == 0;
  const float invE = 1.f / (float)a.E;
  const int g_begin = blockIdx.y * a.genes_per_cta;
  const int g_end = min(a.G, g_begin + a.genes_per_cta);
  constexpr float LN2 = 0.69314718055994530942f;

  // the thread's spots: sub-tile s, half h -> n = nw + 16 s + 2 r + h ; invalid spots read a valid column of y and have EF' = 0
  int col[P4_SUB][2];                                         // columns of y: 32-bit (Ntot < 2^31)
  if (!fast_cols) {
#pragma unroll
    for (int s = 0; s < P4_SUB; ++s)
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int nc = min(nw + 16 * s + 2 * r + h, a.B - 1);
        col[s][h] = HAS_IDX ? (int)a.idx[nc] : nc;
      }
  }

  // y in accumulator-fragment layout: register q = 4 tt + i of sub-tile s <-> gene gblk + 8 tt + 2c + (i & 1), spot half i >> 1.
  // Rows past the gene range re-read the range's last row (masked when consumed: only the last block of a range is ragged), so the
  // loads carry no predicate and no select and really are in flight for a whole block.
  float yreg[P4_SUB][8];
  const YT* ybase = reinterpret_cast<const YT*>(a.y);      // a.y carries the caller's pointer whatever its element type
  const int ld = (int)a.y_ld;                          // a row of y is shorter than 2^31 entries
  const int ld8 = 8 * ld;
  auto load_y = [&](int s, int gblk) {
    if (fast_cols && gblk + 16 <= g_end) {
      // interior block: the four rows 2c, 2c + 1, 2c + 8, 2c + 9 from one base pointer (one 32 x 32 -> 64-bit multiply-add, three adds)
      const YT* p0 = ybase + (int64_t)(gblk + 2 * c) * ld + (nw + 16 * s + 2 * r);
      const YT* p1 = p0 + ld;
      const YT* p2 = p0 + ld8;
      const YT* p3 = p2 + ld;
      y_load2<YT>(p0, yreg[s][0], yreg[s][2]); y_load2<YT>(p1, yreg[s][1], yreg[s][3]);
      y_load2<YT>(p2, yreg[s][4], yreg[s][6]); y_load2<YT>(p3, yreg[s][5], yreg[s][7]);
      return;
    }
    // ragged block / gathered columns: four clamped row pointers
    const YT* rowp[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int g = min(gblk + 8 * (j >> 1) + 2 * c + (j & 1), g_end - 1);
      rowp[j] = ybase + (int64_t)g * ld;
    }
    if (!HAS_IDX && block_full) {
#pragma unroll
      for (int q = 0; q < 8; ++q) yreg[s][q] = y_load1<YT>(rowp[2 * (q >> 2) + (q & 1)] + (nw + 16 * s + 2 * r) + ((q >> 1) & 1));
    } else {
#pragma unroll
      for (int q = 0; q < 8; ++q) yreg[s][q] = y_load1<YT>(rowp[2 * (q >> 2) + (q & 1)] + col[s][(q >> 1) & 1]);
    }
  };
#pragma unroll
  for (int s = 0; s < P4_SUB; ++s) load_y(s, g_begin);

  double ll = 0.0;
  for (int e = 0; e < a.E; ++e) {
    // operand fragments of the sample: A1 = EF'^T [16 spots x 16 factors] (rate), A3 = EF' [16 factors x 16 spots] (d/dW);
    // register k of A1 <-> spot half k & 1, factors 2c + 8 (k >> 1) + {0, 1}
    uint32_t a1h[P4_SUB][4], a1l[P4_SUB][4], a3h[P4_SUB][4], a3l[P4_SUB][4];
    float d2[P4_SUB][2][4];
#pragma unroll
    for (int s = 0; s < P4_SUB; ++s) {
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int n = nw + 16 * s + 2 * r + (k & 1);
        a1h[s][k] = 0u; a1l[s][k] = 0u;
        if (n < a.B) {
          const int64_t o = (((int64_t)e * a.B + n) * 16 + 2 * c + 8 * (k >> 1)) >> 1;
          a1h[s][k] = reinterpret_cast<const uint32_t*>(w.efh)[o];
          a1l[s][k] = reinterpret_cast<const uint32_t*>(w.efl)[o];
        }
      }
    }
#pragma unroll
    for (int s = 0; s < P4_SUB; ++s) {
      a3h[s][0] = movmatrix_t(a1h[s][0]); a3h[s][1] = movmatrix_t(a1h[s][2]);
      a3h[s][2] = movmatrix_t(a1h[s][1]); a3h[s][3] = movmatrix_t(a1h[s][3]);
      a3l[s][0] = movmatrix_t(a1l[s][0]); a3l[s][1] = movmatrix_t(a1l[s][2]);
      a3l[s][2] = movmatrix_t(a1l[s][1]); a3l[s][3] = movmatrix_t(a1l[s][3]);
#pragma unroll
      for (int lt = 0; lt < 2; ++lt)
#pragma unroll
        for (int i = 0; i < 4; ++i) d2[s][lt][i] = 0.f;
    }

    for (int g0 = g_begin; g0 < g_end; g0 += P4_GCH) {
      __syncthreads();                              // the previous chunk's reduction is done with sAcc; every warp is done with sW
      {                                             // stage the chunk's loadings: thread <-> (gene tid / 4, factors 4 (tid & 3) ..+3)
        const int gi = tid >> 2, lq = (tid & 3) * 4;
        uint2 vh = make_uint2(0u, 0u), vl = make_uint2(0u, 0u);
        if (g0 + gi < g_end) {
          vh = *reinterpret_cast<const uint2*>(w.wh + (int64_t)(g0 + gi) * 16 + lq);
          vl = *reinterpret_cast<const uint2*>(w.wl + (int64_t)(g0 + gi) * 16 + lq);
        }
        *reinterpret_cast<uint2*>(&sWh[gi][lq]) = vh;
        *reinterpret_cast<uint2*>(&sWl[gi][lq]) = vl;
        if constexpr (NB) {
          if (tid < P4_GCH)
            nbS[tid] = g0 + tid < g_end ? reinterpret_cast<const float2*>(a.nbg)[g0 + tid] : make_float2(1.f, 1.f);
        }
      }
      __syncthreads();
      const int nblk = min(P4_GCH / 16, (g_end - g0 + 15) >> 4);
      float llc = 0.f, llg = 0.f;
#pragma unroll 1
      for (int jb = 0; jb < nblk; ++jb) {
        const int gblk = g0 + 16 * jb;
        // next block in (sample, gene) order, for the y prefetch
        int gnext = gblk + 16;
        if (gnext >= g_end) gnext = (e + 1 < a.E) ? g_begin : -1;
        const bool ragged = gblk + 16 > g_end || !block_full;          // uniform: some of the 16 x 32 elements are not there
        // ldmatrix row addresses.  rate: B[k = factor][n = gene], matrices (genes 0-7, l 0-7), (genes 0-7, l 8-15), (genes 8-15, l 0-7),
        // (genes 8-15, l 8-15); d/dEF': B[k = gene][n = factor], transposed on load: (genes 0-7, l 0-7), (genes 8-15, l 0-7), (genes 0-7,
        // l 8-15), (genes 8-15, l 8-15).  The fragments are (re)loaded per sub-tile right before their MMAs to keep them short-lived.
        const int mi = lane >> 3, row = lane & 7;
        const int o1 = (16 * jb + (mi >> 1) * 8 + row) * P4_WLD + (mi & 1) * 8;
        const int o2 = (16 * jb + (mi & 1) * 8 + row) * P4_WLD + (mi >> 1) * 8;
        float d3[2][4];
#pragma unroll
        for (int tt = 0; tt < 2; ++tt)
#pragma unroll
          for (int i = 0; i < 4; ++i) d3[tt][i] = 0.f;
#pragma unroll
        for (int s = 0; s < P4_SUB; ++s) {
          float c1[2][4];
          {
            uint32_t b1h[4], b1l[4];
            ldmatrix_x4(b1h, &sWh[0][0] + o1);
            ldmatrix_x4(b1l, &sWl[0][0] + o1);
#pragma unroll
            for (int tt = 0; tt < 2; ++tt) {
#pragma unroll
              for (int i = 0; i < 4; ++i) c1[tt][i] = 0.f;
              mma_bf16(c1[tt], a1l[s], b1h[2 * tt], b1h[2 * tt + 1]);
              mma_bf16(c1[tt], a1h[s], b1l[2 * tt], b1l[2 * tt + 1]);
              mma_bf16(c1[tt], a1h[s], b1h[2 * tt], b1h[2 * tt + 1]);
            }
          }
          if (ragged) {                             // genes past the range / spots past the minibatch carry no count
#pragma unroll
            for (int q = 0; q < 8; ++q)
              if (gblk + 8 * (q >> 2) + 2 * c + (q & 1) >= g_end || nw + 16 * s + 2 * r + ((q >> 1) & 1) >= a.B) yreg[s][q] = 0.f;
          }
          // element-wise on the rate fragment
          float t[8];
          if constexpr (NB) {
            // d log NB / d r = (y - r) / (r (1 + q)), q = r / theta; llg collects the natural-log terms with the opposite sign.
            // The table terms of counts >= 64 and non-integer y are zero here and come from nb_slow in the pass below.
            // dth: d ll / d theta of the thread's four genes over its two spots of the sub-tile; slot j <-> gene
            // gblk + 8 (j >> 1) + 2c + (j & 1) (register q of a fragment is slot 2 (q >> 2) + (q & 1))
            float dth[4] = {0.f, 0.f, 0.f, 0.f};
            unsigned slow = 0u;
#pragma unroll
            for (int q = 0; q < 8; ++q) {
              const float y = yreg[s][q];
              const float2 nb = nbS[16 * jb + 8 * (q >> 2) + 2 * c + (q & 1)];
              const int yi = (int)min((unsigned)__float2int_rz(y), 63u);     // negative or huge -> 63, which fails the comparison
              const bool ok = (float)yi == y;
              const int g = min(gblk + 8 * (q >> 2) + 2 * c + (q & 1), g_end - 1);
              float2 tv = __ldg(reinterpret_cast<const float2*>(a.tab) + (int64_t)g * 64 + yi);
              if (!ok) { tv = make_float2(0.f, 0.f); slow |= 1u << q; }
              const float rate = fmaxf(c1[q >> 2][q & 3], 1e-30f);
              const float qq = rate * nb.y;
              const float l1p = nb_log1p(qq);
              float rd;
              asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rd) : "f"(fmaf(rate, qq, rate)));
              const float ud = (y - rate) * rd;
              llc = fmaf(y, __log2f(rate), llc);
              llg += fmaf(y + nb.x, l1p, -tv.x);
              t[q] = ud * invE;
              dth[2 * (q >> 2) + (q & 1)] += tv.y - fmaf(ud, qq, l1p);
            }
#pragma unroll 1
            while (slow) {                          // one call site, not unrolled: it keeps the call's register cost off the hot path
              const int q = __ffs(slow) - 1, j = 2 * (q >> 2) + (q & 1);
              slow &= slow - 1u;
              float y = 0.f;
#pragma unroll
              for (int k = 0; k < 8; ++k) y = k == q ? yreg[s][k] : y;
              const double2 sl = nb_slow((double)y, (double)nbS[16 * jb + 8 * (j >> 1) + 2 * c + (j & 1)].x, a.with_lgamma);
              llg -= (float)sl.x;
#pragma unroll
              for (int k = 0; k < 4; ++k) dth[k] += k == j ? (float)sl.y : 0.f;
            }
            // sum the four slots over the 8 lanes of equal c (lane bits 2-4) in 4 shuffles; lane bits 4 and 3 end up naming the
            // slot.  Summed per sub-tile (the first one writes), so the four accumulators live only through this element step.
            const bool hi16 = lane & 16, hi8 = lane & 8;
            float k0 = hi16 ? dth[2] : dth[0], k1 = hi16 ? dth[3] : dth[1];
            k0 += __shfl_xor_sync(0xffffffffu, hi16 ? dth[0] : dth[2], 16);
            k1 += __shfl_xor_sync(0xffffffffu, hi16 ? dth[1] : dth[3], 16);
            float k = hi8 ? k1 : k0;
            k += __shfl_xor_sync(0xffffffffu, hi8 ? k0 : k1, 8);
            k += __shfl_xor_sync(0xffffffffu, k, 4);
            if ((lane & 4) == 0) {
              float* d = &dS[warp][16 * jb + 8 * (lane >> 4) + 2 * c + ((lane >> 3) & 1)];
              *d = s == 0 ? k : *d + k;
            }
          } else {
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            const float y = yreg[s][q];
            const float rate = fmaxf(c1[q >> 2][q & 3], 1e-30f);
            float rinv;
            asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rinv) : "f"(rate));
            llc = fmaf(y, __log2f(rate), llc);
            t[q] = fmaf(y * invE, rinv, -invE);
          }
          }
          if (!NB && a.with_lgamma) {
            // log(y!) from the table, branch-free: the entry of min(trunc(y), 63), exact whenever y is an integer count below 64
            // (lfact[0] = lfact[1] = 0); anything else (y >= 64, non-integer y) is detected by comparing back and redone exactly.
            bool exact = true;
            float lg8 = 0.f;
#pragma unroll
            for (int q = 0; q < 8; ++q) {
              const float y = yreg[s][q];
              const int yi = (int)min((unsigned)__float2int_rz(y), 63u);       // negative or huge -> 63, which fails the comparison
              exact = exact && ((float)yi == y);
              lg8 += lfact[yi];
            }
            if (!exact) {
              lg8 = 0.f;
#pragma unroll
              for (int q = 0; q < 8; ++q) {
                const float y = yreg[s][q];
                const int yi = (int)min((unsigned)__float2int_rz(y), 63u);
                lg8 += ((float)yi == y) ? lfact[yi] : lfact_slow(y);
              }
            }
            llg += lg8;
          }
          if (gnext >= 0) load_y(s, gnext);         // the sub-tile's y registers are free: fetch the next block's values into them
          // t' as the A fragment [16 spots x 16 genes]: a0 = tile 0 rows r, a1 = tile 0 rows r + 8, a2 / a3 = tile 1
          uint32_t th[4], tl[4];
          split_bf16x2(t[0], t[1], th[0], tl[0]);
          split_bf16x2(t[2], t[3], th[1], tl[1]);
          split_bf16x2(t[4], t[5], th[2], tl[2]);
          split_bf16x2(t[6], t[7], th[3], tl[3]);
          {
            uint32_t b2h[4], b2l[4];
            ldmatrix_x4_t(b2h, &sWh[0][0] + o2);
            ldmatrix_x4_t(b2l, &sWl[0][0] + o2);
#pragma unroll
            for (int lt = 0; lt < 2; ++lt) {
              mma_bf16(d2[s][lt], tl, b2h[2 * lt], b2h[2 * lt + 1]);
              mma_bf16(d2[s][lt], th, b2l[2 * lt], b2l[2 * lt + 1]);
              mma_bf16(d2[s][lt], th, b2h[2 * lt], b2h[2 * lt + 1]);
            }
          }
          // t'^T as B fragments [16 spots x 8 genes] of the two gene tiles
#pragma unroll
          for (int tt = 0; tt < 2; ++tt) {
            const uint32_t bh0 = movmatrix_t(th[2 * tt]), bh1 = movmatrix_t(th[2 * tt + 1]);
            const uint32_t bl0 = movmatrix_t(tl[2 * tt]), bl1 = movmatrix_t(tl[2 * tt + 1]);
            mma_bf16(d3[tt], a3l[s], bh0, bh1);
            mma_bf16(d3[tt], a3h[s], bl0, bl1);
            mma_bf16(d3[tt], a3h[s], bh0, bh1);
          }
        }
        // D3[l = r (+8)][gene = 16 jb + 8 tt + 2c (+1)] of this warp's 32 spots
#pragma unroll
        for (int tt = 0; tt < 2; ++tt) {
          *reinterpret_cast<float2*>(&sAcc[warp][r][16 * jb + 8 * tt + 2 * c]) = make_float2(d3[tt][0], d3[tt][1]);
          *reinterpret_cast<float2*>(&sAcc[warp][r + 8][16 * jb + 8 * tt + 2 * c]) = make_float2(d3[tt][2], d3[tt][3]);
        }
      }
      ll += (double)((llc * LN2 - llg) * invE);
      __syncthreads();
      const int nvalid = min(P4_GCH, g_end - g0) * a.F;
      for (int i = tid; i < nvalid; i += P4_THREADS) {
        const int gi = i / a.F, f = i - gi * a.F;
        float v = 0.f;
#pragma unroll
        for (int w8 = 0; w8 < P4_WARPS; ++w8) v += sAcc[w8][f][gi];
        float* dst = a.gW_part + ((int64_t)blockIdx.x * a.G + g0 + gi) * a.F + f;
        *dst = e == 0 ? v : *dst + v;
      }
      if constexpr (NB) {
        if (tid < min(P4_GCH, g_end - g0)) {
          float v = 0.f;
#pragma unroll
          for (int w8 = 0; w8 < P4_WARPS; ++w8) v += dS[w8][tid];
          float* dst = a.gD_part + (int64_t)blockIdx.x * a.G + g0 + tid;
          *dst = e == 0 ? v : *dst + v;
        }
      }
    }
    // D2[n][l] of the sample leaves the registers: (n = r + 8 (i >> 1), l = 8 lt + 2c + (i & 1)) pairs as float2
#pragma unroll
    for (int s = 0; s < P4_SUB; ++s)
#pragma unroll
      for (int lt = 0; lt < 2; ++lt)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int n = nw + 16 * s + 2 * r + h;
          if (n < a.B) {
            float2* dst = reinterpret_cast<float2*>(w.d2 + ((int64_t)e * a.B + n) * 16 + 8 * lt + 2 * c);
            const float2 v = make_float2(d2[s][lt][2 * h], d2[s][lt][2 * h + 1]);
            if (a.atomic_out) atomicAdd(dst, v); else *dst = v;
          }
        }
  }
  const double tot = block_sum<double>(ll, red);
  if (tid == 0) a.ll_part[blockIdx.y * gridDim.x + blockIdx.x] = tot;
}


// blocks [0, gw_blocks): gW[g, f] = (softplus'(W[g, f]) or 1) * sum_b gW_part[b, g, f]; blocks [gw_blocks, ...): 64 spots each, all samples:
// gF = EF' D2 -> d/dmean, d/dspread, d/dV and sum_g r.  The last block to finish sums the log-likelihood partials (fixed order).
// NB: blocks [gw_blocks + spot_blocks, ...) reduce the d/dD partials, 256 genes each; ll has no sum_g r term.
template <bool NB>
__global__ void __launch_bounds__(256) poisson_post4_kernel(const K7Args<float, NB> a, const Poisson4Ws w, float* __restrict__ gW, int nbx,
                                                            int nby, int gw_blocks, int spot_blocks, double* __restrict__ ll_out) {
  __shared__ double red[32];
  __shared__ float wsum[16];
  __shared__ bool last;
  const int tid = threadIdx.x;
  if (NB && (int)blockIdx.x >= gw_blocks + spot_blocks) {
    if constexpr (NB) {                     // gD[g] = softplus'(D[g]) / E * sum_b gD_part[b, g], in a fixed order
      const int g = (blockIdx.x - gw_blocks - spot_blocks) * 256 + tid;
      if (g < a.G) {
        float s0 = 0.f, s1 = 0.f;
        int b = 0;
        for (; b + 1 < nbx; b += 2) { s0 += a.gD_part[(int64_t)b * a.G + g]; s1 += a.gD_part[(int64_t)(b + 1) * a.G + g]; }
        if (b < nbx) s0 += a.gD_part[(int64_t)b * a.G + g];
        a.gD[g] = softplus_grad(a.D[g]) * (s0 + s1) / (float)a.E;
      }
    }
  } else if ((int)blockIdx.x < gw_blocks) {
    // 64 outputs per block; thread (o, p) adds the partials of the CTAs b = p, p + 4, ... (independent loads, 256-byte rows)
    __shared__ float part[4][64];
    const int64_t GF = (int64_t)a.G * a.F, i = (int64_t)blockIdx.x * 64 + (tid & 63);
    const int p = tid >> 6;
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
    if (i < GF) {
      int b = p;
      for (; b + 12 < nbx; b += 16) {
        s0 += a.gW_part[(int64_t)b * GF + i];
        s1 += a.gW_part[(int64_t)(b + 4) * GF + i];
        s2 += a.gW_part[(int64_t)(b + 8) * GF + i];
        s3 += a.gW_part[(int64_t)(b + 12) * GF + i];
      }
      for (; b < nbx; b += 4) s0 += a.gW_part[(int64_t)b * GF + i];
    }
    part[p][tid & 63] = (s0 + s1) + (s2 + s3);
    __syncthreads();
    if (tid < 64 && i < GF) {
      const float s = (part[0][tid] + part[1][tid]) + (part[2][tid] + part[3][tid]);
      gW[i] = a.w_softplus ? s * softplus_grad(a.W[i]) : s;
    }
  } else {
    if (!NB && tid < 16) {
      float v = 0.f;
      for (int by = 0; by < nby; ++by) v += w.wsum[by * 16 + tid];
      wsum[tid] = v;
    }
    __syncthreads();
    const int sb = blockIdx.x - gw_blocks, n = sb * 64 + (tid >> 2), lq = (tid & 3) * 4;
    float rs = 0.f, gsum = 0.f, vraw = 0.f, spV = 1.f;
    if (n < a.B) {
      vraw = a.V[a.idx ? a.idx[n] : (int64_t)n];
      spV = softplus(vraw);
      float gm[4] = {0.f, 0.f, 0.f, 0.f}, gs[4] = {0.f, 0.f, 0.f, 0.f}, sdv[4];
      for (int e = 0; e < a.E; ++e) {
        float ev[4], epsv[4];
        poisson_ef4(a, e, n, lq, spV, ev, epsv, sdv);
        const float4 d = *reinterpret_cast<const float4*>(w.d2 + ((int64_t)e * a.B + n) * 16 + lq);
        const float dv[4] = {d.x, d.y, d.z, d.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float gF = ev[j] * dv[j];
          gm[j] += gF;
          gs[j] = fmaf(gF, epsv[j], gs[j]);
          gsum += gF;
          if constexpr (!NB) rs = fmaf(ev[j], wsum[lq + j], rs);
        }
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int f = lq + j;
        if (f < a.F) {
          const int64_t o = (int64_t)f * a.B + n;
          float gsp = gs[j];
          if (f < a.n_var) gsp = a.spread[o] >= a.clamp_min ? gsp / (2.f * sdv[j]) : 0.f;   // d sd / d var = 1 / (2 sd) where not clamped
          a.gmean[o] = gm[j];
          a.gspread[o] = gsp;
        }
      }
    }
    // d ll / d V[n] = softplus'(V) / softplus(V) * sum_e sum_l gF_e[l, n]   (sum_g (y - r) = E sum_l EF'_l D2_l; 1/E is inside t')
    gsum += __shfl_xor_sync(0xffffffffu, gsum, 1);
    gsum += __shfl_xor_sync(0xffffffffu, gsum, 2);
    if (n < a.B && (tid & 3) == 0) a.gV[n] = softplus_grad(vraw) * gsum / spV;
    if constexpr (!NB) {
      const double tot = block_sum<double>((double)rs, red);
      if (tid == 0) w.rs_part[sb] = tot;
    }
  }
  // last block done: ll = sum(main partials) - sum(rate sums) / E
  __threadfence();
  __syncthreads();
  if (tid == 0) last = atomicAdd(w.ticket, 1u) == gridDim.x - 1;
  __syncthreads();
  if (!last) return;
  __threadfence();
  double s = 0.0;
  for (int i = tid; i < nbx * nby; i += 256) s += __ldcg(a.ll_part + i);
  if constexpr (!NB) {
    double rsum = 0.0;
    for (int i = tid; i < spot_blocks; i += 256) rsum += __ldcg(w.rs_part + i);
    s -= rsum / (double)a.E;
  }
  s = block_sum<double>(s, red);
  if (tid == 0) ll_out[0] = s;
}


// gW[g,f] = (softplus'(W[g,f]) or 1) * sum_b gW_part[b,g,f]
template <typename T>
__global__ void poisson_gw_reduce_kernel(const T* __restrict__ part, const T* __restrict__ W, T* __restrict__ gW, int64_t GF, int nb,
                                         int w_softplus) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= GF) return;
  T s = T(0);
  for (int b = 0; b < nb; ++b) s += part[(int64_t)b * GF + e];
  gW[e] = w_softplus ? s * softplus_grad(W[e]) : s;
}

__global__ void sum_double_kernel(const double* __restrict__ part, int n, double* __restrict__ out) {
  __shared__ double red[32];
  double s = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) s += part[i];
  s = block_sum<double>(s, red);
  if (threadIdx.x == 0) out[0] = s;
}

// K7-NB per-gene terms, in double: theta = softplus(D), 1 / theta, and for k < 64
//   Lambda_g[k] = sum_{j<k} log1p(j / theta) = lgamma(k + theta) - lgamma(theta) - k log theta   (minus log k! with_lgamma)
//   Psi_g[k]    = sum_{j<k} 1 / (theta + j)  = psi(k + theta) - psi(theta)
// Four genes per 256-thread block, thread <-> (gene, k); each prefix is summed in the same order by its own thread.
template <typename T>
__global__ void __launch_bounds__(256) negbin_tables_kernel(const T* __restrict__ D, int G, int with_lgamma, T* __restrict__ nbg,
                                                            T* __restrict__ tab) {
  __shared__ double sl[4][64], sp[4][64];
  const int k = threadIdx.x & 63, gl = threadIdx.x >> 6, g = blockIdx.x * 4 + gl;
  const double th = g < G ? softplus((double)D[g]) : 1.0;
  sl[gl][k] = ::log1p(k / th);                      // log(theta + k) - log theta, without the cancellation
  sp[gl][k] = 1.0 / (th + k);
  __syncthreads();
  if (g >= G) return;
  double lam = 0.0, psi = 0.0;
  for (int j = 0; j < k; ++j) { lam += sl[gl][j]; psi += sp[gl][j]; }
  if (with_lgamma) lam -= ::lgamma(k + 1.0);
  tab[((int64_t)g * 64 + k) * 2] = (T)lam;
  tab[((int64_t)g * 64 + k) * 2 + 1] = (T)psi;
  if (k < 2) nbg[(int64_t)g * 2 + k] = (T)(k == 0 ? th : 1.0 / th);
}

// gD[g] = softplus'(D[g]) / E * sum_b part[b, g] (poisson_kernel2 path; the tensor-core path does this in poisson_post4_kernel<true>)
template <typename T>
__global__ void negbin_gd_reduce_kernel(const T* __restrict__ part, const T* __restrict__ D, T* __restrict__ gD, int G, int nb, int E) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= G) return;
  T s = T(0);
  for (int b = 0; b < nb; ++b) s += part[(int64_t)b * G + g];
  gD[g] = softplus_grad(D[g]) * s / T(E);
}

template <typename T, int FMAX> constexpr size_t poisson_smem2() {
  return ((sizeof(T) * PZ_GCH * (P2_SPOTS + 1) + 15) / 16) * 16 + sizeof(T) * (FMAX * P2_SPOTS + PZ_GCH * FMAX + 4 * PZ_GCH * FMAX);
}
static bool poisson_use_v4(int F, bool is_f32) { return is_f32 && F <= 16; }     // tensor-core kernels; anything else runs kernel2
template <typename T, int FMAX, typename A> int poisson_launch(const A& a, dim3 grid, cudaStream_t st) {
  constexpr size_t smem = poisson_smem2<T, FMAX>();
  void (*kern)(const A) = poisson_kernel2<T, FMAX, std::is_same<A, NegBinArgs<T>>::value>;
  GPZ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<grid, P2_THREADS, smem, st>>>(a);
  GPZ_CHECK_LAUNCH();
  return GPZ_OK;
}

static void poisson_grid(int G, int F, int B, bool is_f32, int* nbx, int* nby, int* gpc) {
  if (poisson_use_v4(F, is_f32)) {        // 256 spots per CTA, gene ranges in whole 16-gene blocks, about four waves of 2 CTAs per SM
    *nbx = (int)cdiv(B, P4_SPOTS);
    const int blocks = (int)cdiv(G, 16);
    int by = 1;
    if (*nbx < 1184) by = (int)min((int64_t)blocks, (int64_t)max(1, 1184 / (*nbx > 0 ? *nbx : 1)));
    const int bpc = (int)cdiv(blocks, by);
    *gpc = bpc * 16;
    *nby = (int)cdiv(G, *gpc);
    return;
  }
  *nbx = (int)cdiv(B, P2_SPOTS);
  const int chunks = (int)cdiv(G, PZ_GCH);
  int by = 1;
  if (*nbx < 1184) by = (int)min((int64_t)chunks, cdiv(1184, *nbx > 0 ? *nbx : 1));
  const int cpc = (int)cdiv(chunks, by);
  *gpc = cpc * PZ_GCH;
  *nby = (int)cdiv(G, *gpc);
}

// workspace: ll partials (double) | gW partials [nbx][G][F] | (v4) the Poisson4Ws arrays
static size_t poisson_ll_slots(int nbx, int nby) { return ((size_t)nbx * nby + 2 + 1) & ~(size_t)1; }   // keeps what follows 16-byte aligned
static size_t poisson_ws_bytes(int G, int F, int B, int E, bool is_f32, size_t elt, int nbx, int nby) {
  size_t b = sizeof(double) * poisson_ll_slots(nbx, nby) + (elt * (size_t)nbx * G * F + 15) / 16 * 16;
  if (poisson_use_v4(F, is_f32)) {
    const size_t EB16 = 16 * (size_t)(E > 0 ? E : 1) * B;
    b += 2 * sizeof(uint16_t) * 16 * (size_t)G + 2 * sizeof(uint16_t) * EB16 + sizeof(float) * EB16 + sizeof(float) * 16 * (size_t)nby +
         sizeof(double) * (size_t)cdiv(B, 64) + 16;
  }
  return b;
}
// K7-NB appends: gD partials [nbx][G] | per-gene terms [G][2] | tables [G][64][2]
static size_t negbin_extra_bytes(int G, size_t elt, int nbx) { return (elt * (size_t)nbx * G + 15) / 16 * 16 + elt * 130 * (size_t)G; }
static size_t negbin_ws_bytes(int G, int F, int B, int E, bool is_f32, size_t elt, int nbx, int nby) {
  return (poisson_ws_bytes(G, F, B, E, is_f32, elt, nbx, nby) + 15) / 16 * 16 + negbin_extra_bytes(G, elt, nbx);
}

// y_kind: element type of y — 0 = T (the reference's format), 1 = uint8, 2 = int16, 3 = int32 (fp32 tensor-core kernel only).
// A = PoissonArgs<T> runs K7; A = NegBinArgs<T> runs K7-NB (same grid and kernels' structure, plus the per-gene tables and gD).
template <typename T, typename A>
int poisson_fwdbwd(A a, T* gW, double* ll_out, void* ws, size_t ws_bytes, cudaStream_t st, int y_kind = 0) {
  constexpr bool NB = std::is_same<A, NegBinArgs<T>>::value;
  if (a.F < 1 || a.F > 32 || a.E < 1 || a.G < 1) return GPZ_ERR_UNSUPPORTED;
  if (y_kind < 0 || y_kind > 3 || (y_kind != 0 && !poisson_use_v4(a.F, std::is_same<T, float>::value))) return GPZ_ERR_UNSUPPORTED;
  if (a.B == 0) {                       // empty minibatch: ll = 0, no gradient
    GPZ_CUDA(cudaMemsetAsync(ll_out, 0, sizeof(double), st));
    GPZ_CUDA(cudaMemsetAsync(gW, 0, sizeof(T) * (size_t)a.G * a.F, st));
    if constexpr (NB) GPZ_CUDA(cudaMemsetAsync(a.gD, 0, sizeof(T) * (size_t)a.G, st));
    return GPZ_OK;
  }
  int nbx, nby, gpc;
  poisson_grid(a.G, a.F, a.B, std::is_same<T, float>::value, &nbx, &nby, &gpc);
  const size_t base = poisson_ws_bytes(a.G, a.F, a.B, a.E, std::is_same<T, float>::value, sizeof(T), nbx, nby);
  const size_t need = NB ? negbin_ws_bytes(a.G, a.F, a.B, a.E, std::is_same<T, float>::value, sizeof(T), nbx, nby) : base;
  if (ws_bytes < need) return GPZ_ERR_BADARG;
  a.ll_part = reinterpret_cast<double*>(ws);
  a.gW_part = reinterpret_cast<T*>(a.ll_part + poisson_ll_slots(nbx, nby));
  a.genes_per_cta = gpc;
  a.atomic_out = nby > 1;
  if constexpr (NB) {
    unsigned char* pn = reinterpret_cast<unsigned char*>(ws) + (base + 15) / 16 * 16;
    a.gD_part = reinterpret_cast<T*>(pn); pn += (sizeof(T) * (size_t)nbx * a.G + 15) / 16 * 16;
    T* nbg = reinterpret_cast<T*>(pn);
    T* tab = nbg + 2 * (size_t)a.G;
    a.nbg = nbg; a.tab = tab;
    negbin_tables_kernel<T><<<(unsigned)cdiv(a.G, 4), 256, 0, st>>>(a.D, a.G, a.with_lgamma, nbg, tab);
    GPZ_CHECK_LAUNCH();
  }
  if (a.atomic_out && !poisson_use_v4(a.F, std::is_same<T, float>::value)) {
    GPZ_CUDA(cudaMemsetAsync(a.gV, 0, sizeof(T) * a.B, st));
    GPZ_CUDA(cudaMemsetAsync(a.gmean, 0, sizeof(T) * a.B * a.F, st));
    GPZ_CUDA(cudaMemsetAsync(a.gspread, 0, sizeof(T) * a.B * a.F, st));
  }
  dim3 grid(nbx, nby);
  int rc;
  if constexpr (std::is_same<T, float>::value) {
    if (poisson_use_v4(a.F, true)) {       // fp32, F <= 16: contractions on the tensor cores
      unsigned char* p4 = reinterpret_cast<unsigned char*>(a.gW_part) + (sizeof(T) * (size_t)nbx * a.G * a.F + 15) / 16 * 16;
      const size_t EB16 = 16 * (size_t)a.E * a.B;
      const int spot_blocks = (int)cdiv(a.B, 64), gw_blocks = (int)cdiv((int64_t)a.G * a.F, 64);
      Poisson4Ws w;
      w.d2 = reinterpret_cast<float*>(p4); p4 += sizeof(float) * EB16;
      w.wsum = reinterpret_cast<float*>(p4); p4 += sizeof(float) * 16 * (size_t)nby;
      w.rs_part = reinterpret_cast<double*>(p4); p4 += sizeof(double) * (size_t)spot_blocks;       // 8-byte aligned: every block above is a multiple of 64 B
      w.efh = reinterpret_cast<uint16_t*>(p4); p4 += sizeof(uint16_t) * EB16;
      w.efl = reinterpret_cast<uint16_t*>(p4); p4 += sizeof(uint16_t) * EB16;
      w.wh = reinterpret_cast<uint16_t*>(p4); p4 += sizeof(uint16_t) * 16 * (size_t)a.G;
      w.wl = reinterpret_cast<uint16_t*>(p4); p4 += sizeof(uint16_t) * 16 * (size_t)a.G;
      w.ticket = reinterpret_cast<unsigned int*>(p4);
      poisson_prep4_kernel<<<nby + a.E * spot_blocks, 256, 0, st>>>(a, w, nby, spot_blocks);
      GPZ_CHECK_LAUNCH();
#define GPZ_P4_LAUNCH(YT)                                                              \
  do {                                                                                 \
    if (a.idx) poisson_kernel4<true, YT, NB><<<grid, P4_THREADS, 0, st>>>(a, w);       \
    else poisson_kernel4<false, YT, NB><<<grid, P4_THREADS, 0, st>>>(a, w);            \
  } while (0)
      if (y_kind == 1) GPZ_P4_LAUNCH(uint8_t);
      else if (y_kind == 2) GPZ_P4_LAUNCH(int16_t);
      else if (y_kind == 3) GPZ_P4_LAUNCH(int32_t);
      else GPZ_P4_LAUNCH(float);
#undef GPZ_P4_LAUNCH
      GPZ_CHECK_LAUNCH();
      const int gd_blocks = NB ? (int)cdiv(a.G, 256) : 0;       // NB: the d/dD reduction
      poisson_post4_kernel<NB><<<gw_blocks + spot_blocks + gd_blocks, 256, 0, st>>>(a, w, gW, nbx, nby, gw_blocks, spot_blocks, ll_out);
      GPZ_CHECK_LAUNCH();
      return GPZ_OK;
    }
  }
  if (a.F <= 4) rc = poisson_launch<T, 4>(a, grid, st);
  else if (a.F <= 12) rc = poisson_launch<T, 12>(a, grid, st);
  else if (a.F <= 20) rc = poisson_launch<T, 20>(a, grid, st);
  else rc = poisson_launch<T, 32>(a, grid, st);
  if (rc) return rc;
  const int64_t GF = (int64_t)a.G * a.F;
  poisson_gw_reduce_kernel<T><<<(unsigned)cdiv(GF, 256), 256, 0, st>>>(a.gW_part, a.W, gW, GF, nbx, a.w_softplus);
  GPZ_CHECK_LAUNCH();
  if constexpr (NB) {
    negbin_gd_reduce_kernel<T><<<(unsigned)cdiv(a.G, 256), 256, 0, st>>>(a.gD_part, a.D, a.gD, a.G, nbx, a.E);
    GPZ_CHECK_LAUNCH();
  }
  sum_double_kernel<<<1, 256, 0, st>>>(a.ll_part, nbx * nby, ll_out);
  GPZ_CHECK_LAUNCH();
  return GPZ_OK;
}

// rate[e,g,n] = softplus(V[col]) * sum_f w(W[g,f]) exp(F[e,f,n]) -- the compatibility path that materialises
// pY.rate for callers of model.forward() (likelihoods.py:83-85); not used by the fused ELBO.
template <typename T>
__global__ void poisson_rate_kernel(const T* __restrict__ W, int w_softplus, const T* __restrict__ V, const int64_t* __restrict__ idx,
                                    const T* __restrict__ Fs, T* __restrict__ rate, int G, int F, int B, int E) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  const int e = blockIdx.z;
  if (n >= B) return;
  const T spV = softplus(V[idx ? idx[n] : (int64_t)n]);
  const int g0 = blockIdx.y * 32, g1 = min(G, g0 + 32);
  for (int g = g0; g < g1; ++g) {
    T zr = T(0);
    for (int f = 0; f < F; ++f) {
      T w = W[(int64_t)g * F + f];
      if (w_softplus) w = softplus(w);
      zr = fma(w, Num<T>::exp(Fs[((int64_t)e * F + f) * B + n]), zr);
    }
    rate[((int64_t)e * G + g) * B + n] = spV * zr;
  }
}

// ---- K7-CSC: the same outputs from sparse counts (spot-major compressed columns: indptr[N+1], genes[nnz], values[nnz]) --------
// With s_n = softplus(V_n), w = softplus(W) (or raw W), c_f = sum_g w_gf, eps_efn = s_n exp(F_efn), r_egn = sum_f w_gf eps_efn and
// t_egn = y_gn / (E r_egn) on the nonzeros only, the y = 0 entries contribute only -r, whose sums close through c_f:
//   ll          = sum_nz [ (1/E) sum_e y log r - lgamma(y+1) ] - (1/E) sum_{e,n,f} c_f eps_efn
//   d/dF_efn    = eps_efn ( sum_{g in nz(n)} t_egn w_gf - c_f / E )
//   d/dw_gf     = sum_e sum_{n in nz(g)} t_egn eps_efn - u_f,          u_f = (1/E) sum_{e,n} eps_efn
//   d/dV_n      = softplus'(V_n) / s_n ( sum_{g in nz(n)} y_gn - (1/E) sum_{e,f} c_f eps_efn )
// so the work per step is O(nnz F + B F + G F) whatever the density.  The "-1" the dense kernels take per element is taken here
// once per (spot, factor) and once per factor: near a fit the two sides nearly cancel, so c_f, u_f, ll, the per-spot
// sum_g t w and the final combination of the per-CTA d/dw partials are all carried in double.
// Mapping: one warp per spot (lanes stride over the spot's nonzeros; lane f owns factor f of the spot's per-spot terms), a fixed
// range of spots per CTA.  d/dw is scattered into a per-CTA G x F shared-memory accumulator when it fits (summed afterwards by
// csc_reduce_kernel in a fixed order), else into one G x F double accumulator in global memory by atomics.
constexpr int CSC_MAX_WARPS = 16;
// 512 threads; 256 for F > 12, whose F double accumulators per lane need more than the 128 registers a 512-thread CTA allows
template <int FMAX> constexpr int csc_threads() { return FMAX > 12 ? 256 : 512; }
constexpr size_t CSC_SMEM_MAX = 160 * 1024;      // per-CTA d/dw accumulator limit: G F <= 40960 in fp32 (config 2's 2000 x 20 fits)

template <typename T> struct CscArgs {
  const int64_t* indptr; const int32_t* genes; const void* values;
  const int64_t* idx;
  const T* W; int w_softplus; const T* V; const T* mean; const T* spread; const T* eps;
  int G, F, B, E, n_var; T clamp_min; int with_lgamma;
  // workspace
  const T* w;                  // [G][FMAX] softplus(W) or W, factors >= F zero
  const double* c;             // [F] column sums of w
  double* ll_part;             // [nbx]
  double* u_part;              // [nbx][F]
  T* gw_part;                  // [nbx][G][F] (shared-memory path) or null
  double* gw_acc;              // [G][F] (atomic path) or null
  int spots_per_cta;
  // outputs
  T* gV; T* gmean; T* gspread;
};

// blocks [0, F): c_f = sum_g w_gf in double; blocks [F, ...): the padded rows of w
template <typename T, int FMAX>
__global__ void __launch_bounds__(256) csc_prep_kernel(const T* __restrict__ W, int w_softplus, int G, int F, T* __restrict__ w,
                                                       double* __restrict__ c) {
  __shared__ double red[32];
  if ((int)blockIdx.x < F) {
    const int f = blockIdx.x;
    double s = 0.0;
    for (int g = threadIdx.x; g < G; g += blockDim.x) {
      const T v = W[(int64_t)g * F + f];
      s += (double)(w_softplus ? softplus(v) : v);
    }
    s = block_sum<double>(s, red);
    if (threadIdx.x == 0) c[f] = s;
    return;
  }
  const int64_t i = (int64_t)(blockIdx.x - F) * blockDim.x + threadIdx.x;
  if (i >= (int64_t)G * FMAX) return;
  const int64_t g = i / FMAX;
  const int f = (int)(i - g * FMAX);
  T v = T(0);
  if (f < F) {
    v = W[g * F + f];
    if (w_softplus) v = softplus(v);
  }
  w[i] = v;
}

template <typename YT, typename T> __device__ __forceinline__ T csc_value(const void* p, int64_t k) {
  return (T)reinterpret_cast<const YT*>(p)[k];
}
// four consecutive elements of a 16-byte aligned row
__device__ __forceinline__ void ld4(const float* p, float (&o)[4]) {
  const float4 v = *reinterpret_cast<const float4*>(p);
  o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w;
}
__device__ __forceinline__ void ld4(const double* p, double (&o)[4]) {
  const double2 v0 = reinterpret_cast<const double2*>(p)[0], v1 = reinterpret_cast<const double2*>(p)[1];
  o[0] = v0.x; o[1] = v0.y; o[2] = v1.x; o[3] = v1.y;
}
__device__ __forceinline__ void ld4_nc(const float* p, float (&o)[4]) {
  const float4 v = __ldg(reinterpret_cast<const float4*>(p));
  o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w;
}
__device__ __forceinline__ void ld4_nc(const double* p, double (&o)[4]) {
  const double2 v0 = __ldg(reinterpret_cast<const double2*>(p)), v1 = __ldg(reinterpret_cast<const double2*>(p) + 1);
  o[0] = v0.x; o[1] = v0.y; o[2] = v1.x; o[3] = v1.y;
}

template <typename T, typename YT, int FMAX, bool SMEM_ACC>
__global__ void __launch_bounds__(csc_threads<FMAX>(), 1) poisson_csc_kernel(const CscArgs<T> a) {
  constexpr int CSC_THREADS = csc_threads<FMAX>(), CSC_WARPS = CSC_THREADS / 32;
  extern __shared__ __align__(16) unsigned char csc_smem[];
  T* sAcc = reinterpret_cast<T*>(csc_smem);                     // [G][F] (SMEM_ACC)
  __shared__ double red[32];
  __shared__ double sU[CSC_MAX_WARPS][32];
  __shared__ __align__(16) T sEf[CSC_MAX_WARPS][32];                  // eps_e[:] of the warp's current spot (read as broadcasts)
  __shared__ T lfact[64];                                         // log(y!) for integer counts y < 64

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int F = a.F, GF = a.G * a.F;
  if (tid < 64) lfact[tid] = Num<T>::lgamma(T(tid + 1));
  if (SMEM_ACC)
    for (int i = tid; i < GF; i += CSC_THREADS) sAcc[i] = T(0);
  __syncthreads();

  const T invE = T(1) / T(a.E);
  const double cf = lane < F ? a.c[lane] : 0.0;
  double ll = 0.0, u = 0.0;                                       // u: lane f's share of u_f
  const int b_begin = blockIdx.x * a.spots_per_cta, b_end = min(a.B, b_begin + a.spots_per_cta);
  for (int b = b_begin + warp; b < b_end; b += CSC_WARPS) {
    const int64_t col = a.idx ? a.idx[b] : (int64_t)b;
    const int64_t p0 = a.indptr[col], p1 = a.indptr[col + 1];
    const T vraw = a.V[col];
    const T spV = softplus(vraw);
    // lane f: this spot's variational parameters of factor f
    T mu = T(0), sd = T(0), sp = T(0);
    if (lane < F) {
      const int64_t o = (int64_t)lane * a.B + b;
      mu = a.mean[o];
      sp = a.spread[o];
      sd = lane < a.n_var ? Num<T>::sqrt(sp > a.clamp_min ? sp : a.clamp_min) : sp;
    }
    T gm = T(0), gs = T(0);
    double ysum = 0.0, rsum = 0.0;                                // sum_nz y;  sum_e sum_f c_f eps_ef
    for (int e = 0; e < a.E; ++e) {
      T epsv = T(0), ev = T(0);
      if (lane < F) {
        epsv = a.eps[((int64_t)e * F + lane) * a.B + b];
        ev = spV * Num<T>::exp(fma(epsv, sd, mu));
      }
      const T* sE = sEf[warp];
      __syncwarp();                                               // the previous spot / sample is done with sE
      if (lane < FMAX) sEf[warp][lane] = ev;                      // lanes >= F hold 0
      __syncwarp();
      rsum += warp_sum<double>(cf * (double)ev);
      u += (double)ev;
      double acc[FMAX];                                           // sum over the lane's nonzeros of t w_f
#pragma unroll
      for (int f = 0; f < FMAX; ++f) acc[f] = 0.0;
      double llc = 0.0;
      for (int64_t k = p0 + lane; k < p1; k += 32) {
        const int g = a.genes[k];
        const T y = csc_value<YT, T>(a.values, k);
        const T* wr = a.w + (int64_t)g * FMAX;
        T r = T(0);
#pragma unroll
        for (int f4 = 0; f4 < FMAX; f4 += 4) {
          T w4[4], e4[4];
          ld4_nc(wr + f4, w4);
          ld4(sE + f4, e4);
#pragma unroll
          for (int j = 0; j < 4; ++j) r = fma(w4[j], e4[j], r);
        }
        const T t = fast_div(y, r) * invE;
        T lp = y * fast_log(r) * invE;
        if (e == 0) {
          if (a.with_lgamma) {
            const int yi = (int)y;
            lp -= (yi >= 0 && yi < 64 && T(yi) == y) ? lfact[yi] : Num<T>::lgamma(y + T(1));
          }
          ysum += (double)y;
        }
        llc += (double)lp;
        // second pass over the row (reloaded from L1 rather than held: keeps the F double accumulators spill-free)
#pragma unroll
        for (int f4 = 0; f4 < FMAX; f4 += 4) {
          T w4[4], e4[4];
          ld4(wr + f4, w4);
          ld4(sE + f4, e4);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int f = f4 + j;
            acc[f] += (double)(t * w4[j]);
            if (f < F) {
              const T gw = t * e4[j];
              if (SMEM_ACC) atomicAdd(sAcc + g * F + f, gw);
              else atomicAdd(a.gw_acc + (int64_t)g * F + f, (double)gw);
            }
          }
        }
      }
      ll += llc;
      // lane f: d ll / d F_ef = eps_ef (sum_g t w_f - c_f / E)
      double mine = 0.0;
#pragma unroll
      for (int f = 0; f < FMAX; ++f) {
        const double v = warp_sum<double>(acc[f]);
        if (lane == f) mine = v;
      }
      if (lane < F) {
        const T gF = (T)((double)ev * (mine - cf * (double)invE));
        gm += gF;
        gs = fma(gF, epsv, gs);
      }
    }
    ysum = warp_sum<double>(ysum);
    if (lane == 0) {
      ll -= rsum * (double)invE;
      a.gV[b] = (T)((double)(softplus_grad(vraw) / spV) * (ysum - rsum * (double)invE));
    }
    if (lane < F) {
      const int64_t o = (int64_t)lane * a.B + b;
      if (lane < a.n_var) gs = sp >= a.clamp_min ? gs / (T(2) * sd) : T(0);   // spread is a variance: d sd / d var = 1 / (2 sd)
      a.gmean[o] = gm;
      a.gspread[o] = gs;
    }
  }

  // per-CTA partials: ll, u_f, and the d/dw accumulator
  sU[warp][lane] = u;
  const double tot = block_sum<double>(ll, red);                  // its barriers also publish sU and the shared atomics
  if (tid == 0) a.ll_part[blockIdx.x] = tot;
  if (tid < F) {
    double s = 0.0;
    for (int w8 = 0; w8 < CSC_WARPS; ++w8) s += sU[w8][tid];
    a.u_part[(int64_t)blockIdx.x * F + tid] = s * (double)invE;
  }
  if (SMEM_ACC)
    for (int i = tid; i < GF; i += CSC_THREADS) a.gw_part[(int64_t)blockIdx.x * GF + i] = sAcc[i];
}

// gW[g, f] = (softplus'(W) or 1) * (sum of the d/dw partials - u_f), all sums in double and in a fixed order; block 0 also sums ll
template <typename T>
__global__ void __launch_bounds__(256) csc_reduce_kernel(const CscArgs<T> a, int nbx, T* __restrict__ gW, double* __restrict__ ll_out) {
  __shared__ double u[32];
  __shared__ double red[32];
  const int tid = threadIdx.x;
  if (tid < a.F) {
    double s = 0.0;
    for (int b = 0; b < nbx; ++b) s += a.u_part[(int64_t)b * a.F + tid];
    u[tid] = s;
  }
  if (blockIdx.x == 0) {
    double s = 0.0;
    for (int b = tid; b < nbx; b += blockDim.x) s += a.ll_part[b];
    s = block_sum<double>(s, red);                                // also the barrier that publishes u
    if (tid == 0) ll_out[0] = s;
  } else {
    __syncthreads();
  }
  // 64 outputs per block; thread (o, p) adds the partials of the CTAs b = p, p + 4, ... with four independent accumulators
  __shared__ double part[4][64];
  const int64_t GF = (int64_t)a.G * a.F, i = (int64_t)blockIdx.x * 64 + (tid & 63);
  const int p = tid >> 6;
  double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
  if (i < GF && a.gw_part) {
    int b = p;
    for (; b + 12 < nbx; b += 16) {
      s0 += (double)a.gw_part[(int64_t)b * GF + i];
      s1 += (double)a.gw_part[(int64_t)(b + 4) * GF + i];
      s2 += (double)a.gw_part[(int64_t)(b + 8) * GF + i];
      s3 += (double)a.gw_part[(int64_t)(b + 12) * GF + i];
    }
    for (; b < nbx; b += 4) s0 += (double)a.gw_part[(int64_t)b * GF + i];
  }
  part[p][tid & 63] = (s0 + s1) + (s2 + s3);
  __syncthreads();
  if (tid >= 64 || i >= GF) return;
  const double s = a.gw_part ? (part[0][tid] + part[1][tid]) + (part[2][tid] + part[3][tid]) : a.gw_acc[i];
  const T d = (T)(s - u[i % a.F]);
  gW[i] = a.w_softplus ? d * softplus_grad(a.W[i]) : d;
}

static int csc_fmax(int F) { return F <= 4 ? 4 : F <= 12 ? 12 : F <= 20 ? 20 : 32; }
static int csc_nbx(int B) {                   // one CTA per SM (the per-CTA d/dw partials are G F each), at least 16 spots per CTA
  static int nsm = 0;
  if (nsm == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) nsm = 148;
  }
  return (int)max((int64_t)1, min(cdiv(B, 16), (int64_t)nsm));
}
static bool csc_smem_acc(int G, int F, size_t elt) { return elt * (size_t)G * F <= CSC_SMEM_MAX; }
static size_t align16(size_t b) { return (b + 15) / 16 * 16; }
// workspace: ll_part [nbx] | u_part [nbx][F] | c [F] (doubles) | w [G][FMAX] | d/dw partials [nbx][G][F] T or accumulator [G][F] double
static size_t csc_ws_bytes(int G, int F, int B, size_t elt) {
  const int nbx = csc_nbx(B);
  size_t b = align16(sizeof(double) * ((size_t)nbx * (F + 1) + F)) + align16(elt * (size_t)G * csc_fmax(F));
  b += csc_smem_acc(G, F, elt) ? align16(elt * (size_t)nbx * G * F) : align16(sizeof(double) * (size_t)G * F);
  return b;
}

template <typename T, typename YT, int FMAX> int csc_launch_main(const CscArgs<T>& a, int nbx, cudaStream_t st) {
  if (a.gw_part) {
    const size_t smem = sizeof(T) * (size_t)a.G * a.F;
    GPZ_CUDA(cudaFuncSetAttribute(poisson_csc_kernel<T, YT, FMAX, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    poisson_csc_kernel<T, YT, FMAX, true><<<nbx, csc_threads<FMAX>(), smem, st>>>(a);
  } else {
    poisson_csc_kernel<T, YT, FMAX, false><<<nbx, csc_threads<FMAX>(), 0, st>>>(a);
  }
  GPZ_CHECK_LAUNCH();
  return GPZ_OK;
}
template <typename T, int FMAX> int csc_launch(CscArgs<T> a, int count_kind, int nbx, double* wbase_c, cudaStream_t st) {
  csc_prep_kernel<T, FMAX><<<(unsigned)(a.F + cdiv((int64_t)a.G * FMAX, 256)), 256, 0, st>>>(a.W, a.w_softplus, a.G, a.F,
                                                                                              const_cast<T*>(a.w), wbase_c);
  GPZ_CHECK_LAUNCH();
  switch (count_kind) {
    case 1: return csc_launch_main<T, uint8_t, FMAX>(a, nbx, st);
    case 2: return csc_launch_main<T, int16_t, FMAX>(a, nbx, st);
    case 3: return csc_launch_main<T, int32_t, FMAX>(a, nbx, st);
    default: return csc_launch_main<T, T, FMAX>(a, nbx, st);
  }
}

template <typename T>
int poisson_fwdbwd_csc(CscArgs<T> a, int count_kind, int64_t n_total, T* gW, double* ll_out, void* ws, size_t ws_bytes, cudaStream_t st) {
  if (a.F < 1 || a.F > 32 || a.E < 1 || a.G < 1) return GPZ_ERR_UNSUPPORTED;
  if (count_kind < 0 || count_kind > 3 || a.B < 0 || (!a.idx && a.B != n_total)) return GPZ_ERR_BADARG;
  if (a.B == 0) {                       // empty minibatch: ll = 0, no gradient
    GPZ_CUDA(cudaMemsetAsync(ll_out, 0, sizeof(double), st));
    GPZ_CUDA(cudaMemsetAsync(gW, 0, sizeof(T) * (size_t)a.G * a.F, st));
    return GPZ_OK;
  }
  if (ws_bytes < csc_ws_bytes(a.G, a.F, a.B, sizeof(T))) return GPZ_ERR_BADARG;
  const int nbx = csc_nbx(a.B), fmax = csc_fmax(a.F);
  unsigned char* p = reinterpret_cast<unsigned char*>(ws);
  a.ll_part = reinterpret_cast<double*>(p);
  a.u_part = a.ll_part + nbx;
  double* c = a.u_part + (size_t)nbx * a.F;
  a.c = c;
  p += align16(sizeof(double) * ((size_t)nbx * (a.F + 1) + a.F));
  a.w = reinterpret_cast<T*>(p);
  p += align16(sizeof(T) * (size_t)a.G * fmax);
  a.gw_part = nullptr; a.gw_acc = nullptr;
  if (csc_smem_acc(a.G, a.F, sizeof(T))) {
    a.gw_part = reinterpret_cast<T*>(p);
  } else {
    a.gw_acc = reinterpret_cast<double*>(p);
    GPZ_CUDA(cudaMemsetAsync(a.gw_acc, 0, sizeof(double) * (size_t)a.G * a.F, st));
  }
  a.spots_per_cta = (int)cdiv(a.B, nbx);
  int rc;
  if (fmax == 4) rc = csc_launch<T, 4>(a, count_kind, nbx, c, st);
  else if (fmax == 12) rc = csc_launch<T, 12>(a, count_kind, nbx, c, st);
  else if (fmax == 20) rc = csc_launch<T, 20>(a, count_kind, nbx, c, st);
  else rc = csc_launch<T, 32>(a, count_kind, nbx, c, st);
  if (rc) return rc;
  csc_reduce_kernel<T><<<(unsigned)max((int64_t)1, cdiv((int64_t)a.G * a.F, 64)), 256, 0, st>>>(a, nbx, gW, ll_out);
  GPZ_CHECK_LAUNCH();
  return GPZ_OK;
}

}  // namespace gpz

using namespace gpz;

#define GPZ_POISSON_IMPL(SUF, T)                                                                                       \
  extern "C" int64_t gpz_poisson_workspace_bytes_##SUF(int G, int F, int B, int E) {                                   \
    int nbx, nby, gpc;                                                                                                 \
    poisson_grid(G, F, B, sizeof(T) == 4, &nbx, &nby, &gpc);                                                           \
    return (int64_t)poisson_ws_bytes(G, F, B, E, sizeof(T) == 4, sizeof(T), nbx, nby);                                 \
  }                                                                                                                    \
  extern "C" int gpz_poisson_fwdbwd_##SUF(const T* y, int64_t y_ld, const int64_t* idx, const T* W, int w_softplus,    \
                                          const T* V, const T* mean, const T* spread, const T* eps, int G, int F,      \
                                          int B, int E, int n_var, T clamp_min, int with_lgamma, double* ll, T* gW,    \
                                          T* gV, T* gmean, T* gspread, void* ws, int64_t ws_bytes, void* stream) {     \
    PoissonArgs<T> a;                                                                                                  \
    a.y = y; a.y_ld = y_ld; a.idx = idx; a.W = W; a.w_softplus = w_softplus; a.V = V; a.mean = mean;                   \
    a.spread = spread; a.eps = eps; a.G = G; a.F = F; a.B = B; a.E = E; a.n_var = n_var; a.clamp_min = clamp_min;      \
    a.with_lgamma = with_lgamma; a.gV = gV; a.gmean = gmean; a.gspread = gspread;                                      \
    return poisson_fwdbwd<T>(a, gW, ll, ws, (size_t)ws_bytes, (cudaStream_t)stream);                                   \
  }                                                                                                                    \
  extern "C" int gpz_poisson_rate_##SUF(const T* W, int w_softplus, const T* V, const int64_t* idx, const T* Fs,       \
                                        T* rate, int G, int F, int B, int E, void* stream) {                           \
    if (B == 0 || G == 0 || E == 0) return GPZ_OK;                                                                     \
    poisson_rate_kernel<T><<<dim3((unsigned)cdiv(B, 128), (unsigned)cdiv(G, 32), E), 128, 0, (cudaStream_t)stream>>>(  \
        W, w_softplus, V, idx, Fs, rate, G, F, B, E);                                                                  \
    GPZ_CHECK_LAUNCH();                                                                                                \
    return GPZ_OK;                                                                                                     \
  }

GPZ_POISSON_IMPL(f32, float)
GPZ_POISSON_IMPL(f64, double)

// counts stored as uint8 / int16 / int32 (y_kind 1 / 2 / 3; 0 = float): same outputs and workspace as gpz_poisson_fwdbwd_f32
extern "C" int gpz_poisson_fwdbwd_yt_f32(const void* y, int y_kind, int64_t y_ld, const int64_t* idx, const float* W, int w_softplus,
                                         const float* V, const float* mean, const float* spread, const float* eps, int G, int F, int B,
                                         int E, int n_var, float clamp_min, int with_lgamma, double* ll, float* gW, float* gV,
                                         float* gmean, float* gspread, void* ws, int64_t ws_bytes, void* stream) {
  PoissonArgs<float> a;
  a.y = reinterpret_cast<const float*>(y); a.y_ld = y_ld; a.idx = idx; a.W = W; a.w_softplus = w_softplus; a.V = V; a.mean = mean;
  a.spread = spread; a.eps = eps; a.G = G; a.F = F; a.B = B; a.E = E; a.n_var = n_var; a.clamp_min = clamp_min;
  a.with_lgamma = with_lgamma; a.gV = gV; a.gmean = gmean; a.gspread = gspread;
  return poisson_fwdbwd<float>(a, gW, ll, ws, (size_t)ws_bytes, (cudaStream_t)stream, y_kind);
}

// K7-NB: the Poisson arguments plus D (G, raw dispersion) and the output gD (G)
template <typename T>
static NegBinArgs<T> negbin_args(const T* y, int64_t y_ld, const int64_t* idx, const T* W, int w_softplus, const T* V, const T* D,
                                 const T* mean, const T* spread, const T* eps, int G, int F, int B, int E, int n_var, T clamp_min,
                                 int with_lgamma, T* gV, T* gD, T* gmean, T* gspread) {
  NegBinArgs<T> a;
  a.y = y; a.y_ld = y_ld; a.idx = idx; a.W = W; a.w_softplus = w_softplus; a.V = V; a.mean = mean;
  a.spread = spread; a.eps = eps; a.G = G; a.F = F; a.B = B; a.E = E; a.n_var = n_var; a.clamp_min = clamp_min;
  a.with_lgamma = with_lgamma; a.gV = gV; a.gmean = gmean; a.gspread = gspread;
  a.D = D; a.gD = gD;
  return a;
}

#define GPZ_NEGBIN_IMPL(SUF, T)                                                                                        \
  extern "C" int64_t gpz_negbin_workspace_bytes_##SUF(int G, int F, int B, int E) {                                    \
    int nbx, nby, gpc;                                                                                                 \
    poisson_grid(G, F, B, sizeof(T) == 4, &nbx, &nby, &gpc);                                                           \
    return (int64_t)negbin_ws_bytes(G, F, B, E, sizeof(T) == 4, sizeof(T), nbx, nby);                                  \
  }                                                                                                                    \
  extern "C" int gpz_negbin_fwdbwd_##SUF(const T* y, int64_t y_ld, const int64_t* idx, const T* W, int w_softplus,     \
                                         const T* V, const T* D, const T* mean, const T* spread, const T* eps, int G,  \
                                         int F, int B, int E, int n_var, T clamp_min, int with_lgamma, double* ll,     \
                                         T* gW, T* gV, T* gD, T* gmean, T* gspread, void* ws, int64_t ws_bytes,        \
                                         void* stream) {                                                               \
    const NegBinArgs<T> a = negbin_args<T>(y, y_ld, idx, W, w_softplus, V, D, mean, spread, eps, G, F, B, E, n_var,    \
                                           clamp_min, with_lgamma, gV, gD, gmean, gspread);                            \
    return poisson_fwdbwd<T>(a, gW, ll, ws, (size_t)ws_bytes, (cudaStream_t)stream);                                   \
  }

GPZ_NEGBIN_IMPL(f32, float)
GPZ_NEGBIN_IMPL(f64, double)

extern "C" int gpz_negbin_fwdbwd_yt_f32(const void* y, int y_kind, int64_t y_ld, const int64_t* idx, const float* W, int w_softplus,
                                        const float* V, const float* D, const float* mean, const float* spread, const float* eps, int G,
                                        int F, int B, int E, int n_var, float clamp_min, int with_lgamma, double* ll, float* gW,
                                        float* gV, float* gD, float* gmean, float* gspread, void* ws, int64_t ws_bytes, void* stream) {
  const NegBinArgs<float> a = negbin_args<float>(reinterpret_cast<const float*>(y), y_ld, idx, W, w_softplus, V, D, mean, spread, eps,
                                                 G, F, B, E, n_var, clamp_min, with_lgamma, gV, gD, gmean, gspread);
  return poisson_fwdbwd<float>(a, gW, ll, ws, (size_t)ws_bytes, (cudaStream_t)stream, y_kind);
}

namespace gpz {
__global__ void digamma_kernel(const double* __restrict__ x, double* __restrict__ out, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = nb_digamma(x[i]);
}
__global__ void lgamma_kernel(const double* __restrict__ x, double* __restrict__ out, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = nb_lgamma(x[i]);
}
}  // namespace gpz

// the NB kernels' own digamma / lgamma (x > 0), element-wise, for testing them against a reference
extern "C" int gpz_digamma_f64(const double* x, double* out, int64_t n, void* stream) {
  if (n <= 0) return GPZ_OK;
  digamma_kernel<<<(unsigned)cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>(x, out, n);
  GPZ_CHECK_LAUNCH();
  return GPZ_OK;
}
extern "C" int gpz_lgamma_f64(const double* x, double* out, int64_t n, void* stream) {
  if (n <= 0) return GPZ_OK;
  lgamma_kernel<<<(unsigned)cdiv(n, 256), 256, 0, (cudaStream_t)stream>>>(x, out, n);
  GPZ_CHECK_LAUNCH();
  return GPZ_OK;
}

// sparse counts (K7-CSC): count_kind 0 = T, 1 = uint8, 2 = int16, 3 = int32
#define GPZ_POISSON_CSC_IMPL(SUF, T)                                                                                    \
  extern "C" int64_t gpz_poisson_csc_workspace_bytes_##SUF(int G, int F, int B, int E) {                                \
    (void)E;                                                                                                            \
    return (int64_t)csc_ws_bytes(G, F, B, sizeof(T));                                                                   \
  }                                                                                                                     \
  extern "C" int gpz_poisson_fwdbwd_csc_##SUF(const int64_t* indptr, const int32_t* genes, const void* counts,          \
                                              int count_kind, int64_t n_total, const int64_t* idx, const T* W,           \
                                              int w_softplus, const T* V, const T* mean, const T* spread, const T* eps,  \
                                              int G, int F, int B, int E, int n_var, T clamp_min, int with_lgamma,       \
                                              double* ll, T* gW, T* gV, T* gmean, T* gspread, void* ws, int64_t ws_bytes, \
                                              void* stream) {                                                            \
    CscArgs<T> a;                                                                                                       \
    a.indptr = indptr; a.genes = genes; a.values = counts; a.idx = idx; a.W = W; a.w_softplus = w_softplus; a.V = V;   \
    a.mean = mean; a.spread = spread; a.eps = eps; a.G = G; a.F = F; a.B = B; a.E = E; a.n_var = n_var;                 \
    a.clamp_min = clamp_min; a.with_lgamma = with_lgamma; a.gV = gV; a.gmean = gmean; a.gspread = gspread;              \
    return poisson_fwdbwd_csc<T>(a, count_kind, n_total, gW, ll, ws, (size_t)ws_bytes, (cudaStream_t)stream);          \
  }

GPZ_POISSON_CSC_IMPL(f32, float)
GPZ_POISSON_CSC_IMPL(f64, double)
