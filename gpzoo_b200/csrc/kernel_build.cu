// K1: fused pairwise-distance + covariance kernel-matrix build and its backward.
//
// Replaces  torch.cdist(X,Z)**2 -> expand(L) -> /l^2 -> exp -> *sigma^2   (kernels.py:114-130, 141-155)
// and the multi-group form with group-distance scaling (kernels.py:172-191, 204-228); the covariance kinds and their formulas are
// listed once, with their code, in the block below.
// d^2 is a direct sum of squared differences (never |x|^2+|z|^2-2xz), which is
// what makes fp32 results track the fp64 reference (SURVEY.md §0).  Output layout L x n1 x n2, n2 contiguous.
// HBM-bound: one pass writes 4*L*n1*n2 bytes; each thread owns 4 consecutive j and streams float4 stores.
#include <climits>
#include <type_traits>

#include "common.cuh"
#include "gpzoo_b200.h"
#include "umma_gemm.h"

namespace gpz {

constexpr int KB_DMAX = 4;      // spatial dimension supported by the kernels (reference uses D = 1 or 2)
constexpr int KB_LMAX = 32;     // factors handled per launch by the backward (host loops over chunks)
constexpr int KB_ROWS = 16;     // rows (i) per CTA
constexpr int KB_THREADS = 256;
constexpr int KB_VEC = 4;       // consecutive j per thread
constexpr int KB_GMAX = 64;     // max number of groups (r2 table kept in shared memory)

template <typename T> struct KBArgs {
  const T* x1; const T* x2;         // n1 x D, n2 x D
  const T* sigma; const T* ls;      // L
  const T* a;                       // L  group-difference coefficient (already squared / abs'd by the host); MG only
  const T* r2;                      // ng x ng squared embedding distances; MG only
  const int64_t* g1; const int64_t* g2;
  int n1, n2, D, L, ng;
  T p_half;                         // input_dim / 2
  T jitter;                         // added to K[l,i,i] (add_jitter, utilities.py:407-418); 0 for cross matrices
  int kind;                         // 0: RBF (squared exponential); 1 / 2 / 3: Matern-3/2 / -1/2 / -5/2, no groups
};

// ---- The covariance kinds.  Everything kind-specific lives in this block: a kind is added here and in the host dispatch
// (kb_dispatch_kind), nowhere else.  r = |x1_i - x2_j|, d2 = r^2:
//
//   kind 0, RBF:  K[l,i,j] = sigma_l^2 exp(-0.5 d2 / (ls_l^2 den)) / den^(p/2),  den = a_l r2[g1_i, g2_j] + 1 with groups,
//                 den = 1 without (p/2 = p_half, input_dim / 2)
//   kind 1, Matern-3/2 (kernels.py:6-30, batched_Matern32):  K[l,i,j] = sigma_l^2 (1 + v) exp(-v),            v = sqrt(3) r / ls_l
//   kind 2, Matern-1/2 (exponential, batched_Matern12):        K[l,i,j] = sigma_l^2 exp(-v),                  v = r / ls_l
//   kind 3, Matern-5/2 (batched_Matern52):                     K[l,i,j] = sigma_l^2 (1 + v + v^2/3) exp(-v),  v = sqrt(5) r / ls_l
//
// Only the RBF has a multi-group form (as in the reference).  The backward needs K0 (K without jitter) and the slope u with
// dK/dx1 = -u (x1 - x2); with e = sigma^2 exp(-v) for the Matern kinds:
//   kind 0:  u = K0 / (ls^2 den)
//   kind 1:  K0 = (1 + v) e,            u = (3 / ls^2) e                 (finite at r = 0)
//   kind 2:  K0 = e,                    u = e / (ls r), 0 at r = 0        (the sub-gradient 0 at the cusp)
//   kind 3:  K0 = (1 + v + v^2/3) e,    u = (5 / (3 ls^2)) (1 + v) e     (finite at r = 0)
//
// ARD (per-dimension lengthscales ls[l,d], no groups): every kind is evaluated at unit lengthscale on the scaled squared
// distance s2 = sum_d (x1_d - x2_d)^2 / ls[l,d]^2, which takes the place of d2 above.  With u from kb_terms at unit lengthscale
// (dK/ds2 = -u/2):  dK/dx1_d = -u (x1_d - x2_d) / ls_d^2,  dK/dls_d = u (x1_d - x2_d)^2 / ls_d^3.  Equal ls[l,d] give the
// isotropic kernel.

// s_c[l] of the kernels: -1/(2 ls^2) for the RBF, the factor of r in v for the Matern kinds
template <typename T, int KIND> __device__ __forceinline__ T kb_coeff(T ls) {
  return KIND == 1 ? Num<T>::sqrt(T(3)) / ls : KIND == 2 ? T(1) / ls : KIND == 3 ? Num<T>::sqrt(T(5)) / ls : T(-0.5) / (ls * ls);
}

// forward: K without jitter, exact functions; c = kb_coeff(ls_l), s2 = sigma_l^2; a_l and r2 are used with groups only
template <typename T, bool MG, int KIND>
__device__ __forceinline__ T kb_value(T c, T s2, T a_l, T r2, T d2, T p_half) {
  if (MG) {
    // one reciprocal per entry (MUFU.RCP in fp32: the two IEEE divisions held the multi-group build at 20 % of HBM peak)
    const T den = fma(a_l, r2, T(1));
    const T idn = fast_div(T(1), den);
    const T sc = p_half == T(1) ? idn : Num<T>::pow(den, -p_half);
    return s2 * Num<T>::exp(c * d2 * idn) * sc;
  } else if (KIND == 1) {
    const T vv = c * Num<T>::sqrt(d2);
    return s2 * (T(1) + vv) * Num<T>::exp(-vv);
  } else if (KIND == 2) {
    return s2 * Num<T>::exp(-c * Num<T>::sqrt(d2));
  } else if (KIND == 3) {
    const T vv = c * Num<T>::sqrt(d2);
    return s2 * fma(vv * T(1.0 / 3.0), vv, T(1) + vv) * Num<T>::exp(-vv);
  }
  return s2 * Num<T>::exp(c * d2);
}

// backward: K0, u times the upstream gradient g, and (groups) idn = 1/den.  The recomputed K uses the MUFU exponential in fp32
// (error ~1e-6 relative on entries that only enter sums with a 1e-4 parity tolerance; fp64 stays exact): the backward is
// issue-bound, not DRAM-bound, and expf's range reduction was a third of its instructions.
template <typename T> struct KBTerms { T k0, u, idn; };
template <typename T, bool MG, int KIND>
__device__ __forceinline__ KBTerms<T> kb_terms(T c, T s2, T a_l, T r2, T d2, T p_half, T g) {
  T k0, idn = T(1), ee = T(0), ir = T(0);
  if (MG) {
    const T den = fma(a_l, r2, T(1));
    idn = fast_div(T(1), den);
    const T sc = p_half == T(1) ? idn : Num<T>::pow(den, -p_half);
    k0 = s2 * fast_exp(c * d2 * idn) * sc;
  } else if (KIND == 1) {
    const T vv = c * Num<T>::sqrt(d2);
    ee = s2 * fast_exp(-vv);
    k0 = (T(1) + vv) * ee;
  } else if (KIND == 2) {
    ir = d2 > T(0) ? Num<T>::rsqrt(d2) : T(0);      // 1/r; 0 at r = 0 (a d2 below 1e-38 is 0 under -ftz)
    ee = s2 * fast_exp(-c * d2 * ir);               // r = d2 / r
    k0 = ee;
  } else if (KIND == 3) {
    const T vv = c * Num<T>::sqrt(d2);
    ee = s2 * fast_exp(-vv);
    ir = T(1) + vv;
    k0 = fma(vv * T(1.0 / 3.0), vv, ir) * ee;
  } else {
    k0 = s2 * fast_exp(c * d2);
  }
  const T gk = g * k0;
  const T u = KIND == 1 ? g * ee * c * c                        // G s2 exp(-v) 3 / ls^2
            : KIND == 2 ? gk * c * ir                           // G K0 / (ls r)
            : KIND == 3 ? g * ee * ir * c * c * T(1.0 / 3.0)    // G s2 (1 + v) exp(-v) 5 / (3 ls^2)
                        : gk * (T(-2) * c) * idn;               // G K0 / (ls^2 den)
  return {k0, u, idn};
}

// ---- Tile pieces shared by the kernels.

// ARD: 1/ls[l,d]^2 of factors l0 .. l0 + n - 1 into s_il2[l * KB_DMAX + d], 0 past D (a.ls is L x D)
template <typename T>
__device__ __forceinline__ void kb_stage_il2(const KBArgs<T>& a, int tid, int l0, int n, T* s_il2) {
  for (int e = tid; e < n * KB_DMAX; e += KB_THREADS) {
    const int l = e / KB_DMAX, d = e % KB_DMAX;
    const T ls = d < a.D ? a.ls[(int64_t)(l0 + l) * a.D + d] : T(1);
    s_il2[e] = d < a.D ? T(1) / (ls * ls) : T(0);
  }
}

// factors l0 .. l0 + n - 1 into shared memory (s_c = kb_coeff, s_s2 = sigma^2, s_a with groups) and, with groups, the r^2
// table, with ARD s_il2 (kb_coeff then at unit lengthscale); tid = threadIdx.x, the caller synchronises
template <typename T, bool MG, int KIND, bool ARD = false>
__device__ __forceinline__ void kb_stage(const KBArgs<T>& a, int tid, int l0, int n, T* s_c, T* s_s2, T* s_a, T* s_r2,
                                         T* s_il2 = nullptr) {
  if (ARD) kb_stage_il2(a, tid, l0, n, s_il2);
  for (int l = tid; l < n; l += KB_THREADS) {
    const T ls = ARD ? T(1) : a.ls[l0 + l], sg = a.sigma[l0 + l];
    s_c[l] = kb_coeff<T, KIND>(ls);
    s_s2[l] = sg * sg;
    if (MG) s_a[l] = a.a[l0 + l];
  }
  if (MG) for (int e = tid; e < a.ng * a.ng; e += KB_THREADS) s_r2[e] = a.r2[e];
}

// the thread's columns j0 .. j0 + nv - 1 (points and groups; zeros past nv and past D)
template <typename T, bool MG, int VEC>
__device__ __forceinline__ void kb_load_cols(const KBArgs<T>& a, int64_t j0, int nv, T (&xj)[KB_DMAX][VEC], int (&gj)[VEC]) {
#pragma unroll
  for (int v = 0; v < VEC; ++v) {
#pragma unroll
    for (int d = 0; d < KB_DMAX; ++d) xj[d][v] = (v < nv && d < a.D) ? a.x2[(j0 + v) * a.D + d] : T(0);
    gj[v] = (MG && v < nv) ? (int)a.g2[j0 + v] : 0;
  }
}

// squared distances of row i to the thread's columns
template <typename T, int VEC>
__device__ __forceinline__ void kb_row_d2(const KBArgs<T>& a, int i, const T (&xj)[KB_DMAX][VEC], T (&d2)[VEC]) {
#pragma unroll
  for (int v = 0; v < VEC; ++v) d2[v] = T(0);
#pragma unroll
  for (int d = 0; d < KB_DMAX; ++d) {
    if (d < a.D) {
      const T xi = a.x1[(int64_t)i * a.D + d];
#pragma unroll
      for (int v = 0; v < VEC; ++v) { const T df = xi - xj[d][v]; d2[v] = fma(df, df, d2[v]); }
    }
  }
}

// ARD: per-dimension squared differences of row i to the thread's columns (0 past D, where x2's columns are 0 as well)
template <typename T, int VEC>
__device__ __forceinline__ void kb_row_sq(const KBArgs<T>& a, int i, const T (&xj)[KB_DMAX][VEC], T (&sq)[KB_DMAX][VEC]) {
#pragma unroll
  for (int d = 0; d < KB_DMAX; ++d) {
    const T xi = d < a.D ? a.x1[(int64_t)i * a.D + d] : T(0);
#pragma unroll
    for (int v = 0; v < VEC; ++v) { const T df = xi - xj[d][v]; sq[d][v] = df * df; }
  }
}

// ARD: scaled squared distances s2 = sum_d sq_d il2_d of one factor (il2 = s_il2 + l * KB_DMAX).  KB_DMAX terms whatever D
// (sq and il2 are 0 past D): a switch on D per factor, measured, made the Matern kinds' forward slower still
template <typename T, int VEC>
__device__ __forceinline__ void kb_scaled_d2(const T* il2, const T (&sq)[KB_DMAX][VEC], T (&s2)[VEC]) {
  T w[KB_DMAX];
#pragma unroll
  for (int d = 0; d < KB_DMAX; ++d) w[d] = il2[d];
#pragma unroll
  for (int v = 0; v < VEC; ++v) {
    s2[v] = sq[0][v] * w[0];
#pragma unroll
    for (int d = 1; d < KB_DMAX; ++d) s2[v] = fma(sq[d][v], w[d], s2[v]);
  }
}

// group r^2 of row i and the thread's columns (groups only)
template <typename T, bool MG, int VEC>
__device__ __forceinline__ void kb_row_r2(const KBArgs<T>& a, int i, const T* s_r2, const int (&gj)[VEC], T (&r2)[VEC]) {
  if (MG) {
    const int gi = (int)a.g1[i];
#pragma unroll
    for (int v = 0; v < VEC; ++v) r2[v] = s_r2[gi * a.ng + gj[v]];
  }
}

template <typename T> struct Vec4 { T v[4]; };

// fp64 Matern-1/2: without a register target ptxas settles on 64 registers and spills; 3 CTAs per SM (<= 80 registers) keep
// it spill-free like Matern-3/2.  A min-blocks value of 0 is no bound at all, so every other instantiation compiles as before.
// ARD: per-dimension lengthscales (see the kinds block); the row keeps its per-dimension squared differences, s2 per factor.
// Those take ~20 more registers, and the 3-CTA bound made the fp64 ARD Matern-1/2 spill, so ARD has no bound.
template <typename T, bool MG, bool ALIGNED, int KIND = 0, bool ARD = false>
__global__ void __launch_bounds__(KB_THREADS, (KIND == 2 && sizeof(T) == 8 && !ARD) ? 3 : 0) kbuild_fwd_kernel(const KBArgs<T> a, T* __restrict__ out, T* __restrict__ out_lo) {
  __shared__ T s_c[KB_LMAX * 8], s_s2[KB_LMAX * 8], s_a[KB_LMAX * 8];
  __shared__ T s_r2[MG ? KB_GMAX * KB_GMAX : 1];
  __shared__ __align__(16) T s_il2[ARD ? KB_LMAX * 8 * KB_DMAX : 1];
  const int tid = threadIdx.x;
  kb_stage<T, MG, KIND, ARD>(a, tid, 0, a.L, s_c, s_s2, s_a, s_r2, s_il2);
  __syncthreads();

  const int64_t j0 = ((int64_t)blockIdx.x * KB_THREADS + tid) * KB_VEC;
  if (j0 >= a.n2) return;
  const int nv = (int)min((int64_t)KB_VEC, a.n2 - j0);
  T xj[KB_DMAX][KB_VEC];
  int gj[KB_VEC];
  kb_load_cols<T, MG>(a, j0, nv, xj, gj);
  const int i0 = blockIdx.y * KB_ROWS, i1 = min(i0 + KB_ROWS, a.n1);
  for (int i = i0; i < i1; ++i) {
    T d2[KB_VEC], r2[KB_VEC], sq[ARD ? KB_DMAX : 1][KB_VEC];
    if constexpr (ARD) kb_row_sq(a, i, xj, sq);
    else kb_row_d2(a, i, xj, d2);
    kb_row_r2<T, MG>(a, i, s_r2, gj, r2);
    for (int l = 0; l < a.L; ++l) {
      const T c = s_c[l], s2 = s_s2[l];
      if constexpr (ARD) kb_scaled_d2(s_il2 + l * KB_DMAX, sq, d2);
      Vec4<T> k;
#pragma unroll
      for (int v = 0; v < KB_VEC; ++v) {
        T val = kb_value<T, MG, KIND>(c, s2, MG ? s_a[l] : T(0), MG ? r2[v] : T(0), d2[v], a.p_half);
        if (a.jitter != T(0) && (int64_t)i == j0 + v) val += a.jitter;
        k.v[v] = val;
      }
      T* o = out + ((int64_t)l * a.n1 + i) * a.n2 + j0;
      if (ALIGNED && nv == KB_VEC) {
        if (sizeof(T) == 4) {
          __stcs(reinterpret_cast<float4*>(o), make_float4((float)k.v[0], (float)k.v[1], (float)k.v[2], (float)k.v[3]));
        } else {
          __stcs(reinterpret_cast<double2*>(o), make_double2((double)k.v[0], (double)k.v[1]));
          __stcs(reinterpret_cast<double2*>(o) + 1, make_double2((double)k.v[2], (double)k.v[3]));
        }
      } else {
        for (int v = 0; v < nv; ++v) o[v] = k.v[v];
      }
      if (sizeof(T) == 4 && out_lo != nullptr) {          // lo = x - tf32_trunc(x): second operand of the split-TF32 GEMMs
        float lo[KB_VEC];
#pragma unroll
        for (int v = 0; v < KB_VEC; ++v) {
          const float x = (float)k.v[v];
          lo[v] = x - __uint_as_float(__float_as_uint(x) & 0xFFFFE000u);
        }
        float* ol = reinterpret_cast<float*>(out_lo) + ((int64_t)l * a.n1 + i) * a.n2 + j0;
        if (ALIGNED && nv == KB_VEC) __stcs(reinterpret_cast<float4*>(ol), make_float4(lo[0], lo[1], lo[2], lo[3]));
        else for (int v = 0; v < nv; ++v) ol[v] = lo[v];
      }
    }
  }
}

// fp32 build written directly as the fp16 operand planes of the split-FP16 tensor-core GEMMs (csrc/umma_gemm.cu):
// out_h + out_l ~= K * scale[l], scale[l] = the power of two that puts sigma_l^2 (+|jitter|), the largest possible entry,
// in (2^14, 2^15].  4 bytes per entry leave the SM (half of K + lo plane in fp32); each thread owns 8 consecutive j and
// streams one 16-byte store per plane, row and factor.
constexpr int KB_VEC8 = 8;
template <bool MG, int KIND = 0, bool ARD = false>
__global__ void __launch_bounds__(KB_THREADS) kbuild_fwd_h_kernel(const KBArgs<float> a, __half* __restrict__ out_h,
                                                                  __half* __restrict__ out_l, float* __restrict__ out_scale) {
  __shared__ float s_c[KB_LMAX * 8], s_s2[KB_LMAX * 8], s_a[KB_LMAX * 8], s_sc[KB_LMAX * 8];
  __shared__ float s_r2[MG ? KB_GMAX * KB_GMAX : 1];
  __shared__ __align__(16) float s_il2[ARD ? KB_LMAX * 8 * KB_DMAX : 1];
  // kb_stage's loop with s_sc and out_scale: written out, since a per-factor hook inside kb_stage reschedules the multi-group kernel
  const int tid = threadIdx.x;
  if (ARD) kb_stage_il2(a, tid, 0, a.L, s_il2);
  for (int l = tid; l < a.L; l += KB_THREADS) {
    const float ls = ARD ? 1.f : a.ls[l], sg = a.sigma[l];
    s_c[l] = kb_coeff<float, KIND>(ls);
    s_s2[l] = sg * sg;
    s_sc[l] = gpz_pow2_scale(sg * sg + fabsf(a.jitter));
    if (MG) s_a[l] = a.a[l];
    if (blockIdx.x == 0 && blockIdx.y == 0) out_scale[l] = s_sc[l];
  }
  if (MG) for (int e = tid; e < a.ng * a.ng; e += KB_THREADS) s_r2[e] = a.r2[e];
  __syncthreads();

  const int64_t j0 = ((int64_t)blockIdx.x * KB_THREADS + tid) * KB_VEC8;
  if (j0 >= a.n2) return;                        // n2 % 8 == 0 (checked by the host): whole vectors only
  float xj[KB_DMAX][KB_VEC8];
  int gj[KB_VEC8];
  kb_load_cols<float, MG>(a, j0, KB_VEC8, xj, gj);
  const int i0 = blockIdx.y * KB_ROWS, i1 = min(i0 + KB_ROWS, a.n1);
  for (int i = i0; i < i1; ++i) {
    float d2[KB_VEC8], r2[KB_VEC8], sq[ARD ? KB_DMAX : 1][KB_VEC8];
    if constexpr (ARD) kb_row_sq(a, i, xj, sq);
    else kb_row_d2(a, i, xj, d2);
    kb_row_r2<float, MG>(a, i, s_r2, gj, r2);
    for (int l = 0; l < a.L; ++l) {
      const float c = s_c[l], s2 = s_s2[l], sc = s_sc[l];
      if constexpr (ARD) kb_scaled_d2(s_il2 + l * KB_DMAX, sq, d2);
      float k[KB_VEC8];
#pragma unroll
      for (int v = 0; v < KB_VEC8; ++v) {
        float val = kb_value<float, MG, KIND>(c, s2, MG ? s_a[l] : 0.f, MG ? r2[v] : 0.f, d2[v], a.p_half);
        if (a.jitter != 0.f && (int64_t)i == j0 + v) val += a.jitter;
        k[v] = val * sc;
      }
      uint4 h, lo;
      { const __half2 hh = __floats2half2_rn(k[0], k[1]); const float2 f = __half22float2(hh);
        const __half2 ll = __floats2half2_rn(k[0] - f.x, k[1] - f.y);
        h.x = *reinterpret_cast<const uint32_t*>(&hh); lo.x = *reinterpret_cast<const uint32_t*>(&ll); }
      { const __half2 hh = __floats2half2_rn(k[2], k[3]); const float2 f = __half22float2(hh);
        const __half2 ll = __floats2half2_rn(k[2] - f.x, k[3] - f.y);
        h.y = *reinterpret_cast<const uint32_t*>(&hh); lo.y = *reinterpret_cast<const uint32_t*>(&ll); }
      { const __half2 hh = __floats2half2_rn(k[4], k[5]); const float2 f = __half22float2(hh);
        const __half2 ll = __floats2half2_rn(k[4] - f.x, k[5] - f.y);
        h.z = *reinterpret_cast<const uint32_t*>(&hh); lo.z = *reinterpret_cast<const uint32_t*>(&ll); }
      { const __half2 hh = __floats2half2_rn(k[6], k[7]); const float2 f = __half22float2(hh);
        const __half2 ll = __floats2half2_rn(k[6] - f.x, k[7] - f.y);
        h.w = *reinterpret_cast<const uint32_t*>(&hh); lo.w = *reinterpret_cast<const uint32_t*>(&ll); }
      const int64_t o = ((int64_t)l * a.n1 + i) * a.n2 + j0;
      __stcs(reinterpret_cast<uint4*>(out_h + o), h);
      __stcs(reinterpret_cast<uint4*>(out_l + o), lo);
    }
  }
}

// Backward: given G = dLoss/dK (L x n1 x n2) recompute K0 (K without jitter) and, with u from kb_terms, reduce
//   g_sigma[l] += (2/sigma_l) sum G K0
//   g_ls[l]    += sum G u d2 / ls
//   g_a[l]     += sum G K0 (0.5 d2/(ls^2 den^2) - p_half/den) r2             (MG)
//   g_x1[i,:]  -= sum_{l,j} G u (x1_i - x2_j) ;  g_x2[j,:] += same
// One CTA covers KB_ROWS rows x (KB_THREADS*4) columns; the L accumulators live in registers.
// The position gradients stay products of u with the direct differences: |u (x1 - x2)| <= K0 / ls for Matern-1/2, so
// near-coincident points are harmless (an x1 sum(u) - sum(u x2) form would cancel catastrophically).
// ARD: u at unit lengthscale on s2; g_ls (L x D) += sum G u (x1_d - x2_d)^2 (later divided by ls_d^3), and the position
// weights are per dimension, w_d = sum_l G u / ls[l,d]^2.
template <typename T, bool MG, bool ALIGNED, int LMAX, int KIND = 0, bool ARD = false>
__global__ void __launch_bounds__(KB_THREADS, (sizeof(T) == 4 && LMAX <= 12) ? 2 : 1) kbuild_bwd_kernel(const KBArgs<T> a, const T* __restrict__ G, int l0, int Lc,
                                                                 double* __restrict__ g_x1, T* __restrict__ g_x2,
                                                                 double* __restrict__ g_sigma, double* __restrict__ g_ls,
                                                                 double* __restrict__ g_a) {
  __shared__ T s_c[LMAX], s_s2[LMAX], s_a[LMAX];
  __shared__ T s_r2[MG ? KB_GMAX * KB_GMAX : 1];
  __shared__ double s_red[32];
  __shared__ T s_row[KB_ROWS][KB_DMAX][KB_THREADS / 32];
  __shared__ __align__(16) T s_il2[ARD ? LMAX * KB_DMAX : 1];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  kb_stage<T, MG, KIND, ARD>(a, tid, l0, Lc, s_c, s_s2, s_a, s_r2, s_il2);
  __syncthreads();

  const int64_t j0 = ((int64_t)blockIdx.x * KB_THREADS + tid) * KB_VEC;
  const int nv = j0 < a.n2 ? (int)min((int64_t)KB_VEC, a.n2 - j0) : 0;
  T xj[KB_DMAX][KB_VEC];
  int gj[KB_VEC];
  kb_load_cols<T, MG>(a, j0, nv, xj, gj);
  T acc_s[LMAX], acc_l[LMAX], acc_a[MG ? LMAX : 1];
#pragma unroll
  for (int l = 0; l < LMAX; ++l) { acc_s[l] = T(0); acc_l[l] = T(0); if (MG) acc_a[l] = T(0); }
  T acc_d[ARD ? LMAX : 1][KB_DMAX];                    // ARD: sum G u (x1_d - x2_d)^2 per factor and dimension
  if constexpr (ARD) {
#pragma unroll
    for (int l = 0; l < LMAX; ++l)
#pragma unroll
      for (int d = 0; d < KB_DMAX; ++d) acc_d[l][d] = T(0);
  }
  T gx2[KB_DMAX][KB_VEC];
#pragma unroll
  for (int d = 0; d < KB_DMAX; ++d)
#pragma unroll
    for (int v = 0; v < KB_VEC; ++v) gx2[d][v] = T(0);

  const int i0 = blockIdx.y * KB_ROWS, i1 = min(i0 + KB_ROWS, a.n1);
  for (int i = i0; i < i1; ++i) {
    T df[KB_DMAX][KB_VEC], d2[KB_VEC], r2[KB_VEC], w[KB_VEC];   // w = sum_l G u
    T wd[KB_DMAX][KB_VEC];                                       // ARD: w_d = sum_l G u / ls[l,d]^2
#pragma unroll
    for (int v = 0; v < KB_VEC; ++v) { d2[v] = T(0); w[v] = T(0); r2[v] = T(0); }
    if constexpr (ARD) {
#pragma unroll
      for (int d = 0; d < KB_DMAX; ++d)
#pragma unroll
        for (int v = 0; v < KB_VEC; ++v) wd[d][v] = T(0);
    }
#pragma unroll
    for (int d = 0; d < KB_DMAX; ++d) {
      const T xi = d < a.D ? a.x1[(int64_t)i * a.D + d] : T(0);
#pragma unroll
      for (int v = 0; v < KB_VEC; ++v) { df[d][v] = xi - xj[d][v]; d2[v] = fma(df[d][v], df[d][v], d2[v]); }
    }
    kb_row_r2<T, MG>(a, i, s_r2, gj, r2);
    if (nv > 0) {
      // phase 1: issue every load of this row (one 16-byte vector per factor) before any is used
      T g[LMAX][KB_VEC];
#pragma unroll
      for (int l = 0; l < LMAX; ++l) {
        const T* gp = G + ((int64_t)(l0 + (l < Lc ? l : 0)) * a.n1 + i) * a.n2 + j0;
        if (ALIGNED && nv == KB_VEC) {
          if (sizeof(T) == 4) {
            const float4 t = __ldcs(reinterpret_cast<const float4*>(gp));
            g[l][0] = t.x; g[l][1] = t.y; g[l][2] = t.z; g[l][3] = t.w;
          } else {
            const double2 t0 = __ldcs(reinterpret_cast<const double2*>(gp));
            const double2 t1 = __ldcs(reinterpret_cast<const double2*>(gp) + 1);
            g[l][0] = t0.x; g[l][1] = t0.y; g[l][2] = t1.x; g[l][3] = t1.y;
          }
        } else {
#pragma unroll
          for (int v = 0; v < KB_VEC; ++v) g[l][v] = v < nv ? gp[v] : T(0);
        }
      }
      // phase 2: recompute K and accumulate
#pragma unroll
      for (int l = 0; l < LMAX; ++l) {
        if constexpr (ARD) {
          if (l >= Lc) continue;
          // the squared differences are formed again per factor: kept per row, their registers made the fp32 kernels spill
          T il2[KB_DMAX];
#pragma unroll
          for (int d = 0; d < KB_DMAX; ++d) il2[d] = s_il2[l * KB_DMAX + d];
#pragma unroll
          for (int v = 0; v < KB_VEC; ++v) {
            T s2d = df[0][v] * il2[0] * df[0][v];
#pragma unroll
            for (int d = 1; d < KB_DMAX; ++d) s2d = fma(df[d][v] * il2[d], df[d][v], s2d);
            const KBTerms<T> t = kb_terms<T, false, KIND>(s_c[l], s_s2[l], T(0), T(0), s2d, a.p_half, g[l][v]);
            acc_s[l] = fma(g[l][v], t.k0, acc_s[l]);
#pragma unroll
            for (int d = 0; d < KB_DMAX; ++d) {
              acc_d[l][d] = fma(t.u * df[d][v], df[d][v], acc_d[l][d]);
              wd[d][v] = fma(t.u, il2[d], wd[d][v]);
            }
          }
        } else if (l < Lc) {
          const T c = s_c[l], s2 = s_s2[l];
#pragma unroll
          for (int v = 0; v < KB_VEC; ++v) {
            const KBTerms<T> t = kb_terms<T, MG, KIND>(c, s2, MG ? s_a[l] : T(0), r2[v], d2[v], a.p_half, g[l][v]);
            const T gk = g[l][v] * t.k0;
            acc_s[l] += gk;
            acc_l[l] = fma(t.u, d2[v], acc_l[l]);          // later divided by ls
            if (MG) acc_a[l] = fma(gk * r2[v], (T(-1) * c * d2[v] * t.idn - a.p_half) * t.idn, acc_a[l]);
            w[v] += t.u;
          }
        }
      }
    }
    // row reduction for g_x1[i,:]
#pragma unroll
    for (int d = 0; d < KB_DMAX; ++d) {
      if (d < a.D) {
        T r = T(0);
#pragma unroll
        for (int v = 0; v < KB_VEC; ++v) {
          const T wv = ARD ? wd[d][v] : w[v];
          r = fma(wv, df[d][v], r); gx2[d][v] = fma(wv, df[d][v], gx2[d][v]);
        }
        r = warp_sum(r);
        if (lane == 0) s_row[i - i0][d][warp] = r;
      }
    }
  }
  __syncthreads();
  if (g_x1 != nullptr) {
    for (int e = tid; e < (i1 - i0) * a.D; e += KB_THREADS) {
      const int ii = e / a.D, d = e % a.D;
      double r = 0.0;
#pragma unroll
      for (int wv = 0; wv < KB_THREADS / 32; ++wv) r += (double)s_row[ii][d][wv];
      atomicAdd(g_x1 + (int64_t)(i0 + ii) * a.D + d, -r);
    }
  }
  if (g_x2 != nullptr) {
    for (int v = 0; v < nv; ++v)
#pragma unroll
      for (int d = 0; d < KB_DMAX; ++d)
        if (d < a.D) atomicAdd(g_x2 + (j0 + v) * a.D + d, gx2[d][v]);
  }
#pragma unroll
  for (int l = 0; l < LMAX; ++l) {
    if (l < Lc) {                                   // uniform across the block
      double v = block_sum<double>((double)acc_s[l], s_red);
      if (tid == 0) atomicAdd(g_sigma + l0 + l, v);
      if constexpr (ARD) {
#pragma unroll
        for (int d = 0; d < KB_DMAX; ++d) {
          if (d < a.D) {
            v = block_sum<double>((double)acc_d[l][d], s_red);
            if (tid == 0) atomicAdd(g_ls + (int64_t)(l0 + l) * a.D + d, v);
          }
        }
      } else {
        v = block_sum<double>((double)acc_l[l], s_red);
        if (tid == 0) atomicAdd(g_ls + l0 + l, v);
        if (MG) {
          v = block_sum<double>((double)acc_a[l], s_red);
          if (tid == 0) atomicAdd(g_a + l0 + l, v);
        }
      }
    }
  }
}

// ARD: g_sigma = 2 S/sigma, g_ls[l,d] = Sl[l,d]/ls[l,d]^3 (LD = L * D entries), g_x1 = ws_x1
template <typename T>
__global__ void kbuild_bwd_ard_finalize_kernel(const double* __restrict__ ws, const T* __restrict__ sigma, const T* __restrict__ ls,
                                               int L, int LD, int n1D, T* __restrict__ g_sigma, T* __restrict__ g_ls,
                                               T* __restrict__ g_x1) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e < L) g_sigma[e] = (T)(2.0 * ws[e] / (double)sigma[e]);
  if (e < LD) { const double l = (double)ls[e]; g_ls[e] = (T)(ws[L + e] / (l * l * l)); }
  if (g_x1 != nullptr && e < n1D) g_x1[e] = (T)ws[L + LD + e];
}

// double accumulators -> outputs:  g_sigma = 2 S/sigma, g_ls = Sl/ls, g_a = Sa, g_x1 = ws_x1
template <typename T>
__global__ void kbuild_bwd_finalize_kernel(const double* __restrict__ ws, const T* __restrict__ sigma, const T* __restrict__ ls, int L,
                                           int n1D, T* __restrict__ g_sigma, T* __restrict__ g_ls, T* __restrict__ g_a,
                                           T* __restrict__ g_x1) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e < L) {
    g_sigma[e] = (T)(2.0 * ws[e] / (double)sigma[e]);
    g_ls[e] = (T)(ws[L + e] / (double)ls[e]);
    if (g_a != nullptr) g_a[e] = (T)ws[2 * L + e];
  }
  if (g_x1 != nullptr && e < n1D) g_x1[e] = (T)ws[3 * L + e];
}

// plain Euclidean distance matrix (n1 x n2) by direct differences: kernel(X, Z, return_distance=True)
// (kernels.py:118-124) without cdist's matmul path.
template <typename T>
__global__ void cdist_kernel(const T* __restrict__ x1, const T* __restrict__ x2, T* __restrict__ out, int n1, int n2, int D) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= (int64_t)n1 * n2) return;
  const int i = (int)(e / n2), j = (int)(e % n2);
  T d2 = T(0);
  for (int d = 0; d < D; ++d) { const T df = x1[(int64_t)i * D + d] - x2[(int64_t)j * D + d]; d2 = fma(df, df, d2); }
  out[e] = Num<T>::sqrt(d2);
}

// ---- Host dispatch: runtime values -> the compile-time parameters of the kernels.  Every instantiated kernel is reached here.
template <int V> using kb_int = std::integral_constant<int, V>;

// (kind, groups, ARD) -> f(std::bool_constant<MG>, kb_int<KIND>, std::bool_constant<ARD>) for the nine supported forms: the
// RBF with and without groups, the three Matern kinds (which have no multi-group form in the reference), and the four kinds
// with per-dimension lengthscales (no groups); GPZ_ERR_UNSUPPORTED for anything else
template <typename F> int kb_dispatch_kind(int kind, bool mg, bool ard, F&& f) {
  if (mg) return kind == 0 && !ard ? f(std::true_type{}, kb_int<0>{}, std::false_type{}) : GPZ_ERR_UNSUPPORTED;
  const auto with_ard = [&](auto kd) { return ard ? f(std::false_type{}, kd, std::true_type{}) : f(std::false_type{}, kd, std::false_type{}); };
  switch (kind) {
    case 0: return with_ard(kb_int<0>{});
    case 1: return with_ard(kb_int<1>{});
    case 2: return with_ard(kb_int<2>{});
    case 3: return with_ard(kb_int<3>{});
    default: return GPZ_ERR_UNSUPPORTED;
  }
}

template <typename F> int kb_dispatch_aligned(bool al, F&& f) { return al ? f(std::true_type{}) : f(std::false_type{}); }

// factors per backward launch: the RBF's register accumulators are sized to L (4 / 8 / 12 / 16, else KB_LMAX);
// the Matern kinds always take KB_LMAX.  ARD keeps 1 + KB_DMAX accumulators per factor: with 3 factors the fp32 kernels (two
// CTAs per SM, <= 128 registers) use 120-127 registers and do not spill; with 4 the Matern-3/2 and -5/2 ones spilled 8 B
constexpr int KB_LMAX_ARD = 3;
template <int KIND, bool ARD, typename F> int kb_dispatch_lmax(int L, F&& f) {
  if constexpr (ARD) return f(kb_int<KB_LMAX_ARD>{});
  else if constexpr (KIND != 0) return f(kb_int<KB_LMAX>{});
  else if (L <= 4) return f(kb_int<4>{});
  else if (L <= 8) return f(kb_int<8>{});
  else if (L <= 12) return f(kb_int<12>{});
  else if (L <= 16) return f(kb_int<16>{});
  else return f(kb_int<KB_LMAX>{});
}

// sizes every entry point supports: 1 <= D <= KB_DMAX, 1 <= L <= l_max, and 1..KB_GMAX groups when there are groups
template <typename T> bool kb_sizes_ok(const KBArgs<T>& a, int l_max) {
  return a.D >= 1 && a.D <= KB_DMAX && a.L >= 1 && a.L <= l_max && (a.g1 == nullptr || (a.ng >= 1 && a.ng <= KB_GMAX));
}

// ard: a.ls holds L x D per-dimension lengthscales (no groups)
template <typename T>
int kbuild_fwd(const KBArgs<T>& a, T* out, T* out_lo, cudaStream_t st, bool ard = false) {
  if (!kb_sizes_ok(a, KB_LMAX * 8)) return GPZ_ERR_UNSUPPORTED;
  if (a.n1 == 0 || a.n2 == 0) return GPZ_OK;
  const bool al = (a.n2 % KB_VEC == 0) && ((reinterpret_cast<uintptr_t>(out) & 31) == 0) &&
                  ((reinterpret_cast<uintptr_t>(out_lo) & 15) == 0);
  const dim3 grid((unsigned)cdiv(a.n2, (int64_t)KB_THREADS * KB_VEC), (unsigned)cdiv(a.n1, KB_ROWS));
  return kb_dispatch_kind(a.kind, a.g1 != nullptr, ard, [&](auto mg, auto kind, auto ardc) {
    return kb_dispatch_aligned(al, [&](auto aligned) {
      kbuild_fwd_kernel<T, decltype(mg)::value, decltype(aligned)::value, decltype(kind)::value, decltype(ardc)::value>
          <<<grid, KB_THREADS, 0, st>>>(a, out, out_lo);
      GPZ_CHECK_LAUNCH();
      return GPZ_OK;
    });
  });
}

// fp16-plane forward (fp32 arithmetic): see kbuild_fwd_h_kernel
int kbuild_fwd_h(const KBArgs<float>& a, void* out_h, void* out_l, float* out_scale, cudaStream_t st, bool ard = false) {
  if (!kb_sizes_ok(a, KB_LMAX * 8)) return GPZ_ERR_UNSUPPORTED;
  if (a.n2 % KB_VEC8 || (reinterpret_cast<uintptr_t>(out_h) & 15) || (reinterpret_cast<uintptr_t>(out_l) & 15)) return GPZ_ERR_UNSUPPORTED;
  if (a.n1 == 0 || a.n2 == 0) return GPZ_OK;
  const dim3 grid((unsigned)cdiv(a.n2, (int64_t)KB_THREADS * KB_VEC8), (unsigned)cdiv(a.n1, KB_ROWS));
  return kb_dispatch_kind(a.kind, a.g1 != nullptr, ard, [&](auto mg, auto kd, auto ardc) {
    kbuild_fwd_h_kernel<decltype(mg)::value, decltype(kd)::value, decltype(ardc)::value>
        <<<grid, KB_THREADS, 0, st>>>(a, (__half*)out_h, (__half*)out_l, out_scale);
    GPZ_CHECK_LAUNCH();
    return GPZ_OK;
  });
}

// ws: 3 L + n1 D doubles (sigma, ls, a, x1 sums); with ard L + L D + n1 D (sigma, the L x D ls sums, x1)
template <typename T>
int kbuild_bwd(const KBArgs<T>& a, const T* G, T* g_x1, T* g_x2, T* g_sigma, T* g_ls, T* g_a, double* ws, cudaStream_t st,
               bool ard = false) {
  if (!kb_sizes_ok(a, INT_MAX)) return GPZ_ERR_UNSUPPORTED;
  const int n1D = a.n1 * a.D, nls = ard ? a.L * a.D : a.L;
  GPZ_CUDA(cudaMemsetAsync(ws, 0, sizeof(double) * ((ard ? 1 : 2) * (size_t)a.L + nls + n1D), st));
  if (g_x2) GPZ_CUDA(cudaMemsetAsync(g_x2, 0, sizeof(T) * a.n2 * a.D, st));
  double* w_sigma = ws; double* w_ls = ws + a.L; double* w_a = ws + 2 * a.L;
  double* w_x1 = ard ? ws + a.L + nls : ws + 3 * a.L;
  if (a.n1 > 0 && a.n2 > 0) {
    const bool al = (a.n2 % KB_VEC == 0) && ((reinterpret_cast<uintptr_t>(G) & 31) == 0);
    const dim3 grid((unsigned)cdiv(a.n2, (int64_t)KB_THREADS * KB_VEC), (unsigned)cdiv(a.n1, KB_ROWS));
    const int rc = kb_dispatch_kind(a.kind, a.g1 != nullptr, ard, [&](auto mg, auto kind, auto ardc) {
      return kb_dispatch_lmax<decltype(kind)::value, decltype(ardc)::value>(a.L, [&](auto lmax) {
        return kb_dispatch_aligned(al, [&](auto aligned) {
          constexpr int LMAX = decltype(lmax)::value;
          // g_x1/g_x2 accumulate over all l-chunks (atomics), so every chunk launch adds its share
          for (int l0 = 0; l0 < a.L; l0 += LMAX) {
            kbuild_bwd_kernel<T, decltype(mg)::value, decltype(aligned)::value, LMAX, decltype(kind)::value, decltype(ardc)::value>
                <<<grid, KB_THREADS, 0, st>>>(a, G, l0, min(LMAX, a.L - l0), w_x1, g_x2, w_sigma, w_ls, w_a);
            GPZ_CHECK_LAUNCH();
          }
          return GPZ_OK;
        });
      });
    });
    if (rc != GPZ_OK) return rc;
  }
  const int tot = max(nls, n1D);
  if (ard) kbuild_bwd_ard_finalize_kernel<T><<<(unsigned)cdiv(tot, 256), 256, 0, st>>>(ws, a.sigma, a.ls, a.L, nls, n1D, g_sigma, g_ls, g_x1);
  else kbuild_bwd_finalize_kernel<T><<<(unsigned)cdiv(tot, 256), 256, 0, st>>>(ws, a.sigma, a.ls, a.L, n1D, g_sigma, g_ls, g_a, g_x1);
  GPZ_CHECK_LAUNCH();
  return GPZ_OK;
}

}  // namespace gpz

using namespace gpz;

#define GPZ_KB_IMPL(SUF, T)                                                                                        \
  extern "C" int gpz_kernel_build_fwd_##SUF(const T* x1, const T* x2, const T* sigma, const T* ls, const T* a,     \
                                            const T* r2, const int64_t* g1, const int64_t* g2, int n1, int n2,     \
                                            int D, int L, int ng, int kind, T p_half, T jitter, T* out, T* out_lo, \
                                            void* stream) {                                                        \
    KBArgs<T> k{x1, x2, sigma, ls, a, r2, g1, g2, n1, n2, D, L, ng, p_half, jitter, kind};                         \
    return kbuild_fwd<T>(k, out, out_lo, (cudaStream_t)stream);                                                    \
  }                                                                                                                \
  extern "C" int gpz_kernel_build_bwd_##SUF(const T* x1, const T* x2, const T* sigma, const T* ls, const T* a,     \
                                            const T* r2, const int64_t* g1, const int64_t* g2, int n1, int n2,     \
                                            int D, int L, int ng, int kind, T p_half, const T* G, T* g_x1, T* g_x2, \
                                            T* g_sigma, T* g_ls, T* g_a, double* ws, void* stream) {               \
    KBArgs<T> k{x1, x2, sigma, ls, a, r2, g1, g2, n1, n2, D, L, ng, p_half, T(0), kind};                           \
    return kbuild_bwd<T>(k, G, g_x1, g_x2, g_sigma, g_ls, g_a, ws, (cudaStream_t)stream);                          \
  }                                                                                                                \
  extern "C" int gpz_kernel_build_ard_fwd_##SUF(const T* x1, const T* x2, const T* sigma, const T* ls, int n1,     \
                                                int n2, int D, int L, int kind, T jitter, T* out, T* out_lo,       \
                                                void* stream) {                                                    \
    KBArgs<T> k{x1, x2, sigma, ls, nullptr, nullptr, nullptr, nullptr, n1, n2, D, L, 0, T(1), jitter, kind};       \
    return kbuild_fwd<T>(k, out, out_lo, (cudaStream_t)stream, true);                                              \
  }                                                                                                                \
  extern "C" int gpz_kernel_build_ard_bwd_##SUF(const T* x1, const T* x2, const T* sigma, const T* ls, int n1,     \
                                                int n2, int D, int L, int kind, const T* G, T* g_x1, T* g_x2,      \
                                                T* g_sigma, T* g_ls, double* ws, void* stream) {                   \
    KBArgs<T> k{x1, x2, sigma, ls, nullptr, nullptr, nullptr, nullptr, n1, n2, D, L, 0, T(1), T(0), kind};         \
    return kbuild_bwd<T>(k, G, g_x1, g_x2, g_sigma, g_ls, nullptr, ws, (cudaStream_t)stream, true);                \
  }                                                                                                                \
  extern "C" int gpz_cdist_##SUF(const T* x1, const T* x2, T* out, int n1, int n2, int D, void* stream) {          \
    const int64_t total = (int64_t)n1 * n2;                                                                        \
    if (total == 0) return GPZ_OK;                                                                                 \
    cdist_kernel<T><<<(unsigned)cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(x1, x2, out, n1, n2, D);         \
    GPZ_CHECK_LAUNCH();                                                                                            \
    return GPZ_OK;                                                                                                 \
  }

GPZ_KB_IMPL(f32, float)
GPZ_KB_IMPL(f64, double)

extern "C" int gpz_kernel_build_fwd_h_f32(const float* x1, const float* x2, const float* sigma, const float* ls, const float* a,
                                          const float* r2, const int64_t* g1, const int64_t* g2, int n1, int n2, int D, int L,
                                          int ng, int kind, float p_half, float jitter, void* out_h, void* out_l,
                                          float* out_scale, void* stream) {
  const KBArgs<float> k{x1, x2, sigma, ls, a, r2, g1, g2, n1, n2, D, L, ng, p_half, jitter, kind};
  return kbuild_fwd_h(k, out_h, out_l, out_scale, (cudaStream_t)stream);
}

extern "C" int gpz_kernel_build_ard_fwd_h_f32(const float* x1, const float* x2, const float* sigma, const float* ls, int n1,
                                              int n2, int D, int L, int kind, float jitter, void* out_h, void* out_l,
                                              float* out_scale, void* stream) {
  const KBArgs<float> k{x1, x2, sigma, ls, nullptr, nullptr, nullptr, nullptr, n1, n2, D, L, 0, 1.f, jitter, kind};
  return kbuild_fwd_h(k, out_h, out_l, out_scale, (cudaStream_t)stream, true);
}
