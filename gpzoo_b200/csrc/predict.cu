// K3/K4: whitened triangular products and the fused SVGP predictive mean / variance.
//
// Reference (gp.py:218-225, utilities.py:382-397):  W^T = Kzz^-1 Kzx via cholesky_solve (two TRSMs),
// mean = W mu, cov = Kxx + sum((W (S - Kzz)) o W).  With Lc = chol(Kzz), Linv = Lc^-1, T = Linv Lu,
// q = Linv mu the same quantities are (SURVEY.md App. A.1, exact algebra):
//     A = Linv Kzx          (lower-triangular product  == TRSM  Lc A = Kzx)
//     C = T^T A             (upper-triangular product  == Lu^T Lc^-T A)
//     mean[n] = sum_m q[m] A[m,n]
//     var[n]  = Kxx[n] - sum_m A[m,n]^2 + sum_m C[m,n]^2
// which needs 2 M^2 N flops instead of 6 M^2 N and never forms S - Kzz (no cancellation).
//
// Backward (App. A.5), given gm = dL/dmean, gv = dL/dvar (L x N):
//     gC = 2 C diag(gv)                    gT   = tril(A gC^T)           gq = A gm
//     gA = T gC - 2 A diag(gv) + q gm^T    gKzx = Linv^T gA              gLinv = tril(gA Kzx^T)
//     gKxx = gv
#include "gemm_simt.cuh"
#include "gpzoo_b200.h"
#include "umma_gemm.h"

namespace gpz {

// mean / var column reductions over m.  One thread per column n, rows streamed coalesced.
template <typename T>
__global__ void __launch_bounds__(256) predict_reduce_kernel(const T* __restrict__ A, const T* __restrict__ C,
                                                              const T* __restrict__ q, const T* __restrict__ kxx,
                                                              T* __restrict__ mean, T* __restrict__ var, int M, int N) {
  extern __shared__ unsigned char smem_raw[];
  T* sq = reinterpret_cast<T*>(smem_raw);
  const int l = blockIdx.y;
  for (int m = threadIdx.x; m < M; m += blockDim.x) sq[m] = q[(int64_t)l * M + m];
  __syncthreads();
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  const T* a = A + (int64_t)l * M * N + n;
  const T* c = C + (int64_t)l * M * N + n;
  T mu = T(0), s_a = T(0), s_c = T(0);
#pragma unroll 4
  for (int m = 0; m < M; ++m) {
    const T av = a[(int64_t)m * N], cv = c[(int64_t)m * N];
    mu = fma(sq[m], av, mu);
    s_a = fma(av, av, s_a);
    s_c = fma(cv, cv, s_c);
  }
  mean[(int64_t)l * N + n] = mu;
  var[(int64_t)l * N + n] = kxx[(int64_t)l * N + n] - s_a + s_c;
}

// backward prologue, one pass over A and C:  C <- gC = 2 C gv ;  gA0 = -2 A gv + q gm^T
template <typename T>
__global__ void __launch_bounds__(256) predict_bwd_prep_kernel(const T* __restrict__ A, T* __restrict__ C, const T* __restrict__ q,
                                                                const T* __restrict__ gm, const T* __restrict__ gv,
                                                                T* __restrict__ gA, T* __restrict__ Clo, int M, int N,
                                                                int rows_per_cta) {
  const int l = blockIdx.z;
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  const T gmn = gm[(int64_t)l * N + n], gvn = gv[(int64_t)l * N + n];
  const int m0 = blockIdx.y * rows_per_cta, m1 = min(m0 + rows_per_cta, M);
  for (int m = m0; m < m1; ++m) {
    const int64_t e = ((int64_t)l * M + m) * N + n;
    const T av = A[e], cv = C[e];
    const T gc = T(2) * cv * gvn;
    C[e] = gc;
    if (sizeof(T) == 4 && Clo != nullptr) {
      const float x = (float)gc;
      reinterpret_cast<float*>(Clo)[e] = x - __uint_as_float(__float_as_uint(x) & 0xFFFFE000u);
    }
    gA[e] = fma(q[(int64_t)l * M + m], gmn, T(-2) * av * gvn);
  }
}

// out[l,m] = sum_n A[l,m,n] v[l,n]      (gq = A gm); one CTA per row, 4 independent accumulators per thread
template <typename T>
__global__ void __launch_bounds__(256) rowdot_kernel(const T* __restrict__ A, const T* __restrict__ v, T* __restrict__ out, int M, int N) {
  __shared__ T red[32];
  const int m = blockIdx.x, l = blockIdx.y;
  const T* a = A + ((int64_t)l * M + m) * N;
  const T* vv = v + (int64_t)l * N;
  T acc0 = T(0), acc1 = T(0), acc2 = T(0), acc3 = T(0);
  int n = threadIdx.x;
  for (; n + 3 * 256 < N; n += 4 * 256) {
    const T a0 = a[n], a1 = a[n + 256], a2 = a[n + 512], a3 = a[n + 768];
    acc0 = fma(a0, vv[n], acc0);
    acc1 = fma(a1, vv[n + 256], acc1);
    acc2 = fma(a2, vv[n + 512], acc2);
    acc3 = fma(a3, vv[n + 768], acc3);
  }
  for (; n < N; n += 256) acc0 = fma(a[n], vv[n], acc0);
  T acc = block_sum<T>((acc0 + acc1) + (acc2 + acc3), red);
  if (threadIdx.x == 0) out[(int64_t)l * M + m] = acc;
}

// out[l,j] = sum_k A[l,k,j] v[l,k]      (A^T v for row-major A): a CTA owns 32 columns, its 8 thread rows stride over k
template <typename T>
__global__ void __launch_bounds__(256) coldot_kernel(const T* __restrict__ A, const T* __restrict__ v, T* __restrict__ out, int K, int N) {
  __shared__ T red[8][33];
  const int l = blockIdx.y, tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int j = blockIdx.x * 32 + tx;
  const T* a = A + (int64_t)l * K * N + j;
  const T* vv = v + (int64_t)l * K;
  T acc0 = T(0), acc1 = T(0);
  if (j < N) {
    int k = ty;
    for (; k + 8 < K; k += 16) {
      acc0 = fma(a[(int64_t)k * N], vv[k], acc0);
      acc1 = fma(a[(int64_t)(k + 8) * N], vv[k + 8], acc1);
    }
    if (k < K) acc0 = fma(a[(int64_t)k * N], vv[k], acc0);
  }
  red[ty][tx] = acc0 + acc1;
  __syncthreads();
  if (ty == 0 && j < N) {
    T sacc = T(0);
#pragma unroll
    for (int r = 0; r < 8; ++r) sacc += red[r][tx];
    out[(int64_t)l * N + j] = sacc;
  }
}

template <typename T>
int predict_fwd(const T* Kzx, const T* Linv, const T* Tm, const T* q, const T* kxx, T* A, T* C, T* mean, T* var,
                int M, int N, int L, cudaStream_t st) {
  const int64_t sMM = (int64_t)M * M, sMN = (int64_t)M * N;
  int rc = gemm<T>(st, false, false, M, N, M, T(1), Linv, M, sMM, Kzx, N, sMN, T(0), A, N, sMN, L, 1, 0, 0);
  if (rc) return rc;
  rc = gemm<T>(st, true, false, M, N, M, T(1), Tm, M, sMM, A, N, sMN, T(0), C, N, sMN, L, 2, 0, 0);
  if (rc) return rc;
  predict_reduce_kernel<T><<<dim3((unsigned)cdiv(N, 256), L), 256, sizeof(T) * M, st>>>(A, C, q, kxx, mean, var, M, N);
  GPZ_CHECK_LAUNCH();
  return GPZ_OK;
}

// gT and gLinv must be zero-initialised by the caller (only their lower triangles are written, split-K atomics).
template <typename T>
int predict_bwd(const T* Kzx, const T* Linv, const T* Tm, const T* q, const T* A, T* C, const T* gm, const T* gv,
                T* gA, T* gKzx, T* gLinv, T* gT, T* gq, int M, int N, int L, cudaStream_t st) {
  const int64_t sMM = (int64_t)M * M, sMN = (int64_t)M * N;
  const int rows = 64;
  predict_bwd_prep_kernel<T><<<dim3((unsigned)cdiv(N, 256), (unsigned)cdiv(M, rows), L), 256, 0, st>>>(A, C, q, gm, gv, gA, (T*)nullptr, M, N, rows);
  GPZ_CHECK_LAUNCH();
  rowdot_kernel<T><<<dim3(M, L), 256, 0, st>>>(A, gm, gq, M, N);
  GPZ_CHECK_LAUNCH();
  // split the long reduction over the N spots so the small M x M outputs still fill the GPU
  int splitk = 1;
  {
    const int64_t tiles = cdiv(M, GemmCfg<T>::BM) * cdiv(M, GemmCfg<T>::BN) * L / 2 + 1;
    while (splitk < 16 && tiles * splitk < 148 * 4 && N / (splitk * 2) >= 512) splitk *= 2;
  }
  // gT = tril(A gC^T)
  int rc = gemm<T>(st, false, true, M, M, N, T(1), A, N, sMN, C, N, sMN, T(0), gT, M, sMM, L, 0, 0, 1, splitk > 1 ? splitk : 1);
  if (rc) return rc;
  // gA += T gC
  rc = gemm<T>(st, false, false, M, N, M, T(1), Tm, M, sMM, C, N, sMN, T(1), gA, N, sMN, L, 1, 0, 0);
  if (rc) return rc;
  // gKzx = Linv^T gA
  rc = gemm<T>(st, true, false, M, N, M, T(1), Linv, M, sMM, gA, N, sMN, T(0), gKzx, N, sMN, L, 2, 0, 0);
  if (rc) return rc;
  // gLinv = tril(gA Kzx^T)
  rc = gemm<T>(st, false, true, M, M, N, T(1), gA, N, sMN, Kzx, N, sMN, T(0), gLinv, M, sMM, L, 0, 0, 1, splitk > 1 ? splitk : 1);
  return rc;
}

// ---- tensor-core (tcgen05, split-TF32) variant of the same two entry points, fp32 only ----------------------------
// ws layout (floats): [Linv_lo | TT | TT_lo | T_lo | LinvT | LinvT_lo] (each L*M*M) then [sumA2 | sumC2] (each L*N).
// The column reductions of the predictive mean / variance and the row reduction gq = A gm are fused into the GEMM
// epilogues (umma_gemm.cu epi_mode 1..3), so A and C are never re-read for them.
static int tc_gemm(cudaStream_t st, int bk, int m, int n, int k, const float* A, const float* Alo, int64_t lda, int64_t sA,
                   const float* B, const float* Blo, int64_t ldb, int64_t sB, float* D, float* Dlo, int64_t ldd, int64_t sD,
                   int batch, int a_tri, int d_tri, int splitk, const UmmaEpilogue* epi = nullptr) {
  return umma_gemm_ex(bk, m, n, k, 1.0f, A, Alo, lda, sA, B, Blo, ldb, sB, nullptr, D, Dlo, ldd, sD, batch, a_tri, 0, d_tri, splitk,
                      3, epi, (void*)st);
}

__global__ void predict_var_kernel(const float* __restrict__ kxx, const float* __restrict__ sA2, const float* __restrict__ sC2,
                                   float* __restrict__ var, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) var[i] = kxx[i] - sA2[i] + sC2[i];
}

// C <- gC = 2 C gv  and its lo part
__global__ void __launch_bounds__(256) predict_scale_kernel(float* __restrict__ C, float* __restrict__ Clo, const float* __restrict__ gv,
                                                             int M, int N) {
  const int l = blockIdx.z;
  const int n4 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (n4 >= N) return;
  const float4 g = *reinterpret_cast<const float4*>(gv + (int64_t)l * N + n4);
  const int m0 = blockIdx.y * 16, m1 = min(m0 + 16, M);
  for (int m = m0; m < m1; ++m) {
    const int64_t e = ((int64_t)l * M + m) * N + n4;
    float4 c = *reinterpret_cast<const float4*>(C + e);
    c.x *= 2.f * g.x; c.y *= 2.f * g.y; c.z *= 2.f * g.z; c.w *= 2.f * g.w;
    *reinterpret_cast<float4*>(C + e) = c;
    float4 lo;
    lo.x = c.x - __uint_as_float(__float_as_uint(c.x) & 0xFFFFE000u);
    lo.y = c.y - __uint_as_float(__float_as_uint(c.y) & 0xFFFFE000u);
    lo.z = c.z - __uint_as_float(__float_as_uint(c.z) & 0xFFFFE000u);
    lo.w = c.w - __uint_as_float(__float_as_uint(c.w) & 0xFFFFE000u);
    *reinterpret_cast<float4*>(Clo + e) = lo;
  }
}

static int predict_fwd_tc(const float* Kzx, const float* Kzx_lo, const float* Linv, const float* Tm, const float* q, const float* kxx,
                          float* A, float* A_lo, float* C, float* mean, float* var, float* ws, int M, int N, int L, cudaStream_t st) {
  const int64_t sMM = (int64_t)M * M, sMN = (int64_t)M * N, W = sMM * L, LN = (int64_t)L * N;
  float* Linv_lo = ws; float* TT = ws + W; float* TT_lo = ws + 2 * W;
  float* sA2 = ws + 6 * W; float* sC2 = sA2 + LN;
  int rc = gpz_tf32_lo_f32(Linv, Linv_lo, W, (void*)st);
  if (rc) return rc;
  rc = gpz_transpose_lo_f32(Tm, TT, TT_lo, M, L, (void*)st);
  if (rc) return rc;
  GPZ_CUDA(cudaMemsetAsync(sA2, 0, sizeof(float) * 2 * LN, st));
  GPZ_CUDA(cudaMemsetAsync(mean, 0, sizeof(float) * LN, st));
  // A = Linv Kzx  (lower-triangular product == TRSM Lc A = Kzx); epilogue: sum_m A^2 and mean = sum_m q_m A
  UmmaEpilogue e1{1, nullptr, q, nullptr, nullptr, sA2, mean, nullptr};
  rc = tc_gemm(st, 0, M, N, M, Linv, Linv_lo, M, sMM, Kzx, Kzx_lo, N, sMN, A, A_lo, N, sMN, L, 1, 0, 1, &e1);
  if (rc) return rc;
  // C = T^T A     (upper-triangular product); epilogue: sum_m C^2
  UmmaEpilogue e2{2, nullptr, nullptr, nullptr, nullptr, sC2, nullptr, nullptr};
  rc = tc_gemm(st, 0, M, N, M, TT, TT_lo, M, sMM, A, A_lo, N, sMN, C, nullptr, N, sMN, L, 2, 0, 1, &e2);
  if (rc) return rc;
  predict_var_kernel<<<(unsigned)cdiv(LN, 256), 256, 0, st>>>(kxx, sA2, sC2, var, LN);
  GPZ_CHECK_LAUNCH();
  return GPZ_OK;
}

static int predict_bwd_tc(const float* Kzx, const float* Kzx_lo, const float* Linv, const float* Tm, const float* q, const float* A,
                          const float* A_lo, float* C, float* C_lo, const float* gm, const float* gv, float* gA, float* gA_lo,
                          float* gKzx, float* gLinv, float* gT, float* gq, float* ws, int M, int N, int L, cudaStream_t st) {
  const int64_t sMM = (int64_t)M * M, sMN = (int64_t)M * N, W = sMM * L;
  float* T_lo = ws + 3 * W; float* LinvT = ws + 4 * W; float* LinvT_lo = ws + 5 * W;
  int rc = gpz_tf32_lo_f32(Tm, T_lo, W, (void*)st);
  if (rc) return rc;
  rc = gpz_transpose_lo_f32(Linv, LinvT, LinvT_lo, M, L, (void*)st);
  if (rc) return rc;
  // C <- gC = 2 C gv (+ lo part)
  predict_scale_kernel<<<dim3((unsigned)cdiv(N, 1024), (unsigned)cdiv(M, 16), L), 256, 0, st>>>(C, C_lo, gv, M, N);
  GPZ_CHECK_LAUNCH();
  GPZ_CUDA(cudaMemsetAsync(gq, 0, sizeof(float) * (size_t)L * M, st));
  int splitk = 1;
  {
    const int64_t tiles = cdiv(M, 128) * cdiv(M, 256) * L / 2 + 1;
    while (splitk < 32 && tiles * splitk < 148 * 2 && N / (splitk * 2) >= 1024) splitk *= 2;
  }
  // gT = tril(A gC^T)   (reduction over the N spots, both operands K-major)
  rc = tc_gemm(st, 1, M, M, N, A, A_lo, N, sMN, C, C_lo, N, sMN, gT, nullptr, M, sMM, L, 0, 1, splitk);
  if (rc) return rc;
  // gA = T gC - 2 A gv + q gm^T ;  gq = A gm     (both in the epilogue, which reads the A tile once)
  UmmaEpilogue e3{3, A, q, gv, gm, nullptr, nullptr, gq};
  rc = tc_gemm(st, 0, M, N, M, Tm, T_lo, M, sMM, C, C_lo, N, sMN, gA, gA_lo, N, sMN, L, 1, 0, 1, &e3);
  if (rc) return rc;
  // gKzx = Linv^T gA
  rc = tc_gemm(st, 0, M, N, M, LinvT, LinvT_lo, M, sMM, gA, gA_lo, N, sMN, gKzx, nullptr, N, sMN, L, 2, 0, 1);
  if (rc) return rc;
  // gLinv = tril(gA Kzx^T)
  return tc_gemm(st, 1, M, M, N, gA, gA_lo, N, sMN, Kzx, Kzx_lo, N, sMN, gLinv, nullptr, M, sMM, L, 0, 1, splitk);
}


// ---- tensor-core (tcgen05, split-FP16) variant: the default fp32 hot path ------------------------------------------------
// Every N-proportional operand travels as a pair of fp16 planes (hi, lo) of x * s[l] (s[l] a power of two, 22 significant
// bits, 4 bytes per entry) instead of fp32 + lo plane (8 bytes); the GEMMs run at the f16 tensor-core rate (2x tf32).
// Scales come from upper bounds that are available BEFORE the producing kernel runs, so every epilogue can write the planes
// of its output directly:
//   Kzx  : |K| <= sigma^2                                   (kernel_build.cu writes the planes and sK)
//   A    : |A[:,n]|_2^2 = k_n^T (Kzz + jitter I)^-1 k_n <= Kxx[n]   (Schur complement of a PSD kernel)  ->  bound 2 sqrt(max Kxx)
//   C    : |C[m,n]| <= |T[:,m]|_2 |A[:,n]|_2 <= sqrt(M) max|T| sqrt(max Kxx)      (bound x 2; max|C| is also tracked exactly)
//   A diag(2 gv) : 2 max|A| max|gv|                          (written by the gA epilogue, feeds gT)
//   gA   : |T|_inf 2 max|C| max|gv| + 2 max|A| max|gv| + max|q| max|gm|
//   Linv, T (M x M): exact max from a reduction pass.
// A bound that is 2^10 too loose still leaves the fp16 subnormal floor 2^-30 below the largest entry, i.e. below fp32 epsilon
// relative to the matrix norm; a violated bound produces inf/NaN (never a silently saturated value).
// ws_h (halfs): [Linv_h | Linv_l | LinvT_h | LinvT_l | T_h | T_l | TT_h | TT_l], each L*M*M.
// ws_f (floats): [sumA2 (L*N) | sumC2 (L*N) | stats (16 slots of L)], slots:
enum { ST_S_LINV = 0, ST_S_T, ST_S_A, ST_S_AW, ST_S_GA, ST_AMAX_LINV, ST_AMAX_T, ST_AMAX_A, ST_AMAX_C, ST_TINF, ST_AMAX_GV,
       ST_AMAX_GM, ST_AMAX_Q, ST_AMAX_KXX, ST_AMAX_GA, ST_S_C, ST_SLOTS };

// max |x[l,:]| of up to three L x n arrays in one launch: grid (chunks, L, arrays), atomicMax on the float bits
struct Amax3 { const float* x[3]; int n[3]; unsigned int* out[3]; };
__global__ void __launch_bounds__(256) amax3_kernel(const Amax3 a) {
  const int l = blockIdx.y, w = blockIdx.z;
  const float* x = a.x[w] + (int64_t)l * a.n[w];
  float m = 0.f;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < a.n[w]; i += gridDim.x * blockDim.x) m = fmaxf(m, fabsf(x[i]));
#pragma unroll
  for (int sh = 16; sh > 0; sh >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, sh));
  if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(a.out[w] + l, __float_as_uint(m));
}

// sA[l] from max Kxx[l,:], sC[l] from max|T| as well
__global__ void predict_h_fwd_scales_kernel(float* __restrict__ stats, int L, int M) {
  const int l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l >= L) return;
  const float rk = sqrtf(stats[ST_AMAX_KXX * L + l]);
  stats[ST_S_A * L + l] = gpz_pow2_scale(2.f * rk);
  stats[ST_S_C * L + l] = gpz_pow2_scale(2.f * sqrtf((float)M) * stats[ST_AMAX_T * L + l] * rk);
}

// max_i sum_j |T[l,i,j]|: one warp per row
__global__ void __launch_bounds__(256) rowabs_max_kernel(const float* __restrict__ T, unsigned int* __restrict__ out, int M) {
  const int l = blockIdx.y, row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= M) return;
  const float* t = T + ((int64_t)l * M + row) * M;
  float s = 0.f;
  for (int j = lane; j < M; j += 32) s += fabsf(t[j]);
  s = warp_sum(s);
  if (lane == 0 && s > 0.f) atomicMax(out + l, __float_as_uint(s));
}

// the scales of gC and gA from the tracked maxima
__global__ void predict_h_bwd_scales_kernel(float* __restrict__ stats, int L) {
  const int l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l >= L) return;
  const float a_A = stats[ST_AMAX_A * L + l], a_C = stats[ST_AMAX_C * L + l], tinf = stats[ST_TINF * L + l];
  const float a_gv = stats[ST_AMAX_GV * L + l], a_gm = stats[ST_AMAX_GM * L + l], a_q = stats[ST_AMAX_Q * L + l];
  const float b_gC = 2.f * a_C * a_gv;                      // |C diag(2 gv)|
  const float b_gA = tinf * b_gC + 2.f * a_A * a_gv + a_q * a_gm;
  stats[ST_S_AW * L + l] = gpz_pow2_scale(2.f * a_A * a_gv);  // A diag(2 gv)
  stats[ST_S_GA * L + l] = gpz_pow2_scale(b_gA);
}

// S (lower triangle valid) -> full symmetric S and its tf32 lo plane
__global__ void __launch_bounds__(256) sym_lo_kernel(float* __restrict__ S, float* __restrict__ S_lo, int M) {
  const int i = blockIdx.x, l = blockIdx.y;
  const int64_t mat = (int64_t)l * M * M;
  for (int j = threadIdx.x; j < M; j += blockDim.x) {
    const float v = j <= i ? S[mat + (int64_t)i * M + j] : S[mat + (int64_t)j * M + i];
    if (j > i) S[mat + (int64_t)i * M + j] = v;
    S_lo[mat + (int64_t)i * M + j] = v - __uint_as_float(__float_as_uint(v) & 0xFFFFE000u);
  }
}
static Umma16Args h_args(int bk, int m, int n, int k, const __half* Ah, const __half* Al, int64_t lda, int64_t sA, const float* sa,
                         const __half* Bh, const __half* Bl, int64_t ldb, int64_t sB, const float* sb, int64_t ldd, int64_t sD,
                         int batch, int a_tri, int d_tri, int splitk) {
  Umma16Args g{};
  g.b_kmajor = bk; g.m = m; g.n = n; g.k = k; g.alpha = 1.0f;
  g.Ah = Ah; g.Al = Al; g.lda = lda; g.sA = sA; g.sa = sa;
  g.Bh = Bh; g.Bl = Bl; g.ldb = ldb; g.sB = sB; g.sb = sb;
  g.ldd = ldd; g.sD = sD; g.batch = batch; g.a_tri = a_tri; g.d_tri = d_tri; g.splitk = splitk; g.n_terms = 3;
  return g;
}

static int predict_fwd_h(const __half* Kh, const __half* Kl, const float* sK, const float* Linv, const float* Tm, const float* q,
                         const float* kxx, __half* Ah, __half* Al, __half* Ch, __half* Cl, float* mean, float* var, __half* ws_h,
                         float* ws_f, int M, int N, int L, cudaStream_t st) {
  const int64_t sMM = (int64_t)M * M, sMN = (int64_t)M * N, W = sMM * L, LN = (int64_t)L * N;
  __half* Linv_h = ws_h; __half* Linv_l = ws_h + W;
  __half* LinvT_h = ws_h + 2 * W; __half* LinvT_l = ws_h + 3 * W;
  __half* T_h = ws_h + 4 * W; __half* T_l = ws_h + 5 * W; __half* TT_h = ws_h + 6 * W; __half* TT_l = ws_h + 7 * W;
  float* sA2 = ws_f; float* sC2 = ws_f + LN; float* stats = ws_f + 2 * LN;
  unsigned int* ustats = reinterpret_cast<unsigned int*>(stats);
  GPZ_CUDA(cudaMemsetAsync(ws_f, 0, sizeof(float) * (2 * LN + (size_t)ST_SLOTS * L), st));
  GPZ_CUDA(cudaMemsetAsync(mean, 0, sizeof(float) * LN, st));
  int rc = split16_amax(Linv, sMM, L, ustats + ST_AMAX_LINV * L, (void*)st);
  if (rc) return rc;
  rc = split16_planes(Linv, M, M, L, ustats + ST_AMAX_LINV * L, stats + ST_S_LINV * L, Linv_h, Linv_l, LinvT_h, LinvT_l, (void*)st);
  if (rc) return rc;
  rc = split16_amax(Tm, sMM, L, ustats + ST_AMAX_T * L, (void*)st);
  if (rc) return rc;
  rc = split16_planes(Tm, M, M, L, ustats + ST_AMAX_T * L, stats + ST_S_T * L, T_h, T_l, TT_h, TT_l, (void*)st);
  if (rc) return rc;
  rc = split16_amax(kxx, N, L, ustats + ST_AMAX_KXX * L, (void*)st);
  if (rc) return rc;
  predict_h_fwd_scales_kernel<<<(unsigned)cdiv(L, 64), 64, 0, st>>>(stats, L, M);
  GPZ_CHECK_LAUNCH();
  // A = Linv Kzx  (lower-triangular product == TRSM Lc A = Kzx); epilogue: sum_m A^2, mean = sum_m q_m A, max |A|
  UmmaEpilogue e1{1, nullptr, q, nullptr, nullptr, sA2, mean, nullptr};
  Umma16Args g1 = h_args(0, M, N, M, Linv_h, Linv_l, M, sMM, stats + ST_S_LINV * L, Kh, Kl, N, sMN, sK, N, sMN, L, 1, 0, 1);
  g1.Dh = Ah; g1.Dl = Al; g1.sd = stats + ST_S_A * L; g1.amax = ustats + ST_AMAX_A * L; g1.epi = &e1;
  rc = umma_gemm16_ex(g1, (void*)st);
  if (rc) return rc;
  // C = T^T A     (upper-triangular product), kept as fp16 planes for the backward; epilogue: sum_m C^2, max |C|
  UmmaEpilogue e2{2, nullptr, nullptr, nullptr, nullptr, sC2, nullptr, nullptr};
  Umma16Args g2 = h_args(0, M, N, M, TT_h, TT_l, M, sMM, stats + ST_S_T * L, Ah, Al, N, sMN, stats + ST_S_A * L, N, sMN, L, 2, 0, 1);
  g2.Dh = Ch; g2.Dl = Cl; g2.sd = stats + ST_S_C * L; g2.amax = ustats + ST_AMAX_C * L; g2.epi = &e2;
  rc = umma_gemm16_ex(g2, (void*)st);
  if (rc) return rc;
  predict_var_kernel<<<(unsigned)cdiv(LN, 256), 256, 0, st>>>(kxx, sA2, sC2, var, LN);
  GPZ_CHECK_LAUNCH();
  return GPZ_OK;
}

static int predict_bwd_h(const __half* Kh, const __half* Kl, const float* sK, const float* Tm, const float* q, const __half* Ah,
                         const __half* Al, const __half* Ch, const __half* Cl, const float* gm, const float* gv, __half* AWh,
                         __half* AWl, __half* gAh, __half* gAl, float* gKzx, float* gLinv, float* gT, float* gq, __half* ws_h,
                         float* ws_f, float* ws_m, int M, int N, int L, cudaStream_t st) {
  if (ws_m != nullptr && (gT != nullptr || gLinv != nullptr)) return GPZ_ERR_BADARG;
  const int64_t sMM = (int64_t)M * M, sMN = (int64_t)M * N, W = sMM * L, LN = (int64_t)L * N;
  __half* LinvT_h = ws_h + 2 * W; __half* LinvT_l = ws_h + 3 * W;
  __half* T_h = ws_h + 4 * W; __half* T_l = ws_h + 5 * W;
  float* stats = ws_f + 2 * LN;
  unsigned int* ustats = reinterpret_cast<unsigned int*>(stats);
  const float* sA = stats + ST_S_A * L; const float* sAW = stats + ST_S_AW * L; const float* sgA = stats + ST_S_GA * L;
  const float* sC = stats + ST_S_C * L;
  // (the backward may run more than once on the same forward state: reset the maxima it accumulates)
  GPZ_CUDA(cudaMemsetAsync(ustats + ST_TINF * L, 0, sizeof(unsigned int) * 4 * (size_t)L, st));      // TINF, GV, GM, Q are adjacent
  GPZ_CUDA(cudaMemsetAsync(ustats + ST_AMAX_GA * L, 0, sizeof(unsigned int) * (size_t)L, st));
  rowabs_max_kernel<<<dim3((unsigned)cdiv(M, 8), L), 256, 0, st>>>(Tm, ustats + ST_TINF * L, M);
  GPZ_CHECK_LAUNCH();
  Amax3 am{{gv, gm, q}, {N, N, M}, {ustats + ST_AMAX_GV * L, ustats + ST_AMAX_GM * L, ustats + ST_AMAX_Q * L}};
  amax3_kernel<<<dim3(16, L, 3), 256, 0, st>>>(am);
  GPZ_CHECK_LAUNCH();
  predict_h_bwd_scales_kernel<<<(unsigned)cdiv(L, 64), 64, 0, st>>>(stats, L);
  GPZ_CHECK_LAUNCH();
  GPZ_CUDA(cudaMemsetAsync(gq, 0, sizeof(float) * (size_t)L * M, st));
  int splitk = 1;
  {
    const int64_t tiles = cdiv(M, 128) * cdiv(M, 256) * L / 2 + 1;
    while (splitk < 32 && tiles * splitk < 148 * 2 && N / (splitk * 2) >= 1024) splitk *= 2;
  }
  // gA = T C diag(2 gv) - A diag(2 gv) + q gm^T = 2 gv o (T C - A) + q gm^T  straight from the unweighted C planes (the column
  // weights commute out of the product); the same epilogue, which reads the A planes once, also gives gq = A gm and writes
  // AW = A diag(2 gv) as planes for the reduction below
  UmmaEpilogue e3{4, nullptr, q, gv, gm, nullptr, nullptr, gq};
  Umma16Args g3 = h_args(0, M, N, M, T_h, T_l, M, sMM, stats + ST_S_T * L, Ch, Cl, N, sMN, sC, N, sMN, L, 1, 0, 1);
  g3.Dh = gAh; g3.Dl = gAl; g3.sd = sgA; g3.amax = ustats + ST_AMAX_GA * L; g3.epi = &e3; g3.AuxH = Ah; g3.AuxL = Al; g3.saux = sA;
  g3.D2h = AWh; g3.D2l = AWl; g3.sd2 = sAW;
  int rc = umma_gemm16_ex(g3, (void*)st);
  if (rc) return rc;
  if (ws_m == nullptr) {
    // two reductions over the N spots:  gT = tril(AW C^T),  gLinv = tril(gA Kzx^T)
    Umma16Args g4 = h_args(1, M, M, N, AWh, AWl, N, sMN, sAW, Ch, Cl, N, sMN, sC, M, sMM, L, 0, 1, splitk);
    g4.D = gT;
    rc = umma_gemm16_ex(g4, (void*)st);
    if (rc) return rc;
    Umma16Args g5 = h_args(0, M, N, M, LinvT_h, LinvT_l, M, sMM, stats + ST_S_LINV * L, gAh, gAl, N, sMN, sgA, N, sMN, L, 2, 0, 1);
    g5.D = gKzx;
    rc = umma_gemm16_ex(g5, (void*)st);
    if (rc) return rc;
    Umma16Args g6 = h_args(1, M, M, N, gAh, gAl, N, sMN, sgA, Kh, Kl, N, sMN, sK, M, sMM, L, 0, 1, splitk);
    g6.D = gLinv;
    return umma_gemm16_ex(g6, (void*)st);
  }
  // merged backward (csrc/chain.cu takes S1 and gq from here): ONE reduction over the N spots, S1 = A diag(2 gv) A^T (symmetric,
  // lower triangle computed, then mirrored with its lo plane), instead of the two above
  float* S1 = ws_m; float* S1_lo = ws_m + W;
  GPZ_CUDA(cudaMemsetAsync(S1, 0, sizeof(float) * W, st));
  Umma16Args g4 = h_args(1, M, M, N, AWh, AWl, N, sMN, sAW, Ah, Al, N, sMN, sA, M, sMM, L, 0, 1, splitk);
  g4.D = S1;
  rc = umma_gemm16_ex(g4, (void*)st);
  if (rc) return rc;
  // gKzx = Linv^T gA
  Umma16Args g5 = h_args(0, M, N, M, LinvT_h, LinvT_l, M, sMM, stats + ST_S_LINV * L, gAh, gAl, N, sMN, sgA, N, sMN, L, 2, 0, 1);
  g5.D = gKzx;
  rc = umma_gemm16_ex(g5, (void*)st);
  if (rc) return rc;
  sym_lo_kernel<<<dim3(M, L), 256, 0, st>>>(S1, S1_lo, M);
  GPZ_CHECK_LAUNCH();
  return GPZ_OK;
}

}  // namespace gpz

using namespace gpz;

extern "C" int gpz_svgp_predict_tc_supported(int M, int N) { return (M % 4 == 0 && N % 4 == 0 && M >= 64 && N >= 256) ? 1 : 0; }

extern "C" int gpz_svgp_predict_fwd_tc_f32(const float* Kzx, const float* Kzx_lo, const float* Linv, const float* T, const float* q,
                                           const float* kxx, float* A, float* A_lo, float* C, float* mean, float* var, float* ws,
                                           int M, int N, int L, void* stream) {
  if (!gpz_svgp_predict_tc_supported(M, N) || L <= 0) return GPZ_ERR_UNSUPPORTED;
  return predict_fwd_tc(Kzx, Kzx_lo, Linv, T, q, kxx, A, A_lo, C, mean, var, ws, M, N, L, (cudaStream_t)stream);
}
extern "C" int gpz_svgp_predict_bwd_tc_f32(const float* Kzx, const float* Kzx_lo, const float* Linv, const float* T, const float* q,
                                           const float* A, const float* A_lo, float* C, float* C_lo, const float* gm, const float* gv,
                                           float* gA, float* gA_lo, float* gKzx, float* gLinv, float* gT, float* gq, float* ws, int M,
                                           int N, int L, void* stream) {
  if (!gpz_svgp_predict_tc_supported(M, N) || L <= 0) return GPZ_ERR_UNSUPPORTED;
  return predict_bwd_tc(Kzx, Kzx_lo, Linv, T, q, A, A_lo, C, C_lo, gm, gv, gA, gA_lo, gKzx, gLinv, gT, gq, ws, M, N, L,
                        (cudaStream_t)stream);
}

// split-FP16 tensor-core variant (see predict_fwd_h): planes are fp16, ws_h holds 8 L*M*M halfs, ws_f 2 L*N + 16 L floats
// row of the stats block (L floats each, starting at ws_f + 2 L N) holding: 0 scale of A, 1 max|A|, 2 max|C|, 3 scale of gA,
// 4 max|gA|, 5 scale of C  (read by the host-side overflow guard); -1 for an unknown id
extern "C" int gpz_svgp_predict_h_stat_row(int which) {
  switch (which) {
    case 0: return ST_S_A;
    case 1: return ST_AMAX_A;
    case 2: return ST_AMAX_C;
    case 3: return ST_S_GA;
    case 4: return ST_AMAX_GA;
    case 5: return ST_S_C;
    default: return -1;
  }
}
extern "C" int gpz_svgp_predict_h_supported(int M, int N) { return (M % 8 == 0 && N % 8 == 0 && M >= 64 && N >= 256) ? 1 : 0; }
extern "C" int gpz_svgp_predict_fwd_h_f32(const void* Kh, const void* Kl, const float* sK, const float* Linv, const float* T,
                                          const float* q, const float* kxx, void* Ah, void* Al, void* Ch, void* Cl, float* mean,
                                          float* var, void* ws_h, float* ws_f, int M, int N, int L, void* stream) {
  if (!gpz_svgp_predict_h_supported(M, N) || L <= 0) return GPZ_ERR_UNSUPPORTED;
  return predict_fwd_h((const __half*)Kh, (const __half*)Kl, sK, Linv, T, q, kxx, (__half*)Ah, (__half*)Al, (__half*)Ch, (__half*)Cl,
                       mean, var, (__half*)ws_h, ws_f, M, N, L, (cudaStream_t)stream);
}
extern "C" int gpz_svgp_predict_bwd_h_f32(const void* Kh, const void* Kl, const float* sK, const float* T, const float* q,
                                          const void* Ah, const void* Al, const void* Ch, const void* Cl, const float* gm,
                                          const float* gv, void* AWh, void* AWl, void* gAh, void* gAl, float* gKzx, float* gLinv,
                                          float* gT, float* gq, void* ws_h, float* ws_f, float* ws_m, int M, int N, int L,
                                          void* stream) {
  if (!gpz_svgp_predict_h_supported(M, N) || L <= 0) return GPZ_ERR_UNSUPPORTED;
  return predict_bwd_h((const __half*)Kh, (const __half*)Kl, sK, T, q, (const __half*)Ah, (const __half*)Al, (const __half*)Ch,
                       (const __half*)Cl, gm, gv, (__half*)AWh, (__half*)AWl, (__half*)gAh, (__half*)gAl, gKzx, gLinv, gT, gq,
                       (__half*)ws_h, ws_f, ws_m, M, N, L, (cudaStream_t)stream);
}

#define GPZ_PREDICT_IMPL(SUF, T)                                                                                      \
  extern "C" int gpz_svgp_predict_fwd_##SUF(const T* Kzx, const T* Linv, const T* Tm, const T* q, const T* kxx, T* A, \
                                            T* C, T* mean, T* var, int M, int N, int L, void* stream) {               \
    if (M <= 0 || L <= 0 || N < 0) return GPZ_ERR_BADARG;                                                             \
    if (N == 0) return GPZ_OK;                                                                                        \
    return predict_fwd<T>(Kzx, Linv, Tm, q, kxx, A, C, mean, var, M, N, L, (cudaStream_t)stream);                     \
  }                                                                                                                   \
  extern "C" int gpz_svgp_predict_bwd_##SUF(const T* Kzx, const T* Linv, const T* Tm, const T* q, const T* A, T* C,   \
                                            const T* gm, const T* gv, T* gA, T* gKzx, T* gLinv, T* gT, T* gq, int M,  \
                                            int N, int L, void* stream) {                                             \
    if (M <= 0 || L <= 0 || N < 0) return GPZ_ERR_BADARG;                                                             \
    if (N == 0) return GPZ_OK;                                                                                        \
    return predict_bwd<T>(Kzx, Linv, Tm, q, A, C, gm, gv, gA, gKzx, gLinv, gT, gq, M, N, L, (cudaStream_t)stream);    \
  }

GPZ_PREDICT_IMPL(f32, float)
GPZ_PREDICT_IMPL(f64, double)

// batched matrix-vector products: trans == 0: out[l,i] = sum_k A[l,i,k] v[l,k] (A: rows x cols);  trans != 0: out[l,j] = sum_k A[l,k,j] v[l,k]
#define GPZ_GEMV_IMPL(SUF, T)                                                                                         \
  extern "C" int gpz_gemv_##SUF(int trans, const T* A, const T* v, T* out, int rows, int cols, int L, void* stream) { \
    if (rows <= 0 || cols <= 0 || L <= 0) return GPZ_OK;                                                              \
    cudaStream_t st = (cudaStream_t)stream;                                                                           \
    if (!trans) rowdot_kernel<T><<<dim3(rows, L), 256, 0, st>>>(A, v, out, rows, cols);                               \
    else coldot_kernel<T><<<dim3((unsigned)cdiv(cols, 32), L), 256, 0, st>>>(A, v, out, rows, cols);                   \
    GPZ_CHECK_LAUNCH();                                                                                               \
    return GPZ_OK;                                                                                                    \
  }
GPZ_GEMV_IMPL(f32, float)
GPZ_GEMV_IMPL(f64, double)
