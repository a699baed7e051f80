// The O(M^3) chain of one SVGP step as TWO C-ABI calls (fp32, M >= 128): everything between the jittered Kzz and the
// whitened operands of the predictive kernels, and its hand-written backward.
//
// Reference (gp.py:208-221 + torch kl.py MVN||MVN + their autograd):  Lc = cholesky(Kzz + jitter I);  Lu = lower_cholesky(raw);
// cholesky_solve / solve_triangular against Lc.  Here (DESIGN.md §2):
//     forward :  (Lc, Linv) = chol_inv(Kzz)      Lu = tril(raw,-1) + diag(exp(diag raw))      T = Linv Lu      q = Linv mu
//                kl = sum log diag Lc - sum diag raw + 0.5 (|T|_F^2 + |q|^2 - M)
//     backward:  gT += gkl T ;  gq += gkl q
//                gLu  = tril(Linv^T gT) - gkl / diag(Lu)  (+ incoming)        gmu = Linv^T gq
//                gLinv = gLinv_in + tril(gT Lu^T)                             (the rank-1 part tril(gq mu^T) is applied below)
//                gLc  = -tril(Linv^T gLinv Linv^T) - tril(gmu q^T) + gkl / diag(Lc)  (+ incoming)
//                P    = Phi(Lc^T gLc)   (tril, diagonal halved)               gKzz = Linv^T P Linv
// gKzz is returned WITHOUT symmetrisation: its only consumer contracts it with the symmetric dKzz/dtheta, for which
// <S, dK> == <(S + S^T)/2, dK>.  The eight M x M x M products run on the tcgen05 split-TF32 GEMM (csrc/umma_gemm.cu) with the
// triangular structure of every operand / result declared; operand lo planes are written by the producing GEMM's epilogue or
// by the few fused element-wise kernels below, so a step issues ~25 launches here instead of ~70 (ATen adds / fills included).
#include "common.cuh"
#include "gpzoo_b200.h"
#include "umma_gemm.h"

namespace gpz {

// forward prep, one 32 x 32 tile per CTA: Linv_lo ; LinvT, LinvT_lo ; LcT, LcT_lo ; Lu = lct(raw), Lu_lo
__global__ void __launch_bounds__(256) chain_prep_kernel(const float* __restrict__ Linv, const float* __restrict__ Lc,
                                                          const float* __restrict__ raw, float* __restrict__ Linv_lo,
                                                          float* __restrict__ LinvT, float* __restrict__ LinvT_lo,
                                                          float* __restrict__ LcT, float* __restrict__ LcT_lo, float* __restrict__ Lu,
                                                          float* __restrict__ Lu_lo, int M) {
  __shared__ float t1[32][33], t2[32][33];
  const int64_t mat = (int64_t)blockIdx.z * M * M;
  const int bx = blockIdx.x * 32, by = blockIdx.y * 32, tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int r = ty; r < 32; r += 8) {
    const int i = by + r, j = bx + tx;
    float a = 0.f, b = 0.f;
    if (i < M && j < M) {
      const int64_t o = mat + (int64_t)i * M + j;
      a = j <= i ? Linv[o] : 0.f;
      b = j <= i ? Lc[o] : 0.f;
      Linv_lo[o] = tf32_lo_part(a);
      const float x = j <= i ? raw[o] : 0.f;
      const float lu = j < i ? x : (j == i ? expf(x) : 0.f);
      Lu[o] = lu;
      Lu_lo[o] = tf32_lo_part(lu);
    }
    t1[r][tx] = a;
    t2[r][tx] = b;
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    const int i = bx + r, j = by + tx;            // transposed output (i, j) = input (j, i)
    if (i < M && j < M) {
      const int64_t o = mat + (int64_t)i * M + j;
      const float a = t1[tx][r], b = t2[tx][r];
      LinvT[o] = a; LinvT_lo[o] = tf32_lo_part(a);
      LcT[o] = b;   LcT_lo[o] = tf32_lo_part(b);
    }
  }
}

// backward prep: gT = tril(gT_in) + gkl T (and its lo plane, zeros above the diagonal) ; gq = gq_in + gkl q
__global__ void __launch_bounds__(256) chain_bwd_prep_kernel(const float* __restrict__ gT_in, const float* __restrict__ gq_in,
                                                              const float* __restrict__ gkl, const float* __restrict__ T,
                                                              const float* __restrict__ q, float* __restrict__ gT,
                                                              float* __restrict__ gT_lo, float* __restrict__ gq, int M) {
  const int i = blockIdx.x, l = blockIdx.y;
  const int64_t row = ((int64_t)l * M + i) * M;
  const float g = gkl ? gkl[l] : 0.f;
  for (int j = threadIdx.x; j < M; j += blockDim.x) {
    float v = 0.f;
    if (j <= i) v = (gT_in ? gT_in[row + j] : 0.f) + g * T[row + j];
    gT[row + j] = v;
    gT_lo[row + j] = tf32_lo_part(v);
  }
  if (threadIdx.x == 0) gq[(int64_t)l * M + i] = (gq_in ? gq_in[(int64_t)l * M + i] : 0.f) + g * q[(int64_t)l * M + i];
}

// graw = lct_bwd(U + gLu_in - gkl / diag(Lu)):  tril(.,-1) + diag(. * Lu_ii)
__global__ void __launch_bounds__(256) chain_glu_kernel(const float* __restrict__ U, const float* __restrict__ gLu_in,
                                                         const float* __restrict__ gkl, const float* __restrict__ Lu,
                                                         float* __restrict__ graw, int M) {
  const int i = blockIdx.x, l = blockIdx.y;
  const int64_t row = ((int64_t)l * M + i) * M;
  const float g = gkl ? gkl[l] : 0.f;
  for (int j = threadIdx.x; j < M; j += blockDim.x) {
    float v = 0.f;
    if (j <= i) {
      v = U[row + j] + (gLu_in ? gLu_in[row + j] : 0.f);
      if (j == i) { const float d = Lu[row + j]; v = (v - g / d) * d; }
    }
    graw[row + j] = v;
  }
}

// mode 0:  X = tril(X0) - tril(rowv colv^T) + tril(add) + diag(gkl / diag(Dg))      (gLc assembly)
// mode 1:  X = Phi(X0) = tril(X0) with the diagonal halved
// both write X in place together with its lo plane (zeros above the diagonal)
__global__ void __launch_bounds__(256) chain_trifix_kernel(float* __restrict__ X, float* __restrict__ X_lo, int mode,
                                                            const float* __restrict__ rowv, const float* __restrict__ colv,
                                                            const float* __restrict__ add, const float* __restrict__ gkl,
                                                            const float* __restrict__ Dg, int M) {
  const int i = blockIdx.x, l = blockIdx.y;
  const int64_t row = ((int64_t)l * M + i) * M;
  const float g = (mode == 0 && gkl) ? gkl[l] : 0.f;
  const float rv = (mode == 0) ? rowv[(int64_t)l * M + i] : 0.f;
  for (int j = threadIdx.x; j < M; j += blockDim.x) {
    float v = 0.f;
    if (j <= i) {
      v = X[row + j];
      if (mode == 0) {
        v -= rv * colv[(int64_t)l * M + j];
        if (add) v += add[row + j];
        if (j == i) v += g / Dg[row + j];
      } else if (j == i) {
        v *= 0.5f;
      }
    }
    X[row + j] = v;
    X_lo[row + j] = tf32_lo_part(v);
  }
}

// V = V0 + gkl T (lower) with its lo plane
__global__ void __launch_bounds__(256) chain_v_kernel(float* __restrict__ V, float* __restrict__ V_lo, const float* __restrict__ T,
                                                       const float* __restrict__ gkl, int M) {
  const int i = blockIdx.x, l = blockIdx.y;
  const int64_t row = ((int64_t)l * M + i) * M;
  const float g = gkl ? gkl[l] : 0.f;
  for (int j = threadIdx.x; j < M; j += blockDim.x) {
    const float v = j <= i ? V[row + j] + g * T[row + j] : 0.f;      // (the product above wrote the lower triangle only)
    V[row + j] = v;
    V_lo[row + j] = tf32_lo_part(v);
  }
}

// gq = gqp + gkl q
__global__ void chain_gq_kernel(const float* __restrict__ gqp, const float* __restrict__ gkl, const float* __restrict__ q,
                                float* __restrict__ gq, int M, int L) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e < M * L) gq[e] = gqp[e] + (gkl ? gkl[e / M] : 0.f) * q[e];
}

// G2 = tril(YS + YS^T - S1 + gkl Y + q gqp^T) with its lo plane (zeros above the diagonal); 32 x 32 tiles through shared memory
__global__ void __launch_bounds__(256) chain_g2_kernel(const float* __restrict__ YS, const float* __restrict__ S1, const float* __restrict__ Y,
                                                        const float* __restrict__ q, const float* __restrict__ gqp,
                                                        const float* __restrict__ gkl, float* __restrict__ G2, float* __restrict__ G2_lo,
                                                        int M) {
  __shared__ float t[32][33];
  const int64_t mat = (int64_t)blockIdx.z * M * M;
  const int bx = blockIdx.x * 32, by = blockIdx.y * 32, tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const float g = gkl ? gkl[blockIdx.z] : 0.f;
  for (int r = ty; r < 32; r += 8) {                          // t[r][c] = YS[bx + r][by + c]  (the transposed tile)
    const int i = bx + r, j = by + tx;
    t[r][tx] = (i < M && j < M) ? YS[mat + (int64_t)i * M + j] : 0.f;
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    const int i = by + r, j = bx + tx;
    if (i < M && j < M) {
      const int64_t o = mat + (int64_t)i * M + j;
      float v = 0.f;
      if (j <= i) v = YS[o] + t[tx][r] - S1[o] + g * Y[o] + q[(int64_t)blockIdx.z * M + i] * gqp[(int64_t)blockIdx.z * M + j];
      G2[o] = v;
      G2_lo[o] = tf32_lo_part(v);
    }
  }
}

static int tcg(cudaStream_t st, int bk, int M, int L, float alpha, const float* A, const float* Alo, const float* B, const float* Blo,
               const float* Cin, float* D, float* Dlo, int a_tri, int b_tri, int d_tri) {
  const int64_t s = (int64_t)M * M;
  return umma_gemm_ex(bk, M, M, M, alpha, A, Alo, M, s, B, Blo, M, s, Cin, D, Dlo, M, s, L, a_tri, b_tri, d_tri, 1, 3, nullptr, (void*)st);
}

}  // namespace gpz

using namespace gpz;

// aux: 6 L M M floats  [Linv_lo | LinvT | LinvT_lo | LcT | LcT_lo | Lu_lo]   (saved for the backward)
// ws : 5 L M M floats (Cholesky scratch incl. the lo planes of the tensor-core variant) + L doubles
extern "C" int gpz_svgp_chain_supported(int M) { return (M >= 128 && M % 4 == 0) ? 1 : 0; }

extern "C" int gpz_svgp_chain_fwd_f32(float* Kzz, const float* Lu_raw, const float* mu, float* Lc, float* Linv, float* Lu, float* T,
                                      float* q, float* kl, float* aux, float* ws, int M, int L, int chol_tc, int* info, void* stream) {
  if (!gpz_svgp_chain_supported(M) || L <= 0) return GPZ_ERR_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t W = (int64_t)M * M * L;
  float* Linv_lo = aux; float* LinvT = aux + W; float* LinvT_lo = aux + 2 * W; float* LcT = aux + 3 * W; float* LcT_lo = aux + 4 * W;
  float* Lu_lo = aux + 5 * W;
  int rc = chol_tc ? gpz_chol_inv_tc_f32(Kzz, Lc, Linv, ws, ws + W, M, L, info, stream)
                   : gpz_chol_inv_f32(Kzz, Lc, Linv, ws, M, L, info, stream);
  if (rc) return rc;
  chain_prep_kernel<<<dim3((unsigned)cdiv(M, 32), (unsigned)cdiv(M, 32), L), 256, 0, st>>>(Linv, Lc, Lu_raw, Linv_lo, LinvT, LinvT_lo, LcT,
                                                                                            LcT_lo, Lu, Lu_lo, M);
  GPZ_CHECK_LAUNCH();
  GPZ_CUDA(cudaMemsetAsync(T, 0, sizeof(float) * W, st));
  rc = tcg(st, 0, M, L, 1.0f, Linv, Linv_lo, Lu, Lu_lo, nullptr, T, nullptr, 1, 1, 1);          // T = Linv Lu (lower x lower -> lower)
  if (rc) return rc;
  rc = gpz_gemv_f32(0, Linv, mu, q, M, M, L, stream);                                            // q = Linv mu
  if (rc) return rc;
  return gpz_mvn_kl_fwd_f32(T, q, Lc, Lu, kl, reinterpret_cast<double*>(ws), M, L, stream);
}

// ws: 12 L M M + 2 L M floats.  Any incoming gradient may be NULL.  gKzz (L x M x M, not symmetrised), gLu_raw, gmu are outputs.
extern "C" int gpz_svgp_chain_bwd_f32(const float* Lc, const float* Linv, const float* Lu, const float* T, const float* q,
                                      const float* mu, const float* aux, const float* gLc_in, const float* gLinv_in,
                                      const float* gLu_in, const float* gT_in, const float* gq_in, const float* gkl_in, float* gKzz,
                                      float* gLu_raw, float* gmu, float* ws, int M, int L, void* stream) {
  if (!gpz_svgp_chain_supported(M) || L <= 0) return GPZ_ERR_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t W = (int64_t)M * M * L;
  const float* Linv_lo = aux; const float* LinvT = aux + W; const float* LinvT_lo = aux + 2 * W; const float* LcT = aux + 3 * W;
  const float* LcT_lo = aux + 4 * W; const float* Lu_lo = aux + 5 * W;
  float* gT = ws; float* gT_lo = ws + W; float* U = ws + 2 * W; float* gLinv = ws + 3 * W; float* gLinv_lo = ws + 4 * W;
  float* t1 = ws + 5 * W; float* t1_lo = ws + 6 * W; float* gLc = ws + 7 * W; float* gLc_lo = ws + 8 * W;
  float* P = ws + 9 * W; float* P_lo = ws + 10 * W; float* t2_lo = ws + 11 * W; float* gq = ws + 12 * W;
  float* t2 = U;                                   // U is dead once gLu_raw has been formed
  const dim3 rows(M, L);
  chain_bwd_prep_kernel<<<rows, 256, 0, st>>>(gT_in, gq_in, gkl_in, T, q, gT, gT_lo, gq, M);
  GPZ_CHECK_LAUNCH();
  // the buffers written through lower-triangular epilogues keep zeros above the diagonal
  GPZ_CUDA(cudaMemsetAsync(U, 0, sizeof(float) * W, st));
  GPZ_CUDA(cudaMemsetAsync(gLinv, 0, sizeof(float) * 6 * W, st));      // gLinv, gLinv_lo, t1, t1_lo, gLc, gLc_lo
  GPZ_CUDA(cudaMemsetAsync(P, 0, sizeof(float) * W, st));
  int rc = tcg(st, 0, M, L, 1.0f, LinvT, LinvT_lo, gT, gT_lo, nullptr, U, nullptr, 2, 1, 1);     // U = tril(Linv^T gT)
  if (rc) return rc;
  chain_glu_kernel<<<rows, 256, 0, st>>>(U, gLu_in, gkl_in, Lu, gLu_raw, M);
  GPZ_CHECK_LAUNCH();
  rc = gpz_gemv_f32(1, Linv, gq, gmu, M, M, L, stream);                                           // gmu = Linv^T gq
  if (rc) return rc;
  // gLinv = gLinv_in + tril(gT Lu^T)
  rc = tcg(st, 1, M, L, 1.0f, gT, gT_lo, Lu, Lu_lo, gLinv_in, gLinv, gLinv_lo, 1, 2, 1);
  if (rc) return rc;
  rc = tcg(st, 0, M, L, 1.0f, LinvT, LinvT_lo, gLinv, gLinv_lo, nullptr, t1, t1_lo, 2, 1, 1);     // t1 = tril(Linv^T gLinv)
  if (rc) return rc;
  rc = tcg(st, 1, M, L, -1.0f, t1, t1_lo, Linv, Linv_lo, nullptr, gLc, nullptr, 1, 2, 1);         // gLc0 = -tril(t1 Linv^T)
  if (rc) return rc;
  chain_trifix_kernel<<<rows, 256, 0, st>>>(gLc, gLc_lo, 0, gmu, q, gLc_in, gkl_in, Lc, M);
  GPZ_CHECK_LAUNCH();
  rc = tcg(st, 0, M, L, 1.0f, LcT, LcT_lo, gLc, gLc_lo, nullptr, P, nullptr, 2, 1, 1);            // P0 = tril(Lc^T gLc)
  if (rc) return rc;
  chain_trifix_kernel<<<rows, 256, 0, st>>>(P, P_lo, 1, nullptr, nullptr, nullptr, nullptr, nullptr, M);
  GPZ_CHECK_LAUNCH();
  rc = tcg(st, 0, M, L, 1.0f, LinvT, LinvT_lo, P, P_lo, nullptr, t2, t2_lo, 2, 1, 0);             // t2 = Linv^T P
  if (rc) return rc;
  return tcg(st, 0, M, L, 1.0f, t2, t2_lo, Linv, Linv_lo, nullptr, gKzz, nullptr, 0, 1, 0);        // gKzz = t2 Linv
}

// Merged backward of predict + chain (fp32): the predictive backward hands over S1 = A diag(2 gv) A^T (full symmetric, with its
// lo plane) and gqp = A gm instead of gT and gLinv.  With C = T^T A, Kzx = Lc A and Lc^T Linv^T = I, Lu^T Linv^T = T^T:
//     gq = gqp + gkl q ;  gmu = Linv^T gq
//     Y = T T^T ;  V = (S1 + gkl I) T ;  gLu = tril(Linv^T V) - gkl / diag(Lu)  (+ incoming)
//     G2 = Y S1 + S1 Y - S1 + gkl Y + q gqp^T
//     gLc = gkl / diag(Lc) - tril(Linv^T G2) - tril(gmu q^T)  (+ incoming) ;  P = Phi(Lc^T gLc) ;  gKzz = Linv^T P Linv
// i.e. 8 M x M x M products and ONE reduction over the spots, where the predictive backward alone needs two (gT and gLinv).
// ws: 13 L M M + 2 L M floats.
extern "C" int gpz_svgp_chain_bwd_s1_f32(const float* Lc, const float* Linv, const float* Lu, const float* T, const float* q,
                                         const float* mu, const float* aux, const float* S1, const float* S1_lo, const float* gqp,
                                         const float* gkl_in, const float* gLc_in, const float* gLu_in, float* gKzz, float* gLu_raw,
                                         float* gmu, float* ws, int M, int L, void* stream) {
  if (!gpz_svgp_chain_supported(M) || L <= 0) return GPZ_ERR_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t W = (int64_t)M * M * L;
  const float* Linv_lo = aux; const float* LinvT = aux + W; const float* LinvT_lo = aux + 2 * W; const float* LcT = aux + 3 * W;
  const float* LcT_lo = aux + 4 * W;
  float* T_lo = ws; float* Y = ws + W; float* Y_lo = ws + 2 * W; float* V = ws + 3 * W; float* V_lo = ws + 4 * W; float* U = ws + 5 * W;
  float* YS = ws + 6 * W; float* G2 = ws + 7 * W; float* G2_lo = ws + 8 * W; float* gLc = ws + 9 * W; float* gLc_lo = ws + 10 * W;
  float* P = ws + 11 * W; float* P_lo = ws + 12 * W; float* gq = ws + 13 * W;
  float* t2 = YS; float* t2_lo = Y_lo;                   // YS / Y_lo are dead once G2 has been formed
  (void)mu;
  const dim3 rows(M, L);
  const dim3 tiles((unsigned)cdiv(M, 32), (unsigned)cdiv(M, 32), L);
  int rc = gpz_tf32_lo_f32(T, T_lo, W, stream);
  if (rc) return rc;
  chain_gq_kernel<<<(unsigned)cdiv((int64_t)M * L, 256), 256, 0, st>>>(gqp, gkl_in, q, gq, M, L);
  GPZ_CHECK_LAUNCH();
  rc = gpz_gemv_f32(1, Linv, gq, gmu, M, M, L, stream);                                           // gmu = Linv^T gq
  if (rc) return rc;
  rc = tcg(st, 1, M, L, 1.0f, T, T_lo, T, T_lo, nullptr, Y, Y_lo, 1, 2, 0);                        // Y = T T^T (op(B) = T^T)
  if (rc) return rc;
  rc = tcg(st, 0, M, L, 1.0f, S1, S1_lo, T, T_lo, nullptr, V, nullptr, 0, 1, 1);                   // V0 = tril(S1 T)
  if (rc) return rc;
  chain_v_kernel<<<rows, 256, 0, st>>>(V, V_lo, T, gkl_in, M);                                    // V = tril((S1 + gkl I) T)
  GPZ_CHECK_LAUNCH();
  rc = tcg(st, 0, M, L, 1.0f, LinvT, LinvT_lo, V, V_lo, nullptr, U, nullptr, 2, 1, 1);             // U = tril(Linv^T V)
  if (rc) return rc;
  chain_glu_kernel<<<rows, 256, 0, st>>>(U, gLu_in, gkl_in, Lu, gLu_raw, M);
  GPZ_CHECK_LAUNCH();
  rc = tcg(st, 0, M, L, 1.0f, Y, Y_lo, S1, S1_lo, nullptr, YS, nullptr, 0, 0, 0);                  // YS = Y S1 (full)
  if (rc) return rc;
  chain_g2_kernel<<<tiles, 256, 0, st>>>(YS, S1, Y, q, gqp, gkl_in, G2, G2_lo, M);
  GPZ_CHECK_LAUNCH();
  rc = tcg(st, 0, M, L, -1.0f, LinvT, LinvT_lo, G2, G2_lo, nullptr, gLc, nullptr, 2, 1, 1);        // gLc0 = -tril(Linv^T G2)
  if (rc) return rc;
  chain_trifix_kernel<<<rows, 256, 0, st>>>(gLc, gLc_lo, 0, gmu, q, gLc_in, gkl_in, Lc, M);       // - tril(gmu q^T) + gkl / diag(Lc) + incoming
  GPZ_CHECK_LAUNCH();
  rc = tcg(st, 0, M, L, 1.0f, LcT, LcT_lo, gLc, gLc_lo, nullptr, P, nullptr, 2, 1, 1);            // P0 = tril(Lc^T gLc)
  if (rc) return rc;
  chain_trifix_kernel<<<rows, 256, 0, st>>>(P, P_lo, 1, nullptr, nullptr, nullptr, nullptr, nullptr, M);
  GPZ_CHECK_LAUNCH();
  rc = tcg(st, 0, M, L, 1.0f, LinvT, LinvT_lo, P, P_lo, nullptr, t2, t2_lo, 2, 1, 0);             // t2 = Linv^T P
  if (rc) return rc;
  return tcg(st, 0, M, L, 1.0f, t2, t2_lo, Linv, Linv_lo, nullptr, gKzz, nullptr, 0, 1, 0);        // gKzz = t2 Linv
}
