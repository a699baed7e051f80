/* gpzoo_b200 C ABI — the drop-in boundary of the B200-native sparse-GP ELBO hot path.
 *
 * The reference (luisdiaz1997/GPzoo) has no FFI: its boundary is the PyTorch nn.Module surface
 * (gpzoo.kernels / gpzoo.gp / gpzoo.likelihoods).  The host side of this project keeps that surface in
 * Python (package gpzoo_b200) and reaches the CUDA kernels exclusively through the entry points below,
 * loaded with ctypes from libgpzoo_b200.so.  Each entry point names the reference call site it replaces
 * (paths relative to the reference's gpzoo/ directory).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer borrowed from the caller (the library never allocates or frees);
 *     scratch space is passed in and sized by the matching *_workspace_bytes query;
 *   - tensors are row-major, innermost dimension contiguous; batch (factor) index L outermost;
 *   - `stream` is a cudaStream_t passed as void*; all work is asynchronous on that stream;
 *   - return value: 0 on success, -cudaError_t on a CUDA failure, <= -1000 for argument errors;
 *   - suffix _f32 / _f64 selects the arithmetic type (fp64 exists for the 1e-10 parity check);
 *   - no global state; re-entrant; thread-safe per stream.
 */
#ifndef GPZOO_B200_H
#define GPZOO_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif


int gpz_abi_version(void);
/* cudaGetErrorString for -rc, or a library message for rc <= -1000 */
const char* gpz_error_string(int rc);
/* number of CUDA kernels launched by this library in this process (bench.py reports it as gpu_launches) */
long long gpz_launch_count(void);

/* ---- K1 kernel-matrix build: kernels.py:114-130 (RBF), 141-155 (NSF_RBF), 172-191 (MGGP_RBF),
 *      204-228 (MGGP_NSF_RBF); jitter = utilities.py:407-418 (add_jitter) fused on the diagonal.
 *      out[l,i,j] = sigma_l^2 exp(-0.5 |x1_i-x2_j|^2/(ls_l^2 den))/den^p_half (+ jitter if i==j),
 *      den = a_l r2[g1_i,g2_j] + 1.  Pass a=r2=g1=g2=NULL, ng=0 for the plain RBF.
 *      kind = 0: the RBF forms above; kind = 1: Matern-3/2, kernels.py:6-30 (batched_Matern32),
 *      out[l,i,j] = sigma_l^2 (1 + v) exp(-v), v = sqrt(3) |x1_i-x2_j| / ls_l (no groups; its gradients are finite at |x1-x2| = 0);
 *      kind = 2: Matern-1/2 (exponential), out[l,i,j] = sigma_l^2 exp(-|x1_i-x2_j| / ls_l) (no groups; the backward takes the
 *      sub-gradient 0 at |x1-x2| = 0); kind = 3: Matern-5/2, out[l,i,j] = sigma_l^2 (1 + v + v^2/3) exp(-v),
 *      v = sqrt(5) |x1_i-x2_j| / ls_l (no groups).  Other kinds, and kinds 1-3 with groups, return GPZ_ERR_UNSUPPORTED.
 *      out_lo (optional, f32 only): lo = out - tf32_trunc(out), the second operand of the split-TF32 GEMMs. */
int gpz_kernel_build_fwd_f32(const float* x1, const float* x2, const float* sigma, const float* ls, const float* a,
                             const float* r2, const int64_t* g1, const int64_t* g2, int n1, int n2, int D, int L, int ng, int kind,
                             float p_half, float jitter, float* out, float* out_lo, void* stream);
int gpz_kernel_build_fwd_f64(const double* x1, const double* x2, const double* sigma, const double* ls, const double* a,
                             const double* r2, const int64_t* g1, const int64_t* g2, int n1, int n2, int D, int L, int ng, int kind,
                             double p_half, double jitter, double* out, double* out_lo, void* stream);
/* backward of the above (autograd of kernels.py forward): G = dLoss/dout; g_x1/g_x2/g_a may be NULL.
 * ws: 3*L + n1*D doubles of scratch (parameter and x1 gradients are accumulated in fp64). */
int gpz_kernel_build_bwd_f32(const float* x1, const float* x2, const float* sigma, const float* ls, const float* a,
                             const float* r2, const int64_t* g1, const int64_t* g2, int n1, int n2, int D, int L, int ng, int kind,
                             float p_half, const float* G, float* g_x1, float* g_x2, float* g_sigma, float* g_ls, float* g_a,
                             double* ws, void* stream);
int gpz_kernel_build_bwd_f64(const double* x1, const double* x2, const double* sigma, const double* ls, const double* a,
                             const double* r2, const int64_t* g1, const int64_t* g2, int n1, int n2, int D, int L, int ng, int kind,
                             double p_half, const double* G, double* g_x1, double* g_x2, double* g_sigma, double* g_ls,
                             double* g_a, double* ws, void* stream);
/* ---- K1 with per-dimension (ARD) lengthscales, every kind, no groups (csrc/kernel_build.cu):
 *      ls is L x D (row-major); s2 = sum_d (x1_i,d - x2_j,d)^2 / ls[l,d]^2, r = sqrt(s2);
 *      kind = 0: out[l,i,j] = sigma_l^2 exp(-s2/2); kind = 1: sigma_l^2 (1 + v) exp(-v), v = sqrt(3) r;
 *      kind = 2: sigma_l^2 exp(-r) (the backward takes the sub-gradient 0 at r = 0); kind = 3: sigma_l^2 (1 + v + v^2/3) exp(-v),
 *      v = sqrt(5) r; (+ jitter if i==j).  Equal ls[l,d] = ls_l give gpz_kernel_build_fwd of the same kind.
 *      Kinds outside 0-3, D outside 1-4 and L outside the limits of the isotropic calls return GPZ_ERR_UNSUPPORTED.
 *      out_lo and the fwd_h planes and out_scale (sigma_l^2 + |jitter| in (2^14, 2^15]) are as in the isotropic calls.
 *      bwd: g_ls is L x D; g_x1/g_x2 may be NULL; ws: L + L*D + n1*D doubles of scratch. */
int gpz_kernel_build_ard_fwd_f32(const float* x1, const float* x2, const float* sigma, const float* ls, int n1, int n2, int D,
                                 int L, int kind, float jitter, float* out, float* out_lo, void* stream);
int gpz_kernel_build_ard_fwd_f64(const double* x1, const double* x2, const double* sigma, const double* ls, int n1, int n2, int D,
                                 int L, int kind, double jitter, double* out, double* out_lo, void* stream);
int gpz_kernel_build_ard_fwd_h_f32(const float* x1, const float* x2, const float* sigma, const float* ls, int n1, int n2, int D,
                                   int L, int kind, float jitter, void* out_h, void* out_l, float* out_scale, void* stream);
int gpz_kernel_build_ard_bwd_f32(const float* x1, const float* x2, const float* sigma, const float* ls, int n1, int n2, int D,
                                 int L, int kind, const float* G, float* g_x1, float* g_x2, float* g_sigma, float* g_ls,
                                 double* ws, void* stream);
int gpz_kernel_build_ard_bwd_f64(const double* x1, const double* x2, const double* sigma, const double* ls, int n1, int n2, int D,
                                 int L, int kind, const double* G, double* g_x1, double* g_x2, double* g_sigma, double* g_ls,
                                 double* ws, void* stream);
/* kernels.py:118,123-124 (return_distance=True): Euclidean distances n1 x n2 */
int gpz_cdist_f32(const float* x1, const float* x2, float* out, int n1, int n2, int D, void* stream);
int gpz_cdist_f64(const double* x1, const double* x2, double* out, int n1, int n2, int D, void* stream);

/* ---- K2 batched Cholesky fused with the triangular inverse: gp.py:213, 360, 55, 270 (torch.linalg.cholesky).  With
 *      X = Lc^-1 the two triangular solves of gp.py:218 (torch.cholesky_solve) and the solves inside kl_divergence(qU,pU)
 *      (torch kl.py) become triangular products.  W = copy of Kzz (destroyed), outputs Lc and X = Lc^-1 (both lower, upper
 *      triangle zero), tmp = L x M x M scratch; info[l] = 0 or (1-based) index of the first non-positive pivot of factor l. */
int gpz_chol_inv_f32(float* W, float* Lc, float* X, float* tmp, int M, int L, int* info, void* stream);
int gpz_chol_inv_f64(double* W, double* Lc, double* X, double* tmp, int M, int L, int* info, void* stream);
/* the same for large M in fp32 (M % 4 == 0): 256-wide panels whose diagonal blocks run on the cluster kernel of gpz_chol_inv and
 * every larger product on the tcgen05 split-TF32 GEMM in place; lo_ws: 4 L M M floats of scratch (lo planes shadowing W, Lc, X, tmp) */
int gpz_chol_inv_tc_f32(float* W, float* Lc, float* X, float* tmp, float* lo_ws, int M, int L, int* info, void* stream);
/* strided-batched D = alpha op(A) op(B) + beta D with triangular-structure skipping (see csrc/gemm_simt.cuh):
 * S = Lu Lu^T (gp.py:221), W@(S-Kzz) (utilities.py:395) and the O(M^3) backward products are built from it. */
int gpz_gemm_f32(int ta, int tb, int m, int n, int k, float alpha, const float* A, int64_t lda, int64_t sA, const float* B,
                 int64_t ldb, int64_t sB, float beta, float* D, int64_t ldd, int64_t sD, int batch, int a_tri, int b_tri,
                 int d_tri, int splitk, void* stream);
int gpz_gemm_f64(int ta, int tb, int m, int n, int k, double alpha, const double* A, int64_t lda, int64_t sA,
                 const double* B, int64_t ldb, int64_t sB, double beta, double* D, int64_t ldd, int64_t sD, int batch,
                 int a_tri, int b_tri, int d_tri, int splitk, void* stream);
/* batched matrix-vector products (q = Lc^-1 mu and its backward; torch kl.py _batch_mahalanobis's solve):
 * trans == 0: out[l,i] = sum_k A[l,i,k] v[l,k];  trans != 0: out[l,j] = sum_k A[l,k,j] v[l,k];  A is L x rows x cols */
int gpz_gemv_f32(int trans, const float* A, const float* v, float* out, int rows, int cols, int L, void* stream);
int gpz_gemv_f64(int trans, const double* A, const double* v, double* out, int rows, int cols, int L, void* stream);
/* The whole O(M^3) chain of one SVGP step in two calls (fp32, M >= 128, M % 4 == 0; csrc/chain.cu).  Replaces gp.py:208-221
 * (add_jitter is fused upstream, torch.linalg.cholesky, transform_to(lower_cholesky)), the solve_triangular calls inside
 * kl_divergence(qU, pU) (utilities.py:481,616 -> torch kl.py) and the autograd of all of them.
 *   fwd: Kzz (L x M x M, jittered, DESTROYED) -> Lc, Linv = Lc^-1, Lu, T = Linv Lu, q = Linv mu, kl[L];
 *        aux: 6 L M M floats kept for the backward; ws: L M M floats (5 L M M with chol_tc != 0) scratch; info[L] as LAPACK.
 *   bwd: incoming gradients of (Lc, Linv, Lu, T, q, kl) (any may be NULL; triangular ones are read in their lower triangle)
 *        -> gKzz (L x M x M, NOT symmetrised: contract it with a symmetric dKzz), gLu_raw, gmu; ws: 12 L M M + 2 L M floats. */
int gpz_svgp_chain_supported(int M);
int gpz_svgp_chain_fwd_f32(float* Kzz, const float* Lu_raw, const float* mu, float* Lc, float* Linv, float* Lu, float* T, float* q,
                           float* kl, float* aux, float* ws, int M, int L, int chol_tc, int* info, void* stream);
int gpz_svgp_chain_bwd_f32(const float* Lc, const float* Linv, const float* Lu, const float* T, const float* q, const float* mu,
                           const float* aux, const float* gLc_in, const float* gLinv_in, const float* gLu_in, const float* gT_in,
                           const float* gq_in, const float* gkl_in, float* gKzz, float* gLu_raw, float* gmu, float* ws, int M,
                           int L, void* stream);

/* Merged backward of the predictive op and the chain (fp32): gpz_svgp_predict_bwd_h_f32 called with gT = gLinv = NULL and
 * ws_m = [S1 | S1_lo] (2 L M M floats) leaves S1 = A diag(2 gv) A^T (full symmetric) and gq = A gm; this call turns them, gkl and
 * optional incoming gradients of Lc / Lu into gKzz (not symmetrised), gLu_raw, gmu with 8 M x M x M products (csrc/chain.cu).
 * ws: 13 L M M + 2 L M floats. */
int gpz_svgp_chain_bwd_s1_f32(const float* Lc, const float* Linv, const float* Lu, const float* T, const float* q, const float* mu,
                              const float* aux, const float* S1, const float* S1_lo, const float* gqp, const float* gkl_in,
                              const float* gLc_in, const float* gLu_in, float* gKzz, float* gLu_raw, float* gmu, float* ws, int M,
                              int L, void* stream);

/* gp.py:220 transform_to(lower_cholesky): out = tril(raw,-1) + diag(exp(diag raw)), and its backward */
int gpz_lower_cholesky_fwd_f32(const float* raw, float* out, int M, int L, void* stream);
int gpz_lower_cholesky_fwd_f64(const double* raw, double* out, int M, int L, void* stream);
int gpz_lower_cholesky_bwd_f32(const float* g, const float* out, float* graw, int M, int L, void* stream);
int gpz_lower_cholesky_bwd_f64(const double* g, const double* out, double* graw, int M, int L, void* stream);
/* mode 0: tril with halved diagonal (Cholesky backward Phi); 1: (X+X^T)/2 (out != in); 2: tril */
int gpz_tri_op_f32(const float* in, float* out, int M, int L, int mode, void* stream);
int gpz_tri_op_f64(const double* in, double* out, int M, int L, int mode, void* stream);

/* ---- K3/K4 fused predictive mean and variance: gp.py:218-225 + utilities.py:382-397 (svgp_forward).
 *      Inputs Kzx (L x M x N), Linv = Lc^-1, T = Linv Lu, q = Linv mu, kxx (L x N).
 *      Outputs A = Linv Kzx, C = T^T A (both L x M x N, kept for the backward), mean, var (L x N). */
int gpz_svgp_predict_fwd_f32(const float* Kzx, const float* Linv, const float* T, const float* q, const float* kxx,
                             float* A, float* C, float* mean, float* var, int M, int N, int L, void* stream);
int gpz_svgp_predict_fwd_f64(const double* Kzx, const double* Linv, const double* T, const double* q, const double* kxx,
                             double* A, double* C, double* mean, double* var, int M, int N, int L, void* stream);
/* backward; C is overwritten (becomes gC), gA is scratch (L x M x N); gLinv and gT must be zero-filled by the caller */
int gpz_svgp_predict_bwd_f32(const float* Kzx, const float* Linv, const float* T, const float* q, const float* A, float* C,
                             const float* gm, const float* gv, float* gA, float* gKzx, float* gLinv, float* gT, float* gq,
                             int M, int N, int L, void* stream);
int gpz_svgp_predict_bwd_f64(const double* Kzx, const double* Linv, const double* T, const double* q, const double* A,
                             double* C, const double* gm, const double* gv, double* gA, double* gKzx, double* gLinv,
                             double* gT, double* gq, int M, int N, int L, void* stream);

/* tensor-core (tcgen05 split-TF32) variant of the two calls above, fp32 only.  Kzx_lo: lo part of Kzx (kernel_build out_lo);
 * A_lo, C_lo, gA_lo: L x M x N scratch kept between forward and backward / inside the backward; ws: 6*L*M*M + 2*L*N floats
 * (the same buffer must be passed to forward and backward).  gLinv and gT must be zero-filled by the caller. */
int gpz_svgp_predict_tc_supported(int M, int N);
int gpz_svgp_predict_fwd_tc_f32(const float* Kzx, const float* Kzx_lo, const float* Linv, const float* T, const float* q,
                                const float* kxx, float* A, float* A_lo, float* C, float* mean, float* var, float* ws, int M, int N,
                                int L, void* stream);
int gpz_svgp_predict_bwd_tc_f32(const float* Kzx, const float* Kzx_lo, const float* Linv, const float* T, const float* q,
                                const float* A, const float* A_lo, float* C, float* C_lo, const float* gm, const float* gv, float* gA,
                                float* gA_lo, float* gKzx, float* gLinv, float* gT, float* gq, float* ws, int M, int N, int L,
                                void* stream);

/* ---- K5 KL(qU || pU): utilities.py:481,616 -> torch kl.py MVN||MVN, from the whitened T, q (T lower triangular);
 *      ws: L doubles of scratch */
int gpz_mvn_kl_fwd_f32(const float* T, const float* q, const float* Lc, const float* Lu, float* kl, double* ws, int M, int L,
                       void* stream);
int gpz_mvn_kl_fwd_f64(const double* T, const double* q, const double* Lc, const double* Lu, double* kl, double* ws, int M,
                       int L, void* stream);
int gpz_mvn_kl_bwd_f32(const float* g, const float* T, const float* q, const float* Lc, const float* Lu, float* gT, float* gq,
                       float* gLc, float* gLu, int M, int L, void* stream);
int gpz_mvn_kl_bwd_f64(const double* g, const double* T, const double* q, const double* Lc, const double* Lu, double* gT,
                       double* gq, double* gLc, double* gLu, int M, int L, void* stream);

/* ---- K6 VNNGP (gp.py:19-122).  neighbors: idx[n,:] = the K inducing points nearest to x_n, ascending distance, ties to the
 *      lower index (gp.py:64 argsort(cdist)[:, :K]).  fwd: per point and factor the K x K system
 *      kzz = Kzz[l][nn,nn] + jitter I, w = kzz^-1 kxz, mean = w.mu[nn], var = kxx + w^T S[nn,nn] w - w.kxz  (gp.py:67-106).
 *      bwd: scatter-adds dL/dKzz, dL/dS (L x M x M), dL/dmu (L x M), dL/dZ (M x D, through kxz) and gsl = [dL/dsigma | dL/dls]
 *      (2L doubles, through kxz); all outputs are zero-filled by the call.  K <= 16. */
int gpz_vnngp_neighbors_f32(const float* X, const float* Z, int64_t* idx, int N, int M, int D, int K, void* stream);
int gpz_vnngp_neighbors_f64(const double* X, const double* Z, int64_t* idx, int N, int M, int D, int K, void* stream);
int gpz_vnngp_fwd_f32(const float* X, const float* Z, const float* sigma, const float* ls, const float* Kzz, const float* S,
                      const float* mu, const float* kxx, const int64_t* nn, int N, int M, int D, int L, int K, float jitter,
                      float* mean, float* var, void* stream);
int gpz_vnngp_fwd_f64(const double* X, const double* Z, const double* sigma, const double* ls, const double* Kzz, const double* S,
                      const double* mu, const double* kxx, const int64_t* nn, int N, int M, int D, int L, int K, double jitter,
                      double* mean, double* var, void* stream);
int gpz_vnngp_bwd_f32(const float* X, const float* Z, const float* sigma, const float* ls, const float* Kzz, const float* S,
                      const float* mu, const float* kxx, const int64_t* nn, int N, int M, int D, int L, int K, float jitter,
                      const float* gm, const float* gv, float* gKzz, float* gS, float* gmu, float* gZ, double* gsl, void* stream);
int gpz_vnngp_bwd_f64(const double* X, const double* Z, const double* sigma, const double* ls, const double* Kzz, const double* S,
                      const double* mu, const double* kxx, const int64_t* nn, int N, int M, int D, int L, int K, double jitter,
                      const double* gm, const double* gv, double* gKzz, double* gS, double* gmu, double* gZ, double* gsl,
                      void* stream);

/* ---- K7 fused Poisson log-likelihood + loading contraction, forward and backward in one pass:
 *      likelihoods.py:49-53 (get_rate), 80-97 (NSF2), 110-145 (Hybrid_NSF2), 226-253 (NSF), 304-330 (Hybrid_NSF);
 *      utilities.py:479,507,611-614 (ELBO reduction); torch poisson.py log_prob.
 *      spread[f,:] is a variance (clamped at clamp_min, gp.py:228/378/118) for f < n_var and a std-dev otherwise.
 *      ll: one double on the device.  ws sized by gpz_poisson_workspace_bytes_*. */
int64_t gpz_poisson_workspace_bytes_f32(int G, int F, int B, int E);
int64_t gpz_poisson_workspace_bytes_f64(int G, int F, int B, int E);
int gpz_poisson_fwdbwd_f32(const float* y, int64_t y_ld, const int64_t* idx, const float* W, int w_softplus, const float* V,
                           const float* mean, const float* spread, const float* eps, int G, int F, int B, int E, int n_var,
                           float clamp_min, int with_lgamma, double* ll, float* gW, float* gV, float* gmean, float* gspread,
                           void* ws, int64_t ws_bytes, void* stream);
int gpz_poisson_fwdbwd_f64(const double* y, int64_t y_ld, const int64_t* idx, const double* W, int w_softplus,
                           const double* V, const double* mean, const double* spread, const double* eps, int G, int F, int B,
                           int E, int n_var, double clamp_min, int with_lgamma, double* ll, double* gW, double* gV,
                           double* gmean, double* gspread, void* ws, int64_t ws_bytes, void* stream);
/* compatibility path: materialise pY.rate (E x G x B) for callers of model.forward() (likelihoods.py:83-85) */
/* the same with the counts stored as integers: y_kind 1 = uint8, 2 = int16, 3 = int32 (0 = float).  Lossless for count data, a
 * quarter / half of the HBM traffic and of the host upload.  fp32, F <= 16 (the tensor-core kernel); GPZ_ERR_UNSUPPORTED otherwise. */
int gpz_poisson_fwdbwd_yt_f32(const void* y, int y_kind, int64_t y_ld, const int64_t* idx, const float* W, int w_softplus, const float* V,
                              const float* mean, const float* spread, const float* eps, int G, int F, int B, int E, int n_var,
                              float clamp_min, int with_lgamma, double* ll, float* gW, float* gV, float* gmean, float* gspread,
                              void* ws, int64_t ws_bytes, void* stream);
/* K7-CSC: the same call on sparse counts, whose work scales with the nonzeros instead of G x N.  The count matrix is stored as
 * spot-major compressed columns (AnnData's N x G CSR): spot n owns entries indptr[n] .. indptr[n+1] (int64, n_total + 1 of them)
 * of genes (int32, in [0, G), ascending and unique within a spot) and counts (count_kind 0 = T, 1 = uint8, 2 = int16,
 * 3 = int32; non-negative, no explicit zeros needed).  idx (B or NULL; NULL requires B == n_total) picks the columns of the
 * resident matrix, no gather copy.  The y = 0 entries enter in closed form through the column sums of the loadings; c_f, u_f,
 * ll and the final combination of the d/dW partials are carried in double.  Outputs and conventions as gpz_poisson_fwdbwd_*;
 * F <= 32 (GPZ_ERR_UNSUPPORTED otherwise), any E.  ws sized by gpz_poisson_csc_workspace_bytes_*. */
int64_t gpz_poisson_csc_workspace_bytes_f32(int G, int F, int B, int E);
int64_t gpz_poisson_csc_workspace_bytes_f64(int G, int F, int B, int E);
int gpz_poisson_fwdbwd_csc_f32(const int64_t* indptr, const int32_t* genes, const void* counts, int count_kind, int64_t n_total,
                               const int64_t* idx, const float* W, int w_softplus, const float* V, const float* mean,
                               const float* spread, const float* eps, int G, int F, int B, int E, int n_var, float clamp_min,
                               int with_lgamma, double* ll, float* gW, float* gV, float* gmean, float* gspread, void* ws,
                               int64_t ws_bytes, void* stream);
int gpz_poisson_fwdbwd_csc_f64(const int64_t* indptr, const int32_t* genes, const void* counts, int count_kind, int64_t n_total,
                               const int64_t* idx, const double* W, int w_softplus, const double* V, const double* mean,
                               const double* spread, const double* eps, int G, int F, int B, int E, int n_var, double clamp_min,
                               int with_lgamma, double* ll, double* gW, double* gV, double* gmean, double* gspread, void* ws,
                               int64_t ws_bytes, void* stream);
/* K7-NB: the same call with a negative-binomial likelihood, one dispersion per gene, theta_g = softplus(D_g):
 *   log NB(y | r, theta) = lgamma(y + theta) - lgamma(theta) - lgamma(y + 1) + y log(r / (theta + r)) - theta log1p(r / theta)
 *   ll = mean_e sum_{g,n} log NB; with_lgamma = 0 drops only lgamma(y + 1).  D (G, raw) is an input, gD = d ll / d D (G) an
 *   output; every other argument and output as gpz_poisson_fwdbwd_*.  Dense counts only.  ws sized by gpz_negbin_workspace_bytes_*. */
int64_t gpz_negbin_workspace_bytes_f32(int G, int F, int B, int E);
int64_t gpz_negbin_workspace_bytes_f64(int G, int F, int B, int E);
int gpz_negbin_fwdbwd_f32(const float* y, int64_t y_ld, const int64_t* idx, const float* W, int w_softplus, const float* V,
                          const float* D, const float* mean, const float* spread, const float* eps, int G, int F, int B, int E,
                          int n_var, float clamp_min, int with_lgamma, double* ll, float* gW, float* gV, float* gD, float* gmean,
                          float* gspread, void* ws, int64_t ws_bytes, void* stream);
int gpz_negbin_fwdbwd_f64(const double* y, int64_t y_ld, const int64_t* idx, const double* W, int w_softplus, const double* V,
                          const double* D, const double* mean, const double* spread, const double* eps, int G, int F, int B, int E,
                          int n_var, double clamp_min, int with_lgamma, double* ll, double* gW, double* gV, double* gD,
                          double* gmean, double* gspread, void* ws, int64_t ws_bytes, void* stream);
/* counts stored as integers (y_kind as gpz_poisson_fwdbwd_yt_f32; fp32, F <= 16) */
int gpz_negbin_fwdbwd_yt_f32(const void* y, int y_kind, int64_t y_ld, const int64_t* idx, const float* W, int w_softplus,
                             const float* V, const float* D, const float* mean, const float* spread, const float* eps, int G, int F,
                             int B, int E, int n_var, float clamp_min, int with_lgamma, double* ll, float* gW, float* gV, float* gD,
                             float* gmean, float* gspread, void* ws, int64_t ws_bytes, void* stream);
/* K7-G: the Gaussian factor model of RSF / FA (csrc/gaussian.cu), y_gn ~ N(bias_g + sum_f W_gf F_fn, s_g^2), s = softplus(noise),
 *   real-valued y (G x Ntot, row stride y_ld), real loadings W (G x F), bias and raw noise (G).  The expectation over
 *   q(F) = N(mean, v) is exact, so there are no samples:
 *   ll = sum_{g,n} [ -1/2 log 2 pi - log s_g - (y_gn - bias_g - sum_f W_gf mean_fn)^2 / (2 s_g^2) ] - 1/2 sum_{g,f} W_gf^2 V_f / s_g^2,
 *   V_f = sum_n v_fn.  spread as gpz_poisson_fwdbwd_* (v = max(spread, clamp_min) for f < n_var, spread^2 otherwise); idx (B or
 *   NULL) gathers y[:, idx]; nothing is rescaled by Ntot / B.  Outputs: ll (one double), gW, gbias, gnoise (G x F, G, G), gmean,
 *   gspread (F x B).  y is read once and nothing of size G x B is written; partials are summed in a fixed order (no atomics).
 *   1 <= F <= 32, 0 <= n_var <= F, and y_ld >= B without idx; GPZ_ERR_UNSUPPORTED otherwise.  ws sized by
 *   gpz_gaussian_workspace_bytes_*. */
int64_t gpz_gaussian_workspace_bytes_f32(int G, int F, int B);
int64_t gpz_gaussian_workspace_bytes_f64(int G, int F, int B);
int gpz_gaussian_fwdbwd_f32(const float* y, int64_t y_ld, const int64_t* idx, const float* W, const float* bias, const float* noise,
                            const float* mean, const float* spread, int G, int F, int B, int n_var, float clamp_min, double* ll,
                            float* gW, float* gbias, float* gnoise, float* gmean, float* gspread, void* ws, int64_t ws_bytes,
                            void* stream);
int gpz_gaussian_fwdbwd_f64(const double* y, int64_t y_ld, const int64_t* idx, const double* W, const double* bias,
                            const double* noise, const double* mean, const double* spread, int G, int F, int B, int n_var,
                            double clamp_min, double* ll, double* gW, double* gbias, double* gnoise, double* gmean,
                            double* gspread, void* ws, int64_t ws_bytes, void* stream);
/* the digamma and lgamma of the K7-NB kernels (x > 0), element-wise over n doubles on the device */
int gpz_digamma_f64(const double* x, double* out, int64_t n, void* stream);
int gpz_lgamma_f64(const double* x, double* out, int64_t n, void* stream);
int gpz_poisson_rate_f32(const float* W, int w_softplus, const float* V, const int64_t* idx, const float* F, float* rate,
                         int G, int nF, int B, int E, void* stream);
int gpz_poisson_rate_f64(const double* W, int w_softplus, const double* V, const int64_t* idx, const double* F, double* rate,
                         int G, int nF, int B, int E, void* stream);

/* ---- tcgen05 / TMA batched GEMM in split-TF32 arithmetic (fp32 hot path of K3/K4 and their backward; csrc/umma_gemm.cu).
 *      D = alpha A op(B) (+ Cin), A m x k K-major; op(B): b_kmajor=0 -> B is k x n (n contiguous), 1 -> B is n x k.
 *      Alo/Blo: lo = x - tf32_trunc(x) parts (n_terms=3) or NULL (n_terms=1); Dlo (optional) receives the lo part of D.
 *      Replaces the cuBLAS GEMMs behind torch.cholesky_solve / W@(S-Kzz) (gp.py:218, utilities.py:395) and autograd's. */
int gpz_umma_gemm_supported(int b_kmajor, int m, int n, int k, int64_t lda, int64_t ldb, int64_t ldd);
int gpz_umma_gemm_f32(int b_kmajor, int m, int n, int k, float alpha, const float* A, const float* Alo, int64_t lda, int64_t sA,
                      const float* B, const float* Blo, int64_t ldb, int64_t sB, const float* Cin, float* D, float* Dlo,
                      int64_t ldd, int64_t sD, int batch, int a_tri, int b_tri, int d_tri, int splitk, int n_terms, void* stream);
/* lo = x - tf32_trunc(x) (flat array);  xt = x^T per M x M matrix with optional lo part */
int gpz_tf32_lo_f32(const float* x, float* lo, int64_t n, void* stream);
int gpz_transpose_lo_f32(const float* x, float* xt, float* xt_lo, int M, int L, void* stream);

/* ---- the same GEMM in split-FP16 arithmetic (twice the tensor-core rate of split-TF32 at the same ~2^-22 accuracy).
 *      Operands are pairs of fp16 planes (hi, lo) of x * s[b]: hi = rn(x s), lo = rn(x s - hi), s[b] a per-batch power of two
 *      in device memory chosen from a bound on max |x| so that nothing overflows (gpz_split16 picks it from the exact max).
 *      The kernel issues hi*lo + lo*hi + hi*hi into one TMEM accumulator and undoes the scales in the epilogue.
 *      Outputs (each optional): D fp32 (+ Cin, an fp32 addend that may alias D); (Dh, Dl) fp16 planes of D * sd[b];
 *      amax[b] = max |D| as float bits (atomicMax).  a_tri / b_tri / d_tri: op(A) / op(B) / D lower (1) or upper (2) triangular. */
int gpz_split16_f32(const float* x, int rows, int cols, int batch, void* h, void* l, void* hT, void* lT, float* scale,
                    void* amax_ws, void* stream);
int gpz_umma_gemm16_f32(int b_kmajor, int m, int n, int k, float alpha, const void* Ah, const void* Al, int64_t lda, int64_t sA,
                        const float* sa, const void* Bh, const void* Bl, int64_t ldb, int64_t sB, const float* sb,
                        const float* Cin, float* D, void* Dh, void* Dl, const float* sd, void* amax, int64_t ldd, int64_t sD,
                        int batch, int a_tri, int b_tri, int d_tri, int splitk, int n_terms, void* stream);

/* split-FP16 K1 forward and SVGP predictive op (the default fp32 hot path; csrc/kernel_build.cu, csrc/predict.cu):
 *      kernel_build_fwd_h writes K as fp16 planes (out_h + out_l ~= K * out_scale[l], 4 bytes per entry) instead of fp32;
 *      predict_fwd_h / predict_bwd_h are gpz_svgp_predict_fwd/bwd (gp.py:218-225, utilities.py:382-397 and their autograd)
 *      on those planes: A, C, gA and AW = A diag(2 gv) (scratch of the backward) travel as fp16 planes as well; gKzx, gLinv, gT,
 *      gq, mean, var are fp32.  The backward never forms gC = C diag(2 gv): gA = 2 gv o (T C - A) + q gm^T comes straight from
 *      the unweighted C planes (column weights commute out of the product), gT = tril(AW C^T).
 *      ws_h: 8 L M M halfs, ws_f: 2 L N + 16 L floats, both written by fwd and read by bwd; gT and gLinv zero-initialised. */
int gpz_kernel_build_fwd_h_f32(const float* x1, const float* x2, const float* sigma, const float* ls, const float* a,
                               const float* r2, const int64_t* g1, const int64_t* g2, int n1, int n2, int D, int L, int ng, int kind,
                               float p_half, float jitter, void* out_h, void* out_l, float* out_scale, void* stream);
int gpz_svgp_predict_h_supported(int M, int N);
/* row (of L floats, counted from ws_f + 2 L N) of: 0 scale of A, 1 max|A|, 2 max|C|, 3 scale of gA, 4 max|gA|, 5 scale of C —
 * what the host-side overflow guard of the fp16 planes reads */
int gpz_svgp_predict_h_stat_row(int which);
int gpz_svgp_predict_fwd_h_f32(const void* Kh, const void* Kl, const float* sK, const float* Linv, const float* T, const float* q,
                               const float* kxx, void* Ah, void* Al, void* Ch, void* Cl, float* mean, float* var, void* ws_h,
                               float* ws_f, int M, int N, int L, void* stream);
int gpz_svgp_predict_bwd_h_f32(const void* Kh, const void* Kl, const float* sK, const float* T, const float* q, const void* Ah,
                               const void* Al, const void* Ch, const void* Cl, const float* gm, const float* gv, void* AWh, void* AWl,
                               void* gAh, void* gAl, float* gKzx, float* gLinv, float* gT, float* gq, void* ws_h, float* ws_f,
                               float* ws_m, int M, int N, int L, void* stream);
/*      ws_m NULL: the backward runs the two reductions over the N spots gT = tril(AW C^T), gLinv = tril(gA Kzx^T).
 *      ws_m = [S1 | S1_lo] (2 L M M floats), which requires gT = gLinv = NULL (GPZ_ERR_BADARG otherwise): it runs ONE reduction,
 *      S1 = A diag(2 gv) A^T, for gpz_svgp_chain_bwd_s1_f32. */

/* ---- training-step update (SURVEY §8(f) row 1): multi-tensor Adam in one launch (torch.optim.Adam without weight decay /
 *      amsgrad; utilities.py:621 optimizer.step()) with the reference's post-step clamp W.clamp_(min=0) (utilities.py:623) fused in
 *      for the tensors flagged in clamp0.  The pointer tables are HOST arrays of device pointers; step counts from 1. */
int gpz_adam_step_f32(int n_tensors, void* const* params, void* const* grads, void* const* exp_avg, void* const* exp_avg_sq,
                      const int64_t* numel, const int* clamp0, double lr, double beta1, double beta2, double eps, int step,
                      void* stream);
int gpz_adam_step_f64(int n_tensors, void* const* params, void* const* grads, void* const* exp_avg, void* const* exp_avg_sq,
                      const int64_t* numel, const int* clamp0, double lr, double beta1, double beta2, double eps, int step,
                      void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GPZOO_B200_H */
