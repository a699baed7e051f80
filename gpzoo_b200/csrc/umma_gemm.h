// Internal (non-ABI) entries of the tcgen05 GEMMs with the fused epilogues used by csrc/predict.cu.
#pragma once
#include <cuda_fp16.h>
#include <stdint.h>

struct UmmaEpilogue {
  int mode;              // see Params::epi_mode in umma_gemm.cu
  const float* Aux; const float* rowv; const float* colv1; const float* colv2;
  float* col1; float* col2; float* rowacc;
};

// split-TF32 arithmetic on fp32 operands (x, lo)
int umma_gemm_ex(int b_kmajor, int m, int n, int k, float alpha, const float* A, const float* Alo, int64_t lda, int64_t sA,
                 const float* B, const float* Blo, int64_t ldb, int64_t sB, const float* Cin, float* D, float* Dlo, int64_t ldd,
                 int64_t sD, int batch, int a_tri, int b_tri, int d_tri, int splitk, int n_terms, const UmmaEpilogue* epi,
                 void* stream, int max_ctas = 0);     // max_ctas > 0: at most that many persistent CTAs (leaves SMs to other streams)

// split-FP16 arithmetic: operands are fp16 planes (hi, lo) of x * s[b], s[b] a per-batch power of two kept in device memory
struct Umma16Args {
  int b_kmajor, m, n, k;
  float alpha;
  const __half* Ah; const __half* Al; int64_t lda, sA; const float* sa;     // A: m x k, k contiguous
  const __half* Bh; const __half* Bl; int64_t ldb, sB; const float* sb;     // B: k x n (n contiguous) or, b_kmajor, n x k
  float* D; int64_t ldd, sD;                                                // optional fp32 output
  const float* Cin;                                                         // optional fp32 addend (same layout as D; may be D)
  int b_tri;                                                                // op(B) (k x n) lower (1) / upper (2) triangular
  __half* Dh; __half* Dl; const float* sd;                                  // optional fp16 (hi, lo) output of D * sd[b]
  unsigned int* amax;                                                       // optional per-batch max |D| (float bits)
  int batch, a_tri, d_tri, splitk, n_terms;
  const UmmaEpilogue* epi;                                                  // fused epilogue (mode 3 may use AuxH/AuxL)
  const __half* AuxH; const __half* AuxL; const float* saux;
  __half* D2h; __half* D2l; const float* sd2;                               // epilogue mode 4: second fp16-plane output
};
int umma_gemm16_ex(const Umma16Args& args, void* stream);

// scale[b] = 2^(15 - ceil(log2 amax[b])) (so that amax * scale is in (2^14, 2^15]); (hi, lo) planes of x * scale and,
// optionally, of the per-matrix transpose.  amax_bits: per-batch max |x| as float bits (computed by split16_amax).
int split16_amax(const float* x, int64_t per_batch, int batch, unsigned int* amax_bits, void* stream);
int split16_planes(const float* x, int rows, int cols, int batch, const unsigned int* amax_bits, float* scale, __half* h, __half* l,
                   __half* hT, __half* lT, void* stream);

__host__ __device__ inline float gpz_pow2_scale(float bound) {
  // power of two s with bound * s in (2^14, 2^15]; 1 for bound == 0 / non-finite
  if (!(bound > 0.f) || bound > 3.0e38f) return 1.0f;
  int e;
  frexpf(bound, &e);                 // bound = f * 2^e, f in [0.5, 1)  ->  bound <= 2^e
  int se = 15 - e;
  se = se < -100 ? -100 : (se > 100 ? 100 : se);
  return ldexpf(1.0f, se);
}
