// tcgen05 / TMEM / TMA batched GEMM in split-precision arithmetic for the fp32 hot path.
//
// The big contractions of the SVGP step (the triangular products that replace cholesky_solve, gp.py:218, and
// svgp_forward, utilities.py:392-395, plus their backward) are genuine dense GEMMs.  The parity target (1e-4 of the
// fp64 reference on gradients, through a Cholesky factor of condition ~100) rules out a single tensor-core pass (TF32: 7.7e-4,
// FP16: 2.9e-4 per GEMM), so every operand travels as a pair (hi, lo) and each k-step issues three MMAs into the same TMEM
// accumulator,  D += hi_A*lo_B ;  D += hi_A*hi_B ;  D += lo_A*hi_B,  which recovers ~2^-22 per product.  Two arithmetics:
//   split-FP16 (template F16, the default): operands are two fp16 planes of x * s[b] (hi = rn(x s), lo = rn(x s - hi), s[b] a
//     per-batch power of two in device memory, 4 bytes per entry), kind::f16 MMAs (K = 16) at the f16 rate;
//   split-TF32: operands are fp32 x plus an fp32 plane lo = x - tf32_trunc(x) (8 bytes per entry; the tensor core truncates x
//     itself), kind::tf32 MMAs (K = 8) at half that rate.  Kept for the M x M x M products and for shapes that are not 8-aligned.
//
//   D[b] (m x n) = alpha * A[b] (m x k, K-major: row-major, k contiguous) * op(B[b]) (+ Cin[b])
//   op(B): B stored k x n with n contiguous ("MN-major", the layout of Kzx / A / gC / gA: L x M x N), or
//          B stored n x k with k contiguous ("K-major", used for the reductions over the N spots).
//
// Persistent: one CTA per SM (320 threads), 128 x 256 output tiles from an atomic counter.  Warp 0: scheduler + TMA producer
// (cp.async.bulk.tensor into a 4-stage ring of 48 KB stages of 64 bytes of k per row; 64B-swizzled K-major tiles, MN-major tiles
// 128B-swizzled in fp16 / 128B(32B-atom)-swizzled in tf32).  Warp 1: allocates the 512 TMEM columns (two accumulators) and issues
// tcgen05.mma (M=128, N=256) from one thread, releasing stages and publishing accumulators with tcgen05.commit.  Warps 2-9:
// epilogue (two warps per TMEM lane quadrant): tcgen05.ld -> XOR-swizzled shared-memory transpose -> scales / fused reductions /
// fp16 split / max tracking -> full-line stores (or fp32 atomics for split-K), overlapping the next tile's MMAs.
// Triangular operands skip whole k-blocks; lower-triangular outputs skip whole tiles and use N=128 MMAs on diagonal tiles.
#include <cuda.h>
#include <cuda_fp16.h>

#include <atomic>

#include "common.cuh"
#include "gpzoo_b200.h"
#include "umma_gemm.h"

namespace gpz {
namespace umma {

// A stage holds 64 bytes of k per row: 16 fp32 (tf32 arithmetic) or 32 fp16 (split-FP16 arithmetic) elements, so the
// byte geometry of the K-major tiles (and the stage size) is the same in both modes.
#ifndef GPZ_UMMA_STAGES
#define GPZ_UMMA_STAGES 4
#endif
#ifndef GPZ_UMMA_EPI_WARPS
#define GPZ_UMMA_EPI_WARPS 8
#endif
// Epilogue modes 3 / 4 read an Aux tile (fp16 planes).  AUX_AHEAD = 1 makes the epilogue warps prefetch the NEXT tile's Aux
// region into L2 (peeking at the scheduler's other slot) instead of the current tile's; measured SLOWER on the B200
// (svgp_predict_bwd_h 3.29 -> 3.46 ms: the extra L2 traffic competes with the two output streams), so it is off.
#ifndef GPZ_UMMA_AUX_AHEAD
#define GPZ_UMMA_AUX_AHEAD 0
#endif
constexpr int BM = 128, BN = 256, BK = 16, BK16 = 32, STAGES = GPZ_UMMA_STAGES;
constexpr int A_BYTES = BM * BK * 4;          // 8 KB   (128 rows x 64 B, SWIZZLE_64B)
constexpr int B_BYTES = BN * BK * 4;          // 16 KB  (K-major: 256 rows x 64 B; MN-major tf32: 8 chunks x 16 k-rows x 128 B;
                                              //         MN-major fp16: 4 chunks x 32 k-rows x 128 B)
constexpr int STAGE_BYTES = 2 * A_BYTES + 2 * B_BYTES;   // raw + lo of both operands = 48 KB
constexpr int EPI_WARPS = GPZ_UMMA_EPI_WARPS;  // EPI_WARPS / 4 epilogue warps per TMEM lane quadrant, each owns an equal share of the tile's columns
constexpr int EPI_CHUNKS = (BN / 32) / (EPI_WARPS / 4);      // 32-column chunks per epilogue warp
static_assert(EPI_WARPS % 4 == 0 && (BN / 32) % (EPI_WARPS / 4) == 0, "epilogue warps must split the tile's column chunks evenly");
constexpr int EPI_BYTES = EPI_WARPS * 32 * 32 * 4;  // per-warp 32 x 32 fp32 staging tile, XOR-swizzled 16-byte columns
constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /*align slack*/ + 256 /*barriers*/ + EPI_BYTES;
constexpr int NTHREADS = 64 + 32 * EPI_WARPS;
static_assert(SMEM_BYTES <= 232448, "shared memory per CTA");
constexpr uint32_t TMEM_COLS = 512;      // two 128 x 256 fp32 accumulators

struct Params {
  float* D; float* Dlo; const float* Cin;
  int m, n, k;
  int64_t ldd, sD;
  int batch, splitk;
  int a_tri, b_tri, d_tri;
  int n_terms;            // 3: split-TF32, 1: plain TF32
  int b_map4d;            // MN-major B loaded with one 4-D box per stage (needs n % 32 == 0)
  // fused epilogues of the SVGP predictive op (csrc/predict.cu); vectors are per batch entry
  //   1: col1[n] += sum_i D[i,n]^2 ; col2[n] += sum_i rowv[i] D[i,n]                     (A = Linv Kzx: sum A^2 and mean)
  //   2: col1[n] += sum_i D[i,n]^2                                                        (C = T^T A: sum C^2)
  //   3: D = acc - 2 Aux[i,n] colv1[n] + rowv[i] colv2[n] ; rowacc[i] += sum_n Aux[i,n] colv2[n]   (gA and gq = A gm)
  //   4: D = 2 colv1[n] (acc - Aux[i,n]) + rowv[i] colv2[n] ; rowacc as 3 ; D2 = 2 colv1[n] Aux[i,n]  (fp16 planes D2h/D2l * sd2)
  //      (gA from the UNweighted C planes: the column weights 2 gv commute out of T C diag(2 gv); D2 = A diag(2 gv) feeds gT)
  int epi_mode;
  const float* Aux; const float* rowv; const float* colv1; const float* colv2;
  float* col1; float* col2; float* rowacc;
  float alpha;
  // split-FP16 mode: operands are (hi, lo) fp16 planes of x * s[b] with per-batch power-of-two scales s
  int bk;                                 // k elements per stage (BK or BK16)
  const float* sa; const float* sb;       // operand scales (nullptr = 1): the accumulator is multiplied by 1/(sa[b] sb[b])
  __half* Dh; __half* Dl; const float* sd;   // optional (hi, lo) fp16 output planes of D * sd[b]  (same ldd / sD as D)
  unsigned int* amax;                     // optional per-batch max |D| (float bits, atomicMax)
  const __half* AuxH; const __half* AuxL; const float* saux;   // epi_mode 3 / 4: Aux given as fp16 planes instead of fp32
  __half* D2h; __half* D2l; const float* sd2;                 // epi_mode 4: second output (same ldd / sD as D)
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t done = 0;
  const uint32_t addr = smem_u32(bar);
  while (!done) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
  }
}
// non-blocking probe of an mbarrier phase (acquire): true when the phase with this parity has completed
__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(done)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return done != 0;
}
__device__ __forceinline__ void tma_load_3d(const CUtensorMap* map, uint64_t* bar, void* dst, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(const CUtensorMap* map, uint64_t* bar, void* dst, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// x * s -> (hi, lo) fp16 pair, hi = rn(x s), lo = rn(x s - hi): 22 significant bits; an out-of-range value becomes inf
// (and the products NaN) so that a violated scale bound is loud, never silently saturated
__device__ __forceinline__ void split_half(float xs, __half& h, __half& l) {
  h = __float2half_rn(xs);
  l = __float2half_rn(xs - __half2float(h));
}
// two values at once with the packed conversions (cvt.rn.f16x2.f32)
__device__ __forceinline__ void split_half2(float a, float b, uint32_t& h, uint32_t& l) {
  const __half2 hh = __floats2half2_rn(a, b);
  const float2 hf = __half22float2(hh);
  const __half2 ll = __floats2half2_rn(a - hf.x, b - hf.y);
  h = *reinterpret_cast<const uint32_t*>(&hh);
  l = *reinterpret_cast<const uint32_t*>(&ll);
}
__device__ __forceinline__ float unpack_sum(uint32_t h, uint32_t l, int hi_half) {
  const unsigned short hs = hi_half ? (unsigned short)(h >> 16) : (unsigned short)(h & 0xffffu);
  const unsigned short ls = hi_half ? (unsigned short)(l >> 16) : (unsigned short)(l & 0xffffu);
  return __half2float(__ushort_as_half(hs)) + __half2float(__ushort_as_half(ls));
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, "
      "%25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
        "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// explicit shared-memory accesses of the epilogue staging tile (the tile's address is derived by integer arithmetic from the
// dynamic shared-memory base, so plain pointer dereferences compile to generic LD.E / ST.E with their longer latency)
__device__ __forceinline__ float4 lds128(uint32_t saddr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(saddr) : "memory");
  return v;
}
__device__ __forceinline__ void sts128(uint32_t saddr, float a, float b, float c, float d) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(saddr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
// tcgen05.ld without the wait (the caller overlaps global prefetches with the TMEM read latency)
__device__ __forceinline__ void tmem_ld32_nowait(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, "
      "%25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
        "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Specialised epilogue of one warp for a tile that lies completely inside the matrix (the common case of the N-proportional
// split-FP16 GEMMs): 4 chunks of 32 columns, everything addressed incrementally, no runtime mode tests in the inner loop.
//   MODE 0: plain   1: + sum_i D^2 and sum_i rowv_i D per column   2: + sum_i D^2   3: D = acc - 2 Aux colv1 + rowv colv2, rowacc
//   OUT_D: fp32 store;  OUT_H: (hi, lo) fp16 planes of D * sd.  MODE 3 reads Aux as fp16 planes (prefetched into L2 by the caller).
template <int MODE, bool OUT_D, bool OUT_H>
__device__ __forceinline__ void epilogue_tile_fast(const Params& p, int b, int i0, int j0, int q, int lane, int c_begin,
                                                   uint32_t tmem_acc, float* epi, float alpha_b, float sd_b, float inv_saux,
                                                   float& amx, float sd2_b = 1.0f) {
  const int lr = lane >> 3, cq = (lane & 7) * 4;
  const int row0 = i0 + q * 32;
  const int64_t ld4 = 4 * p.ldd;
  int64_t o_chunk = (int64_t)b * p.sD + (int64_t)(row0 + lr) * p.ldd + j0 + c_begin * 32 + cq;   // element of (row lr, this lane's 4 columns)
  const int64_t colbase = (int64_t)b * p.n + j0 + c_begin * 32 + cq;
  float racc[8];
  const float* qrow = p.rowv + (int64_t)b * p.m + row0 + lr;      // rowv of row (4 itr + lr): re-read per use (L1), saves 8 registers
  if (MODE == 3 || MODE == 4) {
#pragma unroll
    for (int u = 0; u < 8; ++u) racc[u] = 0.f;
  }
#ifndef GPZ_UMMA_AUX_WIN
#define GPZ_UMMA_AUX_WIN 4                         // rows of the Aux planes held ahead in registers (4 or 8)
#endif
  constexpr int AW = GPZ_UMMA_AUX_WIN;
  static_assert(AW == 4 || AW == 8, "Aux window");
  uint2 axh[AW], axl[AW];                            // Aux planes of AW rows ahead: a rotating window
  const uint32_t srd = smem_u32(epi) + lr * 128;     // staging read: row (4 itr + lr), 16-byte slot (lane & 7) ^ (row & 7)
  const uint32_t swr = smem_u32(epi) + lane * 128;   // staging write: row lane
#pragma unroll 1
  for (int cc = 0; cc < EPI_CHUNKS; ++cc) {
    uint32_t r[32];
    tmem_ld32_nowait(tmem_acc + (uint32_t)((c_begin + cc) * 32), r);
    float4 cv1, cv2;
    if (MODE == 3 || MODE == 4) {
      cv1 = __ldg(reinterpret_cast<const float4*>(p.colv1 + colbase + cc * 32));
      cv2 = __ldg(reinterpret_cast<const float4*>(p.colv2 + colbase + cc * 32));
      // (the Aux region of this warp was prefetched into L2 while the tile before was in the epilogue; every row's slot is
      // refilled with the same row of the NEXT chunk as soon as it is consumed, so a load has a whole chunk to complete: the
      // round-2 capture showed 69 % of the epilogue's samples stalled on these loads with a 4-row window)
      if (cc == 0) {
#pragma unroll
        for (int u = 0; u < AW; ++u) {
          axh[u] = __ldcs(reinterpret_cast<const uint2*>(p.AuxH + o_chunk + u * ld4));
          axl[u] = __ldcs(reinterpret_cast<const uint2*>(p.AuxL + o_chunk + u * ld4));
        }
      }
    }
    tmem_ld_wait();
#pragma unroll
    for (int u = 0; u < 32; u += 4)
      sts128(swr + (((u >> 2) ^ (lane & 7)) << 4), __uint_as_float(r[u]), __uint_as_float(r[u + 1]), __uint_as_float(r[u + 2]),
             __uint_as_float(r[u + 3]));
    __syncwarp();
    float4 cs1 = make_float4(0.f, 0.f, 0.f, 0.f), cs2 = cs1;
#pragma unroll
    for (int itr = 0; itr < 8; ++itr) {
      // row = 4 itr + lr, so row & 7 = (4 (itr & 1) + lr) & 7
      float4 v = lds128(srd + itr * 512 + ((((lane & 7) ^ ((4 * (itr & 1) + lr) & 7))) << 4));
      v.x *= alpha_b; v.y *= alpha_b; v.z *= alpha_b; v.w *= alpha_b;
      const int64_t o = o_chunk + itr * ld4;
      if (MODE == 3 || MODE == 4) {
        const uint2 hh = axh[itr % AW], ll = axl[itr % AW];
        if (AW == 8) {
          if (cc + 1 < EPI_CHUNKS) {                   // the slot is free again: fetch the same row of the next chunk
            axh[itr] = __ldcs(reinterpret_cast<const uint2*>(p.AuxH + o + 32));
            axl[itr] = __ldcs(reinterpret_cast<const uint2*>(p.AuxL + o + 32));
          }
        } else if (itr < 4) {                          // fetch row itr + 4 of this chunk
          axh[itr] = __ldcs(reinterpret_cast<const uint2*>(p.AuxH + o + 4 * ld4));
          axl[itr] = __ldcs(reinterpret_cast<const uint2*>(p.AuxL + o + 4 * ld4));
        } else if (cc + 1 < EPI_CHUNKS) {              // ... and row itr - 4 of the next chunk
          axh[itr - 4] = __ldcs(reinterpret_cast<const uint2*>(p.AuxH + o + 32 - 4 * ld4));
          axl[itr - 4] = __ldcs(reinterpret_cast<const uint2*>(p.AuxL + o + 32 - 4 * ld4));
        }
        float4 ax;
        ax.x = unpack_sum(hh.x, ll.x, 0) * inv_saux; ax.y = unpack_sum(hh.x, ll.x, 1) * inv_saux;
        ax.z = unpack_sum(hh.y, ll.y, 0) * inv_saux; ax.w = unpack_sum(hh.y, ll.y, 1) * inv_saux;
        const float qv = __ldg(qrow + itr * 4);
        if (MODE == 3) {
          v.x += fmaf(qv, cv2.x, -2.f * ax.x * cv1.x);
          v.y += fmaf(qv, cv2.y, -2.f * ax.y * cv1.y);
          v.z += fmaf(qv, cv2.z, -2.f * ax.z * cv1.z);
          v.w += fmaf(qv, cv2.w, -2.f * ax.w * cv1.w);
        } else {
          const float4 w = make_float4(2.f * cv1.x, 2.f * cv1.y, 2.f * cv1.z, 2.f * cv1.w);
          v.x = fmaf(w.x, v.x - ax.x, qv * cv2.x);
          v.y = fmaf(w.y, v.y - ax.y, qv * cv2.y);
          v.z = fmaf(w.z, v.z - ax.z, qv * cv2.z);
          v.w = fmaf(w.w, v.w - ax.w, qv * cv2.w);
          uint2 qh, ql;                                 // D2 = A diag(2 gv)
          split_half2(w.x * ax.x * sd2_b, w.y * ax.y * sd2_b, qh.x, ql.x);
          split_half2(w.z * ax.z * sd2_b, w.w * ax.w * sd2_b, qh.y, ql.y);
          *reinterpret_cast<uint2*>(p.D2h + o) = qh;
          *reinterpret_cast<uint2*>(p.D2l + o) = ql;
        }
        racc[itr] += ax.x * cv2.x + ax.y * cv2.y + ax.z * cv2.z + ax.w * cv2.w;     // reduced over the lanes once per tile
      } else if (MODE != 0) {
        cs1.x = fmaf(v.x, v.x, cs1.x); cs1.y = fmaf(v.y, v.y, cs1.y); cs1.z = fmaf(v.z, v.z, cs1.z); cs1.w = fmaf(v.w, v.w, cs1.w);
        if (MODE == 1) {
          const float qv = __ldg(qrow + itr * 4);
          cs2.x = fmaf(qv, v.x, cs2.x); cs2.y = fmaf(qv, v.y, cs2.y); cs2.z = fmaf(qv, v.z, cs2.z); cs2.w = fmaf(qv, v.w, cs2.w);
        }
      }
      if (OUT_D) *reinterpret_cast<float4*>(p.D + o) = v;
      if (OUT_H) {
        uint2 ph, pl;
        split_half2(v.x * sd_b, v.y * sd_b, ph.x, pl.x);
        split_half2(v.z * sd_b, v.w * sd_b, ph.y, pl.y);
        *reinterpret_cast<uint2*>(p.Dh + o) = ph;
        *reinterpret_cast<uint2*>(p.Dl + o) = pl;
      }
      amx = fmaxf(amx, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
    }
    if (MODE == 1 || MODE == 2) {
#pragma unroll
      for (int sh = 8; sh <= 16; sh <<= 1) {
        cs1.x += __shfl_xor_sync(0xffffffffu, cs1.x, sh); cs1.y += __shfl_xor_sync(0xffffffffu, cs1.y, sh);
        cs1.z += __shfl_xor_sync(0xffffffffu, cs1.z, sh); cs1.w += __shfl_xor_sync(0xffffffffu, cs1.w, sh);
        if (MODE == 1) {
          cs2.x += __shfl_xor_sync(0xffffffffu, cs2.x, sh); cs2.y += __shfl_xor_sync(0xffffffffu, cs2.y, sh);
          cs2.z += __shfl_xor_sync(0xffffffffu, cs2.z, sh); cs2.w += __shfl_xor_sync(0xffffffffu, cs2.w, sh);
        }
      }
      if (lane < 8) {
        float* c1 = p.col1 + colbase + cc * 32;
        atomicAdd(c1, cs1.x); atomicAdd(c1 + 1, cs1.y); atomicAdd(c1 + 2, cs1.z); atomicAdd(c1 + 3, cs1.w);
        if (MODE == 1) {
          float* c2 = p.col2 + colbase + cc * 32;
          atomicAdd(c2, cs2.x); atomicAdd(c2 + 1, cs2.y); atomicAdd(c2 + 2, cs2.z); atomicAdd(c2 + 3, cs2.w);
        }
      }
    }
    __syncwarp();
    o_chunk += 32;
  }
  if (MODE == 3 || MODE == 4) {
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      float rp = racc[u];
      rp += __shfl_xor_sync(0xffffffffu, rp, 1);
      rp += __shfl_xor_sync(0xffffffffu, rp, 2);
      rp += __shfl_xor_sync(0xffffffffu, rp, 4);
      if ((lane & 7) == 0) atomicAdd(p.rowacc + (int64_t)b * p.m + row0 + u * 4 + lr, rp);
    }
  }
}

// shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start>>4 [0,14) | LBO>>4 [16,30) | SBO>>4 [32,46) |
// version=1 [46,48) | layout type [61,64)  (1 = SWIZZLE_128B_BASE32B, 2 = SWIZZLE_128B, 4 = SWIZZLE_64B)
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) |
         ((uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32) | (1ull << 46) | ((uint64_t)layout << 61);
}

struct TileInfo {
  int b, i0, j0, kb0, nkb;     // batch entry, tile origin, first k-block, number of k-blocks (0 = no MMA work)
  int zero;                    // nkb == 0 but the tile is part of the output: the epilogue writes alpha*0 (+Cin)
};

// tile index -> coordinates.  mt (row tile) is the fastest index so that consecutively scheduled tiles share the same
// B column block (L2 reuse); the dynamic scheduler balances the unequal k-ranges of triangular operands.
__device__ __forceinline__ TileInfo tile_info(const Params& p, int t, int mtiles, int ntiles) {
  TileInfo ti;
  const int mt = t % mtiles;
  int r = t / mtiles;
  const int nt = r % ntiles;
  r /= ntiles;
  const int split = r % p.splitk;
  ti.b = r / p.splitk;
  ti.i0 = mt * BM;
  ti.j0 = nt * BN;
  const int i1 = min(ti.i0 + BM, p.m), j1 = min(ti.j0 + BN, p.n);
  ti.kb0 = 0;
  ti.nkb = 0;
  ti.zero = 0;
  if ((p.d_tri == 1 && ti.j0 >= i1) || (p.d_tri == 2 && ti.i0 >= j1)) return ti;
  int k_lo = 0, k_hi = p.k;
  if (p.a_tri == 1) k_hi = min(k_hi, i1);
  if (p.a_tri == 2) k_lo = max(k_lo, ti.i0);
  if (p.b_tri == 1) k_lo = max(k_lo, ti.j0);
  if (p.b_tri == 2) k_hi = min(k_hi, j1);
  const int kb0 = k_lo / p.bk;
  const int nkb_all = k_hi > kb0 * p.bk ? (k_hi - kb0 * p.bk + p.bk - 1) / p.bk : 0;
  int kb_begin = 0, kb_end = nkb_all;
  if (p.splitk > 1) {
    const int chunk = (nkb_all + p.splitk - 1) / p.splitk;
    kb_begin = split * chunk;
    kb_end = min(nkb_all, kb_begin + chunk);
  }
  ti.kb0 = kb0 + kb_begin;
  ti.nkb = max(0, kb_end - kb_begin);
  ti.zero = (ti.nkb == 0 && p.splitk == 1) ? 1 : 0;      // empty k-range of triangular operands: the product is 0
  return ti;
}

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// Persistent kernel: one CTA per SM, tiles handed out by an atomic counter.  The 512 TMEM columns hold two 128 x 256 fp32
// accumulators, so the epilogue of tile i overlaps the MMAs of tile i+1.
// (320 threads are allocated like 384: the register cap is 168 per thread)
template <bool B_KMAJOR, bool F16>
__global__ void __launch_bounds__(NTHREADS, 1)
umma_gemm_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapAlo,
                 const __grid_constant__ CUtensorMap mapB, const __grid_constant__ CUtensorMap mapBlo, const Params p,
                 unsigned int* __restrict__ tile_counter, int total_tiles, int mtiles, int ntiles) {
  extern __shared__ unsigned char smem_raw[];
  __shared__ uint32_t tmem_base_slot;
  __shared__ int sched_tile[2];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* accum_full = empty_bar + STAGES;     // [2]
  uint64_t* accum_empty = accum_full + 2;        // [2]
  uint64_t* sched_full = accum_empty + 2;        // [2]
  uint64_t* sched_empty = sched_full + 2;        // [2]

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(full_bar + s, 1); mbar_init(empty_bar + s, 1); }
    for (int s = 0; s < 2; ++s) {
      mbar_init(accum_full + s, 1);
      mbar_init(accum_empty + s, EPI_WARPS);     // one arrival per epilogue warp
      mbar_init(sched_full + s, 1);
      mbar_init(sched_empty + s, 1 + EPI_WARPS); // MMA thread + epilogue warps
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_slot)), "r"(TMEM_COLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = tmem_base_slot;
  const uint32_t tx_bytes = p.n_terms == 3 ? (uint32_t)STAGE_BYTES : (uint32_t)(A_BYTES + B_BYTES);

  if (warp == 0) {
    // ===== scheduler + TMA producer (one thread) =====
    if (lane == 0) {
      uint32_t it = 0;                                     // running k-block counter across tiles (stage ring position)
      for (uint32_t iter = 0;; ++iter) {
        const int slot = iter & 1;
        mbar_wait(sched_empty + slot, ((iter >> 1) & 1u) ^ 1u);
        const int t = (int)atomicAdd(tile_counter, 1u);
        sched_tile[slot] = t < total_tiles ? t : -1;
        mbar_arrive(sched_full + slot);                    // release: the tile index is visible to the waiters
        if (t >= total_tiles) break;
        const TileInfo ti = tile_info(p, t, mtiles, ntiles);
        for (int kb = 0; kb < ti.nkb; ++kb, ++it) {
          const int s = it % STAGES;
          const uint32_t ph = (it / STAGES) & 1u;
          mbar_wait(empty_bar + s, ph ^ 1u);
          unsigned char* st = smem + s * STAGE_BYTES;
          mbar_expect_tx(full_bar + s, tx_bytes);
          // MN-major B: chunks of CW columns (128 B rows), CHB bytes apart (tf32: 32 cols x 16 k-rows; fp16: 64 x 32)
          constexpr int CW = F16 ? 64 : 32, CHB = F16 ? 4096 : 2048;
          const int kc = (ti.kb0 + kb) * (F16 ? BK16 : BK);
          tma_load_3d(&mapA, full_bar + s, st, kc, ti.i0, ti.b);
          if (B_KMAJOR) {
            tma_load_3d(&mapB, full_bar + s, st + 2 * A_BYTES, kc, ti.j0, ti.b);
          } else if (p.b_map4d) {                  // one box {CW cols, k-rows, BN/CW column chunks}: chunk-major in smem
            tma_load_4d(&mapB, full_bar + s, st + 2 * A_BYTES, 0, kc, ti.j0 / CW, ti.b);
          } else {
#pragma unroll
            for (int c = 0; c < BN / CW; ++c)
              tma_load_3d(&mapB, full_bar + s, st + 2 * A_BYTES + c * CHB, ti.j0 + c * CW, kc, ti.b);
          }
          if (p.n_terms == 3) {
            tma_load_3d(&mapAlo, full_bar + s, st + A_BYTES, kc, ti.i0, ti.b);
            if (B_KMAJOR) {
              tma_load_3d(&mapBlo, full_bar + s, st + 2 * A_BYTES + B_BYTES, kc, ti.j0, ti.b);
            } else if (p.b_map4d) {
              tma_load_4d(&mapBlo, full_bar + s, st + 2 * A_BYTES + B_BYTES, 0, kc, ti.j0 / CW, ti.b);
            } else {
#pragma unroll
              for (int c = 0; c < BN / CW; ++c)
                tma_load_3d(&mapBlo, full_bar + s, st + 2 * A_BYTES + B_BYTES + c * CHB, ti.j0 + c * CW, kc, ti.b);
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (one thread) =====
    if (lane == 0) {
      // instruction descriptor (cute::UMMA::InstrDescriptor): D=F32 [4,6)=1, A=TF32 [7,10)=2, B=TF32 [10,13)=2,
      // a_major [15]=0 (K), b_major [16], N>>3 [17,23), M>>4 [24,29)
      // operand format 2 = TF32, 0 = F16
      const uint32_t fmt = F16 ? 0u : 2u;
      const uint32_t idesc_full = (1u << 4) | (fmt << 7) | (fmt << 10) | ((B_KMAJOR ? 0u : 1u) << 16) | ((uint32_t)(BN >> 3) << 17) |
                             ((uint32_t)(BM >> 4) << 24);
      uint32_t it = 0, acc_iter = 0;
      for (uint32_t iter = 0;; ++iter) {
        const int slot = iter & 1;
        mbar_wait(sched_full + slot, (iter >> 1) & 1u);
        const int t = sched_tile[slot];
        mbar_arrive(sched_empty + slot);
        if (t < 0) break;
        const TileInfo ti = tile_info(p, t, mtiles, ntiles);
        if (ti.nkb == 0) continue;
        const uint32_t as = acc_iter & 1u;
        mbar_wait(accum_empty + as, ((acc_iter >> 1) & 1u) ^ 1u);       // epilogue has drained this accumulator
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t tmem_d = tmem_base + as * (uint32_t)BN;
        // lower-triangular output, tile on the diagonal with its right half above it: a 128-column MMA is enough
        // (the epilogue masks columns > row, so the stale right half of the accumulator is never stored)
        const uint32_t idesc = (p.d_tri == 1 && ti.i0 + BM <= ti.j0 + BN / 2)
                                   ? ((idesc_full & ~(0x3Fu << 17)) | ((uint32_t)(BN >> 4) << 17)) : idesc_full;
        for (int kb = 0; kb < ti.nkb; ++kb, ++it) {
          const int s = it % STAGES;
          const uint32_t ph = (it / STAGES) & 1u;
          mbar_wait(full_bar + s, ph);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t sa = smem_u32(smem + s * STAGE_BYTES);
          const uint32_t sb = sa + 2 * A_BYTES;
#pragma unroll
          for (int ks = 0; ks < 2; ++ks) {
            // K-major SW64: rows of 64 B, 8-row groups 512 B apart; one MMA k-step (8 tf32 / 16 fp16) = 32 B inside the row
            const uint64_t a_raw = make_desc(sa + ks * 32, 16, 512, 4);
            const uint64_t a_lo = make_desc(sa + A_BYTES + ks * 32, 16, 512, 4);
            uint64_t b_raw, b_lo;
            if (B_KMAJOR) {
              b_raw = make_desc(sb + ks * 32, 16, 512, 4);
              b_lo = make_desc(sb + B_BYTES + ks * 32, 16, 512, 4);
            } else if (F16) {
              // MN-major fp16: plain SWIZZLE_128B (layout type 2), atoms of 64 columns (128 B) x 8 k-rows: column chunks
              // 4 KB apart (= LBO), 8-row k groups 1 KB apart (= SBO); one K=16 step = two k groups = 2 KB
              b_raw = make_desc(sb + ks * 2048, 4096, 1024, 2);
              b_lo = make_desc(sb + B_BYTES + ks * 2048, 4096, 1024, 2);
            } else {
              // MN-major tf32 must use SWIZZLE_128B_BASE32B (layout type 1; 32 B chunks swizzled inside a 4-row x 128 B
              // atom): chunks of 32 columns (128 B rows) 2 KB apart (= LBO), 4-row k groups 512 B apart (= SBO);
              // one K=8 step = two k groups = 1 KB
              b_raw = make_desc(sb + ks * 1024, 2048, 512, 1);
              b_lo = make_desc(sb + B_BYTES + ks * 1024, 2048, 512, 1);
            }
            const uint32_t acc0 = (kb > 0 || ks > 0) ? 1u : 0u;
            if (F16) {
              if (p.n_terms == 3) {
                umma_f16(tmem_d, a_raw, b_lo, idesc, acc0);
                umma_f16(tmem_d, a_raw, b_raw, idesc, 1u);
                umma_f16(tmem_d, a_lo, b_raw, idesc, 1u);
              } else {
                umma_f16(tmem_d, a_raw, b_raw, idesc, acc0);
              }
            } else if (p.n_terms == 3) {
              umma_tf32(tmem_d, a_raw, b_lo, idesc, acc0);
              umma_tf32(tmem_d, a_lo, b_raw, idesc, 1u);
              umma_tf32(tmem_d, a_raw, b_raw, idesc, 1u);
            } else {
              umma_tf32(tmem_d, a_raw, b_raw, idesc, acc0);
            }
          }
          umma_commit(empty_bar + s);               // frees the smem stage once these MMAs have read it
        }
        umma_commit(accum_full + as);               // accumulator complete
        ++acc_iter;
      }
    }
  } else {
    // ===== epilogue: warps 2..9, TMEM lane quadrant = warp % 4; warps 2..5 take column chunks 0..3, warps 6..9 chunks 4..7 =====
    const int q = warp & 3;
    const int c_begin = ((warp - 2) >> 2) * EPI_CHUNKS, c_end = c_begin + EPI_CHUNKS;
    const bool vec_ok = (p.ldd % 4 == 0) && ((reinterpret_cast<uintptr_t>(p.D) & 15) == 0) &&
                        (!p.Dlo || (reinterpret_cast<uintptr_t>(p.Dlo) & 15) == 0) &&
                        (!p.Cin || (reinterpret_cast<uintptr_t>(p.Cin) & 15) == 0) && ((p.sD % 4) == 0) &&
                        (!p.Dh || ((reinterpret_cast<uintptr_t>(p.Dh) & 7) == 0 && (reinterpret_cast<uintptr_t>(p.Dl) & 7) == 0)) &&
                        (!p.AuxH || ((reinterpret_cast<uintptr_t>(p.AuxH) & 7) == 0 && (reinterpret_cast<uintptr_t>(p.AuxL) & 7) == 0)) &&
                        (!p.D2h || ((reinterpret_cast<uintptr_t>(p.D2h) & 7) == 0 && (reinterpret_cast<uintptr_t>(p.D2l) & 7) == 0));
    float* epi = reinterpret_cast<float*>(smem + STAGES * STAGE_BYTES + 256) + (warp - 2) * 32 * 32;
    uint32_t acc_iter = 0;
    bool aux_ahead = false;                  // this tile's Aux region was already prefetched into L2 during the tile before
    for (uint32_t iter = 0;; ++iter) {
      const int slot = iter & 1;
      mbar_wait(sched_full + slot, (iter >> 1) & 1u);
      const int t = sched_tile[slot];
      __syncwarp();
      if (lane == 0) mbar_arrive(sched_empty + slot);
      if (t < 0) break;
      const TileInfo ti = tile_info(p, t, mtiles, ntiles);
      const bool has_acc = ti.nkb > 0;
      if (!has_acc && !ti.zero) continue;
      const uint32_t as = acc_iter & 1u;
      if (F16 && (p.epi_mode == 3 || p.epi_mode == 4) && p.AuxH) {
        // pull this warp's part of the Aux planes (32 rows x 128 columns x 2 planes) into L2: of this tile unless that was done
        // a tile ago, and of the NEXT tile when the scheduler has already handed it out (the slot cannot be refilled before this
        // warp arrives on it, so the peek is safe).  With the epilogue as the bottleneck of these modes the hand-out of the
        // current tile comes too late for the prefetch to land before the loads.
        auto aux_prefetch = [&](const TileInfo& tj) {
          const __half* ah = p.AuxH + (int64_t)tj.b * p.sD + (int64_t)(tj.i0 + q * 32 + lane) * p.ldd + tj.j0 + c_begin * 32;
          const __half* al = p.AuxL + (int64_t)tj.b * p.sD + (int64_t)(tj.i0 + q * 32 + lane) * p.ldd + tj.j0 + c_begin * 32;
          asm volatile("prefetch.global.L2 [%0];" ::"l"(ah));
          asm volatile("prefetch.global.L2 [%0];" ::"l"(al));
          if (EPI_CHUNKS > 2) {
            asm volatile("prefetch.global.L2 [%0];" ::"l"(ah + 64));
            asm volatile("prefetch.global.L2 [%0];" ::"l"(al + 64));
          }
        };
        if (!aux_ahead && has_acc && ti.i0 + BM <= p.m && ti.j0 + BN <= p.n) aux_prefetch(ti);
        aux_ahead = false;
        if (GPZ_UMMA_AUX_AHEAD && mbar_test(sched_full + (slot ^ 1), ((iter + 1) >> 1) & 1u)) {
          const int tn = sched_tile[slot ^ 1];
          if (tn >= 0) {
            const TileInfo tj = tile_info(p, tn, mtiles, ntiles);
            if (tj.nkb > 0 && tj.i0 + BM <= p.m && tj.j0 + BN <= p.n) {
              aux_prefetch(tj);
              aux_ahead = true;
            }
          }
        }
      }
      if (has_acc) {
        mbar_wait(accum_full + as, (acc_iter >> 1) & 1u);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      }
      // per-batch scales (powers of two): accumulator -> true value, true value -> fp16 output planes
      float alpha_b = p.alpha;
      if (p.sa) alpha_b *= 1.0f / p.sa[ti.b];
      if (p.sb) alpha_b *= 1.0f / p.sb[ti.b];
      const float sd_b = (p.Dh && p.sd) ? p.sd[ti.b] : 1.0f;
      const float inv_saux = (p.AuxH && p.saux) ? 1.0f / p.saux[ti.b] : 1.0f;
      const float sd2_b = (p.D2h && p.sd2) ? p.sd2[ti.b] : 1.0f;
      float amx = 0.f;
      if (F16 && has_acc && vec_ok && p.splitk == 1 && p.d_tri == 0 && !p.Cin && !p.Dlo && ti.i0 + BM <= p.m && ti.j0 + BN <= p.n) {
        // tile completely inside the matrix: specialised, branch-free inner loops
        const uint32_t tacc = tmem_base + ((uint32_t)(q * 32) << 16) + as * (uint32_t)BN;
        bool done = true;
        if (p.epi_mode == 1 && p.Dh && !p.D) epilogue_tile_fast<1, false, true>(p, ti.b, ti.i0, ti.j0, q, lane, c_begin, tacc, epi, alpha_b, sd_b, inv_saux, amx);
        else if (p.epi_mode == 2 && p.D && !p.Dh) epilogue_tile_fast<2, true, false>(p, ti.b, ti.i0, ti.j0, q, lane, c_begin, tacc, epi, alpha_b, sd_b, inv_saux, amx);
        else if (p.epi_mode == 2 && p.Dh && !p.D) epilogue_tile_fast<2, false, true>(p, ti.b, ti.i0, ti.j0, q, lane, c_begin, tacc, epi, alpha_b, sd_b, inv_saux, amx);
        else if (p.epi_mode == 3 && p.AuxH && p.Dh && !p.D) epilogue_tile_fast<3, false, true>(p, ti.b, ti.i0, ti.j0, q, lane, c_begin, tacc, epi, alpha_b, sd_b, inv_saux, amx);
        else if (p.epi_mode == 4 && p.AuxH && p.Dh && !p.D && p.D2h) epilogue_tile_fast<4, false, true>(p, ti.b, ti.i0, ti.j0, q, lane, c_begin, tacc, epi, alpha_b, sd_b, inv_saux, amx, sd2_b);
        else if (p.epi_mode == 0 && p.D && !p.Dh) epilogue_tile_fast<0, true, false>(p, ti.b, ti.i0, ti.j0, q, lane, c_begin, tacc, epi, alpha_b, sd_b, inv_saux, amx);
        else if (p.epi_mode == 0 && p.Dh && !p.D) epilogue_tile_fast<0, false, true>(p, ti.b, ti.i0, ti.j0, q, lane, c_begin, tacc, epi, alpha_b, sd_b, inv_saux, amx);
        else done = false;
        if (done) {
          if (p.amax) {
#pragma unroll
            for (int sh = 16; sh > 0; sh >>= 1) amx = fmaxf(amx, __shfl_xor_sync(0xffffffffu, amx, sh));
            if (lane == 0 && amx > 0.f) atomicMax(p.amax + ti.b, __float_as_uint(amx));
          }
          asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
          __syncwarp();
          if (lane == 0) mbar_arrive(accum_empty + as);
          ++acc_iter;
          continue;
        }
      }
      const int gi = ti.i0 + q * 32 + lane;
      const int wrow0 = ti.i0 + q * 32;
      float racc[8];                          // mode 3: per-row partial sums of this lane's 8 rows (coalesced path)
      float qreg[8];                          // rowv of this lane's 8 rows (coalesced path)
      float racc_s = 0.f;                     // mode 3, scalar path: row gi
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        racc[u] = 0.f;
        const int rr = wrow0 + u * 4 + (lane >> 3);
        qreg[u] = (p.epi_mode != 0 && p.epi_mode != 2 && rr < p.m) ? p.rowv[(int64_t)ti.b * p.m + rr] : 0.f;
      }
      const float q_s = (p.epi_mode != 0 && p.epi_mode != 2 && gi < p.m) ? p.rowv[(int64_t)ti.b * p.m + gi] : 0.f;
      const int64_t row_off = (int64_t)ti.b * p.sD + (int64_t)gi * p.ldd;
#pragma unroll 1
      for (int c = c_begin; c < c_end; ++c) {
        uint32_t r[32];
        if (has_acc) {
          tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + as * (uint32_t)BN + (uint32_t)(c * 32), r);
        } else {
#pragma unroll
          for (int u = 0; u < 32; ++u) r[u] = 0u;
        }
        const int gj0 = ti.j0 + c * 32;
        // warp-uniform: the whole 32 x 32 block of this warp lies inside the matrix and inside the stored triangle
        const int wi0 = ti.i0 + q * 32;
        const bool warp_full = (wi0 + 32 <= p.m) && (gj0 + 32 <= p.n) &&
                               !((p.d_tri == 1 && gj0 + 31 > wi0) || (p.d_tri == 2 && gj0 < wi0 + 31));
        if (!warp_full && (gi >= p.m || gj0 >= p.n)) continue;
        if (p.splitk > 1) {
          for (int u = 0; u < 32; ++u) {
            const int gj = gj0 + u;
            if (gj >= p.n) break;
            if ((p.d_tri == 1 && gj > gi) || (p.d_tri == 2 && gj < gi)) continue;
            atomicAdd(p.D + row_off + gj, alpha_b * __uint_as_float(r[u]));
          }
        } else if (warp_full && vec_ok) {
          // transpose the 32 x 32 block through shared memory so that every store instruction writes whole 128-byte
          // lines: lane -> (row = 4*it + lane/8, 4 columns at (lane%8)*4)
          // (staging tile: row r keeps its 16-byte column c4 at slot c4 ^ (r & 7): conflict-free both ways without padding)
#pragma unroll
          for (int u = 0; u < 32; u += 4)
            sts128(smem_u32(epi) + lane * 128 + (((u >> 2) ^ (lane & 7)) << 4), __uint_as_float(r[u]), __uint_as_float(r[u + 1]),
                   __uint_as_float(r[u + 2]), __uint_as_float(r[u + 3]));
          __syncwarp();
          const int cq = (lane & 7) * 4;
          float4 cs1 = make_float4(0.f, 0.f, 0.f, 0.f), cs2 = make_float4(0.f, 0.f, 0.f, 0.f);
          float4 cv1 = cs1, cv2 = cs1;
          if (p.epi_mode == 3 || p.epi_mode == 4) {
            cv1 = *reinterpret_cast<const float4*>(p.colv1 + (int64_t)ti.b * p.n + gj0 + cq);
            cv2 = *reinterpret_cast<const float4*>(p.colv2 + (int64_t)ti.b * p.n + gj0 + cq);
          }
#pragma unroll
          for (int itr = 0; itr < 8; ++itr) {
            const int rr = itr * 4 + (lane >> 3);
            float4 v = lds128(smem_u32(epi) + rr * 128 + (((lane & 7) ^ (rr & 7)) << 4));
            v.x *= alpha_b; v.y *= alpha_b; v.z *= alpha_b; v.w *= alpha_b;
            const int64_t o = (int64_t)ti.b * p.sD + (int64_t)(ti.i0 + q * 32 + rr) * p.ldd + gj0 + cq;
            if (p.Cin) {
              const float4 cc = *reinterpret_cast<const float4*>(p.Cin + o);
              v.x += cc.x; v.y += cc.y; v.z += cc.z; v.w += cc.w;
            }
            if (p.epi_mode == 3 || p.epi_mode == 4) {
              float4 ax;
              if (p.AuxH) {
                const uint2 hh = *reinterpret_cast<const uint2*>(p.AuxH + o);
                const uint2 ll = *reinterpret_cast<const uint2*>(p.AuxL + o);
                ax.x = unpack_sum(hh.x, ll.x, 0) * inv_saux; ax.y = unpack_sum(hh.x, ll.x, 1) * inv_saux;
                ax.z = unpack_sum(hh.y, ll.y, 0) * inv_saux; ax.w = unpack_sum(hh.y, ll.y, 1) * inv_saux;
              } else {
                ax = *reinterpret_cast<const float4*>(p.Aux + o);
              }
              const float qv = qreg[itr];
              if (p.epi_mode == 3) {
                v.x += fmaf(qv, cv2.x, -2.f * ax.x * cv1.x);
                v.y += fmaf(qv, cv2.y, -2.f * ax.y * cv1.y);
                v.z += fmaf(qv, cv2.z, -2.f * ax.z * cv1.z);
                v.w += fmaf(qv, cv2.w, -2.f * ax.w * cv1.w);
              } else {
                v.x = fmaf(2.f * cv1.x, v.x - ax.x, qv * cv2.x);
                v.y = fmaf(2.f * cv1.y, v.y - ax.y, qv * cv2.y);
                v.z = fmaf(2.f * cv1.z, v.z - ax.z, qv * cv2.z);
                v.w = fmaf(2.f * cv1.w, v.w - ax.w, qv * cv2.w);
                if (p.D2h) {
                  uint2 qh, ql;
                  split_half2(2.f * cv1.x * ax.x * sd2_b, 2.f * cv1.y * ax.y * sd2_b, qh.x, ql.x);
                  split_half2(2.f * cv1.z * ax.z * sd2_b, 2.f * cv1.w * ax.w * sd2_b, qh.y, ql.y);
                  *reinterpret_cast<uint2*>(p.D2h + o) = qh;
                  *reinterpret_cast<uint2*>(p.D2l + o) = ql;
                }
              }
              float rp = ax.x * cv2.x + ax.y * cv2.y + ax.z * cv2.z + ax.w * cv2.w;
              rp += __shfl_xor_sync(0xffffffffu, rp, 1);
              rp += __shfl_xor_sync(0xffffffffu, rp, 2);
              rp += __shfl_xor_sync(0xffffffffu, rp, 4);
              racc[itr] += rp;
            } else if (p.epi_mode != 0) {
              cs1.x = fmaf(v.x, v.x, cs1.x); cs1.y = fmaf(v.y, v.y, cs1.y); cs1.z = fmaf(v.z, v.z, cs1.z); cs1.w = fmaf(v.w, v.w, cs1.w);
              if (p.epi_mode == 1) {
                const float qv = qreg[itr];
                cs2.x = fmaf(qv, v.x, cs2.x); cs2.y = fmaf(qv, v.y, cs2.y); cs2.z = fmaf(qv, v.z, cs2.z); cs2.w = fmaf(qv, v.w, cs2.w);
              }
            }
            if (p.D) *reinterpret_cast<float4*>(p.D + o) = v;
            if (p.Dlo) {
              float4 lo;
              lo.x = v.x - __uint_as_float(__float_as_uint(v.x) & 0xFFFFE000u);
              lo.y = v.y - __uint_as_float(__float_as_uint(v.y) & 0xFFFFE000u);
              lo.z = v.z - __uint_as_float(__float_as_uint(v.z) & 0xFFFFE000u);
              lo.w = v.w - __uint_as_float(__float_as_uint(v.w) & 0xFFFFE000u);
              *reinterpret_cast<float4*>(p.Dlo + o) = lo;
            }
            if (p.Dh) {
              uint2 ph, pl;
              split_half2(v.x * sd_b, v.y * sd_b, ph.x, pl.x);
              split_half2(v.z * sd_b, v.w * sd_b, ph.y, pl.y);
              *reinterpret_cast<uint2*>(p.Dh + o) = ph;
              *reinterpret_cast<uint2*>(p.Dl + o) = pl;
            }
            if (p.amax) amx = fmaxf(amx, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
          }
          if (p.epi_mode == 1 || p.epi_mode == 2) {
            // column sums over the warp's 32 rows: combine the four row groups (lane/8), then lanes 0..7 own 4 columns each
#pragma unroll
            for (int sh = 8; sh <= 16; sh <<= 1) {
              cs1.x += __shfl_xor_sync(0xffffffffu, cs1.x, sh); cs1.y += __shfl_xor_sync(0xffffffffu, cs1.y, sh);
              cs1.z += __shfl_xor_sync(0xffffffffu, cs1.z, sh); cs1.w += __shfl_xor_sync(0xffffffffu, cs1.w, sh);
              if (p.epi_mode == 1) {
                cs2.x += __shfl_xor_sync(0xffffffffu, cs2.x, sh); cs2.y += __shfl_xor_sync(0xffffffffu, cs2.y, sh);
                cs2.z += __shfl_xor_sync(0xffffffffu, cs2.z, sh); cs2.w += __shfl_xor_sync(0xffffffffu, cs2.w, sh);
              }
            }
            if (lane < 8) {
              float* c1 = p.col1 + (int64_t)ti.b * p.n + gj0 + cq;
              atomicAdd(c1, cs1.x); atomicAdd(c1 + 1, cs1.y); atomicAdd(c1 + 2, cs1.z); atomicAdd(c1 + 3, cs1.w);
              if (p.epi_mode == 1) {
                float* c2 = p.col2 + (int64_t)ti.b * p.n + gj0 + cq;
                atomicAdd(c2, cs2.x); atomicAdd(c2 + 1, cs2.y); atomicAdd(c2 + 2, cs2.z); atomicAdd(c2 + 3, cs2.w);
              }
            }
          }
          __syncwarp();
        } else {
          for (int u = 0; u < 32; ++u) {
            const int gj = gj0 + u;
            if (gj >= p.n) break;
            if ((p.d_tri == 1 && gj > gi) || (p.d_tri == 2 && gj < gi)) continue;
            float v = alpha_b * __uint_as_float(r[u]);
            if (p.Cin) v += p.Cin[row_off + gj];
            if (p.epi_mode == 3 || p.epi_mode == 4) {
              const float ax = p.AuxH ? (__half2float(p.AuxH[row_off + gj]) + __half2float(p.AuxL[row_off + gj])) * inv_saux
                                      : p.Aux[row_off + gj];
              const float g2 = p.colv2[(int64_t)ti.b * p.n + gj];
              const float g1 = p.colv1[(int64_t)ti.b * p.n + gj];
              if (p.epi_mode == 3) {
                v += fmaf(q_s, g2, -2.f * ax * g1);
              } else {
                v = fmaf(2.f * g1, v - ax, q_s * g2);
                if (p.D2h) {
                  __half h2, l2;
                  split_half(2.f * g1 * ax * sd2_b, h2, l2);
                  p.D2h[row_off + gj] = h2;
                  p.D2l[row_off + gj] = l2;
                }
              }
              racc_s = fmaf(ax, g2, racc_s);
            } else if (p.epi_mode != 0) {
              atomicAdd(p.col1 + (int64_t)ti.b * p.n + gj, v * v);
              if (p.epi_mode == 1) atomicAdd(p.col2 + (int64_t)ti.b * p.n + gj, q_s * v);
            }
            if (p.D) p.D[row_off + gj] = v;
            if (p.Dlo) p.Dlo[row_off + gj] = v - __uint_as_float(__float_as_uint(v) & 0xFFFFE000u);
            if (p.Dh) {
              __half h, l;
              split_half(v * sd_b, h, l);
              p.Dh[row_off + gj] = h;
              p.Dl[row_off + gj] = l;
            }
            if (p.amax) amx = fmaxf(amx, fabsf(v));
          }
        }
      }
      if (p.epi_mode == 3 || p.epi_mode == 4) {
        if ((lane & 7) == 0) {
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const int rr = wrow0 + u * 4 + (lane >> 3);
            if (rr < p.m && racc[u] != 0.f) atomicAdd(p.rowacc + (int64_t)ti.b * p.m + rr, racc[u]);
          }
        }
        if (gi < p.m && racc_s != 0.f) atomicAdd(p.rowacc + (int64_t)ti.b * p.m + gi, racc_s);
      }
      if (p.amax) {
#pragma unroll
        for (int sh = 16; sh > 0; sh >>= 1) amx = fmaxf(amx, __shfl_xor_sync(0xffffffffu, amx, sh));
        if (lane == 0 && amx > 0.f) atomicMax(p.amax + ti.b, __float_as_uint(amx));
      }
      if (has_acc) {
        // this warp is done reading the accumulator stage: hand it back to the MMA thread
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive(accum_empty + as);
        ++acc_iter;
      }
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS));
  }
}

// ---- host side --------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(ptr);
  }
  return fn;
}

// K-major operand: rows x k (k contiguous, row stride ld), batch stride sB  ->  3-D map {k, rows, batch}, box {16, box_rows, 1}
static int make_map_kmajor(CUtensorMap* map, const float* base, int rows, int k, int64_t ld, int64_t sB, int batch, int box_rows) {
  EncodeTiledFn enc = encode_fn();
  if (!enc) return GPZ_ERR_UNSUPPORTED;
  cuuint64_t gdim[3] = {(cuuint64_t)k, (cuuint64_t)rows, (cuuint64_t)batch};
  cuuint64_t gstr[2] = {(cuuint64_t)ld * 4, (cuuint64_t)(batch > 1 ? sB : (int64_t)rows * ld) * 4};
  cuuint32_t box[3] = {(cuuint32_t)BK, (cuuint32_t)box_rows, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(base), gdim, gstr, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? GPZ_OK : GPZ_ERR_BADARG;
}

// MN-major operand: k x n (n contiguous, row stride ld)  ->  3-D map {n, k, batch}, box {32, 16, 1} (128 B rows, SWIZZLE_128B_ATOM_32B)
static int make_map_mnmajor(CUtensorMap* map, const float* base, int k, int n, int64_t ld, int64_t sB, int batch) {
  EncodeTiledFn enc = encode_fn();
  if (!enc) return GPZ_ERR_UNSUPPORTED;
  cuuint64_t gdim[3] = {(cuuint64_t)n, (cuuint64_t)k, (cuuint64_t)batch};
  cuuint64_t gstr[2] = {(cuuint64_t)ld * 4, (cuuint64_t)(batch > 1 ? sB : (int64_t)k * ld) * 4};
  cuuint32_t box[3] = {32, (cuuint32_t)BK, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(base), gdim, gstr, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? GPZ_OK : GPZ_ERR_BADARG;
}

// MN-major operand with n % 32 == 0: 4-D view {32, k, n/32, batch} (strides 4 B, ld, 128 B, sB) so that ONE box {32, 16, 8, 1}
// lands chunk-major in shared memory (8 chunks x 16 rows x 128 B) - 1 TMA instruction per stage instead of 8.
static int make_map_mnmajor4d(CUtensorMap* map, const float* base, int k, int n, int64_t ld, int64_t sB, int batch) {
  EncodeTiledFn enc = encode_fn();
  if (!enc) return GPZ_ERR_UNSUPPORTED;
  cuuint64_t gdim[4] = {32, (cuuint64_t)k, (cuuint64_t)(n / 32), (cuuint64_t)batch};
  cuuint64_t gstr[3] = {(cuuint64_t)ld * 4, 128, (cuuint64_t)(batch > 1 ? sB : (int64_t)k * ld) * 4};
  cuuint32_t box[4] = {32, (cuuint32_t)BK, (cuuint32_t)(BN / 32), 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(base), gdim, gstr, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? GPZ_OK : GPZ_ERR_BADARG;
}

// ---- fp16 planes (split-FP16 mode): same byte geometry for K-major tiles; MN-major tiles use plain SWIZZLE_128B ----
static int make_map_kmajor16(CUtensorMap* map, const __half* base, int rows, int k, int64_t ld, int64_t sB, int batch, int box_rows) {
  EncodeTiledFn enc = encode_fn();
  if (!enc) return GPZ_ERR_UNSUPPORTED;
  cuuint64_t gdim[3] = {(cuuint64_t)k, (cuuint64_t)rows, (cuuint64_t)batch};
  cuuint64_t gstr[2] = {(cuuint64_t)ld * 2, (cuuint64_t)(batch > 1 ? sB : (int64_t)rows * ld) * 2};
  cuuint32_t box[3] = {(cuuint32_t)BK16, (cuuint32_t)box_rows, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<__half*>(base), gdim, gstr, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? GPZ_OK : GPZ_ERR_BADARG;
}
// MN-major fp16: 3-D map {n, k, batch}, box {64, 32, 1} (128 B rows)
static int make_map_mnmajor16(CUtensorMap* map, const __half* base, int k, int n, int64_t ld, int64_t sB, int batch) {
  EncodeTiledFn enc = encode_fn();
  if (!enc) return GPZ_ERR_UNSUPPORTED;
  cuuint64_t gdim[3] = {(cuuint64_t)n, (cuuint64_t)k, (cuuint64_t)batch};
  cuuint64_t gstr[2] = {(cuuint64_t)ld * 2, (cuuint64_t)(batch > 1 ? sB : (int64_t)k * ld) * 2};
  cuuint32_t box[3] = {64, (cuuint32_t)BK16, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<__half*>(base), gdim, gstr, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? GPZ_OK : GPZ_ERR_BADARG;
}
// MN-major fp16 with n % 64 == 0: 4-D view {64, k, n/64, batch}, ONE box {64, 32, 4, 1} per stage, chunk-major in smem
static int make_map_mnmajor16_4d(CUtensorMap* map, const __half* base, int k, int n, int64_t ld, int64_t sB, int batch) {
  EncodeTiledFn enc = encode_fn();
  if (!enc) return GPZ_ERR_UNSUPPORTED;
  cuuint64_t gdim[4] = {64, (cuuint64_t)k, (cuuint64_t)(n / 64), (cuuint64_t)batch};
  cuuint64_t gstr[3] = {(cuuint64_t)ld * 2, 128, (cuuint64_t)(batch > 1 ? sB : (int64_t)k * ld) * 2};
  cuuint32_t box[4] = {64, (cuuint32_t)BK16, (cuuint32_t)(BN / 64), 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<__half*>(base), gdim, gstr, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? GPZ_OK : GPZ_ERR_BADARG;
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

constexpr int NUM_COUNTERS = 256;
__device__ unsigned int g_tile_counters[NUM_COUNTERS];

}  // namespace umma
}  // namespace gpz

using namespace gpz;
using namespace gpz::umma;

// common launch: persistent grid, dynamic tile scheduler (one counter per in-flight launch, taken round-robin from a small
// device array)
static int launch_gemm(bool b_kmajor, bool f16, const CUtensorMap& mA, const CUtensorMap& mAlo, const CUtensorMap& mB,
                       const CUtensorMap& mBlo, const Params& p, cudaStream_t st, int max_ctas = 0) {
  const int mtiles = (int)cdiv(p.m, BM), ntiles = (int)cdiv(p.n, BN);
  const int64_t total64 = (int64_t)mtiles * ntiles * p.batch * p.splitk;
  if (total64 > 0x7fffffff) return GPZ_ERR_UNSUPPORTED;
  const int total = (int)total64;
  static unsigned int* counters = nullptr;
  static std::atomic<unsigned int> next_slot{0};
  static int num_sms = 0;
  if (!counters) {
    unsigned int* ptr = nullptr;
    GPZ_CUDA(cudaGetSymbolAddress((void**)&ptr, g_tile_counters));
    counters = ptr;
    int dev = 0;
    GPZ_CUDA(cudaGetDevice(&dev));
    GPZ_CUDA(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev));
    GPZ_CUDA(cudaFuncSetAttribute(umma_gemm_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    GPZ_CUDA(cudaFuncSetAttribute(umma_gemm_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    GPZ_CUDA(cudaFuncSetAttribute(umma_gemm_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    GPZ_CUDA(cudaFuncSetAttribute(umma_gemm_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
  }
  unsigned int* counter = counters + (next_slot.fetch_add(1) % NUM_COUNTERS);
  GPZ_CUDA(cudaMemsetAsync(counter, 0, sizeof(unsigned int), st));
  int grid = total < num_sms ? total : num_sms;
  if (max_ctas > 0 && grid > max_ctas) grid = max_ctas;
  if (f16) {
    if (b_kmajor) umma_gemm_kernel<true, true><<<grid, NTHREADS, SMEM_BYTES, st>>>(mA, mAlo, mB, mBlo, p, counter, total, mtiles, ntiles);
    else umma_gemm_kernel<false, true><<<grid, NTHREADS, SMEM_BYTES, st>>>(mA, mAlo, mB, mBlo, p, counter, total, mtiles, ntiles);
  } else {
    if (b_kmajor) umma_gemm_kernel<true, false><<<grid, NTHREADS, SMEM_BYTES, st>>>(mA, mAlo, mB, mBlo, p, counter, total, mtiles, ntiles);
    else umma_gemm_kernel<false, false><<<grid, NTHREADS, SMEM_BYTES, st>>>(mA, mAlo, mB, mBlo, p, counter, total, mtiles, ntiles);
  }
  GPZ_CHECK_LAUNCH();
  return GPZ_OK;
}


// 1 if the tcgen05 path can take this problem (alignment / divisibility), 0 otherwise (caller uses gpz_gemm_f32)
extern "C" int gpz_umma_gemm_supported(int b_kmajor, int m, int n, int k, int64_t lda, int64_t ldb, int64_t ldd) {
  if (m < 1 || n < 1 || k < 1) return 0;
  if (lda % 4 || ldb % 4) return 0;
  (void)ldd;
  return 1;
}

extern "C" int gpz_umma_gemm_f32(int b_kmajor, int m, int n, int k, float alpha, const float* A, const float* Alo, int64_t lda,
                                 int64_t sA, const float* B, const float* Blo, int64_t ldb, int64_t sB, const float* Cin, float* D,
                                 float* Dlo, int64_t ldd, int64_t sD, int batch, int a_tri, int b_tri, int d_tri, int splitk,
                                 int n_terms, void* stream) {
  return umma_gemm_ex(b_kmajor, m, n, k, alpha, A, Alo, lda, sA, B, Blo, ldb, sB, Cin, D, Dlo, ldd, sD, batch, a_tri, b_tri, d_tri,
                      splitk, n_terms, nullptr, stream);
}

int umma_gemm_ex(int b_kmajor, int m, int n, int k, float alpha, const float* A, const float* Alo, int64_t lda, int64_t sA,
                 const float* B, const float* Blo, int64_t ldb, int64_t sB, const float* Cin, float* D, float* Dlo, int64_t ldd,
                 int64_t sD, int batch, int a_tri, int b_tri, int d_tri, int splitk, int n_terms, const UmmaEpilogue* epi,
                 void* stream, int max_ctas) {
  if (!gpz_umma_gemm_supported(b_kmajor, m, n, k, lda, ldb, ldd)) return GPZ_ERR_UNSUPPORTED;
  if (n_terms != 1 && n_terms != 3) return GPZ_ERR_BADARG;
  if (n_terms == 3 && (!Alo || !Blo)) return GPZ_ERR_BADARG;
  if (!aligned16(A) || !aligned16(B) || (Alo && !aligned16(Alo)) || (Blo && !aligned16(Blo)) || (sA % 4) || (sB % 4))
    return GPZ_ERR_UNSUPPORTED;
  if (splitk < 1) splitk = 1;
  if (splitk > 1 && (Cin || Dlo)) return GPZ_ERR_BADARG;
  CUtensorMap mA, mAlo, mB, mBlo;
  int b_map4d = 0;
  int rc = make_map_kmajor(&mA, A, m, k, lda, sA, batch, BM);
  if (rc) return rc;
  rc = make_map_kmajor(&mAlo, Alo ? Alo : A, m, k, lda, sA, batch, BM);
  if (rc) return rc;
  if (b_kmajor) {
    rc = make_map_kmajor(&mB, B, n, k, ldb, sB, batch, BN);
    if (rc) return rc;
    rc = make_map_kmajor(&mBlo, Blo ? Blo : B, n, k, ldb, sB, batch, BN);
  } else {
    b_map4d = n % 32 == 0 ? 1 : 0;
    if (b_map4d) {
      rc = make_map_mnmajor4d(&mB, B, k, n, ldb, sB, batch);
      if (rc == GPZ_OK) rc = make_map_mnmajor4d(&mBlo, Blo ? Blo : B, k, n, ldb, sB, batch);
      if (rc != GPZ_OK) b_map4d = 0;          // driver refused the 4-D view: fall back to 8 plain boxes
    }
    if (!b_map4d) {
      rc = make_map_mnmajor(&mB, B, k, n, ldb, sB, batch);
      if (rc) return rc;
      rc = make_map_mnmajor(&mBlo, Blo ? Blo : B, k, n, ldb, sB, batch);
    }
  }
  if (rc) return rc;
  Params p;
  p.b_map4d = b_map4d;
  p.epi_mode = epi ? epi->mode : 0;
  p.Aux = epi ? epi->Aux : nullptr; p.rowv = epi ? epi->rowv : nullptr; p.colv1 = epi ? epi->colv1 : nullptr;
  p.colv2 = epi ? epi->colv2 : nullptr; p.col1 = epi ? epi->col1 : nullptr; p.col2 = epi ? epi->col2 : nullptr;
  p.rowacc = epi ? epi->rowacc : nullptr;
  if (p.epi_mode != 0 && (splitk > 1 || d_tri != 0)) return GPZ_ERR_BADARG;
  p.D = D; p.Dlo = Dlo; p.Cin = Cin; p.m = m; p.n = n; p.k = k; p.ldd = ldd; p.sD = sD; p.batch = batch; p.splitk = splitk;
  p.a_tri = a_tri; p.b_tri = b_tri; p.d_tri = d_tri; p.n_terms = n_terms; p.alpha = alpha;
  p.bk = BK; p.sa = nullptr; p.sb = nullptr; p.Dh = nullptr; p.Dl = nullptr; p.sd = nullptr; p.amax = nullptr;
  p.AuxH = nullptr; p.AuxL = nullptr; p.saux = nullptr; p.D2h = nullptr; p.D2l = nullptr; p.sd2 = nullptr;
  if (p.epi_mode == 4) return GPZ_ERR_BADARG;            // split-FP16 only
  return launch_gemm(b_kmajor != 0, false, mA, mAlo, mB, mBlo, p, (cudaStream_t)stream, max_ctas);
}

// split-FP16 GEMM: every operand is a pair of fp16 planes (hi, lo) of x * s[b]; three kind::f16 MMAs per k-step
// (hi*lo + lo*hi + hi*hi) give ~2^-22 relative accuracy per product at twice the MMA rate of split-TF32.
int umma_gemm16_ex(const Umma16Args& g, void* stream) {
  if (g.m < 1 || g.n < 1 || g.k < 1 || g.batch < 1) return GPZ_ERR_BADARG;
  if (g.lda % 8 || g.ldb % 8 || g.sA % 8 || g.sB % 8) return GPZ_ERR_UNSUPPORTED;       // 16-byte global strides for TMA
  if (!aligned16(g.Ah) || !aligned16(g.Al) || !aligned16(g.Bh) || !aligned16(g.Bl)) return GPZ_ERR_UNSUPPORTED;
  int splitk = g.splitk < 1 ? 1 : g.splitk;
  if (splitk > 1 && (g.Dh || !g.D || g.amax)) return GPZ_ERR_BADARG;
  if (!g.D && !g.Dh) return GPZ_ERR_BADARG;
  if (g.Dh && !g.Dl) return GPZ_ERR_BADARG;
  CUtensorMap mA, mAlo, mB, mBlo;
  int b_map4d = 0;
  int rc = make_map_kmajor16(&mA, g.Ah, g.m, g.k, g.lda, g.sA, g.batch, BM);
  if (rc) return rc;
  rc = make_map_kmajor16(&mAlo, g.Al, g.m, g.k, g.lda, g.sA, g.batch, BM);
  if (rc) return rc;
  if (g.b_kmajor) {
    rc = make_map_kmajor16(&mB, g.Bh, g.n, g.k, g.ldb, g.sB, g.batch, BN);
    if (rc) return rc;
    rc = make_map_kmajor16(&mBlo, g.Bl, g.n, g.k, g.ldb, g.sB, g.batch, BN);
  } else {
    b_map4d = (g.n % 64 == 0) ? 1 : 0;
    if (b_map4d) {
      rc = make_map_mnmajor16_4d(&mB, g.Bh, g.k, g.n, g.ldb, g.sB, g.batch);
      if (rc == GPZ_OK) rc = make_map_mnmajor16_4d(&mBlo, g.Bl, g.k, g.n, g.ldb, g.sB, g.batch);
      if (rc != GPZ_OK) b_map4d = 0;
    }
    if (!b_map4d) {
      rc = make_map_mnmajor16(&mB, g.Bh, g.k, g.n, g.ldb, g.sB, g.batch);
      if (rc) return rc;
      rc = make_map_mnmajor16(&mBlo, g.Bl, g.k, g.n, g.ldb, g.sB, g.batch);
    }
  }
  if (rc) return rc;
  Params p;
  const UmmaEpilogue* epi = g.epi;
  p.b_map4d = b_map4d;
  p.epi_mode = epi ? epi->mode : 0;
  p.Aux = epi ? epi->Aux : nullptr; p.rowv = epi ? epi->rowv : nullptr; p.colv1 = epi ? epi->colv1 : nullptr;
  p.colv2 = epi ? epi->colv2 : nullptr; p.col1 = epi ? epi->col1 : nullptr; p.col2 = epi ? epi->col2 : nullptr;
  p.rowacc = epi ? epi->rowacc : nullptr;
  if (p.epi_mode != 0 && (splitk > 1 || g.d_tri != 0)) return GPZ_ERR_BADARG;
  if (g.Cin && (splitk > 1 || !g.D)) return GPZ_ERR_BADARG;
  p.D = g.D; p.Dlo = nullptr; p.Cin = g.Cin; p.m = g.m; p.n = g.n; p.k = g.k; p.ldd = g.ldd; p.sD = g.sD; p.batch = g.batch;
  p.splitk = splitk; p.a_tri = g.a_tri; p.b_tri = g.b_tri; p.d_tri = g.d_tri; p.n_terms = g.n_terms == 1 ? 1 : 3; p.alpha = g.alpha;
  p.bk = BK16; p.sa = g.sa; p.sb = g.sb; p.Dh = g.Dh; p.Dl = g.Dl; p.sd = g.sd; p.amax = g.amax;
  p.AuxH = g.AuxH; p.AuxL = g.AuxL; p.saux = g.saux; p.D2h = g.D2h; p.D2l = g.D2l; p.sd2 = g.sd2;
  if (p.epi_mode == 4 && (!p.AuxH || !p.D2h || !p.D2l)) return GPZ_ERR_BADARG;
  return launch_gemm(g.b_kmajor != 0, true, mA, mAlo, mB, mBlo, p, (cudaStream_t)stream);
}

// lo = x - tf32_trunc(x) for a flat array, and (optionally) the batched transpose of an M x M matrix with its lo part
__global__ void tf32_lo_kernel(const float* __restrict__ x, float* __restrict__ lo, int64_t n) {
  const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i + 3 < n) {
    const float4 v = *reinterpret_cast<const float4*>(x + i);
    float4 o;
    o.x = v.x - __uint_as_float(__float_as_uint(v.x) & 0xFFFFE000u);
    o.y = v.y - __uint_as_float(__float_as_uint(v.y) & 0xFFFFE000u);
    o.z = v.z - __uint_as_float(__float_as_uint(v.z) & 0xFFFFE000u);
    o.w = v.w - __uint_as_float(__float_as_uint(v.w) & 0xFFFFE000u);
    *reinterpret_cast<float4*>(lo + i) = o;
  } else {
    for (int64_t j = i; j < n; ++j) lo[j] = x[j] - __uint_as_float(__float_as_uint(x[j]) & 0xFFFFE000u);
  }
}
__global__ void transpose_lo_kernel(const float* __restrict__ x, float* __restrict__ xt, float* __restrict__ xt_lo, int M) {
  __shared__ float tile[32][33];
  const float* X = x + (int64_t)blockIdx.z * M * M;
  const int bx = blockIdx.x * 32, by = blockIdx.y * 32;
  for (int r = threadIdx.y; r < 32; r += 8) {
    const int i = by + r, j = bx + threadIdx.x;
    tile[r][threadIdx.x] = (i < M && j < M) ? X[(int64_t)i * M + j] : 0.f;
  }
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += 8) {
    const int i = bx + r, j = by + threadIdx.x;          // output (i, j) = input (j, i)
    if (i < M && j < M) {
      const float v = tile[threadIdx.x][r];
      const int64_t o = (int64_t)blockIdx.z * M * M + (int64_t)i * M + j;
      xt[o] = v;
      if (xt_lo) xt_lo[o] = v - __uint_as_float(__float_as_uint(v) & 0xFFFFE000u);
    }
  }
}

extern "C" int gpz_tf32_lo_f32(const float* x, float* lo, int64_t n, void* stream) {
  if (n <= 0) return GPZ_OK;
  if ((reinterpret_cast<uintptr_t>(x) & 15) || (reinterpret_cast<uintptr_t>(lo) & 15)) return GPZ_ERR_UNSUPPORTED;
  tf32_lo_kernel<<<(unsigned)cdiv(cdiv(n, 4), 256), 256, 0, (cudaStream_t)stream>>>(x, lo, n);
  GPZ_CHECK_LAUNCH();
  return GPZ_OK;
}
extern "C" int gpz_transpose_lo_f32(const float* x, float* xt, float* xt_lo, int M, int L, void* stream) {
  dim3 grid((unsigned)cdiv(M, 32), (unsigned)cdiv(M, 32), L);
  transpose_lo_kernel<<<grid, dim3(32, 8), 0, (cudaStream_t)stream>>>(x, xt, xt_lo, M);
  GPZ_CHECK_LAUNCH();
  return GPZ_OK;
}

// ---- split-FP16 operand preparation -----------------------------------------------------------------
namespace gpz {
namespace umma {
__global__ void __launch_bounds__(256) amax_kernel(const float* __restrict__ x, int64_t per_batch, unsigned int* __restrict__ amax) {
  const float* xb = x + (int64_t)blockIdx.y * per_batch;
  float m = 0.f;
  if ((per_batch & 3) == 0 && (reinterpret_cast<uintptr_t>(xb) & 15) == 0) {
    const float4* x4 = reinterpret_cast<const float4*>(xb);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < per_batch / 4; i += (int64_t)gridDim.x * blockDim.x) {
      const float4 v = x4[i];
      m = fmaxf(fmaxf(m, fmaxf(fabsf(v.x), fabsf(v.y))), fmaxf(fabsf(v.z), fabsf(v.w)));
    }
  } else {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < per_batch; i += (int64_t)gridDim.x * blockDim.x)
      m = fmaxf(m, fabsf(xb[i]));
  }
#pragma unroll
  for (int sh = 16; sh > 0; sh >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, sh));
  if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(amax + blockIdx.y, __float_as_uint(m));
}

// planes only (no transpose): 8 consecutive elements per thread, 16-byte stores
__global__ void __launch_bounds__(256) split16_flat_kernel(const float* __restrict__ x, int64_t per_batch,
                                                            const unsigned int* __restrict__ amax, float* __restrict__ scale,
                                                            __half* __restrict__ h, __half* __restrict__ l) {
  const int b = blockIdx.y;
  const float s = gpz_pow2_scale(__uint_as_float(amax[b]));
  if (blockIdx.x == 0 && threadIdx.x == 0) scale[b] = s;
  const int64_t base = (int64_t)b * per_batch;
  for (int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 8; i < per_batch; i += (int64_t)gridDim.x * blockDim.x * 8) {
    const float4 v0 = *reinterpret_cast<const float4*>(x + base + i), v1 = *reinterpret_cast<const float4*>(x + base + i + 4);
    uint4 ph, pl;
    split_half2(v0.x * s, v0.y * s, ph.x, pl.x);
    split_half2(v0.z * s, v0.w * s, ph.y, pl.y);
    split_half2(v1.x * s, v1.y * s, ph.z, pl.z);
    split_half2(v1.z * s, v1.w * s, ph.w, pl.w);
    *reinterpret_cast<uint4*>(h + base + i) = ph;
    *reinterpret_cast<uint4*>(l + base + i) = pl;
  }
}

__global__ void split16_kernel(const float* __restrict__ x, int rows, int cols, const unsigned int* __restrict__ amax,
                               float* __restrict__ scale, __half* __restrict__ h, __half* __restrict__ l, __half* __restrict__ hT,
                               __half* __restrict__ lT) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z;
  const float s = gpz_pow2_scale(__uint_as_float(amax[b]));
  if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0 && threadIdx.y == 0) scale[b] = s;
  const int64_t base = (int64_t)b * rows * cols;
  const int bx = blockIdx.x * 32, by = blockIdx.y * 32;
  for (int r = threadIdx.y; r < 32; r += 8) {
    const int i = by + r, j = bx + threadIdx.x;
    float v = 0.f;
    if (i < rows && j < cols) {
      v = x[base + (int64_t)i * cols + j] * s;
      __half hh, ll;
      split_half(v, hh, ll);
      if (h) { h[base + (int64_t)i * cols + j] = hh; l[base + (int64_t)i * cols + j] = ll; }
    }
    tile[r][threadIdx.x] = v;
  }
  if (!hT) return;
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += 8) {
    const int i = bx + r, j = by + threadIdx.x;          // transposed output (i, j) = input (j, i); shape cols x rows
    if (i < cols && j < rows) {
      __half hh, ll;
      split_half(tile[threadIdx.x][r], hh, ll);
      hT[base + (int64_t)i * rows + j] = hh;
      lT[base + (int64_t)i * rows + j] = ll;
    }
  }
}
}  // namespace umma
}  // namespace gpz

int split16_amax(const float* x, int64_t per_batch, int batch, unsigned int* amax_bits, void* stream) {
  if (per_batch <= 0 || batch <= 0) return GPZ_OK;
  const unsigned chunks = (unsigned)std::min<int64_t>(cdiv(per_batch, 256 * 8), 1024);
  amax_kernel<<<dim3(chunks, batch), 256, 0, (cudaStream_t)stream>>>(x, per_batch, amax_bits);
  GPZ_CHECK_LAUNCH();
  return GPZ_OK;
}
int split16_planes(const float* x, int rows, int cols, int batch, const unsigned int* amax_bits, float* scale, __half* h, __half* l,
                   __half* hT, __half* lT, void* stream) {
  if (rows <= 0 || cols <= 0 || batch <= 0) return GPZ_OK;
  const int64_t per_batch = (int64_t)rows * cols;
  if (!hT && h && per_batch % 8 == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(h) & 15) == 0 &&
      (reinterpret_cast<uintptr_t>(l) & 15) == 0) {
    const unsigned chunks = (unsigned)std::min<int64_t>(cdiv(per_batch, 256 * 8 * 4), 2048);
    split16_flat_kernel<<<dim3(chunks, batch), 256, 0, (cudaStream_t)stream>>>(x, per_batch, amax_bits, scale, h, l);
    GPZ_CHECK_LAUNCH();
    return GPZ_OK;
  }
  dim3 grid((unsigned)cdiv(cols, 32), (unsigned)cdiv(rows, 32), batch);
  split16_kernel<<<grid, dim3(32, 8), 0, (cudaStream_t)stream>>>(x, rows, cols, amax_bits, scale, h, l, hT, lT);
  GPZ_CHECK_LAUNCH();
  return GPZ_OK;
}

// x (batch x rows x cols fp32) -> fp16 planes (h, l) of x * scale[b] and optionally of the transposes; amax_ws: batch uint32 scratch
extern "C" int gpz_split16_f32(const float* x, int rows, int cols, int batch, void* h, void* l, void* hT, void* lT, float* scale,
                               void* amax_ws, void* stream) {
  GPZ_CUDA(cudaMemsetAsync(amax_ws, 0, sizeof(unsigned int) * (size_t)batch, (cudaStream_t)stream));
  int rc = split16_amax(x, (int64_t)rows * cols, batch, (unsigned int*)amax_ws, stream);
  if (rc) return rc;
  return split16_planes(x, rows, cols, batch, (const unsigned int*)amax_ws, scale, (__half*)h, (__half*)l, (__half*)hT, (__half*)lT,
                        stream);
}

extern "C" int gpz_umma_gemm16_f32(int b_kmajor, int m, int n, int k, float alpha, const void* Ah, const void* Al, int64_t lda,
                                   int64_t sA, const float* sa, const void* Bh, const void* Bl, int64_t ldb, int64_t sB,
                                   const float* sb, const float* Cin, float* D, void* Dh, void* Dl, const float* sd, void* amax,
                                   int64_t ldd, int64_t sD, int batch, int a_tri, int b_tri, int d_tri, int splitk, int n_terms,
                                   void* stream) {
  Umma16Args g{};
  g.b_kmajor = b_kmajor; g.m = m; g.n = n; g.k = k; g.alpha = alpha;
  g.Ah = (const __half*)Ah; g.Al = (const __half*)Al; g.lda = lda; g.sA = sA; g.sa = sa;
  g.Bh = (const __half*)Bh; g.Bl = (const __half*)Bl; g.ldb = ldb; g.sB = sB; g.sb = sb;
  g.D = D; g.ldd = ldd; g.sD = sD; g.Dh = (__half*)Dh; g.Dl = (__half*)Dl; g.sd = sd; g.amax = (unsigned int*)amax;
  g.batch = batch; g.a_tri = a_tri; g.b_tri = b_tri; g.d_tri = d_tri; g.splitk = splitk; g.n_terms = n_terms; g.Cin = Cin;
  return umma_gemm16_ex(g, stream);
}
