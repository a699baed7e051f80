// K7-G: fused Gaussian factor-model log-likelihood (RSF / FA) with the loading contraction, forward + backward in one pass over y.
//
// Model: y_gn ~ N(b_g + sum_f W_gf F_fn, s_g^2), s = softplus(noise), tau = 1 / s^2, with independent F_fn ~ q = N(m_fn, v_fn).
// The expectation over q is exact, so there are no samples:
//   r_gn = y_gn - b_g - sum_f W_gf m_fn,   t_gn = tau_g r_gn,   V_f = sum_n v_fn,   kappa_f = -1/2 sum_g tau_g W_gf^2
//   ll            = sum_{g,n} [ -1/2 log 2 pi - log s_g - 1/2 tau_g r_gn^2 ] + sum_f kappa_f V_f
//   d/dm_fn       = sum_g W_gf t_gn                    d/dv_fn = kappa_f
//   d/dW_gf       = sum_n t_gn m_fn - tau_g W_gf V_f   d/db_g  = sum_n t_gn
//   d/dnoise_g    = softplus'(noise_g) ( -B / s_g + (sum_n r_gn^2 + sum_f W_gf^2 V_f) / s_g^3 )
// spread[f, :] is a variance (v = max(spread, clamp_min), gradient passed at equality) for f < n_var and a std-dev (v = spread^2)
// otherwise, as in K7.  This is the E -> infinity limit of mean_E sum Normal(b + W F_e, s).log_prob(y).
//
// Only r (F FMAs), the per-spot d/dm (F), the per-gene sum_n t m (F), sum_n t and sum_n t^2 (= sum_n r^2 / s^4) touch the G x B
// elements; they run in gauss_kernel, which reads y once and writes nothing of size G x B.  V, kappa (gauss_prep_kernel) and the
// tau W V correction, d/dnoise, d/dspread and ll (gauss_finish_kernel, gauss_ll_kernel) are O((G + B) F).  Every partial is summed
// in a fixed order (no atomics); V, kappa, ll, sum_n r^2 and the final d/dW combination are carried in double: near a fit
// sum_n t m and tau W V nearly cancel.
#include "common.cuh"
#include "gpzoo_b200.h"

namespace gpz {

template <typename T> struct GaussArgs {
  const T* y; int64_t y_ld;            // G x Ntot, row stride
  const int64_t* idx;                  // B or null (minibatch gather y[:, idx])
  const T* W; const T* bias; const T* noise;   // G x F, G, G (raw: s = softplus(noise))
  const T* mean; const T* spread;      // F x B
  int G, F, B, n_var;
  T clamp_min;
  // workspace
  double* Vd; double* kap;             // [F] V_f, kappa_f
  double* llg;                         // [G] the gene's share of ll (without the kappa V term)
  double* gt_part;                     // [nbx][G][2] sum_n t, sum_n t^2 over the CTA's spots
  T* gW_part;                          // [nbx][G][F] sum_n t m_f over the CTA's spots
  T* gm_part;                          // [nby][F][B] sum_g W_gf t over the CTA's gene range
  int genes_per_cta;                   // multiple of GS_GCH
  // outputs
  double* ll; T* gW; T* gbias; T* gnoise; T* gmean; T* gspread;
};

// ---- gauss_kernel: two spots per thread (256 spots per CTA), the layout of poisson_kernel2 without its sample loop -------------
// A CTA walks its gene range in chunks of 32 staged in shared memory (W rows, tau, b).  Phase A (thread = two spots, so y rows are
// read coalesced, four genes prefetched ahead): r, t, d/dm accumulated in registers, t parked in shared memory.  Phase B (lane =
// gene, warp = a quarter of the spots): sum_n t m_f, sum_n t, sum_n t^2 from shared memory, written as per-CTA partials.
constexpr int GS_THREADS = 128, GS_SPOTS = 256, GS_GCH = 32, GS_GRP = 4;

template <typename T, int FMAX> constexpr size_t gauss_smem() {
  return ((sizeof(T) * GS_GCH * (GS_SPOTS + 1) + 15) / 16) * 16 + sizeof(T) * (FMAX * GS_SPOTS + GS_GCH * FMAX + 4 * GS_GCH * FMAX);
}

// fp32: four CTAs per SM up to FMAX = 12 (128 registers), three above, where 128 registers would spill
template <typename T, int FMAX>
__global__ void __launch_bounds__(GS_THREADS, sizeof(T) == 4 ? (FMAX > 12 ? 3 : 4) : 1) gauss_kernel(const GaussArgs<T> a) {
  extern __shared__ __align__(16) unsigned char gs_smem[];
  typedef T RowT[GS_SPOTS + 1];
  typedef T RowF[FMAX];
  typedef T AccW[GS_GCH][FMAX];
  RowT* tS = reinterpret_cast<RowT*>(gs_smem);                         // [GS_GCH][GS_SPOTS+1]   t
  RowF* mS = reinterpret_cast<RowF*>(gs_smem + ((sizeof(T) * GS_GCH * (GS_SPOTS + 1) + 15) / 16) * 16);   // [GS_SPOTS][FMAX]
  RowF* sW = mS + GS_SPOTS;                                            // [GS_GCH][FMAX]
  AccW* sAcc = reinterpret_cast<AccW*>(sW + GS_GCH);                   // [4][GS_GCH][FMAX]
  __shared__ T sTau[GS_GCH], sB[GS_GCH];
  __shared__ T sT[GS_THREADS / 32][GS_GCH][2];                         // per-warp sum_n t, sum_n t^2

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n0 = blockIdx.x * GS_SPOTS;
  int nn[2]; bool act[2]; int64_t col[2];
  T pg[2][FMAX];
#pragma unroll
  for (int s2 = 0; s2 < 2; ++s2) {
    nn[s2] = n0 + s2 * GS_THREADS + tid;
    act[s2] = nn[s2] < a.B;
    col[s2] = act[s2] ? (a.idx ? a.idx[nn[s2]] : (int64_t)nn[s2]) : 0;
#pragma unroll
    for (int f = 0; f < FMAX; ++f) {
      pg[s2][f] = T(0);
      mS[s2 * GS_THREADS + tid][f] = (f < a.F && act[s2]) ? a.mean[(int64_t)f * a.B + nn[s2]] : T(0);
    }
  }
  const int g_begin = blockIdx.y * a.genes_per_cta;
  const int g_end = min(a.G, g_begin + a.genes_per_cta);

  // y is prefetched four genes ahead, walking the range's rows in order: the row offset advances by additions, so a load costs
  // one 64-bit add instead of a 64-bit multiply-add per element
  const T* yc[2] = {a.y + col[0], a.y + col[1]};
  int gnext = g_begin;
  int64_t ynoff = (int64_t)g_begin * a.y_ld;
  T ynext[GS_GRP][2];
  auto prefetch = [&]() {
    int64_t off = ynoff;
#pragma unroll
    for (int u = 0; u < GS_GRP; ++u) {
#pragma unroll
      for (int s2 = 0; s2 < 2; ++s2) ynext[u][s2] = (act[s2] && gnext + u < g_end) ? __ldcs(yc[s2] + off) : T(0);
      off += a.y_ld;
    }
    gnext += GS_GRP;
    ynoff = off;
  };
  prefetch();

  for (int g0 = g_begin; g0 < g_end; g0 += GS_GCH) {
    __syncthreads();                               // previous chunk's phase B / flush finished with sW, tS, sAcc, sT
    for (int i = tid; i < GS_GCH * FMAX; i += GS_THREADS) {
      const int gi = i / FMAX, f = i % FMAX;
      sW[gi][f] = (g0 + gi < g_end && f < a.F) ? a.W[(int64_t)(g0 + gi) * a.F + f] : T(0);
    }
    if (tid < GS_GCH) {                            // genes past the range get tau = 0, hence t = 0
      const bool in = g0 + tid < g_end;
      const T s = in ? softplus(a.noise[g0 + tid]) : T(1);
      sTau[tid] = in ? T(1) / (s * s) : T(0);
      sB[tid] = in ? a.bias[g0 + tid] : T(0);
    }
    __syncthreads();
    // ---- phase A: thread = two spots ----
    T m[2][FMAX];                                  // re-read per chunk: not live through phase B
#pragma unroll
    for (int s2 = 0; s2 < 2; ++s2) load_row<FMAX>(&mS[s2 * GS_THREADS + tid][0], m[s2]);
#pragma unroll 1
    for (int gb = 0; gb < GS_GCH; gb += GS_GRP) {
      T yv[GS_GRP][2];
#pragma unroll
      for (int u = 0; u < GS_GRP; ++u) { yv[u][0] = ynext[u][0]; yv[u][1] = ynext[u][1]; }
      prefetch();                                  // genes g0 + gb + 4 ...; past the range's end this loads nothing
#pragma unroll
      for (int u = 0; u < GS_GRP; ++u) {
        const int gi = gb + u;
        T wrow[FMAX];
        load_row<FMAX>(&sW[gi][0], wrow);
        const T tau = sTau[gi], b = sB[gi];
#pragma unroll
        for (int s2 = 0; s2 < 2; ++s2) {
          T z0 = T(0), z1 = T(0);
#pragma unroll
          for (int f = 0; f < FMAX; f += 2) { z0 = fma(wrow[f], m[s2][f], z0); z1 = fma(wrow[f + 1], m[s2][f + 1], z1); }
          const T t = act[s2] ? tau * ((yv[u][s2] - b) - (z0 + z1)) : T(0);
#pragma unroll
          for (int f = 0; f < FMAX; ++f) pg[s2][f] = fma(wrow[f], t, pg[s2][f]);
          tS[gi][s2 * GS_THREADS + tid] = t;
        }
      }
    }
    __syncthreads();
    // ---- phase B: lane = gene, warp = a quarter (64) of the spots ----
    T acc[FMAX];
#pragma unroll
    for (int f = 0; f < FMAX; ++f) acc[f] = T(0);
    T st = T(0), st2 = T(0);
    const int nb = warp * 64;
#pragma unroll 4
    for (int k = 0; k < 64; ++k) {
      const T t = tS[lane][nb + k];
      T mrow[FMAX];
      load_row<FMAX>(&mS[nb + k][0], mrow);
#pragma unroll
      for (int f = 0; f < FMAX; ++f) acc[f] = fma(t, mrow[f], acc[f]);
      st += t;
      st2 = fma(t, t, st2);
    }
#pragma unroll
    for (int f = 0; f < FMAX; ++f) sAcc[warp][lane][f] = acc[f];
    sT[warp][lane][0] = st;
    sT[warp][lane][1] = st2;
    __syncthreads();
    for (int i = tid; i < GS_GCH * a.F; i += GS_THREADS) {
      const int gi = i / a.F, f = i % a.F;
      if (g0 + gi < g_end)
        a.gW_part[((int64_t)blockIdx.x * a.G + g0 + gi) * a.F + f] = sAcc[0][gi][f] + sAcc[1][gi][f] + sAcc[2][gi][f] + sAcc[3][gi][f];
    }
    if (tid < GS_GCH && g0 + tid < g_end) {
      double* dst = a.gt_part + ((int64_t)blockIdx.x * a.G + g0 + tid) * 2;
#pragma unroll
      for (int j = 0; j < 2; ++j)
        dst[j] = ((double)sT[0][tid][j] + (double)sT[1][tid][j]) + ((double)sT[2][tid][j] + (double)sT[3][tid][j]);
    }
  }
#pragma unroll
  for (int s2 = 0; s2 < 2; ++s2) {
    if (!act[s2]) continue;
#pragma unroll
    for (int f = 0; f < FMAX; ++f)
      if (f < a.F) a.gm_part[((int64_t)blockIdx.y * a.F + f) * a.B + nn[s2]] = pg[s2][f];
  }
}

// blocks [0, F): V_f = sum_n v_fn; blocks [F, 2F): kappa_f = -1/2 sum_g W_gf^2 / softplus(noise_g)^2; both in double
template <typename T>
__global__ void __launch_bounds__(256) gauss_prep_kernel(const GaussArgs<T> a) {
  __shared__ double red[32];
  const bool is_v = (int)blockIdx.x < a.F;
  const int f = is_v ? blockIdx.x : blockIdx.x - a.F;
  double s = 0.0;
  if (is_v) {
    for (int n = threadIdx.x; n < a.B; n += blockDim.x) {
      const double sp = (double)a.spread[(int64_t)f * a.B + n];
      s += f < a.n_var ? (sp > (double)a.clamp_min ? sp : (double)a.clamp_min) : sp * sp;
    }
  } else {
    for (int g = threadIdx.x; g < a.G; g += blockDim.x) {
      const double sd = softplus((double)a.noise[g]), w = (double)a.W[(int64_t)g * a.F + f];
      s += w * w / (sd * sd);
    }
    s *= -0.5;
  }
  s = block_sum<double>(s, red);
  if (threadIdx.x == 0) (is_v ? a.Vd : a.kap)[f] = s;
}

// blocks [0, gw_blocks): gW[g, f] = sum_b gW_part[b, g, f] - tau_g W_gf V_f (double), one element per thread;
// blocks [gw_blocks, + gene_blocks): per gene d/db, d/dnoise and the gene's share of ll;
// blocks [..., + spot_blocks): per (f, n) d/dm = sum of the gene ranges' partials, d/dspread = kappa_f (clamp) or 2 kappa_f spread.
template <typename T>
__global__ void __launch_bounds__(256) gauss_finish_kernel(const GaussArgs<T> a, int nbx, int nby, int gw_blocks, int gene_blocks) {
  int bid = blockIdx.x;
  const int64_t GF = (int64_t)a.G * a.F;
  if (bid < gw_blocks) {
    const int64_t e = (int64_t)bid * blockDim.x + threadIdx.x;
    if (e >= GF) return;
    const int g = (int)(e / a.F), f = (int)(e % a.F);
    double s = 0.0;
    for (int b = 0; b < nbx; ++b) s += (double)a.gW_part[(int64_t)b * GF + e];
    const double sd = softplus((double)a.noise[g]);
    a.gW[e] = (T)(s - (double)a.W[e] * a.Vd[f] / (sd * sd));
    return;
  }
  bid -= gw_blocks;
  if (bid < gene_blocks) {
    const int g = bid * blockDim.x + threadIdx.x;
    if (g >= a.G) return;
    double st = 0.0, st2 = 0.0;
    for (int b = 0; b < nbx; ++b) {
      st += a.gt_part[((int64_t)b * a.G + g) * 2];
      st2 += a.gt_part[((int64_t)b * a.G + g) * 2 + 1];
    }
    const double x = (double)a.noise[g], sd = softplus(x), s2 = sd * sd;
    const double R = st2 * s2 * s2;                // sum_n r^2
    double wv = 0.0;
    for (int f = 0; f < a.F; ++f) {
      const double w = (double)a.W[(int64_t)g * a.F + f];
      wv += w * w * a.Vd[f];
    }
    a.gbias[g] = (T)st;
    a.gnoise[g] = (T)(softplus_grad(x) * (-(double)a.B / sd + (R + wv) / (s2 * sd)));
    a.llg[g] = -(double)a.B * (0.91893853320467274178 + ::log(sd)) - 0.5 * R / s2;
    return;
  }
  bid -= gene_blocks;
  const int64_t e = (int64_t)bid * blockDim.x + threadIdx.x;
  if (e >= (int64_t)a.F * a.B) return;
  const int f = (int)(e / a.B);
  T s = T(0);
  for (int j = 0; j < nby; ++j) s += a.gm_part[(int64_t)j * a.F * a.B + e];
  a.gmean[e] = s;
  const T k = (T)a.kap[f], sp = a.spread[e];
  a.gspread[e] = f < a.n_var ? (sp >= a.clamp_min ? k : T(0)) : T(2) * k * sp;
}

// ll = sum_g llg[g] + sum_f kappa_f V_f, in a fixed order
__global__ void __launch_bounds__(256) gauss_ll_kernel(const double* __restrict__ llg, const double* __restrict__ Vd,
                                                       const double* __restrict__ kap, int G, int F, double* __restrict__ out) {
  __shared__ double red[32];
  double s = 0.0;
  for (int g = threadIdx.x; g < G; g += blockDim.x) s += llg[g];
  if ((int)threadIdx.x < F) s += kap[threadIdx.x] * Vd[threadIdx.x];
  s = block_sum<double>(s, red);
  if (threadIdx.x == 0) out[0] = s;
}

// 256 spots per CTA; gene ranges of whole 32-gene chunks, about eight CTAs per SM in all (poisson_kernel2's grid)
static void gauss_grid(int G, int B, int* nbx, int* nby, int* gpc) {
  *nbx = (int)cdiv(B, GS_SPOTS);
  const int chunks = (int)cdiv(G, GS_GCH);
  int by = 1;
  if (*nbx < 1184) by = (int)min((int64_t)chunks, cdiv(1184, *nbx > 0 ? *nbx : 1));
  *gpc = (int)cdiv(chunks, by) * GS_GCH;
  *nby = (int)cdiv(G, *gpc);
}

static size_t a16(size_t n) { return (n + 15) / 16 * 16; }
// workspace: V, kappa [2][F] double | llg [G] double | gt_part [nbx][G][2] double | gW_part [nbx][G][F] T | gm_part [nby][F][B] T
static size_t gauss_ws_bytes(int G, int F, int B, size_t elt) {
  int nbx, nby, gpc;
  gauss_grid(G, B, &nbx, &nby, &gpc);
  return a16(sizeof(double) * 2 * (size_t)F) + a16(sizeof(double) * (size_t)G) + sizeof(double) * 2 * (size_t)nbx * G +
         a16(elt * (size_t)nbx * G * F) + a16(elt * (size_t)nby * F * B);
}

template <typename T, int FMAX> int gauss_launch(const GaussArgs<T>& a, dim3 grid, cudaStream_t st) {
  constexpr size_t smem = gauss_smem<T, FMAX>();
  GPZ_CUDA(cudaFuncSetAttribute(gauss_kernel<T, FMAX>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  gauss_kernel<T, FMAX><<<grid, GS_THREADS, smem, st>>>(a);
  GPZ_CHECK_LAUNCH();
  return GPZ_OK;
}

template <typename T> int gauss_fwdbwd(GaussArgs<T> a, void* ws, size_t ws_bytes, cudaStream_t st) {
  if (a.F < 1 || a.F > 32 || a.G < 1 || a.B < 0 || a.n_var < 0 || a.n_var > a.F) return GPZ_ERR_UNSUPPORTED;
  if (!a.idx && a.y_ld < a.B) return GPZ_ERR_UNSUPPORTED;
  if (ws_bytes < gauss_ws_bytes(a.G, a.F, a.B, sizeof(T))) return GPZ_ERR_BADARG;
  if (a.B == 0) {                       // empty minibatch: ll = 0, no gradient
    GPZ_CUDA(cudaMemsetAsync(a.ll, 0, sizeof(double), st));
    GPZ_CUDA(cudaMemsetAsync(a.gW, 0, sizeof(T) * (size_t)a.G * a.F, st));
    GPZ_CUDA(cudaMemsetAsync(a.gbias, 0, sizeof(T) * (size_t)a.G, st));
    GPZ_CUDA(cudaMemsetAsync(a.gnoise, 0, sizeof(T) * (size_t)a.G, st));
    return GPZ_OK;
  }
  int nbx, nby, gpc;
  gauss_grid(a.G, a.B, &nbx, &nby, &gpc);
  unsigned char* p = reinterpret_cast<unsigned char*>(ws);
  a.Vd = reinterpret_cast<double*>(p); a.kap = a.Vd + a.F; p += a16(sizeof(double) * 2 * (size_t)a.F);
  a.llg = reinterpret_cast<double*>(p); p += a16(sizeof(double) * (size_t)a.G);
  a.gt_part = reinterpret_cast<double*>(p); p += sizeof(double) * 2 * (size_t)nbx * a.G;
  a.gW_part = reinterpret_cast<T*>(p); p += a16(sizeof(T) * (size_t)nbx * a.G * a.F);
  a.gm_part = reinterpret_cast<T*>(p);
  a.genes_per_cta = gpc;

  gauss_prep_kernel<T><<<2 * a.F, 256, 0, st>>>(a);
  GPZ_CHECK_LAUNCH();
  const dim3 grid(nbx, nby);
  int rc;
  if (a.F <= 4) rc = gauss_launch<T, 4>(a, grid, st);
  else if (a.F <= 12) rc = gauss_launch<T, 12>(a, grid, st);
  else if (a.F <= 20) rc = gauss_launch<T, 20>(a, grid, st);
  else rc = gauss_launch<T, 32>(a, grid, st);
  if (rc) return rc;
  const int gw_blocks = (int)cdiv((int64_t)a.G * a.F, 256), gene_blocks = (int)cdiv(a.G, 256);
  const int spot_blocks = (int)cdiv((int64_t)a.F * a.B, 256);
  gauss_finish_kernel<T><<<gw_blocks + gene_blocks + spot_blocks, 256, 0, st>>>(a, nbx, nby, gw_blocks, gene_blocks);
  GPZ_CHECK_LAUNCH();
  gauss_ll_kernel<<<1, 256, 0, st>>>(a.llg, a.Vd, a.kap, a.G, a.F, a.ll);
  GPZ_CHECK_LAUNCH();
  return GPZ_OK;
}

}  // namespace gpz

using namespace gpz;

#define GPZ_GAUSSIAN_IMPL(SUF, T)                                                                                      \
  extern "C" int64_t gpz_gaussian_workspace_bytes_##SUF(int G, int F, int B) {                                        \
    return (int64_t)gauss_ws_bytes(G, F, B, sizeof(T));                                                                \
  }                                                                                                                    \
  extern "C" int gpz_gaussian_fwdbwd_##SUF(const T* y, int64_t y_ld, const int64_t* idx, const T* W, const T* bias,    \
                                           const T* noise, const T* mean, const T* spread, int G, int F, int B,        \
                                           int n_var, T clamp_min, double* ll, T* gW, T* gbias, T* gnoise, T* gmean,   \
                                           T* gspread, void* ws, int64_t ws_bytes, void* stream) {                     \
    GaussArgs<T> a = {};                                                                                               \
    a.y = y; a.y_ld = y_ld; a.idx = idx; a.W = W; a.bias = bias; a.noise = noise; a.mean = mean; a.spread = spread;    \
    a.G = G; a.F = F; a.B = B; a.n_var = n_var; a.clamp_min = clamp_min;                                               \
    a.ll = ll; a.gW = gW; a.gbias = gbias; a.gnoise = gnoise; a.gmean = gmean; a.gspread = gspread;                    \
    return gauss_fwdbwd<T>(a, ws, ws_bytes < 0 ? 0 : (size_t)ws_bytes, (cudaStream_t)stream);                          \
  }

GPZ_GAUSSIAN_IMPL(f32, float)
GPZ_GAUSSIAN_IMPL(f64, double)
