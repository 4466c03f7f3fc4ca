// Backward-pass pieces shared by pdg_backward.cu (parameter and input gradients) and pdg_vjp.cu (input gradients of K
// cotangents): the data-gradient workspace, the tile helpers and the LayerNorm-backward finalize.
#pragma once
#include "pdg_ws.cuh"

namespace pdg {

constexpr int BKB = 16;  // weight k-chunk in backward kernels (3 tiles + 2 chunks fit in 227 KB)
constexpr size_t SMEM_B3T = (size_t)(3 * TM * LDS + 2 * BKB * H) * sizeof(float) + TM * 4 * sizeof(float) + 256;

struct BwdWs {
  int64_t N_pad, E_pad;
  int G;
  char* base;
  size_t total;
  float *cta_grads, *gx, *gagg, *RA, *RB, *ge, *DHM, *DHN, *cs1, *cs2, *cs3, *scal, *gdec, *gs;
  BwdWs(int64_t n, int64_t e, int steps, int g, void* ws) : G(g), base((char*)ws) {
    N_pad = round_up(n, TM);
    E_pad = round_up(e, TM);
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t r = o; o += (size_t)round_up((int64_t)bytes, 256); return (float*)(base + r); };
    const size_t nb = (size_t)N_pad * H * sizeof(float), eb = (size_t)E_pad * H * sizeof(float);
    cta_grads = take((size_t)G * GRADP * sizeof(float));
    gx = take(nb); gagg = take(nb); RA = take(nb); RB = take(nb);
    ge = take(eb); DHM = take(eb); DHN = take(eb);
    cs1 = take((size_t)MAXP * 2 * H * sizeof(float));
    cs2 = take((size_t)MAXP * 2 * H * sizeof(float));
    cs3 = take((size_t)MAXP * 2 * H * sizeof(float));
    scal = take((size_t)(2 + 3 * steps) * 4 * sizeof(float));
    gdec = take((size_t)N_pad * 4 * sizeof(float));
    gs = take(256);  // {S, 1/S} of the fp16 backward (k_grad_scale)
    total = o;
  }
};

// ---- small device helpers ------------------------------------------------------------------
// reduce per-thread column partials (cols tx*4.., 64+tx*4..) over the 16 ty groups; dst[128]
__device__ __forceinline__ void colsum_flush(const float (&v)[8], float* scratch, float* dst, bool add) {
  const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;
  __syncthreads();
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    scratch[ty * H + tx * 4 + j] = v[j];
    scratch[ty * H + 64 + tx * 4 + j] = v[4 + j];
  }
  __syncthreads();
  if (threadIdx.x < H) {
    float s = 0.f;
#pragma unroll
    for (int t = 0; t < 16; ++t) s += scratch[t * H + threadIdx.x];
    dst[threadIdx.x] = add ? dst[threadIdx.x] + s : s;
  }
  __syncthreads();
}
// sum over rows < nvalid of column tid of a smem tile (threads < 128)
__device__ __forceinline__ float tile_colsum(const float* T, int nvalid) {
  float s = 0.f;
  if (threadIdx.x < H)
    for (int r = 0; r < nvalid; ++r) s += T[r * LDS + threadIdx.x];
  return s;
}
// load a [128][128] global tile into smem (row-linear, coalesced): sixteen 16-byte cp.async per thread, all in flight at
// once (a register-staged loop kept four: the tile loads were long-scoreboard stalls).  Every caller has a
// __syncthreads() between this and the first read of T.
__device__ __forceinline__ void tile_load(float* T, const float* __restrict__ src) {
  const int tid = threadIdx.x, c4 = (tid & 31) * 4;
#pragma unroll
  for (int it = 0; it < (TM * H / 4) / NT; ++it) {
    const int r = (tid >> 5) + it * 8;
    cp_async16(T + r * LDS + c4, src + (size_t)r * H + c4);
  }
  cp_async_commit();
  cp_async_wait<0>();
}
// global microtile load
__device__ __forceinline__ void mt_load(float (&m)[8][8], const float* __restrict__ src) { acc_load(m, src, H); }

// ---- LayerNorm-backward finalize (1 block, 8 x 128 threads) ------------------------------------
// thread = (channel j, group g): group g owns the per-CTA partials p = g, g+8, ...; all of its loads are issued
// before the first add (one L2 round trip instead of a dependent chain), sums run in a fixed order, groups are
// combined in a fixed order, and the two 128-channel dot products use a fixed shuffle tree => bit-reproducible.
constexpr int FIN_G = 8;
constexpr int FIN_K = 10;  // partials per thread and pass (80 per pass: two passes for 148 CTAs)
struct LnFinArgs {
  const float* cs;
  int nparts;
  const double* fwd_parts;
  double count;
  const float* lnw;
  float* scal_out;
  float* flat_w;  // accumulated with +=: one writer per array and launch
  float* flat_b;
};
// AFFINE = false: the scalars only (input-gradient passes); flat_w / flat_b are not touched
template <bool AFFINE = true>
__device__ __forceinline__ void ln_finalize_body(const float* __restrict__ cs, int nparts, const double* __restrict__ fwd_parts,
                                                 double count, const float* __restrict__ lnw, float* __restrict__ scal_out,
                                                 float* __restrict__ flat_w, float* __restrict__ flat_b) {
  __shared__ float smf[4];
  __shared__ double pc[FIN_G][H], pcy[FIN_G][H];
  __shared__ double r1[4], r2[4];
  const int j = threadIdx.x & (H - 1), g = threadIdx.x >> 7;
  pdl_sync();
  const LnStat st = ln_stat_block(fwd_parts, count, smf);
  double a0 = 0, b0 = 0;
  for (int base = 0; base < nparts; base += FIN_G * FIN_K) {
    float x[FIN_K], y[FIN_K];
#pragma unroll
    for (int k = 0; k < FIN_K; ++k) {
      const int p = base + g + k * FIN_G;
      x[k] = p < nparts ? cs[(size_t)p * 2 * H + j] : 0.f;
      y[k] = p < nparts ? cs[(size_t)p * 2 * H + H + j] : 0.f;
    }
#pragma unroll
    for (int k = 0; k < FIN_K; ++k) { a0 += (double)x[k]; b0 += (double)y[k]; }
  }
  pc[g][j] = a0;
  pcy[g][j] = b0;
  __syncthreads();
  if (g == 0) {
    double cg = 0, cgy = 0;
#pragma unroll
    for (int k = 0; k < FIN_G; ++k) { cg += pc[k][j]; cgy += pcy[k][j]; }
    const double w = lnw[j];
    const double s1 = warp_sum(w * cg);
    const double s2 = warp_sum(w * cgy);  // producers accumulate g*(y-mu) (centred before the product: no cancellation)
    if ((j & 31) == 0) { r1[j >> 5] = s1; r2[j >> 5] = s2; }
    if (AFFINE) {
      flat_w[j] += (float)((double)st.rstd * cgy);
      flat_b[j] += (float)cg;
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    const double S1 = (r1[0] + r1[1]) + (r1[2] + r1[3]), S2 = (r2[0] + r2[1]) + (r2[2] + r2[3]);
    const double a = st.rstd;
    scal_out[0] = (float)(a * S1 / count);
    scal_out[1] = st.sigma > 0.f ? (float)(a * a * S2 / (count * (double)st.sigma)) : 0.f;
    scal_out[2] = st.mu;
    scal_out[3] = st.rstd;
  }
}

}  // namespace pdg
