// Backward-pass pieces shared by pdg_backward.cu (parameter and input gradients) and pdg_vjp.cu (input gradients of K
// cotangents): the data-gradient workspace and what step t reads, the tile helpers, the LayerNorm-backward finalize and
// the bodies of the decoder, node_update, node_pre and encoder kernels.
#pragma once
#include "pdg_ws.cuh"

namespace pdg {

constexpr int BKB = 16;  // weight k-chunk in backward kernels (3 tiles + 2 chunks fit in 227 KB)
constexpr size_t SMEM_B3T = (size_t)(3 * TM * LDS + 2 * BKB * H) * sizeof(float) + TM * 4 * sizeof(float) + 256;
// the kernel bodies below without weight gradients (pdg_vjp.cu): two tiles + the weight chunks + a [TM][4] (or [TM][8]) row area
constexpr size_t SMEM_V2T = (size_t)(2 * TM * LDS + 2 * BKB * H) * sizeof(float) + TM * 8 * sizeof(float) + 256;

// The data-gradient buffers of one backward pass, in workspace order: the gradient chain between kernels (gx, gagg, ge),
// the receiver-side segment sums RA / RB (adjacent: one memset), the edge kernels' hidden gradients DHM / DHN, the per-CTA
// LayerNorm column sums and the LayerNorm-backward scalars.  BwdWs and VjpWs (pdg_vjp.cu) both lay them out with `take`.
struct DataGradBufs {
  float *gx, *gagg, *RA, *RB, *ge, *DHM, *DHN, *cs1, *cs2, *cs3, *scal;
  template <class Take>
  void take_data_grads(Take& take, int64_t N_pad, int64_t E_pad, int steps) {
    const size_t nb = (size_t)N_pad * H * sizeof(float), eb = (size_t)E_pad * H * sizeof(float);
    gx = take(nb); gagg = take(nb); RA = take(nb); RB = take(nb);
    ge = take(eb); DHM = take(eb); DHN = take(eb);
    cs1 = take((size_t)MAXP * 2 * H * sizeof(float));
    cs2 = take((size_t)MAXP * 2 * H * sizeof(float));
    cs3 = take((size_t)MAXP * 2 * H * sizeof(float));
    scal = take((size_t)(2 + 3 * steps) * 4 * sizeof(float));
  }
};

struct BwdWs : DataGradBufs {
  int64_t N_pad, E_pad;
  int G;
  char* base;
  size_t total;
  float *cta_grads, *gdec, *gs;
  BwdWs(int64_t n, int64_t e, int steps, int g, void* ws) : G(g), base((char*)ws) {
    N_pad = round_up(n, TM);
    E_pad = round_up(e, TM);
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t r = o; o += (size_t)round_up((int64_t)bytes, 256); return (float*)(base + r); };
    cta_grads = take((size_t)G * GRADP * sizeof(float));
    take_data_grads(take, N_pad, E_pad, steps);
    gdec = take((size_t)N_pad * 4 * sizeof(float));
    gs = take(256);  // {S, 1/S} of the fp16 backward (k_grad_scale)
    total = o;
  }
};

// What backward step t of W.T reads: the node_update, edge-step and node_pre arguments, from the forward state W, the
// parameters P, the plan's receiver / sender views and the data-gradient buffers D.  The per-CTA gradient slices and the
// tensor-core operand images are left null: only pdg_backward_inputs has them.
struct BwdStepArgs {
  NodeUpdBwdArgs u;
  EdgeBwdArgs e;
  NodePreBwdArgs n;
};
inline BwdStepArgs bwd_step_args(const FwdWs& W, const float* const* P, const DataGradBufs& D, const int32_t* recv,
                                 const int32_t* send, const int32_t* rowptr, const int32_t* sptr, const int32_t* slist,
                                 int t) {
  const bool last = t == W.T - 1;
  const FwdStepArgs f = fwd_step_args(W, P, recv, send, rowptr, t);  // what forward step t read and wrote
  auto scal = [&](int slot) { return D.scal + slot * 4; };
  BwdStepArgs s = {};
  NodeUpdBwdArgs& u = s.u;
  u.gx = D.gx; u.y3 = f.u.y3_out; u.hq = f.u.hq_out; u.aggraw = f.u.aggraw; u.x_t = f.u.x_t; u.rowptr = rowptr;
  u.scal3 = scal(slot_ln3(t)); u.lnw_n = P[PN_LNW]; u.parts1 = f.u.parts1; u.count1 = f.u.count1;
  u.lnw_e = P[PE_LNW]; u.lnb_e = P[PE_LNB]; u.V1 = P[PN_W0]; u.V2 = P[PN_W2]; u.gagg = D.gagg;
  u.cs1 = D.cs1; u.N = f.u.N; u.n_tiles = f.u.n_tiles;
  EdgeBwdArgs& e = s.e;
  e.e_t = f.e.e_out; e.Pa = f.e.Pa; e.Pb = f.e.Pb; e.gagg = D.gagg; e.ge = D.ge;
  e.y2_t = f.e.y2_out; e.yprev = f.e.yprev; e.parts_prev = f.e.prev_parts; e.count_prev = f.e.prev_count;
  e.recv = recv; e.send = send; e.rowptr = rowptr;
  e.WtE = f.e.WtE; e.b1 = f.e.b1; e.Wt2 = f.e.Wt2; e.b2 = f.e.b2;
  e.W0 = P[PE_W0]; e.W2 = P[PE_W2]; e.lnw = P[PE_LNW];
  e.scal1 = scal(slot_ln1(t)); e.scal2 = last ? nullptr : scal(slot_ln2(t));
  e.DHM = D.DHM; e.DHN = D.DHN; e.RA = D.RA; e.RB = D.RB; e.cs2 = D.cs2;
  e.E = f.e.E; e.n_tiles = f.e.n_tiles; e.last = last ? 1 : 0;
  NodePreBwdArgs& n = s.n;
  n.gx = D.gx; n.RA = D.RA; n.RB = last ? nullptr : D.RB; n.DHM = D.DHM; n.DHN = last ? nullptr : D.DHN;
  n.sptr = sptr; n.slist = slist; n.x_t = f.np.x_out; n.yprev = f.np.yprev;
  n.parts_prev = f.np.prev_parts; n.count_prev = f.np.prev_count; n.W0 = P[PE_W0];
  n.cs3 = D.cs3; n.N = f.u.N; n.n_tiles = f.np.n_tiles;
  return s;
}

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
__device__ __forceinline__ void rmw_add(const float (&acc)[8][8], float* dst, int ld) {
  // dst is this CTA's own gradient slice (one writer): fire-and-forget 128-bit reductions (SASS RED.E.ADD.F32x4) perform the
  // same dst += acc at L2 without the load -> add -> store round trip the thread used to wait for
  const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    float* p = dst + (size_t)(ty * 8 + i) * ld + tx * 4;
    atomicAdd(reinterpret_cast<float4*>(p), make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]));
    atomicAdd(reinterpret_cast<float4*>(p + 64), make_float4(acc[i][4], acc[i][5], acc[i][6], acc[i][7]));
  }
}

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

// ---- kernel bodies of the fp32 backward (pdg_backward.cu, WG = true) and the batched adjoint (pdg_vjp.cu, WG = false) ----
// WG: form the weight gradients as well.  The weight-gradient GEMMs (gemm_colA + rmw_add), the bias sums and the third
// smem tile T2 that only they read exist under WG alone; everything else is one sequence of operations, so the adjoint's
// input gradients have the bits of pdg_backward_inputs.  Shared memory: SMEM_B3T with WG, SMEM_V2T without.

// ---- decoder: g_hd = [hd > 0] (g D2);  gx_T = g_hd D1;  column sums of the LayerNorm that produced x_T's increment ----
//   WG: dD1 = g_hd^T x_T, dD2, d1, d2 into this CTA's gradient slice
template <bool WG>
__device__ __forceinline__ void decoder_bwd_body(const float* __restrict__ g_out, float gscale, const float* __restrict__ hd,
                                                 const float* __restrict__ x_T, const float* __restrict__ y3_last,
                                                 const double* __restrict__ parts_prev, double count_prev,
                                                 const float* __restrict__ D1, const float* __restrict__ D2,
                                                 float* __restrict__ gx, float* __restrict__ cta_grads, float* __restrict__ cs3,
                                                 const int* __restrict__ nzflag, int N, int n_tiles) {
  extern __shared__ __align__(16) float smem[];
  float* T0 = smem;
  float* T1 = T0 + TM * LDS;
  float* T2 = T1 + TM * LDS;
  float* Ws = WG ? T2 + TM * LDS : T2;
  float* gd = Ws + 2 * BKB * H;  // [TM][4] (aliases the index area)
  float* cg = WG ? cta_grads + (size_t)blockIdx.x * GRADP : nullptr;
  const int tid = threadIdx.x, c4 = (tid & 31) * 4;
  if constexpr (WG) pdl_sync();  // the backward launches this kernel with launch_pdl
  const float mu_prev = ln_stat_block(parts_prev, count_prev, gd).mu;
  const bool live = nzflag == nullptr || *nzflag != 0;  // all-zero load case: the output was the constant 0
  float d2w[3][4];
#pragma unroll
  for (int o = 0; o < 3; ++o)
#pragma unroll
    for (int c = 0; c < 4; ++c) d2w[o][c] = D2[o * H + c4 + c];
  float dD2[3] = {0, 0, 0}, dd1 = 0.f, dd2 = 0.f;
  float cgx[8] = {0}, cgy[8] = {0};
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int row0 = tile * TM;
    const int nvalid = min(TM, N - row0);
    if (tid < TM) {
      const int row = row0 + tid;
#pragma unroll
      for (int o = 0; o < 3; ++o) gd[tid * 4 + o] = (row < N && live) ? g_out[row * 3 + o] * gscale : 0.f;
    }
    tile_load(T1, hd + (size_t)row0 * H);
    if constexpr (WG) tile_load(T2, x_T + (size_t)row0 * H);
    __syncthreads();
#pragma unroll 4
    for (int it = 0; it < (TM * H / 4) / NT; ++it) {
      const int r = (tid >> 5) + it * 8;
      const float g0 = gd[r * 4 + 0], g1 = gd[r * 4 + 1], g2 = gd[r * 4 + 2];
      const float4 h = *reinterpret_cast<const float4*>(T1 + r * LDS + c4);
      float4 v;
      v.x = h.x > 0.f ? g0 * d2w[0][0] + g1 * d2w[1][0] + g2 * d2w[2][0] : 0.f;
      v.y = h.y > 0.f ? g0 * d2w[0][1] + g1 * d2w[1][1] + g2 * d2w[2][1] : 0.f;
      v.z = h.z > 0.f ? g0 * d2w[0][2] + g1 * d2w[1][2] + g2 * d2w[2][2] : 0.f;
      v.w = h.w > 0.f ? g0 * d2w[0][3] + g1 * d2w[1][3] + g2 * d2w[2][3] : 0.f;
      *reinterpret_cast<float4*>(T0 + r * LDS + c4) = v;
    }
    float acc[8][8];
    if constexpr (WG) {
      __syncthreads();
      if (tid < H) {
        for (int r = 0; r < nvalid; ++r) {
          const float h = T1[r * LDS + tid];
          dD2[0] = fmaf(gd[r * 4 + 0], h, dD2[0]);
          dD2[1] = fmaf(gd[r * 4 + 1], h, dD2[1]);
          dD2[2] = fmaf(gd[r * 4 + 2], h, dD2[2]);
          dd1 += T0[r * LDS + tid];
        }
      } else if (tid < H + 3) {
        for (int r = 0; r < nvalid; ++r) dd2 += gd[r * 4 + (tid - H)];
      }
      acc_zero(acc);
      gemm_colA(T0, T2, TM, acc);  // dD1[o][k] = sum_r g_hd[r][o] x_T[r][k]
      rmw_add(acc, cg + param_offset(ND_W0), H);
    }
    acc_zero(acc);
    gemm_rowA<BKB>(T0, D1, H, acc, Ws, H);  // gx_T = g_hd D1
    acc_store(acc, gx + (size_t)row0 * H, H);
    float y[8][8];
    mt_load(y, y3_last + (size_t)row0 * H);
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) { cgx[j] += acc[i][j]; cgy[j] = fmaf(acc[i][j], y[i][j] - mu_prev, cgy[j]); }
    __syncthreads();
  }
  if constexpr (WG) {
    if (tid < H) {
#pragma unroll
      for (int o = 0; o < 3; ++o) cg[param_offset(ND_W2) + o * H + tid] += dD2[o];
      cg[param_offset(ND_B0) + tid] += dd1;
    } else if (tid < H + 3) {
      cg[param_offset(ND_B2) + tid - H] += dd2;
    }
  }
  colsum_flush(cgx, T0, cs3 + (size_t)blockIdx.x * 2 * H, false);
  colsum_flush(cgy, T0, cs3 + (size_t)blockIdx.x * 2 * H + H, false);
}

// ---- node_update: dhq = [hq > 0] (dy3 V2);  g_agg = dhq V1[:, :128];  gx += dhq V1[:, 128:] -------------------------
//   WG: dV2 = dy3^T hq, dV1 = dhq^T [message LayerNorm rebuilt from aggraw | x_t], the two biases
template <bool WG>
__device__ __forceinline__ void node_update_bwd_body(NodeUpdBwdArgs a) {
  extern __shared__ __align__(16) float smem[];
  float* T0 = smem;
  float* T1 = T0 + TM * LDS;
  float* T2 = T1 + TM * LDS;
  float* Ws = WG ? T2 + TM * LDS : T2;
  float* smf = Ws + 2 * BKB * H;
  float* cg = WG ? a.cta_grads + (size_t)blockIdx.x * GRADP : nullptr;
  const int tid = threadIdx.x, c4 = (tid & 31) * 4, ty = tid >> 4;
  const LnStat st1 = ln_stat_block(a.parts1, a.count1, smf);
  const float c1 = a.scal3[0], c2 = a.scal3[1], mu3 = a.scal3[2], rstd3 = a.scal3[3];
  const float4 wn = *reinterpret_cast<const float4*>(a.lnw_n + c4);
  float4 we, be;  // message LayerNorm affine (WG: the rebuilt message rows)
  if constexpr (WG) {
    we = *reinterpret_cast<const float4*>(a.lnw_e + c4);
    be = *reinterpret_cast<const float4*>(a.lnb_e + c4);
  }
  float dc2 = 0.f, dc1 = 0.f;
  float cg1[8] = {0}, cgy1[8] = {0};
  for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const int row0 = tile * TM;
    const int nvalid = min(TM, a.N - row0);
    // dy3 -> T0 ; hq -> T1
    // row loads in two batches of eight (all loads of a batch in flight before the first use)
#pragma unroll
    for (int bt = 0; bt < 2; ++bt) {
      float4 lg[8], ly[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int r = (tid >> 5) + (bt * 8 + k) * 8;
        const size_t g = ((size_t)row0 + r) * H + c4;
        lg[k] = make_float4(0.f, 0.f, 0.f, 0.f);
        ly[k] = lg[k];
        if (r < nvalid) {
          lg[k] = *reinterpret_cast<const float4*>(a.gx + g);
          ly[k] = *reinterpret_cast<const float4*>(a.y3 + g);
        }
      }
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int r = (tid >> 5) + (bt * 8 + k) * 8;
        const float4 gg = lg[k], y = ly[k];
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (r < nvalid) {
          v.x = y.x > 0.f ? rstd3 * gg.x * wn.x - c1 - c2 * (y.x - mu3) : 0.f;
          v.y = y.y > 0.f ? rstd3 * gg.y * wn.y - c1 - c2 * (y.y - mu3) : 0.f;
          v.z = y.z > 0.f ? rstd3 * gg.z * wn.z - c1 - c2 * (y.z - mu3) : 0.f;
          v.w = y.w > 0.f ? rstd3 * gg.w * wn.w - c1 - c2 * (y.w - mu3) : 0.f;
        }
        *reinterpret_cast<float4*>(T0 + r * LDS + c4) = v;
      }
    }
    tile_load(T1, a.hq + (size_t)row0 * H);
    float acc[8][8];
    if constexpr (WG) {
      __syncthreads();
      dc2 += tile_colsum(T0, nvalid);
      acc_zero(acc);
      gemm_colA(T0, T1, TM, acc);  // dV2[o][i] = sum_r dy3[r][o] hq[r][i]
      rmw_add(acc, cg + param_offset(PN_W2), H);
    }
    acc_zero(acc);
    gemm_rowA<BKB>(T0, a.V2, H, acc, Ws, H);  // dhq_pre = dy3 V2 (without WG, its first barrier publishes T0 / T1)
    {
      float h[8][8];
      acc_load(h, T1, LDS);
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = h[i][j] > 0.f ? acc[i][j] : 0.f;
    }
    acc_store(acc, T0, LDS);  // dhq
    if constexpr (WG) {
      __syncthreads();  // everyone is done with hq in T1
#pragma unroll
      for (int it = 0; it < (TM * H / 4) / NT; ++it) {  // x_t rows straight into T2 (asynchronous, no registers)
        const int r = (tid >> 5) + it * 8;
        cp_async16(T2 + r * LDS + c4, a.x_t + ((size_t)row0 + r) * H + c4);
      }
      cp_async_commit();
#pragma unroll
      for (int bt = 0; bt < 2; ++bt) {
        float4 ls[8];
        float ldeg[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const int r = (tid >> 5) + (bt * 8 + k) * 8;
          const int row = row0 + r;
          ldeg[k] = row < a.N ? (float)(a.rowptr[row + 1] - a.rowptr[row]) : 0.f;
          ls[k] = *reinterpret_cast<const float4*>(a.aggraw + (size_t)row * H + c4);
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const int r = (tid >> 5) + (bt * 8 + k) * 8;
          const float deg = ldeg[k];
          const float4 s4 = ls[k];
          const float dm = deg * st1.mu;
          float4 v;
          v.x = (s4.x - dm) * st1.rstd * we.x + deg * be.x;
          v.y = (s4.y - dm) * st1.rstd * we.y + deg * be.y;
          v.z = (s4.z - dm) * st1.rstd * we.z + deg * be.z;
          v.w = (s4.w - dm) * st1.rstd * we.w + deg * be.w;
          *reinterpret_cast<float4*>(T1 + r * LDS + c4) = v;
        }
      }
      cp_async_wait<0>();
      __syncthreads();
      dc1 += tile_colsum(T0, nvalid);
      acc_zero(acc);
      gemm_colA(T0, T1, TM, acc);  // dV1[:, :128]
      rmw_add(acc, cg + param_offset(PN_W0), 2 * H);
      acc_zero(acc);
      gemm_colA(T0, T2, TM, acc);  // dV1[:, 128:]
      rmw_add(acc, cg + param_offset(PN_W0) + H, 2 * H);
    }
    acc_zero(acc);
    gemm_rowA<BKB>(T0, a.V1, H, acc, Ws, 2 * H);  // g_agg = dhq V1[:, :128]
    acc_store(acc, a.gagg + (size_t)row0 * H, H);
    {
      float s[8][8];
      mt_load(s, a.aggraw + (size_t)row0 * H);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int row = row0 + ty * 8 + i;
        const float deg = row < a.N ? (float)(a.rowptr[row + 1] - a.rowptr[row]) : 0.f;
#pragma unroll
        for (int j = 0; j < 8; ++j) { cg1[j] = fmaf(deg, acc[i][j], cg1[j]); cgy1[j] = fmaf(acc[i][j], s[i][j] - deg * st1.mu, cgy1[j]); }
      }
    }
    acc_zero(acc);
    gemm_rowA<BKB>(T0, a.V1 + H, H, acc, Ws, 2 * H);  // direct path: dhq V1[:, 128:]
    {
      float g0[8][8];
      mt_load(g0, a.gx + (size_t)row0 * H);
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] += g0[i][j];
    }
    acc_store(acc, a.gx + (size_t)row0 * H, H);
    __syncthreads();
  }
  if constexpr (WG) {
    if (tid < H) {
      cg[param_offset(PN_B2) + tid] += dc2;
      cg[param_offset(PN_B0) + tid] += dc1;
    }
  }
  colsum_flush(cg1, T0, a.cs1 + (size_t)blockIdx.x * 2 * H, false);
  colsum_flush(cgy1, T0, a.cs1 + (size_t)blockIdx.x * 2 * H + H, false);
}

// ---- node_pre: dPa = RA + sum_{send = n} dhn, dPb = RB + sum_{send = n} dhm;  gx += dPa Wa + dPb Wb -------------------
//   WG: dWa = dPa^T x_t, dWb = dPb^T x_t
template <bool WG>
__device__ __forceinline__ void node_pre_bwd_body(NodePreBwdArgs a) {
  extern __shared__ __align__(16) float smem[];
  float* T0 = smem;
  float* T1 = T0 + TM * LDS;
  float* T2 = T1 + TM * LDS;
  float* Ws = WG ? T2 + TM * LDS : T2;
  float* cg = WG ? a.cta_grads + (size_t)blockIdx.x * GRADP : nullptr;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float mu_prev = ln_stat_block(a.parts_prev, a.count_prev, Ws).mu;
  float cgx[8] = {0}, cgy[8] = {0};
  for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const int row0 = tile * TM;
    // dPa = RA + sum_{send = n} dhn ; dPb = RB + sum_{send = n} dhm     (warp per row, lane per float4)
    // The tile's sender lists are ONE contiguous range of send_list: staged in shared memory first (Ws is idle until the
    // GEMMs), so the row loads below carry no dependent index loads.
    int* s_ptr = reinterpret_cast<int*>(Ws);  // [TM + 1]
    int* s_list = s_ptr + TM + 4;             // [SLC]
    constexpr int SLC = 2 * BKB * H - (TM + 4);
    if (tid <= TM) s_ptr[tid] = a.sptr[min(row0 + tid, a.N)];
    __syncthreads();
    const int k_lo = s_ptr[0], k_cnt = s_ptr[TM] - s_ptr[0];
    const bool staged = k_cnt <= SLC;
    if (staged)
      for (int i = tid; i < k_cnt; i += NT) s_list[i] = a.slist[k_lo + i];
    __syncthreads();
    for (int rr = 0; rr < TM / 8; ++rr) {
      const int r = warp * (TM / 8) + rr;
      const int n = row0 + r;
      float4 pa = make_float4(0.f, 0.f, 0.f, 0.f), pb = pa;
      if (n < a.N) {
        pa = *reinterpret_cast<const float4*>(a.RA + (size_t)n * H + lane * 4);
        if (a.RB) pb = *reinterpret_cast<const float4*>(a.RB + (size_t)n * H + lane * 4);
        const int k0 = s_ptr[r], k1 = s_ptr[r + 1];
        // sender rows in batches of GB (a mesh node sends to 6-7 edges: one batch per row): every row load of the batch in
        // flight, then the adds in list order (same summation order as one row at a time => same bits)
        constexpr int GB = 8;
        for (int k = k0; k < k1; k += GB) {
          int id[GB];
          float4 m[GB], q[GB];
#pragma unroll
          for (int j = 0; j < GB; ++j) id[j] = k + j < k1 ? (staged ? s_list[k + j - k_lo] : a.slist[k + j]) : -1;
#pragma unroll
          for (int j = 0; j < GB; ++j) {
            m[j] = make_float4(0.f, 0.f, 0.f, 0.f);
            q[j] = m[j];
            if (id[j] >= 0) {
              const size_t p = (size_t)id[j] * H + lane * 4;
              m[j] = __ldcs(reinterpret_cast<const float4*>(a.DHM + p));
              if (a.DHN) q[j] = __ldcs(reinterpret_cast<const float4*>(a.DHN + p));
            }
          }
#pragma unroll
          for (int j = 0; j < GB; ++j)
            if (id[j] >= 0) {
              pb.x += m[j].x; pb.y += m[j].y; pb.z += m[j].z; pb.w += m[j].w;
              pa.x += q[j].x; pa.y += q[j].y; pa.z += q[j].z; pa.w += q[j].w;
            }
        }
      }
      *reinterpret_cast<float4*>(T0 + r * LDS + lane * 4) = pa;
      *reinterpret_cast<float4*>(T1 + r * LDS + lane * 4) = pb;
    }
    // RA / RB rows of this warp re-zeroed for the next step's segment sums -- in a pass of their own: stores between the
    // gather loads serialise them (measured on the tensor-core kernel, DESIGN section 4b)
    for (int rr = 0; rr < TM / 8; ++rr) {
      const int n = row0 + warp * (TM / 8) + rr;
      if (n < a.N) {
        *reinterpret_cast<float4*>(a.RA + (size_t)n * H + lane * 4) = make_float4(0.f, 0.f, 0.f, 0.f);
        if (a.RB) *reinterpret_cast<float4*>(a.RB + (size_t)n * H + lane * 4) = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
    if constexpr (WG) tile_load(T2, a.x_t + (size_t)row0 * H);
    __syncthreads();  // also: every read of the staged lists in Ws is done before the GEMMs stream weights into it
    float acc[8][8];
    if constexpr (WG) {
      acc_zero(acc);
      gemm_colA(T0, T2, TM, acc);  // dWa[o][k] = sum_r dPa[r][o] x_t[r][k]
      rmw_add(acc, cg + param_offset(PE_W0), 3 * H);
      acc_zero(acc);
      gemm_colA(T1, T2, TM, acc);
      rmw_add(acc, cg + param_offset(PE_W0) + H, 3 * H);
    }
    acc_zero(acc);
    gemm_rowA<BKB>(T0, a.W0, H, acc, Ws, 3 * H);      // dPa Wa
    gemm_rowA<BKB>(T1, a.W0 + H, H, acc, Ws, 3 * H);  // + dPb Wb
    {
      float g0[8][8];
      mt_load(g0, a.gx + (size_t)row0 * H);
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] += g0[i][j];
    }
    acc_store(acc, a.gx + (size_t)row0 * H, H);
    {
      float y[8][8];
      mt_load(y, a.yprev + (size_t)row0 * H);
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) { cgx[j] += acc[i][j]; cgy[j] = fmaf(acc[i][j], y[i][j] - mu_prev, cgy[j]); }
    }
    __syncthreads();
  }
  colsum_flush(cgx, T0, a.cs3 + (size_t)blockIdx.x * 2 * H, false);
  colsum_flush(cgy, T0, a.cs3 + (size_t)blockIdx.x * 2 * H + H, false);
}

// ---- encoders (node: NODE=1, edge: NODE=0): dh0 = [h0 > 0] (dy W2) ----------------------------------------------------
//   WG: dW2 = dy^T h0, dW0 = dh0^T feat, the two biases (the dW0 / db0 walk takes warps 0-3)
//   IG: also write the input gradient dfeat = dh0 W0 of every row, un-standardised (models.py:140-162), one warp per row
//       (warps 4-7 with WG, all eight without):
//   node  gi0 = d/d mean_stress [N,3] (features 0-2), gi1 = d/d pos [N,2] (features 3-4), either may be null;
//   edge  gi0 = d/d edge_attr [E] at perm[row] (PyG edge order; perm is a permutation: plain stores).
template <int NODE, bool WG, bool IG>
__device__ __forceinline__ void encoder_bwd_body(const float* __restrict__ g_in, const float* __restrict__ y_raw,
                                                 const float* __restrict__ scal, const float* __restrict__ lnw,
                                                 const float* __restrict__ mean_stress, const float* __restrict__ pos,
                                                 const int64_t* __restrict__ types, const float* __restrict__ edge_attr,
                                                 const int32_t* __restrict__ perm, const pdg_norm_t& nrm, int scale_in,
                                                 const float* __restrict__ W0, const float* __restrict__ b0,
                                                 const float* __restrict__ W2, float* __restrict__ cta_grads, int off_w0,
                                                 int off_b0, int off_w2, int off_b2, int R, int n_tiles,
                                                 float* __restrict__ gi0, float* __restrict__ gi1) {
  extern __shared__ __align__(16) float smem[];
  float* T0 = smem;
  float* T1 = T0 + TM * LDS;
  float* T2 = T1 + TM * LDS;
  float* Ws = WG ? T2 + TM * LDS : T2;
  float* feat = WG ? T2 : Ws + 2 * BKB * H;  // [TM][8]
  float* cg = WG ? cta_grads + (size_t)blockIdx.x * GRADP : nullptr;
  const int tid = threadIdx.x, c4 = (tid & 31) * 4;
  constexpr int NF = NODE ? 6 : 1;
  if constexpr (WG) pdl_sync();  // the backward launches this kernel with launch_pdl
  const float c1 = scal[0], c2 = scal[1], mu = scal[2], rstd = scal[3];
  const float4 w = *reinterpret_cast<const float4*>(lnw + c4);
  float w0[4][NF], bb0[4];
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    bb0[c] = b0[c4 + c];
#pragma unroll
    for (int j = 0; j < NF; ++j) w0[c][j] = W0[(c4 + c) * NF + j];
  }
  float db2 = 0.f, db0 = 0.f, dW0[NF];
#pragma unroll
  for (int j = 0; j < NF; ++j) dW0[j] = 0.f;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int row0 = tile * TM;
    const int nvalid = min(TM, R - row0);
    if (tid < TM) {
      const int row = row0 + tid;
      float f[8] = {0, 0, 0, 0, 0, 0, 0, 0};
      if (row < R) {
        if (NODE) {
          bool nz;
          node_features(mean_stress, pos, types, nrm, scale_in, row, f, nz);
        } else {
          f[0] = edge_feature(edge_attr[perm[row]], nrm, scale_in);
        }
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) feat[tid * 8 + j] = f[j];
    }
    __syncthreads();
#pragma unroll 4
    for (int it = 0; it < (TM * H / 4) / NT; ++it) {
      const int r = (tid >> 5) + it * 8;
      const size_t g = ((size_t)row0 + r) * H + c4;
      float4 d = make_float4(0.f, 0.f, 0.f, 0.f);
      if (r < nvalid) {
        const float4 gg = *reinterpret_cast<const float4*>(g_in + g);
        const float4 y = *reinterpret_cast<const float4*>(y_raw + g);
        d.x = y.x > 0.f ? rstd * gg.x * w.x - c1 - c2 * (y.x - mu) : 0.f;
        d.y = y.y > 0.f ? rstd * gg.y * w.y - c1 - c2 * (y.y - mu) : 0.f;
        d.z = y.z > 0.f ? rstd * gg.z * w.z - c1 - c2 * (y.z - mu) : 0.f;
        d.w = y.w > 0.f ? rstd * gg.w * w.w - c1 - c2 * (y.w - mu) : 0.f;
      }
      *reinterpret_cast<float4*>(T0 + r * LDS + c4) = d;
      float hv[4];
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        float s = bb0[c];
#pragma unroll
        for (int j = 0; j < NF; ++j) s = fmaf(w0[c][j], feat[r * 8 + j], s);
        hv[c] = fmaxf(s, 0.f);
      }
      *reinterpret_cast<float4*>(T1 + r * LDS + c4) = make_float4(hv[0], hv[1], hv[2], hv[3]);
    }
    float acc[8][8];
    if constexpr (WG) {
      __syncthreads();
      db2 += tile_colsum(T0, nvalid);
      acc_zero(acc);
      gemm_colA(T0, T1, TM, acc);  // dW2[o][i] = sum_r dy[r][o] h0[r][i]
      rmw_add(acc, cg + off_w2, H);
    }
    acc_zero(acc);
    gemm_rowA<BKB>(T0, W2, H, acc, Ws, H);  // dh0_pre = dy W2 (without WG, its first barrier publishes T0 / T1)
    {
      float h[8][8];
      acc_load(h, T1, LDS);
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = h[i][j] > 0.f ? acc[i][j] : 0.f;
    }
    acc_store(acc, T0, LDS);  // dh0
    __syncthreads();
    if (WG && tid < H) {
      for (int r = 0; r < nvalid; ++r) {
        const float d = T0[r * LDS + tid];
        db0 += d;
#pragma unroll
        for (int j = 0; j < NF; ++j) dW0[j] = fmaf(d, feat[r * 8 + j], dW0[j]);
      }
    } else if (IG) {  // dfeat[r] = dh0[r] W0, one warp per row, lane = 4 channels
      constexpr int FW = WG ? H / 32 : 0;  // first warp of this walk: the warps the dW0 walk leaves idle
      constexpr int NI = NODE ? 5 : 1;     // feature 5 (nodes_types) is an integer input: no gradient
      for (int r = (tid - FW * 32) >> 5; r < nvalid; r += (NT - FW * 32) / 32) {
        const float4 d = *reinterpret_cast<const float4*>(T0 + r * LDS + c4);
        float s[NI];
#pragma unroll
        for (int j = 0; j < NI; ++j) {
          s[j] = fmaf(d.w, w0[3][j], fmaf(d.z, w0[2][j], fmaf(d.y, w0[1][j], d.x * w0[0][j])));
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) s[j] += __shfl_xor_sync(0xffffffffu, s[j], o);
        }
        if ((tid & 31) == 0) {
          const int row = row0 + r;
          if (NODE) {
            const float sm = scale_in ? nrm.std_mean_stress : 1.f, sp = scale_in ? nrm.std_pos : 1.f;
            if (gi0 != nullptr) {
              gi0[row * 3 + 0] = s[0] / sm; gi0[row * 3 + 1] = s[1 % NI] / sm; gi0[row * 3 + 2] = s[2 % NI] / sm;
            }
            if (gi1 != nullptr) { gi1[row * 2 + 0] = s[3 % NI] / sp; gi1[row * 2 + 1] = s[4 % NI] / sp; }
          } else {
            gi0[perm[row]] = s[0] / (scale_in ? nrm.std_edge_weight : 1.f);
          }
        }
      }
    }
    __syncthreads();
  }
  if constexpr (WG) {
    if (tid < H) {
      cg[off_b2 + tid] += db2;
      cg[off_b0 + tid] += db0;
#pragma unroll
      for (int j = 0; j < NF; ++j) cg[off_w0 + tid * NF + j] += dW0[j];
    }
  }
}

}  // namespace pdg
