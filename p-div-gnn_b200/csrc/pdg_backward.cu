// Backward pass of EncodeProcessDecode (autograd through reference models.py:288-326).
//
// Recompute-based: the forward (PDG_FLAG_SAVE) keeps only x_t, e_t, the raw LayerNorm
// inputs (y3_t, y2_t, encoder outputs), the raw receiver sums, the node-MLP hidden and
// Pa/Pb; the per-edge hidden activations and messages are rebuilt tile by tile.
//
// Graph-mode LayerNorm backward needs two global scalars per LN instance
//   S1 = sum(g*w),  S2 = sum(g*w*(y-mu));  dy = a*g*w - a*S1/M - a^2*S2*(y-mu)/(M*sigma)
// both follow from per-channel column sums  cg = colsum(g), cgy = colsum(g*(y-mu))  which the
// kernel that PRODUCES g accumulates in its epilogue; a one-block finalize kernel turns
// them into {c1, c2, mu, a} and the LN affine gradients.  For the message LayerNorm the
// column sums come from node-level data only (g is constant over a receiver segment):
//   cg = sum_n deg_n * g_agg[n],  cgy = sum_n g_agg[n] * (aggraw[n] - deg_n*mu).
//
// Weight gradients: each CTA accumulates into its own slice of cta_grads[G][GRADP]
// (no atomics); one final kernel sums the slices in fixed order => deterministic.
// Scatter of d(Pa), d(Pb) to SENDER nodes is a gather over the sender CSR of the plan.
#include <cuda_bf16.h>
#include <stdlib.h>

#include "pdg_bwd.cuh"
#include "pdg_tc_tile.cuh"

namespace pdg {

// ---- LayerNorm-backward finalize (pdg_bwd.cuh) ---------------------------------------------------
__global__ void __launch_bounds__(FIN_G* H)
k_ln_finalize(const float* __restrict__ cs, int nparts, const double* __restrict__ fwd_parts, double count,
              const float* __restrict__ lnw, float* __restrict__ scal_out, float* __restrict__ flat_w,
              float* __restrict__ flat_b) {
  ln_finalize_body(cs, nparts, fwd_parts, count, lnw, scal_out, flat_w, flat_b);
}
// two independent LayerNorm instances in one launch (block 0 / block 1): saves a kernel boundary wherever two
// finalizes are adjacent in the chain.  Their flat_w / flat_b targets must be different arrays.
__global__ void __launch_bounds__(FIN_G* H)
k_ln_finalize2(LnFinArgs a0, LnFinArgs a1) {
  const LnFinArgs& a = blockIdx.x == 0 ? a0 : a1;
  ln_finalize_body(a.cs, a.nparts, a.fwd_parts, a.count, a.lnw, a.scal_out, a.flat_w, a.flat_b);
}

// ---- decoder backward, node_update backward (B3): bodies in pdg_bwd.cuh ------------------------------------------------
__global__ void __launch_bounds__(NT, 1)
k_decoder_bwd(const float* __restrict__ g_out, float gscale, const float* __restrict__ hd, const float* __restrict__ x_T,
              const float* __restrict__ y3_last, const double* __restrict__ parts_prev, double count_prev,
              const float* __restrict__ D1, const float* __restrict__ D2, float* __restrict__ gx,
              float* __restrict__ cta_grads, float* __restrict__ cs3, const int* __restrict__ nzflag, int N, int n_tiles) {
  decoder_bwd_body<true>(g_out, gscale, hd, x_T, y3_last, parts_prev, count_prev, D1, D2, gx, cta_grads, cs3, nzflag, N, n_tiles);
}
__global__ void __launch_bounds__(NT, 1) k_node_update_bwd(NodeUpdBwdArgs a) { node_update_bwd_body<true>(a); }

// ---- B2: edge step backward -----------------------------------------------------------------
__global__ void __launch_bounds__(NT, 1) k_edge_step_bwd(EdgeBwdArgs a) {
  extern __shared__ __align__(16) float smem[];
  float* T0 = smem;
  float* T1 = T0 + TM * LDS;
  float* T2 = T1 + TM * LDS;
  float* Ws = T2 + TM * LDS;
  int* recv_s = (int*)(Ws + 2 * BKB * H);
  int* send_s = recv_s + TM;
  int* smi = send_s + TM;
  unsigned* seg_masks = reinterpret_cast<unsigned*>(smi + 8);
  unsigned char* seg_row = reinterpret_cast<unsigned char*>(seg_masks + 4);  // [TM + 1]
  float seg_dummy = 0.f;
  float* cg = a.cta_grads + (size_t)blockIdx.x * GRADP;
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  const float mu_prev = ln_stat_block(a.parts_prev, a.count_prev, (float*)smi).mu;
  const float c1m = a.scal1[0], c2m = a.scal1[1], mu1 = a.scal1[2], rstd1 = a.scal1[3];
  float c1n = 0.f, c2n = 0.f, mu2 = 0.f, rstd2 = 0.f;
  if (!a.last) { c1n = a.scal2[0]; c2n = a.scal2[1]; mu2 = a.scal2[2]; rstd2 = a.scal2[3]; }
  float bias1[8], bias2[8], lw[8];
  load_cols(bias1, a.b1);
  load_cols(bias2, a.b2);
  load_cols(lw, a.lnw);
  float db2[8] = {0}, db1[8] = {0}, cge[8] = {0}, cgye[8] = {0};
  for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const int row0 = tile * TM;
    const int nvalid = min(TM, a.E - row0);
    if (tid < TM) {
      recv_s[tid] = a.recv[row0 + tid];
      send_s[tid] = a.send[row0 + tid];
    }
    if (tid == 0) {
      // rows this tile reads ~50-100 us from now (dy2, ge read-modify-write, LayerNorm column sums) and the next tile's
      // e_t rows: pulled into L2 by the copy engine so that the register loads later pay L2, not DRAM, latency
      constexpr uint32_t TB = TM * H * sizeof(float);
      if (!a.last) {
        tc::bulk_prefetch_l2(a.y2_t + (size_t)row0 * H, TB);
        tc::bulk_prefetch_l2(a.ge + (size_t)row0 * H, TB);
      }
      tc::bulk_prefetch_l2(a.yprev + (size_t)row0 * H, TB);
      if (tile + (int)gridDim.x < a.n_tiles) tc::bulk_prefetch_l2(a.e_t + ((size_t)row0 + (size_t)gridDim.x * TM) * H, TB);
    }
    tile_load(T0, a.e_t + (size_t)row0 * H);
    __syncthreads();
    const int nseg = tile_segments(recv_s, nvalid, seg_row, seg_masks);
    float acc[8][8];
    // G = e_t We^T + b1 ; hidden activations of both edge-MLP evaluations
    acc_zero(acc);
    gemm_rowA<BKB>(T0, a.WtE, H, acc, Ws, H);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int r = ty * 8 + i;
      const float* par = a.Pa + (size_t)recv_s[r] * H + tx * 4;
      const float* pbs = a.Pb + (size_t)send_s[r] * H + tx * 4;
      const float* pas = a.Pa + (size_t)send_s[r] * H + tx * 4;
      const float* pbr = a.Pb + (size_t)recv_s[r] * H + tx * 4;
      const float4 ar0 = __ldg((const float4*)par), ar1 = __ldg((const float4*)(par + 64));
      const float4 bs0 = __ldg((const float4*)pbs), bs1 = __ldg((const float4*)(pbs + 64));
      const float4 as0 = __ldg((const float4*)pas), as1 = __ldg((const float4*)(pas + 64));
      const float4 br0 = __ldg((const float4*)pbr), br1 = __ldg((const float4*)(pbr + 64));
      const float par_[8] = {ar0.x, ar0.y, ar0.z, ar0.w, ar1.x, ar1.y, ar1.z, ar1.w};
      const float pbs_[8] = {bs0.x, bs0.y, bs0.z, bs0.w, bs1.x, bs1.y, bs1.z, bs1.w};
      const float pas_[8] = {as0.x, as0.y, as0.z, as0.w, as1.x, as1.y, as1.z, as1.w};
      const float pbr_[8] = {br0.x, br0.y, br0.z, br0.w, br1.x, br1.y, br1.z, br1.w};
      float hm[8], hn[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float g = acc[i][j] + bias1[j];
        // same association as the forward: (G + Pa) + Pb
        hm[j] = fmaxf(g + par_[j] + pbs_[j], 0.f);
        hn[j] = fmaxf(g + pas_[j] + pbr_[j], 0.f);
      }
      float* p1 = T1 + r * LDS + tx * 4;
      float* p2 = T2 + r * LDS + tx * 4;
      *reinterpret_cast<float4*>(p1) = make_float4(hm[0], hm[1], hm[2], hm[3]);
      *reinterpret_cast<float4*>(p1 + 64) = make_float4(hm[4], hm[5], hm[6], hm[7]);
      *reinterpret_cast<float4*>(p2) = make_float4(hn[0], hn[1], hn[2], hn[3]);
      *reinterpret_cast<float4*>(p2 + 64) = make_float4(hn[4], hn[5], hn[6], hn[7]);
    }
    // ---- message path: y1 (recomputed) -> dy1 -> T0 ----
    acc_zero(acc);
    gemm_rowA<BKB>(T1, a.Wt2, H, acc, Ws, H);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int r = ty * 8 + i;
      const bool ok = r < nvalid;
      const float* gp = a.gagg + (size_t)recv_s[r] * H + tx * 4;
      const float4 g0 = __ldg((const float4*)gp), g1 = __ldg((const float4*)(gp + 64));
      const float gv[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float y = fmaxf(acc[i][j] + bias2[j], 0.f);
        const float d = (ok && y > 0.f) ? rstd1 * gv[j] * lw[j] - c1m - c2m * (y - mu1) : 0.f;
        acc[i][j] = d;
        db2[j] += d;
      }
    }
    acc_store(acc, T0, LDS);
    __syncthreads();
    acc_zero(acc);
    gemm_colA(T0, T1, TM, acc);  // dW2[o][i] += sum_r dy1[r][o] hm[r][i]
    rmw_add(acc, cg + param_offset(PE_W2), H);
    acc_zero(acc);
    gemm_rowA<BKB>(T0, a.W2, H, acc, Ws, H);  // dhm_pre = dy1 W2
    {
      float h[8][8];
      acc_load(h, T1, LDS);
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = h[i][j] > 0.f ? acc[i][j] : 0.f;
    }
    acc_store(acc, a.DHM + (size_t)row0 * H, H);
    acc_store(acc, T1, LDS);  // dhm (own positions only)
    __syncthreads();
    tile_segsum_warp<false>(T1, recv_s, seg_row, nseg, a.rowptr, row0, nvalid, a.RA, seg_dummy, seg_dummy);
    // ---- edge-update path ----
    if (!a.last) {
      {
        float y[8][8], g[8][8];
        mt_load(y, a.y2_t + (size_t)row0 * H);
        mt_load(g, a.ge + (size_t)row0 * H);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const bool ok = ty * 8 + i < nvalid;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float d = (ok && y[i][j] > 0.f) ? rstd2 * g[i][j] * lw[j] - c1n - c2n * (y[i][j] - mu2) : 0.f;
            acc[i][j] = d;
            db2[j] += d;
          }
        }
      }
      acc_store(acc, T0, LDS);  // dy2 (T0 last read by the dhm GEMM, which ended with a barrier)
      __syncthreads();
      acc_zero(acc);
      gemm_colA(T0, T2, TM, acc);  // dW2 += dy2^T hn
      rmw_add(acc, cg + param_offset(PE_W2), H);
      acc_zero(acc);
      gemm_rowA<BKB>(T0, a.W2, H, acc, Ws, H);
      {
        float h[8][8];
        acc_load(h, T2, LDS);
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[i][j] = h[i][j] > 0.f ? acc[i][j] : 0.f;
      }
      acc_store(acc, a.DHN + (size_t)row0 * H, H);
      acc_store(acc, T2, LDS);  // dhn
      __syncthreads();
      tile_segsum_warp<false>(T2, recv_s, seg_row, nseg, a.rowptr, row0, nvalid, a.RB, seg_dummy, seg_dummy);
      // dG = dhm + dhn -> T1 (own positions)
      {
        float m[8][8];
        acc_load(m, T1, LDS);
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[i][j] += m[i][j];
      }
      __syncthreads();  // segment sums over T1/T2 finished before T1 changes
      acc_store(acc, T1, LDS);
    } else {
      acc_load(acc, T1, LDS);
    }
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) db1[j] += acc[i][j];
    // de_t = ge_{t+1} + dG We ;  column sums for the LayerNorm that produced e_t's increment
    acc_zero(acc);
    gemm_rowA<BKB>(T1, a.W0 + 2 * H, H, acc, Ws, 3 * H);
    if (!a.last) {
      float g[8][8];
      mt_load(g, a.ge + (size_t)row0 * H);
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] += g[i][j];
    }
    acc_store(acc, a.ge + (size_t)row0 * H, H);
    {
      float y[8][8];
      mt_load(y, a.yprev + (size_t)row0 * H);
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) { cge[j] += acc[i][j]; cgye[j] = fmaf(acc[i][j], y[i][j] - mu_prev, cgye[j]); }
    }
    // dWe[o][k] += sum_r dG[r][o] e_t[r][k]
    tile_load(T0, a.e_t + (size_t)row0 * H);
    __syncthreads();
    acc_zero(acc);
    gemm_colA(T1, T0, TM, acc);
    rmw_add(acc, cg + param_offset(PE_W0) + 2 * H, 3 * H);
    __syncthreads();
  }
  colsum_flush(db2, T0, cg + param_offset(PE_B2), true);
  colsum_flush(db1, T0, cg + param_offset(PE_B0), true);
  colsum_flush(cge, T0, a.cs2 + (size_t)blockIdx.x * 2 * H, false);
  colsum_flush(cgye, T0, a.cs2 + (size_t)blockIdx.x * 2 * H + H, false);
}

// ---- node_pre backward (B1), encoder backward (node: NODE=1, edge: NODE=0): bodies in pdg_bwd.cuh ------------------------
// IG: also write the input gradients (d/d mean_stress and d/d pos, or d/d edge_attr).  The <NODE, false> instances are the
// parameter-gradient-only kernels.
__global__ void __launch_bounds__(NT, 1) k_node_pre_bwd(NodePreBwdArgs a) { node_pre_bwd_body<true>(a); }

template <int NODE, bool IG>
__global__ void __launch_bounds__(NT, 1)
k_encoder_bwd(const float* __restrict__ g_in, const float* __restrict__ y_raw, const float* __restrict__ scal,
              const float* __restrict__ lnw, const float* __restrict__ mean_stress, const float* __restrict__ pos,
              const int64_t* __restrict__ types, const float* __restrict__ edge_attr, const int32_t* __restrict__ perm,
              pdg_norm_t nrm, int scale_in, const float* __restrict__ W0, const float* __restrict__ b0,
              const float* __restrict__ W2, float* __restrict__ cta_grads, int off_w0, int off_b0, int off_w2,
              int off_b2, int R, int n_tiles, float* __restrict__ gi0, float* __restrict__ gi1) {
  encoder_bwd_body<NODE, true, IG>(g_in, y_raw, scal, lnw, mean_stress, pos, types, edge_attr, perm, nrm, scale_in, W0, b0, W2,
                                   cta_grads, off_w0, off_b0, off_w2, off_b2, R, n_tiles, gi0, gi1);
}

// ---- final reduction over the per-CTA gradient slices ------------------------------------------
// gs != nullptr: the backward ran on gradients scaled by S = gs[0] (k_grad_scale); gs[1] = 1/S (a power of two: exact)
// blocked != 0 (tensor-core path): the [128][128 nb] weight gradients that leave TMEM through whole-block TMA reduce-adds
// sit in the slices in the staging order (grad_block_offset, pdg_tc_tile.cuh): column block b = columns [128 b, 128 b + 128)
// at block b of the parameter's region, float4 chunks XOR-swizzled by the row.  Flat element i is read from there.
__device__ __forceinline__ int grad_slice_index(int i) {
  constexpr int NB = 7;
  constexpr int pid[NB] = {PE_W0, PE_W2, PN_W0, PN_W2, EE_W2, NE_W2, ND_W0};
  constexpr int nblk[NB] = {3, 1, 2, 1, 1, 1, 1};
#pragma unroll
  for (int k = 0; k < NB; ++k) {
    const int off = param_offset(pid[k]), rel = i - off;
    if (rel >= 0 && rel < H * H * nblk[k]) {
      const int w = H * nblk[k], r = rel / w, cf = rel - r * w;
      return off + (cf >> 7) * (H * H) + grad_block_offset(r, cf & (H - 1));
    }
  }
  return i;
}
__global__ void k_grad_reduce(const float* __restrict__ cta_grads, int G, float* __restrict__ flat, const float* __restrict__ gs,
                              int blocked) {
  pdl_sync();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < PDG_PARAM_ELEMS) {
    const int j = blocked ? grad_slice_index(i) : i;
    float s = flat[i];
    for (int g = 0; g < G; ++g) s += cta_grads[(size_t)g * GRADP + j];
    flat[i] = gs != nullptr ? s * gs[1] : s;
  }
}

// Power-of-two gradient scale of the fp16 tensor-core backward (the GradScaler of gnn_train.py:111,204-207 moved inside
// the operator and decided on the device).  The decoder backward builds its first fp16 tile from g * gscale * S, where
// gscale is the output de-standardisation factor (std_local_stress with PDG_FLAG_SCALE_OUTPUT, else 1), so S is chosen
// from that product: gs[0] = S = 2^(8 - e) with max|g| * |gscale| in [2^(e-1), 2^e), gs[1] = 1/S.  Every gradient-valued
// fp16 tile / row of the backward then sits around 2^8 x (its size relative to d loss / d(standardised output)),
// whatever std_local_stress is: measured along the chain the tiles span 1e-5 .. 4 of that maximum, i.e. 2.5e-3 .. 1e3
// after scaling -- inside fp16's normal range [6.1e-5, 65504] with 2^6 of headroom (conversions saturate, nothing
// becomes inf).  The product is formed in double, so it neither overflows nor rounds across a power of two, and S
// follows a power-of-two rescaling of g exactly.  Every consumer (k_grad_reduce, the input-gradient epilogues) removes
// S alone: gscale is part of the chain rule, S is not.  Zero / non-finite: S = 1.  One block; deterministic.
__global__ void __launch_bounds__(1024) k_grad_scale(const float* __restrict__ g, int n, float gscale, float* __restrict__ gs) {
  pdl_sync();
  __shared__ float red[32];
  float m = 0.f;
  for (int i = threadIdx.x; i < n; i += 1024) m = fmaxf(m, fabsf(g[i]));  // fmaxf drops NaNs; inf handled below
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < 32; ++w) m = fmaxf(m, red[w]);
    int e = 0;
    float S = 1.f, inv = 1.f;
    const double mt = (double)m * fabs((double)gscale);
    if (mt > 0.0 && isfinite(mt)) {
      frexp(mt, &e);  // mt = f * 2^e, f in [0.5, 1)
      int k = 8 - e;
      k = k > 100 ? 100 : (k < -100 ? -100 : k);
      S = ldexpf(1.f, k);
      inv = ldexpf(1.f, -k);
    }
    gs[0] = S;
    gs[1] = inv;
  }
}

}  // namespace pdg

using namespace pdg;

extern "C" size_t pdg_backward_ws_bytes(int64_t n_nodes, int64_t n_edges, int steps) {
  if (steps < 1 || steps > 62) return 0;
  int g = num_sms();
  if (g > MAXP) g = MAXP;
  return BwdWs(n_nodes, n_edges, steps, g, nullptr).total;
}

extern "C" int pdg_backward_inputs(const pdg_params_t* params, const pdg_norm_t* norm, const float* mean_stress,
                                   const float* pos, const int64_t* nodes_types, const float* edge_attr, const void* plan,
                                   int64_t n_nodes, int64_t n_edges, int steps, int flags, int precision, void* fwd_ws,
                                   void* bwd_ws, size_t bwd_ws_bytes, const float* grad_local_stress, float* grads_flat,
                                   float* grad_mean_stress, float* grad_pos, float* grad_edge_attr, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  if (steps < 1 || steps > 62) { set_error("pdg_backward: steps=%d unsupported", steps); return -1; }
  if (!(flags & PDG_FLAG_SAVE)) { set_error("pdg_backward: forward was not run with PDG_FLAG_SAVE"); return -1; }
  if (precision != PDG_PREC_FP32 && precision != PDG_PREC_BF16) { set_error("pdg_backward: unknown precision mode %d", precision); return -1; }
  const bool ig_node = grad_mean_stress != nullptr || grad_pos != nullptr, ig_edge = grad_edge_attr != nullptr;
  int G = num_sms();
  if (G > MAXP) G = MAXP;
  const bool tcm = precision == PDG_PREC_BF16;
  FwdWs W(n_nodes, n_edges, steps, true, fwd_ws, tcm);
  BwdWs B(n_nodes, n_edges, steps, G, bwd_ws);
  if (bwd_ws_bytes < B.total) { set_error("pdg_backward: workspace %zu < %zu", bwd_ws_bytes, B.total); return -1; }
  const int N = (int)n_nodes, E = (int)n_edges, T = steps;
  int32_t *perm, *recv, *send, *rowptr, *sptr, *slist;
  pdg_plan_views(const_cast<void*>(plan), n_nodes, n_edges, &perm, &recv, &send, &rowptr, &sptr, &slist);
  const int nt_n = (int)(W.N_pad / TM), nt_e = (int)(W.E_pad / TM);
  const int grid_n = balanced_grid(nt_n, G), grid_e = balanced_grid(nt_e, G);
  const double cnt_n = (double)N * H, cnt_e = (double)E * H;
  const float* const* P = params->p;
  const int scale_in = (flags & PDG_FLAG_SCALE_INPUT) ? 1 : 0;
  if (set_smem((const void*)k_decoder_bwd, SMEM_B3T)) return -2;
  if (set_smem((const void*)k_node_update_bwd, SMEM_B3T)) return -2;
  if (set_smem((const void*)k_edge_step_bwd, SMEM_B3T)) return -2;
  if (set_smem((const void*)k_node_pre_bwd, SMEM_B3T)) return -2;
  if (set_smem(ig_node ? (const void*)k_encoder_bwd<1, true> : (const void*)k_encoder_bwd<1, false>, SMEM_B3T)) return -2;
  if (set_smem(ig_edge ? (const void*)k_encoder_bwd<0, true> : (const void*)k_encoder_bwd<0, false>, SMEM_B3T)) return -2;

  PDG_CUDA_CHECK(cudaMemsetAsync(B.cta_grads, 0, (size_t)G * GRADP * sizeof(float), st));
  PDG_CUDA_CHECK(cudaMemsetAsync(grads_flat, 0, (size_t)PDG_PARAM_ELEMS * sizeof(float), st));
  auto scal = [&](int slot) { return B.scal + slot * 4; };
  auto flat = [&](int pi) { return grads_flat + param_offset(pi); };

  const float gscale = (flags & PDG_FLAG_SCALE_OUTPUT) ? norm->std_local_stress : 1.f;
  const float* gs = nullptr;
  if (tcm) {  // fp16 gradient tiles: scale the incoming gradient to a fixed magnitude, unscale in k_grad_reduce
    PDG_CUDA_CHECK(launch_pdl(k_grad_scale, dim3(1), dim3(1024), 0, st, grad_local_stress, N * PDG_OUT, gscale, B.gs));
    PDG_LAUNCH_CHECK();
    gs = B.gs;
  }
  {
    ScopedTimer tm_(KC_DEC_BWD, st);
    const int* nzf = (flags & PDG_FLAG_ZERO_CHECK) ? W.nzflag : nullptr;
    const DecArgs d = fwd_dec_args(W, P);  // what the forward's decoder read and saved
    if (tcm) {
      if (launch_decoder_bwd_tc(grad_local_stress, gscale, gs, d.hd_out, d.x_out, d.yprev, d.prev_parts, d.prev_count, d.D2, B.gx,
                                B.cta_grads, B.cs3, nzf, N, nt_n, grid_n, W.img, st)) return -2;
    } else {
      PDG_CUDA_CHECK(launch_pdl(k_decoder_bwd, dim3(grid_n), dim3(NT), SMEM_B3T, st, grad_local_stress, gscale, d.hd_out, d.x_out,
                                d.yprev, d.prev_parts, d.prev_count, P[ND_W0], d.D2, B.gx, B.cta_grads, B.cs3, nzf, N, nt_n));
    }
  }
  PDG_LAUNCH_CHECK();
  // receiver-side segment sums RA / RB (contiguous) start from zero; k_node_pre_bwd* re-zeroes every row it consumes
  PDG_CUDA_CHECK(cudaMemsetAsync(B.RA, 0, 2 * (size_t)W.N_pad * H * sizeof(float), st));
  for (int t = T - 1; t >= 0; --t) {
    const bool last = t == T - 1;
    PDG_CUDA_CHECK(launch_pdl(k_ln_finalize, dim3(1), dim3(FIN_G * H), 0, st, B.cs3, grid_n, W.parts_slot(slot_ln3(t)), cnt_n, P[PN_LNW], scal(slot_ln3(t)),
                                   flat(PN_LNW), flat(PN_LNB)));
    PDG_LAUNCH_CHECK();
    BwdStepArgs s = bwd_step_args(W, P, B, recv, send, rowptr, sptr, slist, t);
    NodeUpdBwdArgs& u = s.u;
    EdgeBwdArgs& e = s.e;
    NodePreBwdArgs& n = s.n;
    u.cta_grads = e.cta_grads = n.cta_grads = B.cta_grads;
    u.x_img = tcm ? W.ximg(t) : nullptr; u.hq_img = tcm ? W.hqimg(t) : nullptr; u.agg_img = tcm ? W.aggimg(t) : nullptr;
    e.e_img = W.eimg_[t];
    n.x_img = tcm ? W.ximg(t) : nullptr;
    {
      ScopedTimer tm_(KC_NODE_UPD_BWD, st);
      if (tcm) {
        if (launch_node_update_bwd_tc(u, W.img, grid_n, st)) return -2;
      } else {
        k_node_update_bwd<<<grid_n, NT, SMEM_B3T, st>>>(u);
      }
    }
    PDG_LAUNCH_CHECK();
    // LayerNorm-backward scalars of the message LN (from this step's node kernel) and of the edge-update LN (from the
    // previous edge kernel): one launch, two blocks.  Both feed edge_net.4.{weight,bias}: block 1 accumulates its share
    // in the (otherwise unused) LN entries of gradient slice 1, which k_grad_reduce adds in at the end.
    {
      float* slice1 = B.cta_grads + (size_t)(G > 1 ? 1 : 0) * GRADP;
      LnFinArgs f1{B.cs1, grid_n, W.parts_slot(slot_ln1(t)), cnt_e, P[PE_LNW], scal(slot_ln1(t)), flat(PE_LNW), flat(PE_LNB)};
      if (!last) {
        LnFinArgs f2{B.cs2, grid_e, W.parts_slot(slot_ln2(t)), cnt_e, P[PE_LNW], scal(slot_ln2(t)),
                     slice1 + param_offset(PE_LNW), slice1 + param_offset(PE_LNB)};
        PDG_CUDA_CHECK(launch_pdl(k_ln_finalize2, dim3(2), dim3(FIN_G * H), 0, st, f1, f2));
      } else {
        PDG_CUDA_CHECK(launch_pdl(k_ln_finalize, dim3(1), dim3(FIN_G * H), 0, st, f1.cs, f1.nparts, f1.fwd_parts, f1.count, f1.lnw,
                                  f1.scal_out, f1.flat_w, f1.flat_b));
      }
      PDG_LAUNCH_CHECK();
    }
    {
      ScopedTimer tm_(KC_EDGE_STEP_BWD, st);
      if (tcm) {
        if (launch_edge_step_bwd_tc3(e, W.img, grid_e, st)) return -2;
      } else {
        k_edge_step_bwd<<<grid_e, NT, SMEM_B3T, st>>>(e);
      }
    }
    PDG_LAUNCH_CHECK();
    {
      ScopedTimer tm_(KC_NODE_PRE_BWD, st);
      if (tcm) {
        if (launch_node_pre_bwd_tc(n, W.img, grid_n, st)) return -2;
      } else {
        k_node_pre_bwd<<<grid_n, NT, SMEM_B3T, st>>>(n);
      }
    }
    PDG_LAUNCH_CHECK();
  }
  // encoders: x_0 = LN(y_nenc), e_0 = LN(y_eenc)
  {
    LnFinArgs fn{B.cs3, grid_n, W.parts_slot(0), cnt_n, P[NE_LNW], scal(0), flat(NE_LNW), flat(NE_LNB)};
    LnFinArgs fe{B.cs2, grid_e, W.parts_slot(1), cnt_e, P[EE_LNW], scal(1), flat(EE_LNW), flat(EE_LNB)};
    PDG_CUDA_CHECK(launch_pdl(k_ln_finalize2, dim3(2), dim3(FIN_G * H), 0, st, fn, fe));
    PDG_LAUNCH_CHECK();
  }
  {
    ScopedTimer tm_(KC_ENC_BWD, st);
    if (tcm) {
      if (launch_node_encoder_bwd_tc(B.gx, W.y_nenc, scal(0), P[NE_LNW], mean_stress, pos, nodes_types, norm, scale_in, P[NE_W0],
                                     P[NE_B0], B.cta_grads, gs, grad_mean_stress, grad_pos, N, nt_n, grid_n, W.img, st)) return -2;
    } else {
      PDG_CUDA_CHECK(launch_pdl(ig_node ? k_encoder_bwd<1, true> : k_encoder_bwd<1, false>, dim3(grid_n), dim3(NT), SMEM_B3T, st, B.gx,
                                W.y_nenc, scal(0), P[NE_LNW], mean_stress, pos, nodes_types, nullptr, nullptr, *norm, scale_in, P[NE_W0],
                                P[NE_B0], P[NE_W2], B.cta_grads, param_offset(NE_W0), param_offset(NE_B0), param_offset(NE_W2),
                                param_offset(NE_B2), N, nt_n, grad_mean_stress, grad_pos));
    }
  }
  PDG_LAUNCH_CHECK();
  {
    ScopedTimer tm_(KC_ENC_BWD, st);
    if (tcm) {
      if (launch_edge_encoder_bwd_tc(B.ge, W.y_eenc, scal(1), P[EE_LNW], edge_attr, perm, norm, scale_in, P[EE_W0], P[EE_B0],
                                     B.cta_grads, gs, grad_edge_attr, E, nt_e, grid_e, W.img, st)) return -2;
    } else {
      (ig_edge ? k_encoder_bwd<0, true> : k_encoder_bwd<0, false>)<<<grid_e, NT, SMEM_B3T, st>>>(
          B.ge, W.y_eenc, scal(1), P[EE_LNW], nullptr, nullptr, nullptr, edge_attr, perm, *norm, scale_in, P[EE_W0], P[EE_B0],
          P[EE_W2], B.cta_grads, param_offset(EE_W0), param_offset(EE_B0), param_offset(EE_W2), param_offset(EE_B2), E, nt_e,
          grad_edge_attr, nullptr);
    }
  }
  PDG_LAUNCH_CHECK();
  {
    ScopedTimer tm_(KC_GRAD_REDUCE, st);
    PDG_CUDA_CHECK(launch_pdl(k_grad_reduce, dim3((PDG_PARAM_ELEMS + 255) / 256), dim3(256), 0, st, B.cta_grads, G, grads_flat, gs, tcm ? 1 : 0));
  }
  PDG_LAUNCH_CHECK();
  return 0;
}

extern "C" int pdg_backward(const pdg_params_t* params, const pdg_norm_t* norm, const float* mean_stress,
                            const float* pos, const int64_t* nodes_types, const float* edge_attr, const void* plan,
                            int64_t n_nodes, int64_t n_edges, int steps, int flags, int precision, void* fwd_ws,
                            void* bwd_ws, size_t bwd_ws_bytes, const float* grad_local_stress, float* grads_flat,
                            void* stream) {
  return pdg_backward_inputs(params, norm, mean_stress, pos, nodes_types, edge_attr, plan, n_nodes, n_edges, steps, flags,
                             precision, fwd_ws, bwd_ws, bwd_ws_bytes, grad_local_stress, grads_flat, nullptr, nullptr, nullptr,
                             stream);
}
