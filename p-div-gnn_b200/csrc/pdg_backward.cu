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

// ---- small device helpers ------------------------------------------------------------------
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

// ---- decoder backward -----------------------------------------------------------------------
__global__ void __launch_bounds__(NT, 1)
k_decoder_bwd(const float* __restrict__ g_out, float gscale, const float* __restrict__ hd, const float* __restrict__ x_T,
              const float* __restrict__ y3_last, const double* __restrict__ parts_prev, double count_prev,
              const float* __restrict__ D1, const float* __restrict__ D2, float* __restrict__ gx,
              float* __restrict__ cta_grads, float* __restrict__ cs3, const int* __restrict__ nzflag, int N, int n_tiles) {
  extern __shared__ __align__(16) float smem[];
  float* T0 = smem;
  float* T1 = T0 + TM * LDS;
  float* T2 = T1 + TM * LDS;
  float* Ws = T2 + TM * LDS;
  float* gd = Ws + 2 * BKB * H;  // [TM][4] (aliases the index area)
  float* cg = cta_grads + (size_t)blockIdx.x * GRADP;
  const int tid = threadIdx.x, c4 = (tid & 31) * 4;
  pdl_sync();
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
    tile_load(T2, x_T + (size_t)row0 * H);
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
    float acc[8][8];
    acc_zero(acc);
    gemm_colA(T0, T2, TM, acc);  // dD1[o][k] = sum_r g_hd[r][o] x_T[r][k]
    rmw_add(acc, cg + param_offset(ND_W0), H);
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
  if (tid < H) {
#pragma unroll
    for (int o = 0; o < 3; ++o) cg[param_offset(ND_W2) + o * H + tid] += dD2[o];
    cg[param_offset(ND_B0) + tid] += dd1;
  } else if (tid < H + 3) {
    cg[param_offset(ND_B2) + tid - H] += dd2;
  }
  colsum_flush(cgx, T0, cs3 + (size_t)blockIdx.x * 2 * H, false);
  colsum_flush(cgy, T0, cs3 + (size_t)blockIdx.x * 2 * H + H, false);
}

// ---- B3: node_update backward -----------------------------------------------------------------
__global__ void __launch_bounds__(NT, 1) k_node_update_bwd(NodeUpdBwdArgs a) {
  extern __shared__ __align__(16) float smem[];
  float* T0 = smem;
  float* T1 = T0 + TM * LDS;
  float* T2 = T1 + TM * LDS;
  float* Ws = T2 + TM * LDS;
  float* smf = Ws + 2 * BKB * H;
  float* cg = a.cta_grads + (size_t)blockIdx.x * GRADP;
  const int tid = threadIdx.x, c4 = (tid & 31) * 4, ty = tid >> 4;
  const LnStat st1 = ln_stat_block(a.parts1, a.count1, smf);
  const float c1 = a.scal3[0], c2 = a.scal3[1], mu3 = a.scal3[2], rstd3 = a.scal3[3];
  const float4 wn = *reinterpret_cast<const float4*>(a.lnw_n + c4);
  const float4 we = *reinterpret_cast<const float4*>(a.lnw_e + c4);
  const float4 be = *reinterpret_cast<const float4*>(a.lnb_e + c4);
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
    __syncthreads();
    dc2 += tile_colsum(T0, nvalid);
    float acc[8][8];
    acc_zero(acc);
    gemm_colA(T0, T1, TM, acc);  // dV2[o][i] = sum_r dy3[r][o] hq[r][i]
    rmw_add(acc, cg + param_offset(PN_W2), H);
    acc_zero(acc);
    gemm_rowA<BKB>(T0, a.V2, H, acc, Ws, H);  // dhq_pre = dy3 V2
    {
      float h[8][8];
      acc_load(h, T1, LDS);
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = h[i][j] > 0.f ? acc[i][j] : 0.f;
    }
    acc_store(acc, T0, LDS);  // dhq
    __syncthreads();          // everyone is done with hq in T1
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
  if (tid < H) {
    cg[param_offset(PN_B2) + tid] += dc2;
    cg[param_offset(PN_B0) + tid] += dc1;
  }
  colsum_flush(cg1, T0, a.cs1 + (size_t)blockIdx.x * 2 * H, false);
  colsum_flush(cgy1, T0, a.cs1 + (size_t)blockIdx.x * 2 * H + H, false);
}

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

// ---- B1: node_pre backward -------------------------------------------------------------------
__global__ void __launch_bounds__(NT, 1) k_node_pre_bwd(NodePreBwdArgs a) {
  extern __shared__ __align__(16) float smem[];
  float* T0 = smem;
  float* T1 = T0 + TM * LDS;
  float* T2 = T1 + TM * LDS;
  float* Ws = T2 + TM * LDS;
  float* cg = a.cta_grads + (size_t)blockIdx.x * GRADP;
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
    tile_load(T2, a.x_t + (size_t)row0 * H);
    __syncthreads();
    float acc[8][8];
    acc_zero(acc);
    gemm_colA(T0, T2, TM, acc);  // dWa[o][k] = sum_r dPa[r][o] x_t[r][k]
    rmw_add(acc, cg + param_offset(PE_W0), 3 * H);
    acc_zero(acc);
    gemm_colA(T1, T2, TM, acc);
    rmw_add(acc, cg + param_offset(PE_W0) + H, 3 * H);
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

// ---- encoder backward (node: NODE=1, edge: NODE=0) -------------------------------------------
// IG: also write the input gradient dfeat = dh0 W0 of every row, un-standardised (models.py:140-162):
//   node  gi0 = d/d mean_stress [N,3] (features 0-2), gi1 = d/d pos [N,2] (features 3-4), either may be null;
//   edge  gi0 = d/d edge_attr [E] at perm[row] (PyG edge order; perm is a permutation: plain stores).
// The <NODE, false> instances are the parameter-gradient-only kernels, unchanged.
template <int NODE, bool IG>
__global__ void __launch_bounds__(NT, 1)
k_encoder_bwd(const float* __restrict__ g_in, const float* __restrict__ y_raw, const float* __restrict__ scal,
              const float* __restrict__ lnw, const float* __restrict__ mean_stress, const float* __restrict__ pos,
              const int64_t* __restrict__ types, const float* __restrict__ edge_attr, const int32_t* __restrict__ perm,
              pdg_norm_t nrm, int scale_in, const float* __restrict__ W0, const float* __restrict__ b0,
              const float* __restrict__ W2, float* __restrict__ cta_grads, int off_w0, int off_b0, int off_w2,
              int off_b2, int R, int n_tiles, float* __restrict__ gi0, float* __restrict__ gi1) {
  extern __shared__ __align__(16) float smem[];
  float* T0 = smem;
  float* T1 = T0 + TM * LDS;
  float* T2 = T1 + TM * LDS;
  float* Ws = T2 + TM * LDS;
  float* feat = T2;  // [TM][8]
  float* cg = cta_grads + (size_t)blockIdx.x * GRADP;
  const int tid = threadIdx.x, c4 = (tid & 31) * 4;
  constexpr int NF = NODE ? 6 : 1;
  pdl_sync();
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
          float m0 = mean_stress[row * 3 + 0], m1 = mean_stress[row * 3 + 1], m2 = mean_stress[row * 3 + 2];
          float p0 = pos[row * 2 + 0], p1 = pos[row * 2 + 1];
          if (scale_in) {
            m0 = (m0 - nrm.mean_mean_stress) / nrm.std_mean_stress;
            m1 = (m1 - nrm.mean_mean_stress) / nrm.std_mean_stress;
            m2 = (m2 - nrm.mean_mean_stress) / nrm.std_mean_stress;
            p0 = (p0 - nrm.mean_pos) / nrm.std_pos;
            p1 = (p1 - nrm.mean_pos) / nrm.std_pos;
          }
          f[0] = m0; f[1] = m1; f[2] = m2; f[3] = p0; f[4] = p1; f[5] = (float)types[row];
        } else {
          float v = edge_attr[perm[row]];
          if (scale_in) v = (v - nrm.mean_edge_weight) / nrm.std_edge_weight;
          f[0] = v;
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
    __syncthreads();
    db2 += tile_colsum(T0, nvalid);
    float acc[8][8];
    acc_zero(acc);
    gemm_colA(T0, T1, TM, acc);  // dW2[o][i] = sum_r dy[r][o] h0[r][i]
    rmw_add(acc, cg + off_w2, H);
    acc_zero(acc);
    gemm_rowA<BKB>(T0, W2, H, acc, Ws, H);  // dh0_pre = dy W2
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
    if (tid < H) {
      for (int r = 0; r < nvalid; ++r) {
        const float d = T0[r * LDS + tid];
        db0 += d;
#pragma unroll
        for (int j = 0; j < NF; ++j) dW0[j] = fmaf(d, feat[r * 8 + j], dW0[j]);
      }
    } else if (IG) {  // warps 4-7, idle in the walk above: dfeat[r] = dh0[r] W0, one warp per row, lane = 4 channels
      constexpr int NI = NODE ? 5 : 1;  // feature 5 (nodes_types) is an integer input: no gradient
      for (int r = (tid - H) >> 5; r < nvalid; r += (NT - H) / 32) {
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
  if (tid < H) {
    cg[off_b2 + tid] += db2;
    cg[off_b0 + tid] += db0;
#pragma unroll
    for (int j = 0; j < NF; ++j) cg[off_w0 + tid * NF + j] += dW0[j];
  }
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

static int set_smem_b(const void* fn, size_t bytes) {
  cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e != cudaSuccess) { set_error("cudaFuncSetAttribute(%zu B smem): %s", bytes, cudaGetErrorString(e)); return -2; }
  return 0;
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
  const float* pk = W.pack;
  const int scale_in = (flags & PDG_FLAG_SCALE_INPUT) ? 1 : 0;
  if (set_smem_b((const void*)k_decoder_bwd, SMEM_B3T)) return -2;
  if (set_smem_b((const void*)k_node_update_bwd, SMEM_B3T)) return -2;
  if (set_smem_b((const void*)k_edge_step_bwd, SMEM_B3T)) return -2;
  if (set_smem_b((const void*)k_node_pre_bwd, SMEM_B3T)) return -2;
  if (set_smem_b(ig_node ? (const void*)k_encoder_bwd<1, true> : (const void*)k_encoder_bwd<1, false>, SMEM_B3T)) return -2;
  if (set_smem_b(ig_edge ? (const void*)k_encoder_bwd<0, true> : (const void*)k_encoder_bwd<0, false>, SMEM_B3T)) return -2;

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
    if (tcm) {
      if (launch_decoder_bwd_tc(grad_local_stress, gscale, gs, W.hd, W.x_[T], W.y3_[T - 1], W.parts_slot(slot_ln3(T - 1)), cnt_n,
                                P[ND_W2], B.gx, B.cta_grads, B.cs3, nzf, N, nt_n, grid_n, W.img, st)) return -2;
    } else {
      PDG_CUDA_CHECK(launch_pdl(k_decoder_bwd, dim3(grid_n), dim3(NT), SMEM_B3T, st, grad_local_stress, gscale, W.hd, W.x_[T],
                                W.y3_[T - 1], W.parts_slot(slot_ln3(T - 1)), cnt_n, P[ND_W0], P[ND_W2], B.gx, B.cta_grads, B.cs3,
                                nzf, N, nt_n));
    }
  }
  PDG_LAUNCH_CHECK();
  // receiver-side segment sums RA / RB (contiguous) start from zero; k_node_pre_bwd* re-zeroes every row it consumes
  PDG_CUDA_CHECK(cudaMemsetAsync(B.RA, 0, 2 * (size_t)W.N_pad * H * sizeof(float), st));
  for (int t = T - 1; t >= 0; --t) {
    const bool last = t == T - 1, first = t == 0;
    PDG_CUDA_CHECK(launch_pdl(k_ln_finalize, dim3(1), dim3(FIN_G * H), 0, st, B.cs3, grid_n, W.parts_slot(slot_ln3(t)), cnt_n, P[PN_LNW], scal(slot_ln3(t)),
                                   flat(PN_LNW), flat(PN_LNB)));
    PDG_LAUNCH_CHECK();
    NodeUpdBwdArgs u;
    u.gx = B.gx; u.y3 = W.y3_[t]; u.hq = W.hq_[t]; u.aggraw = W.aggraw_[t]; u.x_t = W.x_[t]; u.rowptr = rowptr;
    u.scal3 = scal(slot_ln3(t)); u.lnw_n = P[PN_LNW]; u.parts1 = W.parts_slot(slot_ln1(t)); u.count1 = cnt_e;
    u.lnw_e = P[PE_LNW]; u.lnb_e = P[PE_LNB]; u.V1 = P[PN_W0]; u.V2 = P[PN_W2]; u.gagg = B.gagg;
    u.cta_grads = B.cta_grads; u.cs1 = B.cs1; u.N = N; u.n_tiles = nt_n;
    u.x_img = tcm ? W.ximg(t) : nullptr; u.hq_img = tcm ? W.hqimg(t) : nullptr; u.agg_img = tcm ? W.aggimg(t) : nullptr;
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
    EdgeBwdArgs e;
    e.e_t = W.e_[t]; e.e_img = W.eimg_[t]; e.Pa = W.Pa_[t]; e.Pb = W.Pb_[t]; e.gagg = B.gagg; e.ge = B.ge;
    e.y2_t = last ? nullptr : W.y2_[t];
    e.yprev = first ? W.y_eenc : W.y2_[t - 1];
    e.parts_prev = W.parts_slot(first ? 1 : slot_ln2(t - 1)); e.count_prev = cnt_e;
    e.recv = recv; e.send = send; e.rowptr = rowptr;
    e.WtE = pk + PackOffsets::PE_WET; e.b1 = P[PE_B0]; e.Wt2 = pk + PackOffsets::PE_W2T; e.b2 = P[PE_B2];
    e.W0 = P[PE_W0]; e.W2 = P[PE_W2]; e.lnw = P[PE_LNW];
    e.scal1 = scal(slot_ln1(t)); e.scal2 = last ? nullptr : scal(slot_ln2(t));
    e.DHM = B.DHM; e.DHN = B.DHN; e.RA = B.RA; e.RB = B.RB; e.cta_grads = B.cta_grads; e.cs2 = B.cs2;
    e.E = E; e.n_tiles = nt_e; e.last = last ? 1 : 0;
    {
      ScopedTimer tm_(KC_EDGE_STEP_BWD, st);
      if (tcm) {
        if (launch_edge_step_bwd_tc3(e, W.img, grid_e, st)) return -2;
      } else {
        k_edge_step_bwd<<<grid_e, NT, SMEM_B3T, st>>>(e);
      }
    }
    PDG_LAUNCH_CHECK();
    NodePreBwdArgs n;
    n.gx = B.gx; n.RA = B.RA; n.RB = last ? nullptr : B.RB; n.DHM = B.DHM; n.DHN = last ? nullptr : B.DHN;
    n.sptr = sptr; n.slist = slist; n.x_t = W.x_[t]; n.yprev = first ? W.y_nenc : W.y3_[t - 1];
    n.parts_prev = W.parts_slot(first ? 0 : slot_ln3(t - 1)); n.count_prev = cnt_n; n.W0 = P[PE_W0];
    n.cta_grads = B.cta_grads; n.cs3 = B.cs3; n.N = N; n.n_tiles = nt_n;
    n.x_img = tcm ? W.ximg(t) : nullptr;
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
