// Batched reverse-mode derivative (vector-Jacobian products) of EncodeProcessDecode.forward with respect to its
// differentiable inputs, fp32 FFMA tiles: for K cotangents u_k of local_stress, J^T u_k on mean_stress, pos and edge_attr.
//
// One adjoint pass runs the data-gradient path of pdg_backward.cu for K cotangents.  It reads the state that a pdg_forward
// with PDG_FLAG_SAVE kept and never writes the forward workspace, so a later pdg_backward is unaffected.  Everything that
// only serves parameter gradients is dropped: the weight-gradient GEMMs (gemm_colA), the per-CTA gradient slices and
// their reduction, the LayerNorm affine gradients.  Left per cotangent and tile: one data GEMM in the decoder, three in
// node_update, three in the edge step, two in node_pre and one in each encoder.
//
// Each cotangent has a workspace of the data buffers of BwdWs (VjpWs below), one after another at a fixed stride.  The
// decoder, node_update, node_pre and encoder kernels are the backward's own bodies (pdg_bwd.cuh) without weight
// gradients: each wrapper below moves its pointers to cotangent blockIdx.y and runs the body over the x-grid of
// pdg_backward_inputs, so every cotangent fills the same per-CTA column-sum slots.  Both host functions take what step t
// reads from bwd_step_args.  The edge kernel is this file's own: it takes a group of cotangents, computes G, both hidden
// masks and the message y1 once per tile, then loops over the group.  Cotangent k runs the data-gradient operations of
// pdg_backward_inputs in their order, so column k has that call's bits: the weight-gradient GEMMs feed none of them.
#include <algorithm>

#include "pdg_bwd.cuh"

namespace pdg {

// Per-cotangent data buffers of the adjoint pass: those of BwdWs without the per-CTA gradient slices, plus the edge
// kernel's per-thread column partials of the edge-encoder LayerNorm sums (a CTA runs its tiles once for a whole group of
// cotangents, so each cotangent's running partials leave registers between tiles: [MAXP CTAs][16][NT threads]).
struct VjpWs : DataGradBufs {
  int64_t N_pad, E_pad;
  char* base;
  size_t total;
  float* eacc;
  VjpWs(int64_t n, int64_t e, int steps, void* ws) : base((char*)ws) {
    N_pad = round_up(n, TM);
    E_pad = round_up(e, TM);
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t r = o; o += (size_t)round_up((int64_t)bytes, 256); return (float*)(base + r); };
    take_data_grads(take, N_pad, E_pad, steps);
    eacc = take((size_t)MAXP * 16 * NT * sizeof(float));
    total = o;  // a multiple of 256 bytes: every copy stays aligned
  }
};

// ---- LayerNorm-backward scalars {c1, c2, mu, a} of one or two instances (blockIdx.x) for every cotangent (blockIdx.y) ----
__global__ void __launch_bounds__(FIN_G* H) k_ln_finalize_vjp(LnFinArgs a0, LnFinArgs a1, size_t cws) {
  const LnFinArgs& a = blockIdx.x == 0 ? a0 : a1;
  const size_t off = (size_t)blockIdx.y * cws;
  ln_finalize_body<false>(copy_at(a.cs, off), a.nparts, a.fwd_parts, a.count, a.lnw, copy_at(a.scal_out, off), nullptr, nullptr);
}

// ---- decoder, node_update, node_pre, encoders: the bodies of the fp32 backward without weight gradients (pdg_bwd.cuh) for
// cotangent blockIdx.y ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(NT, 1)
k_decoder_vjp(const float* __restrict__ g_out, float gscale, const float* __restrict__ hd, const float* __restrict__ y3_last,
              const double* __restrict__ parts_prev, double count_prev, const float* __restrict__ D1,
              const float* __restrict__ D2, float* __restrict__ gx, float* __restrict__ cs3, const int* __restrict__ nzflag,
              int N, int n_tiles, size_t cws) {
  const size_t off = (size_t)blockIdx.y * cws;
  decoder_bwd_body<false>(g_out + (size_t)blockIdx.y * N * PDG_OUT, gscale, hd, nullptr, y3_last, parts_prev, count_prev, D1, D2,
                          copy_at(gx, off), nullptr, copy_at(cs3, off), nzflag, N, n_tiles);  // g_out: [K][N][3]
}

__global__ void __launch_bounds__(NT, 1) k_node_update_vjp(NodeUpdBwdArgs a, size_t cws) {
  const size_t off = (size_t)blockIdx.y * cws;
  a.gx = copy_at(a.gx, off);
  a.gagg = copy_at(a.gagg, off);
  a.scal3 = copy_at(a.scal3, off);
  a.cs1 = copy_at(a.cs1, off);
  node_update_bwd_body<false>(a);
}

__global__ void __launch_bounds__(NT, 1) k_node_pre_vjp(NodePreBwdArgs a, size_t cws) {
  const size_t off = (size_t)blockIdx.y * cws;
  a.gx = copy_at(a.gx, off);
  a.RA = copy_at(a.RA, off);
  a.RB = copy_at(a.RB, off);
  a.DHM = copy_at(a.DHM, off);
  a.DHN = copy_at(a.DHN, off);
  a.cs3 = copy_at(a.cs3, off);
  node_pre_bwd_body<false>(a);
}

//   node  gi0 = d/d mean_stress [K][N][3], gi1 = d/d pos [K][N][2] (either may be null);
//   edge  gi0 = d/d edge_attr [K][E] at perm[row] (PyG edge order)
template <int NODE>
__global__ void __launch_bounds__(NT, 1)
k_encoder_vjp(const float* __restrict__ g_in, const float* __restrict__ y_raw, const float* __restrict__ scal,
              const float* __restrict__ lnw, const float* __restrict__ mean_stress, const float* __restrict__ pos,
              const int64_t* __restrict__ types, const float* __restrict__ edge_attr, const int32_t* __restrict__ perm,
              pdg_norm_t nrm, int scale_in, const float* __restrict__ W0, const float* __restrict__ b0,
              const float* __restrict__ W2, int R, int n_tiles, float* __restrict__ gi0, float* __restrict__ gi1, size_t cws) {
  const size_t off = (size_t)blockIdx.y * cws;
  if (gi0 != nullptr) gi0 += (size_t)blockIdx.y * R * (NODE ? 3 : 1);
  if (gi1 != nullptr) gi1 += (size_t)blockIdx.y * R * 2;
  encoder_bwd_body<NODE, false, true>(copy_at(g_in, off), y_raw, copy_at(scal, off), lnw, mean_stress, pos, types, edge_attr, perm,
                                      nrm, scale_in, W0, b0, W2, nullptr, 0, 0, 0, 0, R, n_tiles, gi0, gi1);
}

// ---- edge step on a tile of 128 receiver-sorted edges, for a group of C cotangents (blockIdx.y = group) -------------
//   once per tile: G = e_t We^T + b1;  m1 = [G + Pa[recv] + Pb[send] > 0], m2 = [G + Pa[send] + Pb[recv] > 0] (register
//                  bits);  y1 = relu(relu(G + Pa[recv] + Pb[send]) W2^T + b2) -> T0 for the whole group
//   per cotangent: dy1 -> T1;  dhm = m1 (dy1 W2) -> DHM, T1, segment sums RA;
//                  dy2 -> T2;  dhn = m2 (dy2 W2) -> DHN, T2, segment sums RB   (not on the last step);
//                  dG = dhm + dhn -> T1;  ge = ge + dG We  and the column sums of the LayerNorm that produced e_t
struct EdgeVjpArgs {
  EdgeBwdArgs e;  // cotangent 0's buffers (gagg, ge, scal1, scal2, DHM, DHN, RA, RB, cs2) and the primal state
  float* eacc;
  size_t cws;
  int K, C;
};

__global__ void __launch_bounds__(NT, 1) k_edge_step_vjp(EdgeVjpArgs v) {
  extern __shared__ __align__(16) float smem[];
  const EdgeBwdArgs& a = v.e;
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
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  const int k0 = blockIdx.y * v.C, nk = min(v.C, v.K - k0);  // this CTA's cotangents: k0 .. k0 + nk - 1
  const float mu_prev = ln_stat_block(a.parts_prev, a.count_prev, (float*)smi).mu;
  for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const int row0 = tile * TM;
    const int nvalid = min(TM, a.E - row0);
    const bool first_tile = tile == (int)blockIdx.x, last_tile = tile + (int)gridDim.x >= a.n_tiles;
    if (tid < TM) {
      recv_s[tid] = a.recv[row0 + tid];
      send_s[tid] = a.send[row0 + tid];
    }
    tile_load(T0, a.e_t + (size_t)row0 * H);
    __syncthreads();
    const int nseg = tile_segments(recv_s, nvalid, seg_row, seg_masks);
    float acc[8][8];
    // ---- primal part, once per tile for the whole group ----
    acc_zero(acc);
    gemm_rowA<BKB>(T0, a.WtE, H, acc, Ws, H);
    unsigned long long m1 = 0, m2 = 0;
    {
      float bias1[8];
      load_cols(bias1, a.b1);
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
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float g = acc[i][j] + bias1[j];
          // same association as the forward: (G + Pa) + Pb
          const float hm = fmaxf(g + par_[j] + pbs_[j], 0.f);
          const float hn = fmaxf(g + pas_[j] + pbr_[j], 0.f);
          m1 |= (unsigned long long)(hm > 0.f) << (i * 8 + j);
          m2 |= (unsigned long long)(hn > 0.f) << (i * 8 + j);
          acc[i][j] = hm;
        }
      }
    }
    acc_store(acc, T1, LDS);  // hm
    acc_zero(acc);
    gemm_rowA<BKB>(T1, a.Wt2, H, acc, Ws, H);
    {
      float bias2[8];
      load_cols(bias2, a.b2);
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaxf(acc[i][j] + bias2[j], 0.f);
    }
    acc_store(acc, T0, LDS);  // y1: read back by the thread that wrote it, for every cotangent of the group
    // ---- cotangents of the group ----
    for (int c = 0; c < nk; ++c) {
      const size_t off = (size_t)(k0 + c) * v.cws;
      const float* scal1 = copy_at(a.scal1, off);
      const float c1m = scal1[0], c2m = scal1[1], mu1 = scal1[2], rstd1 = scal1[3];
      const float* gagg = copy_at(a.gagg, off);
      float* ge = copy_at(a.ge, off);
      {
        float lw[8], y[8][8];
        load_cols(lw, a.lnw);
        acc_load(y, T0, LDS);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int r = ty * 8 + i;
          const bool ok = r < nvalid;
          const float* gp = gagg + (size_t)recv_s[r] * H + tx * 4;
          const float4 g0 = __ldg((const float4*)gp), g1 = __ldg((const float4*)(gp + 64));
          const float gv[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
#pragma unroll
          for (int j = 0; j < 8; ++j)
            acc[i][j] = (ok && y[i][j] > 0.f) ? rstd1 * gv[j] * lw[j] - c1m - c2m * (y[i][j] - mu1) : 0.f;
        }
      }
      acc_store(acc, T1, LDS);  // dy1
      acc_zero(acc);
      gemm_rowA<BKB>(T1, a.W2, H, acc, Ws, H);  // dhm_pre = dy1 W2
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = (m1 >> (i * 8 + j)) & 1ull ? acc[i][j] : 0.f;
      acc_store(acc, copy_at(a.DHM, off) + (size_t)row0 * H, H);
      acc_store(acc, T1, LDS);  // dhm
      __syncthreads();
      tile_segsum_warp<false>(T1, recv_s, seg_row, nseg, a.rowptr, row0, nvalid, copy_at(a.RA, off), seg_dummy, seg_dummy);
      if (!a.last) {
        {
          const float* scal2 = copy_at(a.scal2, off);
          const float c1n = scal2[0], c2n = scal2[1], mu2 = scal2[2], rstd2 = scal2[3];
          float lw[8], y[8][8], g[8][8];
          load_cols(lw, a.lnw);
          mt_load(y, a.y2_t + (size_t)row0 * H);
          mt_load(g, ge + (size_t)row0 * H);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const bool ok = ty * 8 + i < nvalid;
#pragma unroll
            for (int j = 0; j < 8; ++j)
              acc[i][j] = (ok && y[i][j] > 0.f) ? rstd2 * g[i][j] * lw[j] - c1n - c2n * (y[i][j] - mu2) : 0.f;
          }
        }
        acc_store(acc, T2, LDS);  // dy2
        acc_zero(acc);
        gemm_rowA<BKB>(T2, a.W2, H, acc, Ws, H);
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[i][j] = (m2 >> (i * 8 + j)) & 1ull ? acc[i][j] : 0.f;
        acc_store(acc, copy_at(a.DHN, off) + (size_t)row0 * H, H);
        acc_store(acc, T2, LDS);  // dhn
        __syncthreads();
        tile_segsum_warp<false>(T2, recv_s, seg_row, nseg, a.rowptr, row0, nvalid, copy_at(a.RB, off), seg_dummy, seg_dummy);
        {
          float m[8][8];
          acc_load(m, T1, LDS);
#pragma unroll
          for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[i][j] += m[i][j];
        }
        __syncthreads();  // segment sums over T1/T2 finished before T1 changes
        acc_store(acc, T1, LDS);  // dG
      }
      // de_t = ge_{t+1} + dG We ;  column sums for the LayerNorm that produced e_t's increment
      acc_zero(acc);
      gemm_rowA<BKB>(T1, a.W0 + 2 * H, H, acc, Ws, 3 * H);
      if (!a.last) {
        float g[8][8];
        mt_load(g, ge + (size_t)row0 * H);
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[i][j] += g[i][j];
      }
      acc_store(acc, ge + (size_t)row0 * H, H);
      {
        // this cotangent's running column partials: registers of the thread in pdg_backward, here kept in eacc between
        // tiles (same per-thread order of additions)
        float cge[8] = {0}, cgye[8] = {0};
        float* pe = copy_at(v.eacc, off) + (size_t)blockIdx.x * 16 * NT + tid;
        if (!first_tile)
#pragma unroll
          for (int j = 0; j < 8; ++j) { cge[j] = pe[j * NT]; cgye[j] = pe[(8 + j) * NT]; }
        float y[8][8];
        mt_load(y, a.yprev + (size_t)row0 * H);
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int j = 0; j < 8; ++j) { cge[j] += acc[i][j]; cgye[j] = fmaf(acc[i][j], y[i][j] - mu_prev, cgye[j]); }
        if (last_tile) {
          float* cs2 = copy_at(a.cs2, off) + (size_t)blockIdx.x * 2 * H;
          colsum_flush(cge, Ws, cs2, false);  // Ws is idle between GEMMs
          colsum_flush(cgye, Ws, cs2 + H, false);
        } else {
#pragma unroll
          for (int j = 0; j < 8; ++j) { pe[j * NT] = cge[j]; pe[(8 + j) * NT] = cgye[j]; }
        }
      }
    }
    __syncthreads();
  }
}

}  // namespace pdg

using namespace pdg;

extern "C" size_t pdg_vjp_batched_ws_bytes(int64_t n_nodes, int64_t n_edges, int steps, int n_cotangents) {
  if (steps < 1 || steps > 62 || n_cotangents < 1 || n_cotangents > PDG_VJP_MAX_COTANGENTS) return 0;
  return (size_t)n_cotangents * VjpWs(n_nodes, n_edges, steps, nullptr).total;
}

extern "C" int pdg_vjp_batched(const pdg_params_t* params, const pdg_norm_t* norm, const float* mean_stress, const float* pos,
                               const int64_t* nodes_types, const float* edge_attr, const void* plan, int64_t n_nodes,
                               int64_t n_edges, int steps, int flags, int precision, const void* fwd_ws, void* vjp_ws,
                               size_t vjp_ws_bytes, int n_cotangents, const float* grad_local_stress, float* grad_mean_stress,
                               float* grad_pos, float* grad_edge_attr, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  const int K = n_cotangents;
  if (K < 1 || K > PDG_VJP_MAX_COTANGENTS) {
    set_error("pdg_vjp_batched: n_cotangents=%d outside 1..%d", K, PDG_VJP_MAX_COTANGENTS);
    return -1;
  }
  if (precision != PDG_PREC_FP32) {
    set_error("pdg_vjp_batched: only the fp32 mode (PDG_PREC_FP32) has a batched reverse-mode derivative; the 16-bit "
              "mode's input gradients miss its 2e-2 tolerance");
    return -1;
  }
  if (!(flags & PDG_FLAG_SAVE)) { set_error("pdg_vjp_batched: the forward workspace must come from a pdg_forward with PDG_FLAG_SAVE"); return -1; }
  if (steps < 1 || steps > 62) { set_error("pdg_vjp_batched: steps=%d unsupported", steps); return -1; }
  if (grad_mean_stress == nullptr && grad_pos == nullptr && grad_edge_attr == nullptr) {
    set_error("pdg_vjp_batched: no output requested (grad_mean_stress, grad_pos and grad_edge_attr are all NULL)");
    return -1;
  }
  if (n_nodes <= 0 || n_edges <= 0) { set_error("pdg_vjp_batched: empty graph"); return -1; }
  const FwdWs W(n_nodes, n_edges, steps, true, const_cast<void*>(fwd_ws), false);
  const VjpWs V(n_nodes, n_edges, steps, vjp_ws);
  const size_t cws = V.total;  // bytes between consecutive cotangent workspaces
  if (vjp_ws_bytes < (size_t)K * cws) { set_error("pdg_vjp_batched: workspace %zu < %zu", vjp_ws_bytes, (size_t)K * cws); return -1; }
  const int N = (int)n_nodes, E = (int)n_edges, T = steps;
  int32_t *perm, *recv, *send, *rowptr, *sptr, *slist;
  pdg_plan_views(const_cast<void*>(plan), n_nodes, n_edges, &perm, &recv, &send, &rowptr, &sptr, &slist);
  const int nt_n = (int)(W.N_pad / TM), nt_e = (int)(W.E_pad / TM);
  int G = num_sms();
  if (G > MAXP) G = MAXP;
  const int grid_n = balanced_grid(nt_n, G), grid_e = balanced_grid(nt_e, G);  // the x-grids of pdg_backward_inputs
  // Edge kernel: cotangent groups of C over the SMs the x-grid leaves idle (the rule of pdg_jvp_batched)
  int groups = std::min(K, std::max(1, G / grid_e));
  const int C = (K + groups - 1) / groups;
  groups = (K + C - 1) / C;  // no empty group
  const double cnt_n = (double)N * H, cnt_e = (double)E * H;
  const float* const* P = params->p;
  const int scale_in = (flags & PDG_FLAG_SCALE_INPUT) ? 1 : 0;
  const bool ig_node = grad_mean_stress != nullptr || grad_pos != nullptr, ig_edge = grad_edge_attr != nullptr;
  if (set_smem((const void*)k_decoder_vjp, SMEM_V2T)) return -2;
  if (set_smem((const void*)k_node_update_vjp, SMEM_V2T)) return -2;
  if (set_smem((const void*)k_edge_step_vjp, SMEM_B3T)) return -2;
  if (set_smem((const void*)k_node_pre_vjp, SMEM_V2T)) return -2;
  if (set_smem((const void*)k_encoder_vjp<1>, SMEM_V2T)) return -2;
  if (set_smem((const void*)k_encoder_vjp<0>, SMEM_V2T)) return -2;
  auto scal = [&](int slot) { return V.scal + slot * 4; };
  const dim3 gn(grid_n, K);

  {
    ScopedTimer tm_(KC_VJP_DECODER, st);
    const int* nzf = (flags & PDG_FLAG_ZERO_CHECK) ? W.nzflag : nullptr;
    const float gscale = (flags & PDG_FLAG_SCALE_OUTPUT) ? norm->std_local_stress : 1.f;
    k_decoder_vjp<<<gn, NT, SMEM_V2T, st>>>(grad_local_stress, gscale, W.hd, W.y3_[T - 1], W.parts_slot(slot_ln3(T - 1)), cnt_n,
                                            P[ND_W0], P[ND_W2], V.gx, V.cs3, nzf, N, nt_n, cws);
  }
  PDG_LAUNCH_CHECK();
  // receiver-side segment sums RA / RB (adjacent) of every cotangent start from zero: one strided memset
  PDG_CUDA_CHECK(cudaMemset2DAsync(V.RA, cws, 0, 2 * (size_t)W.N_pad * H * sizeof(float), K, st));
  for (int t = T - 1; t >= 0; --t) {
    const bool last = t == T - 1;
    {
      ScopedTimer tm_(KC_VJP_LN_FIN, st);
      LnFinArgs f3{V.cs3, grid_n, W.parts_slot(slot_ln3(t)), cnt_n, P[PN_LNW], scal(slot_ln3(t)), nullptr, nullptr};
      k_ln_finalize_vjp<<<dim3(1, K), FIN_G * H, 0, st>>>(f3, f3, cws);
    }
    PDG_LAUNCH_CHECK();
    const BwdStepArgs s = bwd_step_args(W, P, V, recv, send, rowptr, sptr, slist, t);
    {
      ScopedTimer tm_(KC_VJP_NODE_UPD, st);
      k_node_update_vjp<<<gn, NT, SMEM_V2T, st>>>(s.u, cws);
    }
    PDG_LAUNCH_CHECK();
    {
      ScopedTimer tm_(KC_VJP_LN_FIN, st);
      LnFinArgs f1{V.cs1, grid_n, W.parts_slot(slot_ln1(t)), cnt_e, P[PE_LNW], scal(slot_ln1(t)), nullptr, nullptr};
      LnFinArgs f2 = f1;
      if (!last) f2 = LnFinArgs{V.cs2, grid_e, W.parts_slot(slot_ln2(t)), cnt_e, P[PE_LNW], scal(slot_ln2(t)), nullptr, nullptr};
      k_ln_finalize_vjp<<<dim3(last ? 1 : 2, K), FIN_G * H, 0, st>>>(f1, f2, cws);
    }
    PDG_LAUNCH_CHECK();
    const EdgeVjpArgs v{s.e, V.eacc, cws, K, C};
    {
      ScopedTimer tm_(KC_VJP_EDGE_STEP, st);
      k_edge_step_vjp<<<dim3(grid_e, groups), NT, SMEM_B3T, st>>>(v);
    }
    PDG_LAUNCH_CHECK();
    {
      ScopedTimer tm_(KC_VJP_NODE_PRE, st);
      k_node_pre_vjp<<<gn, NT, SMEM_V2T, st>>>(s.n, cws);
    }
    PDG_LAUNCH_CHECK();
  }
  // encoders: x_0 = LN(y_nenc), e_0 = LN(y_eenc)
  {
    ScopedTimer tm_(KC_VJP_LN_FIN, st);
    LnFinArgs fn{V.cs3, grid_n, W.parts_slot(0), cnt_n, P[NE_LNW], scal(0), nullptr, nullptr};
    LnFinArgs fe{V.cs2, grid_e, W.parts_slot(1), cnt_e, P[EE_LNW], scal(1), nullptr, nullptr};
    k_ln_finalize_vjp<<<dim3(2, K), FIN_G * H, 0, st>>>(fn, fe, cws);
  }
  PDG_LAUNCH_CHECK();
  if (ig_node) {
    ScopedTimer tm_(KC_VJP_ENC, st);
    k_encoder_vjp<1><<<gn, NT, SMEM_V2T, st>>>(V.gx, W.y_nenc, scal(0), P[NE_LNW], mean_stress, pos, nodes_types, nullptr, nullptr,
                                               *norm, scale_in, P[NE_W0], P[NE_B0], P[NE_W2], N, nt_n, grad_mean_stress, grad_pos,
                                               cws);
  }
  if (ig_node) PDG_LAUNCH_CHECK();
  if (ig_edge) {
    ScopedTimer tm_(KC_VJP_ENC, st);
    k_encoder_vjp<0><<<dim3(grid_e, K), NT, SMEM_V2T, st>>>(V.ge, W.y_eenc, scal(1), P[EE_LNW], nullptr, nullptr, nullptr, edge_attr,
                                                            perm, *norm, scale_in, P[EE_W0], P[EE_B0], P[EE_W2], E, nt_e,
                                                            grad_edge_attr, nullptr, cws);
  }
  if (ig_edge) PDG_LAUNCH_CHECK();
  return 0;
}
