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
// node kernels, the encoders and the decoder take the cotangent index from blockIdx.y over the x-grid of
// pdg_backward_inputs, so every cotangent fills the same per-CTA column-sum slots.  The edge kernel takes a group of
// cotangents, computes G, both hidden masks and the message y1 once per tile, then loops over the group.  Cotangent k runs
// the data-gradient operations of pdg_backward_inputs in their order, so column k has that call's bits: the
// weight-gradient GEMMs feed none of them.
#include <algorithm>

#include "pdg_bwd.cuh"

namespace pdg {

// cotangent k's copy of a cotangent-workspace buffer (or of an output): p + off bytes; nullptr stays nullptr
template <class T>
__device__ __forceinline__ T* cot_at(T* p, size_t off) {
  return p == nullptr ? p : reinterpret_cast<T*>(reinterpret_cast<uintptr_t>(p) + off);
}

// decoder, node kernels: two tiles + the weight chunks + a [TM][4] (or [TM][8]) row area
constexpr size_t SMEM_V2T = (size_t)(2 * TM * LDS + 2 * BKB * H) * sizeof(float) + TM * 8 * sizeof(float) + 256;

// Per-cotangent data buffers of the adjoint pass: those of BwdWs without the per-CTA gradient slices, plus the edge
// kernel's per-thread column partials of the edge-encoder LayerNorm sums (a CTA runs its tiles once for a whole group of
// cotangents, so each cotangent's running partials leave registers between tiles: [MAXP CTAs][16][NT threads]).
struct VjpWs {
  int64_t N_pad, E_pad;
  char* base;
  size_t total;
  float *gx, *gagg, *RA, *RB, *ge, *DHM, *DHN, *cs1, *cs2, *cs3, *scal, *eacc;
  VjpWs(int64_t n, int64_t e, int steps, void* ws) : base((char*)ws) {
    N_pad = round_up(n, TM);
    E_pad = round_up(e, TM);
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t r = o; o += (size_t)round_up((int64_t)bytes, 256); return (float*)(base + r); };
    const size_t nb = (size_t)N_pad * H * sizeof(float), eb = (size_t)E_pad * H * sizeof(float);
    gx = take(nb); gagg = take(nb); RA = take(nb); RB = take(nb);  // RA, RB adjacent: one memset
    ge = take(eb); DHM = take(eb); DHN = take(eb);
    cs1 = take((size_t)MAXP * 2 * H * sizeof(float));
    cs2 = take((size_t)MAXP * 2 * H * sizeof(float));
    cs3 = take((size_t)MAXP * 2 * H * sizeof(float));
    scal = take((size_t)(2 + 3 * steps) * 4 * sizeof(float));
    eacc = take((size_t)MAXP * 16 * NT * sizeof(float));
    total = o;  // a multiple of 256 bytes: every copy stays aligned
  }
};

// ---- LayerNorm-backward scalars {c1, c2, mu, a} of one or two instances (blockIdx.x) for every cotangent (blockIdx.y) ----
__global__ void __launch_bounds__(FIN_G* H) k_ln_finalize_vjp(LnFinArgs a0, LnFinArgs a1, size_t cws) {
  const LnFinArgs& a = blockIdx.x == 0 ? a0 : a1;
  const size_t off = (size_t)blockIdx.y * cws;
  ln_finalize_body<false>(cot_at(a.cs, off), a.nparts, a.fwd_parts, a.count, a.lnw, cot_at(a.scal_out, off), nullptr, nullptr);
}

// ---- decoder: gx_T = ([hd > 0] (g D2)) D1 ; column sums of the LayerNorm that produced x_T's increment ----------------
__global__ void __launch_bounds__(NT, 1)
k_decoder_vjp(const float* __restrict__ g_out, float gscale, const float* __restrict__ hd, const float* __restrict__ y3_last,
              const double* __restrict__ parts_prev, double count_prev, const float* __restrict__ D1,
              const float* __restrict__ D2, float* __restrict__ gx, float* __restrict__ cs3, const int* __restrict__ nzflag,
              int N, int n_tiles, size_t cws) {
  extern __shared__ __align__(16) float smem[];
  g_out += (size_t)blockIdx.y * N * PDG_OUT;  // [K][N][3]
  gx = cot_at(gx, blockIdx.y * cws);
  cs3 = cot_at(cs3, blockIdx.y * cws);
  float* T0 = smem;
  float* T1 = T0 + TM * LDS;
  float* Ws = T1 + TM * LDS;
  float* gd = Ws + 2 * BKB * H;  // [TM][4]
  const int tid = threadIdx.x, c4 = (tid & 31) * 4;
  const float mu_prev = ln_stat_block(parts_prev, count_prev, gd).mu;
  const bool live = nzflag == nullptr || *nzflag != 0;
  float d2w[3][4];
#pragma unroll
  for (int o = 0; o < 3; ++o)
#pragma unroll
    for (int c = 0; c < 4; ++c) d2w[o][c] = D2[o * H + c4 + c];
  float cgx[8] = {0}, cgy[8] = {0};
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int row0 = tile * TM;
    if (tid < TM) {
      const int row = row0 + tid;
#pragma unroll
      for (int o = 0; o < 3; ++o) gd[tid * 4 + o] = (row < N && live) ? g_out[row * 3 + o] * gscale : 0.f;
    }
    tile_load(T1, hd + (size_t)row0 * H);
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
  colsum_flush(cgx, T0, cs3 + (size_t)blockIdx.x * 2 * H, false);
  colsum_flush(cgy, T0, cs3 + (size_t)blockIdx.x * 2 * H + H, false);
}

// ---- node_update: dhq = [hq > 0] (dy3 V2);  g_agg = dhq V1[:, :128];  gx += dhq V1[:, 128:] -------------------------
__global__ void __launch_bounds__(NT, 1) k_node_update_vjp(NodeUpdBwdArgs a, size_t cws) {
  extern __shared__ __align__(16) float smem[];
  const size_t off = (size_t)blockIdx.y * cws;
  float* const gx = cot_at(a.gx, off);
  float* const gagg = cot_at(a.gagg, off);
  const float* const scal3 = cot_at(a.scal3, off);
  float* const cs1 = cot_at(a.cs1, off);
  float* T0 = smem;
  float* T1 = T0 + TM * LDS;
  float* Ws = T1 + TM * LDS;
  float* smf = Ws + 2 * BKB * H;
  const int tid = threadIdx.x, c4 = (tid & 31) * 4, ty = tid >> 4;
  const LnStat st1 = ln_stat_block(a.parts1, a.count1, smf);
  const float c1 = scal3[0], c2 = scal3[1], mu3 = scal3[2], rstd3 = scal3[3];
  const float4 wn = *reinterpret_cast<const float4*>(a.lnw_n + c4);
  float cg1[8] = {0}, cgy1[8] = {0};
  for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const int row0 = tile * TM;
    const int nvalid = min(TM, a.N - row0);
    // dy3 -> T0 ; hq -> T1
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
          lg[k] = *reinterpret_cast<const float4*>(gx + g);
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
    acc_zero(acc);
    gemm_rowA<BKB>(T0, a.V2, H, acc, Ws, H);  // dhq_pre = dy3 V2 (its first barrier publishes T0 / T1)
    {
      float h[8][8];
      acc_load(h, T1, LDS);
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = h[i][j] > 0.f ? acc[i][j] : 0.f;
    }
    acc_store(acc, T0, LDS);  // dhq
    acc_zero(acc);
    gemm_rowA<BKB>(T0, a.V1, H, acc, Ws, 2 * H);  // g_agg = dhq V1[:, :128]
    acc_store(acc, gagg + (size_t)row0 * H, H);
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
      mt_load(g0, gx + (size_t)row0 * H);
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] += g0[i][j];
    }
    acc_store(acc, gx + (size_t)row0 * H, H);
    __syncthreads();
  }
  colsum_flush(cg1, T0, cs1 + (size_t)blockIdx.x * 2 * H, false);
  colsum_flush(cgy1, T0, cs1 + (size_t)blockIdx.x * 2 * H + H, false);
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
      const float* scal1 = cot_at(a.scal1, off);
      const float c1m = scal1[0], c2m = scal1[1], mu1 = scal1[2], rstd1 = scal1[3];
      const float* gagg = cot_at(a.gagg, off);
      float* ge = cot_at(a.ge, off);
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
      acc_store(acc, cot_at(a.DHM, off) + (size_t)row0 * H, H);
      acc_store(acc, T1, LDS);  // dhm
      __syncthreads();
      tile_segsum_warp<false>(T1, recv_s, seg_row, nseg, a.rowptr, row0, nvalid, cot_at(a.RA, off), seg_dummy, seg_dummy);
      if (!a.last) {
        {
          const float* scal2 = cot_at(a.scal2, off);
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
        acc_store(acc, cot_at(a.DHN, off) + (size_t)row0 * H, H);
        acc_store(acc, T2, LDS);  // dhn
        __syncthreads();
        tile_segsum_warp<false>(T2, recv_s, seg_row, nseg, a.rowptr, row0, nvalid, cot_at(a.RB, off), seg_dummy, seg_dummy);
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
        float* pe = cot_at(v.eacc, off) + (size_t)blockIdx.x * 16 * NT + tid;
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
          float* cs2 = cot_at(a.cs2, off) + (size_t)blockIdx.x * 2 * H;
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

// ---- node_pre: dPa = RA + sum_{send = n} dhn, dPb = RB + sum_{send = n} dhm;  gx += dPa Wa + dPb Wb -------------------
__global__ void __launch_bounds__(NT, 1) k_node_pre_vjp(NodePreBwdArgs a, size_t cws) {
  extern __shared__ __align__(16) float smem[];
  const size_t off = (size_t)blockIdx.y * cws;
  float* const gx = cot_at(a.gx, off);
  float* const RA = cot_at(a.RA, off);
  float* const RB = cot_at(a.RB, off);
  const float* const DHM = cot_at(a.DHM, off);
  const float* const DHN = cot_at(a.DHN, off);
  float* const cs3 = cot_at(a.cs3, off);
  float* T0 = smem;
  float* T1 = T0 + TM * LDS;
  float* Ws = T1 + TM * LDS;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float mu_prev = ln_stat_block(a.parts_prev, a.count_prev, Ws).mu;
  float cgx[8] = {0}, cgy[8] = {0};
  for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const int row0 = tile * TM;
    // the tile's sender lists staged in shared memory (as k_node_pre_bwd)
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
        pa = *reinterpret_cast<const float4*>(RA + (size_t)n * H + lane * 4);
        if (RB) pb = *reinterpret_cast<const float4*>(RB + (size_t)n * H + lane * 4);
        const int k0 = s_ptr[r], k1 = s_ptr[r + 1];
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
              m[j] = __ldcs(reinterpret_cast<const float4*>(DHM + p));
              if (DHN) q[j] = __ldcs(reinterpret_cast<const float4*>(DHN + p));
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
    // RA / RB rows re-zeroed for the next step's segment sums
    for (int rr = 0; rr < TM / 8; ++rr) {
      const int n = row0 + warp * (TM / 8) + rr;
      if (n < a.N) {
        *reinterpret_cast<float4*>(RA + (size_t)n * H + lane * 4) = make_float4(0.f, 0.f, 0.f, 0.f);
        if (RB) *reinterpret_cast<float4*>(RB + (size_t)n * H + lane * 4) = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
    __syncthreads();  // every read of the staged lists in Ws is done before the GEMM streams weights into it
    float acc[8][8];
    acc_zero(acc);
    gemm_rowA<BKB>(T0, a.W0, H, acc, Ws, 3 * H);      // dPa Wa
    gemm_rowA<BKB>(T1, a.W0 + H, H, acc, Ws, 3 * H);  // + dPb Wb
    {
      float g0[8][8];
      mt_load(g0, gx + (size_t)row0 * H);
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] += g0[i][j];
    }
    acc_store(acc, gx + (size_t)row0 * H, H);
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
  colsum_flush(cgx, T0, cs3 + (size_t)blockIdx.x * 2 * H, false);
  colsum_flush(cgy, T0, cs3 + (size_t)blockIdx.x * 2 * H + H, false);
}

// ---- encoders (node: NODE=1, edge: NODE=0): dh0 = [h0 > 0] (dy W2);  dfeat = dh0 W0, un-standardised ------------------
//   node  gi0 = d/d mean_stress [K][N][3], gi1 = d/d pos [K][N][2] (either may be null);
//   edge  gi0 = d/d edge_attr [K][E] at perm[row] (PyG edge order)
template <int NODE>
__global__ void __launch_bounds__(NT, 1)
k_encoder_vjp(const float* __restrict__ g_in, const float* __restrict__ y_raw, const float* __restrict__ scal,
              const float* __restrict__ lnw, const float* __restrict__ mean_stress, const float* __restrict__ pos,
              const int64_t* __restrict__ types, const float* __restrict__ edge_attr, const int32_t* __restrict__ perm,
              pdg_norm_t nrm, int scale_in, const float* __restrict__ W0, const float* __restrict__ b0,
              const float* __restrict__ W2, int R, int n_tiles, float* __restrict__ gi0, float* __restrict__ gi1, size_t cws) {
  extern __shared__ __align__(16) float smem[];
  {
    const size_t off = (size_t)blockIdx.y * cws;
    g_in = cot_at(g_in, off);
    scal = cot_at(scal, off);
    if (gi0 != nullptr) gi0 += (size_t)blockIdx.y * R * (NODE ? 3 : 1);
    if (gi1 != nullptr) gi1 += (size_t)blockIdx.y * R * 2;
  }
  float* T0 = smem;
  float* T1 = T0 + TM * LDS;
  float* Ws = T1 + TM * LDS;
  float* feat = Ws + 2 * BKB * H;  // [TM][8]
  const int tid = threadIdx.x, c4 = (tid & 31) * 4;
  constexpr int NF = NODE ? 6 : 1;
  const float c1 = scal[0], c2 = scal[1], mu = scal[2], rstd = scal[3];
  const float4 w = *reinterpret_cast<const float4*>(lnw + c4);
  float w0[4][NF], bb0[4];
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    bb0[c] = b0[c4 + c];
#pragma unroll
    for (int j = 0; j < NF; ++j) w0[c][j] = W0[(c4 + c) * NF + j];
  }
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
    float acc[8][8];
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
    // dfeat[r] = dh0[r] W0: one warp per row, lane = 4 channels (the arithmetic of k_encoder_bwd<NODE, true>)
    constexpr int NI = NODE ? 5 : 1;  // feature 5 (nodes_types) is an integer input: no gradient
    for (int r = tid >> 5; r < nvalid; r += NT / 32) {
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
    __syncthreads();
  }
}

static int set_smem_v(const void* fn, size_t bytes) {
  cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e != cudaSuccess) { set_error("cudaFuncSetAttribute(%zu B smem): %s", bytes, cudaGetErrorString(e)); return -2; }
  return 0;
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
  const float* pk = W.pack;
  const int scale_in = (flags & PDG_FLAG_SCALE_INPUT) ? 1 : 0;
  const bool ig_node = grad_mean_stress != nullptr || grad_pos != nullptr, ig_edge = grad_edge_attr != nullptr;
  if (set_smem_v((const void*)k_decoder_vjp, SMEM_V2T)) return -2;
  if (set_smem_v((const void*)k_node_update_vjp, SMEM_V2T)) return -2;
  if (set_smem_v((const void*)k_edge_step_vjp, SMEM_B3T)) return -2;
  if (set_smem_v((const void*)k_node_pre_vjp, SMEM_V2T)) return -2;
  if (set_smem_v((const void*)k_encoder_vjp<1>, SMEM_V2T)) return -2;
  if (set_smem_v((const void*)k_encoder_vjp<0>, SMEM_V2T)) return -2;
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
    const bool last = t == T - 1, first = t == 0;
    {
      ScopedTimer tm_(KC_VJP_LN_FIN, st);
      LnFinArgs f3{V.cs3, grid_n, W.parts_slot(slot_ln3(t)), cnt_n, P[PN_LNW], scal(slot_ln3(t)), nullptr, nullptr};
      k_ln_finalize_vjp<<<dim3(1, K), FIN_G * H, 0, st>>>(f3, f3, cws);
    }
    PDG_LAUNCH_CHECK();
    NodeUpdBwdArgs u = {};
    u.gx = V.gx; u.y3 = W.y3_[t]; u.hq = W.hq_[t]; u.aggraw = W.aggraw_[t]; u.x_t = W.x_[t]; u.rowptr = rowptr;
    u.scal3 = scal(slot_ln3(t)); u.lnw_n = P[PN_LNW]; u.parts1 = W.parts_slot(slot_ln1(t)); u.count1 = cnt_e;
    u.lnw_e = P[PE_LNW]; u.lnb_e = P[PE_LNB]; u.V1 = P[PN_W0]; u.V2 = P[PN_W2]; u.gagg = V.gagg;
    u.cs1 = V.cs1; u.N = N; u.n_tiles = nt_n;
    {
      ScopedTimer tm_(KC_VJP_NODE_UPD, st);
      k_node_update_vjp<<<gn, NT, SMEM_V2T, st>>>(u, cws);
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
    EdgeVjpArgs v = {};
    EdgeBwdArgs& e = v.e;
    e.e_t = W.e_[t]; e.Pa = W.Pa_[t]; e.Pb = W.Pb_[t]; e.gagg = V.gagg; e.ge = V.ge;
    e.y2_t = last ? nullptr : W.y2_[t];
    e.yprev = first ? W.y_eenc : W.y2_[t - 1];
    e.parts_prev = W.parts_slot(first ? 1 : slot_ln2(t - 1)); e.count_prev = cnt_e;
    e.recv = recv; e.send = send; e.rowptr = rowptr;
    e.WtE = pk + PackOffsets::PE_WET; e.b1 = P[PE_B0]; e.Wt2 = pk + PackOffsets::PE_W2T; e.b2 = P[PE_B2];
    e.W0 = P[PE_W0]; e.W2 = P[PE_W2]; e.lnw = P[PE_LNW];
    e.scal1 = scal(slot_ln1(t)); e.scal2 = last ? nullptr : scal(slot_ln2(t));
    e.DHM = V.DHM; e.DHN = V.DHN; e.RA = V.RA; e.RB = V.RB; e.cs2 = V.cs2;
    e.E = E; e.n_tiles = nt_e; e.last = last ? 1 : 0;
    v.eacc = V.eacc; v.cws = cws; v.K = K; v.C = C;
    {
      ScopedTimer tm_(KC_VJP_EDGE_STEP, st);
      k_edge_step_vjp<<<dim3(grid_e, groups), NT, SMEM_B3T, st>>>(v);
    }
    PDG_LAUNCH_CHECK();
    NodePreBwdArgs n = {};
    n.gx = V.gx; n.RA = V.RA; n.RB = last ? nullptr : V.RB; n.DHM = V.DHM; n.DHN = last ? nullptr : V.DHN;
    n.sptr = sptr; n.slist = slist; n.x_t = W.x_[t]; n.yprev = first ? W.y_nenc : W.y3_[t - 1];
    n.parts_prev = W.parts_slot(first ? 0 : slot_ln3(t - 1)); n.count_prev = cnt_n; n.W0 = P[PE_W0];
    n.cs3 = V.cs3; n.N = N; n.n_tiles = nt_n;
    {
      ScopedTimer tm_(KC_VJP_NODE_PRE, st);
      k_node_pre_vjp<<<gn, NT, SMEM_V2T, st>>>(n, cws);
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
