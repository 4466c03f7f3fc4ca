// Forward-mode derivative (Jacobian-vector product) of EncodeProcessDecode.forward with respect to its differentiable
// inputs: tan_local_stress = d local_stress / d (mean_stress, pos, edge_attr) . (tangents), fp32 FFMA tiles.
//
// The tangent pass runs after a pdg_forward with PDG_FLAG_SAVE and follows the forward kernel by kernel.  It reads the
// saved primal state (x_t, e_t, y2_t, Pa_t, Pb_t, aggraw_t, hq_t, y3_t, y_nenc, y_eenc, hd, the LayerNorm partials, the
// packed weights, the zero-load flag), recomputes what the forward did not keep (the first-layer masks of the encoders,
// G = e_t We^T + b1, the message y1) and never writes the forward workspace, so a later pdg_backward is unaffected.
//
// One pass carries K tangents (pdg_jvp_batched).  Each has a tangent workspace of the single-tangent layout, one after
// another at a fixed stride.  The node kernels and the encoders take the tangent index from blockIdx.y; the edge kernel
// takes a group of tangents, computes the primal part of a tile once and loops over the group.  Tangent k runs the same
// operations in the same order (same x-grid, so the same partial slot; same GEMMs and masks) as a single-tangent pass.
//
// Tangent rules (every one linear in the tangent):
//   Linear   yd = xd W^T                     (no bias)
//   ReLU     yd = yd_pre * [y > 0]           (mask = primal OUTPUT > 0, as torch's forward AD of relu)
//   graph LayerNorm  (y - mu) r w + b,  r = 1 / (sigma + eps):
//            yd_ln = w [(yd - mud) r - (y - mu) r^2 sigmad],  mud = sum(yd) / count,
//            sigmad = sum((y - mu) yd) / (count sigma)  (0 when sigma = 0)
// The primal statistics are final before the tangent pass starts, so every tangent producer accumulates the CENTRED
// sum sum((y - mu) yd) directly (no cancellation of sum(y yd) / count - mu mud); per-CTA fp64 partials {sum yd,
// sum (y - mu) yd} in the slot layout of the forward's, reduced in a fixed order (bit-reproducible).
// The message LayerNorm is pushed through the receiver sum as in pdg_forward.cu:
//   aggd = w [(aggrawd - deg mud1) r1 - (aggraw - deg mu1) r1^2 sigmad1].
#include <algorithm>

#include "pdg_ws.cuh"

namespace pdg {

constexpr int BKJ = 16;  // weight k-chunk of the edge kernel (three tiles + two chunks fit in 227 KB, as k_edge_step_bwd)
constexpr size_t SMEM_JENC = SMEM_1A + TM * 16 * sizeof(float);
constexpr size_t SMEM_JEDGE = (size_t)(3 * TM * LDS + 2 * BKJ * H) * sizeof(float) + 2 * TM * sizeof(int) + 16 * sizeof(double) +
                              8 * sizeof(float) + 4 * sizeof(unsigned) + TM + 1 + 256;
// per tangent of an edge-kernel group: the LayerNorm tangent statistics {mud, c} and the fp64 partials {t1s, t1c, t2s, t2c}
constexpr size_t SMEM_JEDGE_TAN = 2 * sizeof(float) + 4 * sizeof(double);
static_assert(SMEM_JEDGE + PDG_JVP_MAX_TANGENTS * SMEM_JEDGE_TAN <= 227 * 1024, "edge JVP kernel exceeds shared memory");

// Tangent statistics of one LayerNorm instance: mud and c = r^2 sigmad, from the tangent partials and the primal
// statistics st (ln_stat_block of the same slot).  CTA-wide; sm: >= 2 floats.
struct LnTan { float mud, c; };
// one warp: the reduction of ln_tan_block; lane 0 writes {mud, c} to out
__device__ __forceinline__ void ln_tan_warp(const double* __restrict__ tparts, double count, const LnStat& st, float* out) {
  const int lane = threadIdx.x & 31;
  constexpr int K = (MAXP + 31) / 32;
  double2 v[K];
#pragma unroll
  for (int k = 0; k < K; ++k) {
    const int i = lane + 32 * k;
    v[k] = i < MAXP ? reinterpret_cast<const double2*>(tparts)[i] : make_double2(0.0, 0.0);
  }
  double s = 0, sc = 0;
#pragma unroll
  for (int k = 0; k < K; ++k) { s += v[k].x; sc += v[k].y; }
  s = warp_sum(s);
  sc = warp_sum(sc);
  if (lane == 0) {
    const double sigma = (double)st.sigma, r = (double)st.rstd;
    const double sigd = sigma > 0 ? sc / (count * sigma) : 0.0;
    out[0] = (float)(s / count);
    out[1] = (float)(r * r * sigd);
  }
}
__device__ __forceinline__ LnTan ln_tan_block(const double* __restrict__ tparts, double count, const LnStat& st, float* sm) {
  if (threadIdx.x < 32) ln_tan_warp(tparts, count, st, sm);
  __syncthreads();
  LnTan t;
  t.mud = sm[0];
  t.c = sm[1];
  __syncthreads();
  return t;
}

// w [(yd - mud) r - (y - mu) c]  for four columns
__device__ __forceinline__ float4 ln_tan4(const float4 y, const float4 yd, const LnStat& st, const LnTan& tt, const float4 w) {
  float4 v;
  v.x = ((yd.x - tt.mud) * st.rstd - (y.x - st.mu) * tt.c) * w.x;
  v.y = ((yd.y - tt.mud) * st.rstd - (y.y - st.mu) * tt.c) * w.y;
  v.z = ((yd.z - tt.mud) * st.rstd - (y.z - st.mu) * tt.c) * w.z;
  v.w = ((yd.w - tt.mud) * st.rstd - (y.w - st.mu) * tt.c) * w.w;
  return v;
}

// acc = [y > 0] acc with y the primal ReLU output (global rows, pitch H); s / c accumulate sum(acc) and
// sum((y - mu) acc) over rows < nvalid (tangent LayerNorm partials)
__device__ __forceinline__ void relu_mask_stats(float (&acc)[8][8], const float* __restrict__ y, int ld, float mu, int nvalid,
                                                float& s, float& c) {
  const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int r = ty * 8 + i;
    const float4 u = *reinterpret_cast<const float4*>(y + (size_t)r * ld + tx * 4);
    const float4 v = *reinterpret_cast<const float4*>(y + (size_t)r * ld + 64 + tx * 4);
    const float yy[8] = {u.x, u.y, u.z, u.w, v.x, v.y, v.z, v.w};
    const bool ok = r < nvalid;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float d = yy[j] > 0.f ? acc[i][j] : 0.f;
      acc[i][j] = d;
      if (ok) { s += d; c = fmaf(yy[j] - mu, d, c); }
    }
  }
}

__device__ __forceinline__ void finish_partials(float s, float c, double* red, double& ts, double& tc) {
  double ds = s, dc = c;
  block_sum2(ds, dc, red);
  if (threadIdx.x == 0) { ts += ds; tc += dc; }
}

// ------------------------------------------------------------------------------------
// node encoder: hd0 = [W0 f + b0 > 0] (W0 fd), fd = [msd / std_ms, posd / std_pos, 0];  yd = [y_nenc > 0] (hd0 W2^T)
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(NT, 1)
k_node_encoder_jvp(const float* __restrict__ mean_stress, const float* __restrict__ pos, const int64_t* __restrict__ types,
                   pdg_norm_t nrm, int scale_in, const float* __restrict__ tan_ms, const float* __restrict__ tan_pos,
                   const float* __restrict__ W0, const float* __restrict__ b0, const float* __restrict__ Wt2,
                   const float* __restrict__ y_nenc, const double* __restrict__ parts, double count, float* __restrict__ yd_out,
                   double* __restrict__ tparts, int N, int n_tiles, int64_t ms_stride, int64_t pos_stride, size_t tws) {
  extern __shared__ __align__(16) float smem[];
  if (tan_ms != nullptr) tan_ms += blockIdx.y * ms_stride;
  if (tan_pos != nullptr) tan_pos += blockIdx.y * pos_stride;
  yd_out = copy_at(yd_out, blockIdx.y * tws);
  tparts = copy_at(tparts, blockIdx.y * tws);
  float* A = smem;
  float* Ws = A + TM * LDS;
  float* feat = Ws + 2 * BK * H;  // [TM][8] primal features
  float* featd = feat + TM * 8;   // [TM][8] tangent features
  double* red = (double*)(featd + TM * 8);
  float* smf = (float*)(red + 16);
  const int tid = threadIdx.x;
  const int c4 = (tid & 31) * 4;
  float w0[4][6], bb0[4];
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    bb0[c] = b0[c4 + c];
#pragma unroll
    for (int j = 0; j < 6; ++j) w0[c][j] = W0[(c4 + c) * 6 + j];
  }
  const LnStat st = ln_stat_block(parts, count, smf);
  double tot_s = 0, tot_c = 0;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int row0 = tile * TM;
    const int nvalid = min(TM, N - row0);
    if (tid < TM) {
      const int row = row0 + tid;
      float f[6] = {0, 0, 0, 0, 0, 0}, fd[6] = {0, 0, 0, 0, 0, 0};
      if (row < N) {
        bool nz;
        node_features(mean_stress, pos, types, nrm, scale_in, row, f, nz);  // the forward's features: its first-layer mask
        if (tan_ms != nullptr)
#pragma unroll
          for (int j = 0; j < 3; ++j) fd[j] = scale_in ? tan_ms[row * 3 + j] / nrm.std_mean_stress : tan_ms[row * 3 + j];
        if (tan_pos != nullptr)
#pragma unroll
          for (int j = 0; j < 2; ++j) fd[3 + j] = scale_in ? tan_pos[row * 2 + j] / nrm.std_pos : tan_pos[row * 2 + j];
      }
#pragma unroll
      for (int j = 0; j < 6; ++j) { feat[tid * 8 + j] = f[j]; featd[tid * 8 + j] = fd[j]; }
    }
    __syncthreads();
#pragma unroll 2
    for (int it = 0; it < (TM * H / 4) / NT; ++it) {
      const int r = (tid >> 5) + it * 8;
      float v[4];
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        float a = bb0[c], d = 0.f;
#pragma unroll
        for (int j = 0; j < 6; ++j) {
          a = fmaf(w0[c][j], feat[r * 8 + j], a);
          d = fmaf(w0[c][j], featd[r * 8 + j], d);
        }
        v[c] = a > 0.f ? d : 0.f;
      }
      *reinterpret_cast<float4*>(A + r * LDS + c4) = make_float4(v[0], v[1], v[2], v[3]);
    }
    float acc[8][8];
    acc_zero(acc);
    gemm_rowA(A, Wt2, H, acc, Ws);
    float s = 0, c = 0;
    relu_mask_stats(acc, y_nenc + (size_t)row0 * H, H, st.mu, nvalid, s, c);
    acc_store(acc, yd_out + (size_t)row0 * H, H);
    finish_partials(s, c, red, tot_s, tot_c);
  }
  if (tid == 0) { tparts[2 * blockIdx.x] = tot_s; tparts[2 * blockIdx.x + 1] = tot_c; }
}

// ------------------------------------------------------------------------------------
// edge encoder: hd0 = [w0 a + b0 > 0] w0 ad with ad = tan_edge_attr[perm[row]] / std_ew;  yd = [y_eenc > 0] (hd0 W2^T)
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(NT, 1)
k_edge_encoder_jvp(const float* __restrict__ edge_attr, const int32_t* __restrict__ perm, pdg_norm_t nrm, int scale_in,
                   const float* __restrict__ tan_ea, const float* __restrict__ W0, const float* __restrict__ b0,
                   const float* __restrict__ Wt2, const float* __restrict__ y_eenc, const double* __restrict__ parts,
                   double count, float* __restrict__ yd_out, double* __restrict__ tparts, int E, int n_tiles,
                   int64_t ea_stride, size_t tws) {
  extern __shared__ __align__(16) float smem[];
  if (tan_ea != nullptr) tan_ea += blockIdx.y * ea_stride;
  yd_out = copy_at(yd_out, blockIdx.y * tws);
  tparts = copy_at(tparts, blockIdx.y * tws);
  float* A = smem;
  float* Ws = A + TM * LDS;
  float* feat = Ws + 2 * BK * H;  // [TM]
  float* featd = feat + TM;       // [TM]
  double* red = (double*)(feat + TM * 16);
  float* smf = (float*)(red + 16);
  const int tid = threadIdx.x;
  const int c4 = (tid & 31) * 4;
  const float4 w0 = *reinterpret_cast<const float4*>(W0 + c4);
  const float4 bb0 = *reinterpret_cast<const float4*>(b0 + c4);
  const LnStat st = ln_stat_block(parts, count, smf);
  double tot_s = 0, tot_c = 0;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int row0 = tile * TM;
    const int nvalid = min(TM, E - row0);
    if (tid < TM) {
      float a = 0.f, ad = 0.f;
      if (row0 + tid < E) {
        const int src = perm[row0 + tid];
        a = edge_feature(edge_attr[src], nrm, scale_in);
        if (tan_ea != nullptr) ad = scale_in ? tan_ea[src] / nrm.std_edge_weight : tan_ea[src];
      }
      feat[tid] = a;
      featd[tid] = ad;
    }
    __syncthreads();
#pragma unroll 4
    for (int it = 0; it < (TM * H / 4) / NT; ++it) {
      const int r = (tid >> 5) + it * 8;
      const float a = feat[r], ad = featd[r];
      *reinterpret_cast<float4*>(A + r * LDS + c4) =
          make_float4(fmaf(w0.x, a, bb0.x) > 0.f ? w0.x * ad : 0.f, fmaf(w0.y, a, bb0.y) > 0.f ? w0.y * ad : 0.f,
                      fmaf(w0.z, a, bb0.z) > 0.f ? w0.z * ad : 0.f, fmaf(w0.w, a, bb0.w) > 0.f ? w0.w * ad : 0.f);
    }
    float acc[8][8];
    acc_zero(acc);
    gemm_rowA(A, Wt2, H, acc, Ws);
    float s = 0, c = 0;
    relu_mask_stats(acc, y_eenc + (size_t)row0 * H, H, st.mu, nvalid, s, c);
    acc_store(acc, yd_out + (size_t)row0 * H, H);
    finish_partials(s, c, red, tot_s, tot_c);
  }
  if (tid == 0) { tparts[2 * blockIdx.x] = tot_s; tparts[2 * blockIdx.x + 1] = tot_c; }
}

// ------------------------------------------------------------------------------------
// node_pre: xd_t = xd_{t-1} + LN-tangent(y_prev, yd_prev);  Pad = xd_t Wa^T,  Pbd = xd_t Wb^T
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(NT, 1)
k_node_pre_jvp(const float* __restrict__ yprev, const double* __restrict__ prev_parts, const double* __restrict__ tprev_parts,
               double prev_count, const float* __restrict__ lnw, const float* __restrict__ tbase,
               const float* __restrict__ typrev, float* __restrict__ tx_out, const float* __restrict__ WtA,
               const float* __restrict__ WtB, float* __restrict__ tPa, float* __restrict__ tPb, int n_tiles, size_t tws) {
  extern __shared__ __align__(16) float smem[];
  {
    const size_t off = blockIdx.y * tws;
    tprev_parts = copy_at(tprev_parts, off);
    tbase = copy_at(tbase, off);
    typrev = copy_at(typrev, off);
    tx_out = copy_at(tx_out, off);
    tPa = copy_at(tPa, off);
    tPb = copy_at(tPb, off);
  }
  float* A = smem;
  float* Ws = A + TM * LDS;
  float* smf = Ws + 2 * BK * H;
  const int tid = threadIdx.x;
  const int c4 = (tid & 31) * 4;
  const LnStat st = ln_stat_block(prev_parts, prev_count, smf);
  const LnTan tt = ln_tan_block(tprev_parts, prev_count, st, smf);
  const float4 w = *reinterpret_cast<const float4*>(lnw + c4);
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const size_t row0 = (size_t)tile * TM;
#pragma unroll
    for (int bt = 0; bt < 4; ++bt) {
      float4 ly[4], ld[4], lx[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const size_t g = (row0 + (tid >> 5) + (bt * 4 + k) * 8) * H + c4;
        ly[k] = *reinterpret_cast<const float4*>(yprev + g);
        ld[k] = *reinterpret_cast<const float4*>(typrev + g);
        lx[k] = tbase != nullptr ? *reinterpret_cast<const float4*>(tbase + g) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int r = (tid >> 5) + (bt * 4 + k) * 8;
        float4 v = ln_tan4(ly[k], ld[k], st, tt, w);
        v.x += lx[k].x; v.y += lx[k].y; v.z += lx[k].z; v.w += lx[k].w;
        *reinterpret_cast<float4*>(tx_out + (row0 + r) * H + c4) = v;
        *reinterpret_cast<float4*>(A + r * LDS + c4) = v;
      }
    }
    float acc[8][8];
    acc_zero(acc);
    gemm_rowA(A, WtA, H, acc, Ws);
    acc_store(acc, tPa + row0 * H, H);
    acc_zero(acc);
    gemm_rowA(A, WtB, H, acc, Ws);
    acc_store(acc, tPb + row0 * H, H);
  }
}

// ------------------------------------------------------------------------------------
// edge_step: one Processor step of the tangent on a tile of 128 receiver-sorted edges
//   ed_t  = ed_{t-1} + LN-tangent(y2_{t-1})                      (lazy; written in place)
//   G     = e_t We^T + b1,  Gd = ed_t We^T                         (G only for the hidden masks and y1)
//   m1 = [G + Pa[recv] + Pb[send] > 0],  m2 = [G + Pa[send] + Pb[recv] > 0]      (register bits)
//   y1    = relu(relu(G + Pa[recv] + Pb[send]) W2^T + b2)          (recomputed: the forward keeps its segment sums only)
//   y1d   = [y1 > 0] ((m1 (Gd + Pad[recv] + Pbd[send])) W2^T)    -> segment sums into aggrawd, partials LN1
//   y2d   = [y2_t > 0] ((m2 (Gd + Pad[send] + Pbd[recv])) W2^T)  -> in place over yd_prev, partials LN2 (not on the last step)
// A CTA takes a group of C tangents: the primal part (G, both masks, y1) runs once per tile, then each tangent of the
// group runs Gd, y1d and y2d.
// Tiles: T0 e_t -> h1 -> y1 (kept for the whole group);  T1 G, then per tangent h1d -> y1d -> h2d;  T2 ed_t -> Gd.
// Two GEMMs per tile plus three per tangent, against the forward's three.
// ------------------------------------------------------------------------------------
struct EdgeJvpArgs {
  // primal state (forward workspace)
  const float* yprev;
  const double* prev_parts;
  const float* prev_w;
  const float* e_t;
  const float* Pa;
  const float* Pb;
  const float* y2_t;  // nullptr on the last step
  const double* parts1;
  const double* parts2;
  // tangent state
  const double* tprev_parts;
  const float* tbase;  // ed_{t-1} (nullptr at t = 0); same buffer as te_out
  const float* typrev; // same buffer as ty2_out
  float* te_out;
  const float* tPa;
  const float* tPb;
  float* ty2_out;
  float* taggraw;
  double* tparts1;
  double* tparts2;
  const int32_t* recv;
  const int32_t* send;
  const int32_t* rowptr;
  const float* WtE;
  const float* b1;
  const float* Wt2;
  const float* b2;
  double count;
  int E, n_tiles;
  size_t tws;  // bytes between consecutive tangent workspaces
  int K, C;    // tangents of the pass; tangents per CTA group (blockIdx.y = group)
};

// acc = m (Gd + P1d[idx1[row]] + P2d[idx2[row]]), bit i*8+j of m = mask of micro-tile element (i, j)
__device__ __forceinline__ void gather_hidden_tan(float (&acc)[8][8], const float* __restrict__ Gd, const float* __restrict__ P1,
                                                  const int* __restrict__ idx1, const float* __restrict__ P2,
                                                  const int* __restrict__ idx2, unsigned long long m) {
  const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int r = ty * 8 + i;
    const float* p1 = P1 + (size_t)idx1[r] * H + tx * 4;
    const float* p2 = P2 + (size_t)idx2[r] * H + tx * 4;
    const float4 a0 = *reinterpret_cast<const float4*>(p1);
    const float4 a1 = *reinterpret_cast<const float4*>(p1 + 64);
    const float4 c0 = *reinterpret_cast<const float4*>(p2);
    const float4 c1 = *reinterpret_cast<const float4*>(p2 + 64);
    const float4 g0 = *reinterpret_cast<const float4*>(Gd + r * LDS + tx * 4);
    const float4 g1 = *reinterpret_cast<const float4*>(Gd + r * LDS + 64 + tx * 4);
    const float v[8] = {g0.x + a0.x + c0.x, g0.y + a0.y + c0.y, g0.z + a0.z + c0.z, g0.w + a0.w + c0.w,
                        g1.x + a1.x + c1.x, g1.y + a1.y + c1.y, g1.z + a1.z + c1.z, g1.w + a1.w + c1.w};
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = (m >> (i * 8 + j)) & 1ull ? v[j] : 0.f;
  }
}
__device__ __forceinline__ unsigned long long pos_bits(const float (&acc)[8][8]) {
  unsigned long long m = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) m |= (unsigned long long)(acc[i][j] > 0.f) << (i * 8 + j);
  return m;
}

// ed_t = ed_{t-1} + LN-tangent(y2_{t-1}) of one tangent (workspace offset off, statistics tt2 = {mud, c}) on the tile's
// rows -> T2, and to te_out (in place over ed_{t-1}) when the next step reads it
__device__ __forceinline__ void load_ed(const EdgeJvpArgs& a, const LnStat& st, const float* tt2, const float4 w, int row0,
                                        size_t off, float* T2) {
  const int tid = threadIdx.x;
  const int c4 = (tid & 31) * 4;
  LnTan tt;
  tt.mud = tt2[0];
  tt.c = tt2[1];
  const float* tbase = copy_at(a.tbase, off);
  const float* typrev = copy_at(a.typrev, off);
  float* te_out = copy_at(a.te_out, off);
#pragma unroll
  for (int bt = 0; bt < 4; ++bt) {
    float4 ly[4], ld[4], lx[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const size_t g = ((size_t)row0 + (tid >> 5) + (bt * 4 + k) * 8) * H + c4;
      ly[k] = *reinterpret_cast<const float4*>(a.yprev + g);
      ld[k] = *reinterpret_cast<const float4*>(typrev + g);
      lx[k] = tbase != nullptr ? *reinterpret_cast<const float4*>(tbase + g) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int r = (tid >> 5) + (bt * 4 + k) * 8;
      const size_t g = ((size_t)row0 + r) * H + c4;
      float4 v = ln_tan4(ly[k], ld[k], st, tt, w);
      v.x += lx[k].x; v.y += lx[k].y; v.z += lx[k].z; v.w += lx[k].w;
      if (te_out != nullptr) *reinterpret_cast<float4*>(te_out + g) = v;
      *reinterpret_cast<float4*>(T2 + r * LDS + c4) = v;
    }
  }
}

__global__ void __launch_bounds__(NT, 1) k_edge_step_jvp(EdgeJvpArgs a) {
  extern __shared__ __align__(16) float smem[];
  float* T0 = smem;
  float* T1 = T0 + TM * LDS;
  float* T2 = T1 + TM * LDS;
  float* Ws = T2 + TM * LDS;
  int* recv_s = (int*)(Ws + 2 * BKJ * H);
  int* send_s = recv_s + TM;
  double* red = (double*)(send_s + TM);
  float* smf = (float*)(red + 16);
  unsigned* seg_masks = (unsigned*)(smf + 8);
  unsigned char* seg_row = (unsigned char*)(seg_masks + 4);  // [TM + 1]
  // per tangent of the group (SMEM_JEDGE_TAN each, above the 16-byte-aligned end of seg_row)
  double* tsum = (double*)(((uintptr_t)(seg_row + TM + 1) + 15) & ~(uintptr_t)15);  // [C][4] {t1s, t1c, t2s, t2c}
  float* ttan = (float*)(tsum + 4 * a.C);                                           // [C][2] {mud, c}
  const int tid = threadIdx.x;
  const int c4 = (tid & 31) * 4;
  const bool upd = a.ty2_out != nullptr;
  const int k0 = blockIdx.y * a.C, nk = min(a.C, a.K - k0);  // this CTA's tangents: k0 .. k0 + nk - 1
  const LnStat st = ln_stat_block(a.prev_parts, a.count, smf);
  for (int c = tid >> 5; c < nk; c += NT / 32) ln_tan_warp(copy_at(a.tprev_parts, (k0 + c) * a.tws), a.count, st, ttan + 2 * c);
  for (int i = tid; i < 4 * nk; i += NT) tsum[i] = 0.0;
  const float mu1 = ln_stat_block(a.parts1, a.count, smf).mu;  // its barriers publish ttan and tsum
  const float mu2 = upd ? ln_stat_block(a.parts2, a.count, smf).mu : 0.f;
  const float4 w = *reinterpret_cast<const float4*>(a.prev_w + c4);
  for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const int row0 = tile * TM;
    const int nvalid = min(TM, a.E - row0);
    if (tid < TM) {
      recv_s[tid] = a.recv[row0 + tid];
      send_s[tid] = a.send[row0 + tid];
    }
    // ---- primal part, once per tile for the whole group: G = e_t We^T + b1 -> T1, masks, y1 -> T0.  e_t arrives in
    // T0 asynchronously while the group's first ed_t goes to T2 (the primal part does not touch T2) ----
#pragma unroll
    for (int it = 0; it < (TM * H / 4) / NT; ++it) {
      const int r = (tid >> 5) + it * 8;
      cp_async16(T0 + r * LDS + c4, a.e_t + ((size_t)row0 + r) * H + c4);
    }
    cp_async_commit();
    load_ed(a, st, ttan, w, row0, (size_t)k0 * a.tws, T2);
    cp_async_wait<0>();
    __syncthreads();  // recv_s/send_s, T0, T2 visible
    const int nseg = tile_segments(recv_s, nvalid, seg_row, seg_masks);
    float acc[8][8];
    acc_zero(acc);
    gemm_rowA<BKJ>(T0, a.WtE, H, acc, Ws);
    {
      float bias1[8];  // biases are loaded where they are used: kept live across the GEMMs they cost a spill
      load_cols(bias1, a.b1);
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] += bias1[j];
    }
    acc_store(acc, T1, LDS);
    __syncthreads();  // T1 visible
    unsigned long long m2 = 0;
    if (upd) {
      gather_hidden(acc, T1, a.Pa, send_s, a.Pb, recv_s);  // the forward's: its masks
      m2 = pos_bits(acc);
    }
    gather_hidden(acc, T1, a.Pa, recv_s, a.Pb, send_s);
    const unsigned long long m1 = pos_bits(acc);
    acc_store(acc, T0, LDS);
    acc_zero(acc);
    gemm_rowA<BKJ>(T0, a.Wt2, H, acc, Ws);
    {
      float bias2[8];
      load_cols(bias2, a.b2);
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaxf(acc[i][j] + bias2[j], 0.f);
    }
    acc_store(acc, T0, LDS);  // y1 stays in T0 until the group's last tangent; G in T1 is dead (masks are in registers)
    // ---- tangents of the group ----
    for (int c = 0; c < nk; ++c) {
      const size_t off = (size_t)(k0 + c) * a.tws;
      if (c > 0) load_ed(a, st, ttan + 2 * c, w, row0, off, T2);
      // ---- Gd = ed_t We^T -> T2 (ed_t of tangent 0 was loaded with e_t) ----
      acc_zero(acc);
      gemm_rowA<BKJ>(T2, a.WtE, H, acc, Ws);  // its first barrier also makes y1 in T0 visible
      acc_store(acc, T2, LDS);
      __syncthreads();  // T2 visible
      // ---- h1d -> T1 ----
      const float* tPa = copy_at(a.tPa, off);
      const float* tPb = copy_at(a.tPb, off);
      gather_hidden_tan(acc, T2, tPa, recv_s, tPb, send_s, m1);
      acc_store(acc, T1, LDS);
      acc_zero(acc);
      gemm_rowA<BKJ>(T1, a.Wt2, H, acc, Ws);
      {
        float s = 0.f, cc = 0.f;
        relu_mask_stats(acc, T0, LDS, mu1, nvalid, s, cc);  // y1d, partials of LN1
        acc_store(acc, T1, LDS);
        __syncthreads();
        float u0 = 0.f, u1 = 0.f;
        tile_segsum_warp<false>(T1, recv_s, seg_row, nseg, a.rowptr, row0, nvalid, copy_at(a.taggraw, off), u0, u1);
        finish_partials(s, cc, red, tsum[4 * c], tsum[4 * c + 1]);  // its barriers also end every read of T1
      }
      // ---- edge-update tangent (skipped on the last step, as in the forward); h2d -> T1, T0 keeps y1 ----
      if (upd) {
        gather_hidden_tan(acc, T2, tPa, send_s, tPb, recv_s, m2);
        acc_store(acc, T1, LDS);
        acc_zero(acc);
        gemm_rowA<BKJ>(T1, a.Wt2, H, acc, Ws);
        float s = 0.f, cc = 0.f;
        relu_mask_stats(acc, a.y2_t + (size_t)row0 * H, H, mu2, nvalid, s, cc);
        acc_store(acc, copy_at(a.ty2_out, off) + (size_t)row0 * H, H);
        finish_partials(s, cc, red, tsum[4 * c + 2], tsum[4 * c + 3]);
      }
      __syncthreads();
    }
  }
  if (tid == 0) {
    for (int c = 0; c < nk; ++c) {
      const size_t off = (size_t)(k0 + c) * a.tws;
      double* p1 = copy_at(a.tparts1, off);
      p1[2 * blockIdx.x] = tsum[4 * c];
      p1[2 * blockIdx.x + 1] = tsum[4 * c + 1];
      if (a.tparts2 != nullptr) {
        double* p2 = copy_at(a.tparts2, off);
        p2[2 * blockIdx.x] = tsum[4 * c + 2];
        p2[2 * blockIdx.x + 1] = tsum[4 * c + 3];
      }
    }
  }
}

// ------------------------------------------------------------------------------------
// node_update: aggd = w1 [(aggrawd - deg mud1) r1 - (aggraw - deg mu1) c1]
//   hqd = [hq > 0] ([aggd, xd_t] V1^T);  y3d = [y3 > 0] (hqd V2^T)  + partials LN3
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(NT, 1)
k_node_update_jvp(const float* __restrict__ aggraw, const float* __restrict__ taggraw, const int32_t* __restrict__ rowptr,
                  const double* __restrict__ parts1, const double* __restrict__ tparts1, double count1,
                  const float* __restrict__ lnw_e, const float* __restrict__ tx_t, const float* __restrict__ WtA,
                  const float* __restrict__ WtX, const float* __restrict__ hq, const float* __restrict__ Wt2,
                  const float* __restrict__ y3, const double* __restrict__ parts3, double count3, float* __restrict__ ty3_out,
                  double* __restrict__ tparts3, int N, int n_tiles, size_t tws) {
  extern __shared__ __align__(16) float smem[];
  {
    const size_t off = blockIdx.y * tws;
    taggraw = copy_at(taggraw, off);
    tparts1 = copy_at(tparts1, off);
    tx_t = copy_at(tx_t, off);
    ty3_out = copy_at(ty3_out, off);
    tparts3 = copy_at(tparts3, off);
  }
  float* A0 = smem;
  float* A1 = A0 + TM * LDS;
  float* Ws = A1 + TM * LDS;
  double* red = (double*)(Ws + 2 * BK * H);
  float* smf = (float*)(red + 16);
  const int tid = threadIdx.x;
  const int c4 = (tid & 31) * 4;
  const LnStat st = ln_stat_block(parts1, count1, smf);
  const LnTan tt = ln_tan_block(tparts1, count1, st, smf);
  const float mu3 = ln_stat_block(parts3, count3, smf).mu;
  const float4 w = *reinterpret_cast<const float4*>(lnw_e + c4);
  double tot_s = 0, tot_c = 0;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int row0 = tile * TM;
    const int nvalid = min(TM, N - row0);
#pragma unroll
    for (int it = 0; it < (TM * H / 4) / NT; ++it) {  // xd_t rows straight into A1
      const int r = (tid >> 5) + it * 8;
      cp_async16(A1 + r * LDS + c4, tx_t + ((size_t)row0 + r) * H + c4);
    }
    cp_async_commit();
#pragma unroll
    for (int bt = 0; bt < 4; ++bt) {
      float4 ls[4], ld[4];
      float ldeg[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int row = row0 + (tid >> 5) + (bt * 4 + k) * 8;
        ldeg[k] = row < N ? (float)(rowptr[row + 1] - rowptr[row]) : 0.f;
        ls[k] = *reinterpret_cast<const float4*>(aggraw + (size_t)row * H + c4);
        ld[k] = *reinterpret_cast<const float4*>(taggraw + (size_t)row * H + c4);
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int r = (tid >> 5) + (bt * 4 + k) * 8;
        const float deg = ldeg[k], dm = deg * st.mu, dmd = deg * tt.mud;
        const float4 s4 = ls[k], d4 = ld[k];
        float4 v;
        v.x = ((d4.x - dmd) * st.rstd - (s4.x - dm) * tt.c) * w.x;
        v.y = ((d4.y - dmd) * st.rstd - (s4.y - dm) * tt.c) * w.y;
        v.z = ((d4.z - dmd) * st.rstd - (s4.z - dm) * tt.c) * w.z;
        v.w = ((d4.w - dmd) * st.rstd - (s4.w - dm) * tt.c) * w.w;
        *reinterpret_cast<float4*>(A0 + r * LDS + c4) = v;
      }
    }
    cp_async_wait<0>();  // gemm_rowA's first barrier makes A0 / A1 visible
    float acc[8][8];
    acc_zero(acc);
    gemm_rowA(A0, WtA, H, acc, Ws);
    gemm_rowA(A1, WtX, H, acc, Ws);
    float s = 0, c = 0;
    relu_mask_stats(acc, hq + (size_t)row0 * H, H, 0.f, 0, s, c);  // hqd (no statistics: nvalid 0)
    acc_store(acc, A0, LDS);
    acc_zero(acc);
    gemm_rowA(A0, Wt2, H, acc, Ws);
    relu_mask_stats(acc, y3 + (size_t)row0 * H, H, mu3, nvalid, s, c);
    acc_store(acc, ty3_out + (size_t)row0 * H, H);
    finish_partials(s, c, red, tot_s, tot_c);
  }
  if (tid == 0) { tparts3[2 * blockIdx.x] = tot_s; tparts3[2 * blockIdx.x + 1] = tot_c; }
}

// ------------------------------------------------------------------------------------
// decoder: xd_T = xd_{T-1} + LN-tangent(y3_{T-1});  hdd = [hd > 0] (xd_T Wd^T);  outd = (hdd D2^T) out_scale,
// exactly 0 when the zero-load flag is clear (the reference's early exit returns constant zeros)
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(NT, 1)
k_decoder_jvp(const float* __restrict__ yprev, const double* __restrict__ prev_parts, const double* __restrict__ tprev_parts,
              double prev_count, const float* __restrict__ lnw, const float* __restrict__ tbase,
              const float* __restrict__ typrev, const float* __restrict__ WtD, const float* __restrict__ hd,
              const float* __restrict__ D2, float out_scale, float* __restrict__ tout, const int* __restrict__ nzflag, int N,
              int n_tiles, size_t tws) {
  extern __shared__ __align__(16) float smem[];
  {
    const size_t off = blockIdx.y * tws;
    tprev_parts = copy_at(tprev_parts, off);
    tbase = copy_at(tbase, off);
    typrev = copy_at(typrev, off);
    tout += (size_t)blockIdx.y * N * PDG_OUT;  // [K][N][3]
  }
  float* A = smem;
  float* Ws = A + TM * LDS;
  float* smf = Ws + 2 * BK * H;
  const int tid = threadIdx.x;
  const int c4 = (tid & 31) * 4;
  const LnStat st = ln_stat_block(prev_parts, prev_count, smf);
  const LnTan tt = ln_tan_block(tprev_parts, prev_count, st, smf);
  const float4 w = *reinterpret_cast<const float4*>(lnw + c4);
  const bool live = nzflag == nullptr || *nzflag != 0;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const size_t row0 = (size_t)tile * TM;
#pragma unroll 4
    for (int it = 0; it < (TM * H / 4) / NT; ++it) {
      const int r = (tid >> 5) + it * 8;
      const size_t g = (row0 + r) * H + c4;
      float4 v = ln_tan4(*reinterpret_cast<const float4*>(yprev + g), *reinterpret_cast<const float4*>(typrev + g), st, tt, w);
      const float4 x0 = *reinterpret_cast<const float4*>(tbase + g);
      v.x += x0.x; v.y += x0.y; v.z += x0.z; v.w += x0.w;
      *reinterpret_cast<float4*>(A + r * LDS + c4) = v;
    }
    float acc[8][8];
    acc_zero(acc);
    gemm_rowA(A, WtD, H, acc, Ws);
    float s = 0, c = 0;
    relu_mask_stats(acc, hd + row0 * H, H, 0.f, 0, s, c);
    acc_store(acc, A, LDS);
    __syncthreads();
    for (int idx = tid; idx < TM * PDG_OUT; idx += NT) {
      const int r = idx / PDG_OUT, o = idx - r * PDG_OUT;
      const size_t row = row0 + r;
      if (row < (size_t)N) {
        float dsum = 0.f;
        const float* ar = A + r * LDS;
        const float* wr = D2 + o * H;
#pragma unroll 8
        for (int k = 0; k < H; ++k) dsum = fmaf(ar[k], __ldg(wr + k), dsum);
        tout[row * PDG_OUT + o] = live ? dsum * out_scale : 0.f;
      }
    }
    __syncthreads();
  }
}

}  // namespace pdg

using namespace pdg;

// The tangent workspace has the buffers of a forward without PDG_FLAG_SAVE: ping-pong xd, Pad, Pbd, aggrawd, y3d,
// ed updated in place, y2d over yd_eenc; its LayerNorm partials hold the tangent partials.  A batched pass keeps K of
// them one after another (the total is a multiple of 256 bytes, so every copy stays aligned).
extern "C" size_t pdg_jvp_ws_bytes(int64_t n_nodes, int64_t n_edges, int steps) {
  if (steps < 1 || steps > 62) return 0;
  return FwdWs(n_nodes, n_edges, steps, false, nullptr, false).total;
}

extern "C" size_t pdg_jvp_batched_ws_bytes(int64_t n_nodes, int64_t n_edges, int steps, int n_tangents) {
  if (n_tangents < 1 || n_tangents > PDG_JVP_MAX_TANGENTS) return 0;
  return (size_t)n_tangents * pdg_jvp_ws_bytes(n_nodes, n_edges, steps);
}

extern "C" int pdg_jvp_batched(const pdg_params_t* params, const pdg_norm_t* norm, const float* mean_stress, const float* pos,
                               const int64_t* nodes_types, const float* edge_attr, const void* plan, int64_t n_nodes,
                               int64_t n_edges, int steps, int flags, int precision, const void* fwd_ws, void* jvp_ws,
                               size_t jvp_ws_bytes, int n_tangents, const float* tan_mean_stress, int64_t ms_stride,
                               const float* tan_pos, int64_t pos_stride, const float* tan_edge_attr, int64_t ea_stride,
                               float* tan_local_stress, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  const int K = n_tangents;
  if (K < 1 || K > PDG_JVP_MAX_TANGENTS) {
    set_error("pdg_jvp_batched: n_tangents=%d outside 1..%d", K, PDG_JVP_MAX_TANGENTS);
    return -1;
  }
  if (steps < 1 || steps > 62) { set_error("pdg_jvp: steps=%d unsupported", steps); return -1; }
  if (precision != PDG_PREC_FP32) {
    set_error("pdg_jvp: only the fp32 mode (PDG_PREC_FP32) has a forward-mode derivative; the 16-bit mode's per-row "
              "derivatives miss its 2e-2 tolerance");
    return -1;
  }
  if (!(flags & PDG_FLAG_SAVE)) { set_error("pdg_jvp: the forward workspace must come from a pdg_forward with PDG_FLAG_SAVE"); return -1; }
  if (n_nodes <= 0 || n_edges <= 0) { set_error("pdg_jvp: empty graph"); return -1; }
  const FwdWs F(n_nodes, n_edges, steps, true, const_cast<void*>(fwd_ws), false);
  const FwdWs J(n_nodes, n_edges, steps, false, jvp_ws, false);
  const size_t tws = J.total;  // bytes between consecutive tangent workspaces
  if (jvp_ws_bytes < (size_t)K * tws) { set_error("pdg_jvp: workspace %zu < %zu", jvp_ws_bytes, (size_t)K * tws); return -1; }
  const int N = (int)n_nodes, E = (int)n_edges, T = steps;
  int32_t *perm, *recv, *send, *rowptr;
  pdg_plan_views(const_cast<void*>(plan), n_nodes, n_edges, &perm, &recv, &send, &rowptr, nullptr, nullptr);
  const int nt_n = (int)(F.N_pad / TM), nt_e = (int)(F.E_pad / TM);
  int sms = num_sms();
  if (sms > MAXP) sms = MAXP;
  const int grid_n = balanced_grid(nt_n, sms), grid_e = balanced_grid(nt_e, sms);
  // Edge kernel: tangent groups of C over the SMs the x-grid leaves idle.  One group of all K (C = K) shares the primal
  // part of every tile across the K tangents; more groups spread the tangents of a small graph over idle SMs.
  int groups = std::min(K, std::max(1, sms / grid_e));
  const int C = (K + groups - 1) / groups;
  groups = (K + C - 1) / C;  // no empty group
  const size_t smem_edge = SMEM_JEDGE + (size_t)C * SMEM_JEDGE_TAN;
  const double cnt_n = (double)N * H, cnt_e = (double)E * H;

  // tangent partials of all K tangents (one strided memset): slots of CTAs that do not exist must read as zero
  PDG_CUDA_CHECK(cudaMemset2DAsync(J.parts, tws, 0, (size_t)(2 + 3 * T) * MAXP * 2 * sizeof(double), K, st));
  const int* nzflag = (flags & PDG_FLAG_ZERO_CHECK) ? F.nzflag : nullptr;
  const float* const* P = params->p;
  const float* pk = F.pack;
  const int scale_in = (flags & PDG_FLAG_SCALE_INPUT) ? 1 : 0;
  const dim3 gn(grid_n, K), ge(grid_e, K);
  {
    ScopedTimer tm_(KC_JVP_NODE_ENC, st);
    if (launch_named("k_node_encoder_jvp", false, k_node_encoder_jvp, gn, dim3(NT), SMEM_JENC, st, mean_stress, pos, nodes_types,
                     *norm, scale_in, tan_mean_stress, tan_pos, P[NE_W0], P[NE_B0], pk + PackOffsets::NE_W2T, F.y_nenc,
                     F.parts_slot(0), cnt_n, J.y_nenc, J.parts_slot(0), N, nt_n, ms_stride, pos_stride, tws)) return -2;
  }
  PDG_LAUNCH_CHECK();
  {
    ScopedTimer tm_(KC_JVP_EDGE_ENC, st);
    if (launch_named("k_edge_encoder_jvp", false, k_edge_encoder_jvp, ge, dim3(NT), SMEM_JENC, st, edge_attr, perm, *norm, scale_in,
                     tan_edge_attr, P[EE_W0], P[EE_B0], pk + PackOffsets::EE_W2T, F.y_eenc, F.parts_slot(1), cnt_e, J.y_eenc,
                     J.parts_slot(1), E, nt_e, ea_stride, tws)) return -2;
  }
  PDG_LAUNCH_CHECK();
  // step t of the forward on F gives the primal state, on J the tangent state
  for (int t = 0; t < T; ++t) {
    const FwdStepArgs f = fwd_step_args(F, P, recv, send, rowptr, t), j = fwd_step_args(J, P, recv, send, rowptr, t);
    {
      ScopedTimer tm_(KC_JVP_NODE_PRE, st);
      if (launch_named("k_node_pre_jvp", false, k_node_pre_jvp, gn, dim3(NT), SMEM_1A, st, f.np.yprev, f.np.prev_parts,
                       j.np.prev_parts, f.np.prev_count, f.np.lnw, j.np.base, j.np.yprev, j.np.x_out, pk + PackOffsets::PE_WAT,
                       pk + PackOffsets::PE_WBT, j.np.Pa, j.np.Pb, nt_n, tws)) return -2;
    }
    PDG_LAUNCH_CHECK();
    PDG_CUDA_CHECK(cudaMemset2DAsync(J.aggraw_[t], tws, 0, (size_t)J.N_pad * H * sizeof(float), K, st));
    EdgeJvpArgs a;
    a.yprev = f.e.yprev;
    a.prev_parts = f.e.prev_parts;
    a.prev_w = f.e.prev_w;
    a.e_t = f.e.e_out;
    a.Pa = f.e.Pa;
    a.Pb = f.e.Pb;
    a.y2_t = f.e.y2_out;
    a.parts1 = f.e.parts1;
    a.parts2 = f.e.parts2;
    a.tprev_parts = j.e.prev_parts;
    a.tbase = j.e.base;
    a.typrev = j.e.yprev;
    a.te_out = j.e.e_out;  // ed_t is read again only by the next step
    a.tPa = j.e.Pa;
    a.tPb = j.e.Pb;
    a.ty2_out = j.e.y2_out;
    a.taggraw = j.e.aggraw;
    a.tparts1 = j.e.parts1;
    a.tparts2 = j.e.parts2;
    a.recv = recv;
    a.send = send;
    a.rowptr = rowptr;
    a.WtE = f.e.WtE;
    a.b1 = f.e.b1;
    a.Wt2 = f.e.Wt2;
    a.b2 = f.e.b2;
    a.count = f.e.prev_count;
    a.E = E;
    a.n_tiles = nt_e;
    a.tws = tws;
    a.K = K;
    a.C = C;
    {
      ScopedTimer tm_(KC_JVP_EDGE_STEP, st);
      if (launch_named("k_edge_step_jvp", false, k_edge_step_jvp, dim3(grid_e, groups), dim3(NT), smem_edge, st, a)) return -2;
    }
    PDG_LAUNCH_CHECK();
    {
      ScopedTimer tm_(KC_JVP_NODE_UPD, st);
      if (launch_named("k_node_update_jvp", false, k_node_update_jvp, gn, dim3(NT), SMEM_2A, st, f.u.aggraw, j.u.aggraw, rowptr,
                       f.u.parts1, j.u.parts1, f.u.count1, f.u.lnw_e, j.u.x_t, pk + PackOffsets::PN_WAT,
                       pk + PackOffsets::PN_WXT, f.u.hq_out, pk + PackOffsets::PN_W2T, f.u.y3_out, f.u.parts3, cnt_n, j.u.y3_out,
                       j.u.parts3, N, nt_n, tws)) return -2;
    }
    PDG_LAUNCH_CHECK();
  }
  const DecArgs fd = fwd_dec_args(F, P), jd = fwd_dec_args(J, P);
  const bool scale_out = (flags & PDG_FLAG_SCALE_OUTPUT) != 0;
  {
    ScopedTimer tm_(KC_JVP_DECODER, st);
    if (launch_named("k_decoder_jvp", false, k_decoder_jvp, gn, dim3(NT), SMEM_1A, st, fd.yprev, fd.prev_parts, jd.prev_parts,
                     fd.prev_count, fd.lnw, jd.base, jd.yprev, pk + PackOffsets::ND_W0T, fd.hd_out, fd.D2,
                     scale_out ? norm->std_local_stress : 1.f, tan_local_stress, nzflag, N, nt_n, tws)) return -2;
  }
  PDG_LAUNCH_CHECK();
  return 0;
}

extern "C" int pdg_jvp(const pdg_params_t* params, const pdg_norm_t* norm, const float* mean_stress, const float* pos,
                       const int64_t* nodes_types, const float* edge_attr, const void* plan, int64_t n_nodes, int64_t n_edges,
                       int steps, int flags, int precision, const void* fwd_ws, void* jvp_ws, size_t jvp_ws_bytes,
                       const float* tan_mean_stress, const float* tan_pos, const float* tan_edge_attr,
                       float* tan_local_stress, void* stream) {
  return pdg_jvp_batched(params, norm, mean_stress, pos, nodes_types, edge_attr, plan, n_nodes, n_edges, steps, flags,
                         precision, fwd_ws, jvp_ws, jvp_ws_bytes, 1, tan_mean_stress, 0, tan_pos, 0, tan_edge_attr, 0,
                         tan_local_stress, stream);
}
