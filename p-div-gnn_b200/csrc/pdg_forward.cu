// Forward pass of EncodeProcessDecode (reference models.py:288-326) as tile kernels.
//
// fp32 path (PDG_PREC_FP32): every Linear is a 128x128-row-tile FFMA GEMM whose A tile is
// produced in shared memory by the fused prologue (gathers, lazy graph-LayerNorm,
// residual) and whose epilogue does bias/ReLU, LayerNorm partial statistics and the
// receiver-segment sum.  Nothing of size [E,384] / [N,256] ever exists in HBM.
//
// Graph-mode LayerNorm (PyG, SURVEY 2.3a) needs the mean/std of the WHOLE tensor, so a
// producer kernel writes the RAW MLP output plus per-CTA {sum, sumsq} partials and the
// consumer kernel applies (y-mu)/(sigma+eps)*w+b (+ residual) while loading ("lazy LN").
// For the message path the normalisation commutes with the sum over incoming edges:
//   sum_k LN(y_k) = w/(sigma+eps) * (sum_k y_k - deg*mu) + deg*b
// so only the raw segment sums [N,128] are stored, never the per-edge messages.
#include "pdg_ws.cuh"
#include "pdg_tc.cuh"

namespace pdg {

// ------------------------------------------------------------------------------------
// weight pack: W[out][in] -> Wt[in][out]
// ------------------------------------------------------------------------------------
// ------------------------------------------------------------------------------------
// shared pieces
// ------------------------------------------------------------------------------------
struct SmemTile {
  float* A;
  float* Ws;
};
constexpr size_t SMEM_1A = (size_t)(TM * LDS + 2 * BK * H) * sizeof(float) + 1024 + 256;
constexpr size_t SMEM_2A = (size_t)(2 * TM * LDS + 2 * BK * H) * sizeof(float) + 1024 + 256;

// relu(acc + bias) in place; accumulate sum / sumsq over rows < nvalid
__device__ __forceinline__ void bias_relu_stats(float (&acc)[8][8], const float (&bias)[8], int nvalid, float& s,
                                                float& ss) {
  const int ty = threadIdx.x >> 4;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const bool ok = ty * 8 + i < nvalid;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float v = fmaxf(acc[i][j] + bias[j], 0.f);
      acc[i][j] = v;
      if (ok) { s += v; ss = fmaf(v, v, ss); }
    }
  }
}

// Instances (pdg_forward_batched): every fp32 forward kernel is a template on INST.  With INST, instance k = blockIdx.y
// over the x-grid of one pdg_forward; its workspace pointers move by k * iws bytes (one forward workspace per instance)
// and its inputs by k * (element stride).  Without INST (pdg_forward) the offsets and their arguments are not read.

// ------------------------------------------------------------------------------------
// node encoder: format_node_features (models.py:140-152) + node_encoder MLP (:260-266)
// writes RAW relu output + LN partials (slot 0)
// ------------------------------------------------------------------------------------
template <bool INST>
__global__ void __launch_bounds__(NT, 1)
k_node_encoder(const float* __restrict__ mean_stress, const float* __restrict__ pos, const int64_t* __restrict__ types,
               pdg_norm_t nrm, int scale_in, const float* __restrict__ W0, const float* __restrict__ b0,
               const float* __restrict__ Wt2, const float* __restrict__ b2, float* __restrict__ y_out,
               double* __restrict__ parts, int* __restrict__ nzflag, int N, int n_tiles, int64_t ms_stride,
               int64_t pos_stride, size_t iws) {
  extern __shared__ __align__(16) float smem[];
  if constexpr (INST) {
    mean_stress += blockIdx.y * ms_stride;
    pos += blockIdx.y * pos_stride;
    y_out = copy_at(y_out, blockIdx.y * iws);
    parts = copy_at(parts, blockIdx.y * iws);
    nzflag = copy_at(nzflag, blockIdx.y * iws);
  }
  float* A = smem;
  float* Ws = A + TM * LDS;
  float* feat = Ws + 2 * BK * H;       // [TM][8]
  double* red = (double*)(feat + TM * 8);
  const int tid = threadIdx.x;
  const int c4 = (tid & 31) * 4;
  float w0[4][6], bb0[4];
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    bb0[c] = b0[c4 + c];
#pragma unroll
    for (int j = 0; j < 6; ++j) w0[c][j] = W0[(c4 + c) * 6 + j];
  }
  float bias2[8];
  load_cols(bias2, b2);
  pdl_sync();  // Wt2 comes from k_pack_all (the previous launch)
  double tot_s = 0, tot_ss = 0;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int row0 = tile * TM;
    const int nvalid = min(TM, N - row0);
    if (tid < TM) {
      const int row = row0 + tid;
      float f[6] = {0, 0, 0, 0, 0, 0};
      bool nz = false;
      if (row < N) {
        float m0 = mean_stress[row * 3 + 0], m1 = mean_stress[row * 3 + 1], m2 = mean_stress[row * 3 + 2];
        float p0 = pos[row * 2 + 0], p1 = pos[row * 2 + 1];
        nz = m0 != 0.f || m1 != 0.f || m2 != 0.f;  // torch.any(mean_stress), models.py:294 (raw values; NaN counts)
        if (scale_in) {
          m0 = (m0 - nrm.mean_mean_stress) / nrm.std_mean_stress;
          m1 = (m1 - nrm.mean_mean_stress) / nrm.std_mean_stress;
          m2 = (m2 - nrm.mean_mean_stress) / nrm.std_mean_stress;
          p0 = (p0 - nrm.mean_pos) / nrm.std_pos;
          p1 = (p1 - nrm.mean_pos) / nrm.std_pos;
        }
        f[0] = m0; f[1] = m1; f[2] = m2; f[3] = p0; f[4] = p1; f[5] = (float)types[row];
      }
#pragma unroll
      for (int j = 0; j < 6; ++j) feat[tid * 8 + j] = f[j];
      if (nzflag != nullptr && __any_sync(0xffffffffu, nz) && (tid & 31) == 0) atomicOr(nzflag, 1);  // warps 0-3, whole
    }
    __syncthreads();
#pragma unroll 4
    for (int it = 0; it < (TM * H / 4) / NT; ++it) {
      const int r = (tid >> 5) + it * 8;
      float v[4];
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        float a = bb0[c];
#pragma unroll
        for (int j = 0; j < 6; ++j) a = fmaf(w0[c][j], feat[r * 8 + j], a);
        v[c] = fmaxf(a, 0.f);
      }
      *reinterpret_cast<float4*>(A + r * LDS + c4) = make_float4(v[0], v[1], v[2], v[3]);
    }
    float acc[8][8];
    acc_zero(acc);
    gemm_rowA(A, Wt2, H, acc, Ws);
    float s = 0, ss = 0;
    bias_relu_stats(acc, bias2, nvalid, s, ss);
    acc_store(acc, y_out + (size_t)row0 * H, H);
    double ds = s, dss = ss;
    block_sum2(ds, dss, red);
    if (tid == 0) { tot_s += ds; tot_ss += dss; }
  }
  if (tid == 0) { parts[2 * blockIdx.x] = tot_s; parts[2 * blockIdx.x + 1] = tot_ss; }
}

// ------------------------------------------------------------------------------------
// edge encoder: format_edge_features (models.py:154-162, :303-307) + edge_encoder MLP
// (:268-274), edges taken in receiver-sorted order through perm.  RAW output + slot 1.
// ------------------------------------------------------------------------------------
template <bool INST>
__global__ void __launch_bounds__(NT, 1)
k_edge_encoder(const float* __restrict__ edge_attr, const int32_t* __restrict__ perm, pdg_norm_t nrm, int scale_in,
               const float* __restrict__ W0, const float* __restrict__ b0, const float* __restrict__ Wt2,
               const float* __restrict__ b2, float* __restrict__ y_out, double* __restrict__ parts, int E,
               int n_tiles, int64_t ea_stride, size_t iws) {
  extern __shared__ __align__(16) float smem[];
  if constexpr (INST) {
    edge_attr += blockIdx.y * ea_stride;
    y_out = copy_at(y_out, blockIdx.y * iws);
    parts = copy_at(parts, blockIdx.y * iws);
  }
  float* A = smem;
  float* Ws = A + TM * LDS;
  float* feat = Ws + 2 * BK * H;  // [TM]
  double* red = (double*)(feat + TM * 8);
  const int tid = threadIdx.x;
  const int c4 = (tid & 31) * 4;
  const float4 w0 = *reinterpret_cast<const float4*>(W0 + c4);
  const float4 bb0 = *reinterpret_cast<const float4*>(b0 + c4);
  float bias2[8];
  load_cols(bias2, b2);
  double tot_s = 0, tot_ss = 0;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int row0 = tile * TM;
    const int nvalid = min(TM, E - row0);
    if (tid < TM) {
      float a = 0.f;
      if (row0 + tid < E) {
        a = edge_attr[perm[row0 + tid]];
        if (scale_in) a = (a - nrm.mean_edge_weight) / nrm.std_edge_weight;
      }
      feat[tid] = a;
    }
    __syncthreads();
#pragma unroll 4
    for (int it = 0; it < (TM * H / 4) / NT; ++it) {
      const int r = (tid >> 5) + it * 8;
      const float a = feat[r];
      *reinterpret_cast<float4*>(A + r * LDS + c4) =
          make_float4(fmaxf(fmaf(w0.x, a, bb0.x), 0.f), fmaxf(fmaf(w0.y, a, bb0.y), 0.f),
                      fmaxf(fmaf(w0.z, a, bb0.z), 0.f), fmaxf(fmaf(w0.w, a, bb0.w), 0.f));
    }
    float acc[8][8];
    acc_zero(acc);
    gemm_rowA(A, Wt2, H, acc, Ws);
    float s = 0, ss = 0;
    bias_relu_stats(acc, bias2, nvalid, s, ss);
    acc_store(acc, y_out + (size_t)row0 * H, H);
    double ds = s, dss = ss;
    block_sum2(ds, dss, red);
    if (tid == 0) { tot_s += ds; tot_ss += dss; }
  }
  if (tid == 0) { parts[2 * blockIdx.x] = tot_s; parts[2 * blockIdx.x + 1] = tot_ss; }
}

// ------------------------------------------------------------------------------------
// K1 node_pre: x_t = x_{t-1} + LN(y_prev)  (residual of models.py:224 applied lazily),
// then the node-level halves of edge_net layer 1:  Pa = x_t Wa^T, Pb = x_t Wb^T  with
// edge_net.0.weight = [Wa | Wb | We]  (x_i | x_j | edge_attr column blocks, :233-238).
// ------------------------------------------------------------------------------------
template <bool INST>
__global__ void __launch_bounds__(NT, 1)
k_node_pre(const float* __restrict__ base, const float* __restrict__ yprev, const double* __restrict__ prev_parts,
           double prev_count, const float* __restrict__ lnw, const float* __restrict__ lnb, float* __restrict__ x_out,
           const float* __restrict__ WtA, const float* __restrict__ WtB, float* __restrict__ Pa, float* __restrict__ Pb,
           int n_tiles, size_t iws) {
  extern __shared__ __align__(16) float smem[];
  if constexpr (INST) {
    const size_t off = blockIdx.y * iws;
    base = copy_at(base, off);
    yprev = copy_at(yprev, off);
    prev_parts = copy_at(prev_parts, off);
    x_out = copy_at(x_out, off);
    Pa = copy_at(Pa, off);
    Pb = copy_at(Pb, off);
  }
  float* A = smem;
  float* Ws = A + TM * LDS;
  float* smf = Ws + 2 * BK * H;
  const int tid = threadIdx.x;
  const int c4 = (tid & 31) * 4;
  const LnStat st = ln_stat_block(prev_parts, prev_count, smf);
  const float4 w = *reinterpret_cast<const float4*>(lnw + c4);
  const float4 b = *reinterpret_cast<const float4*>(lnb + c4);
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const size_t row0 = (size_t)tile * TM;
    // row loads in two batches of eight: every load of a batch is in flight before its first use (the loop was a
    // long-scoreboard stall with four rows in flight)
#pragma unroll
    for (int bt = 0; bt < 2; ++bt) {
      float4 ly[8], lx[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const size_t g = (row0 + (tid >> 5) + (bt * 8 + k) * 8) * H + c4;
        ly[k] = *reinterpret_cast<const float4*>(yprev + g);
        lx[k] = base != nullptr ? *reinterpret_cast<const float4*>(base + g) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int r = (tid >> 5) + (bt * 8 + k) * 8;
        const size_t g = (row0 + r) * H + c4;
        const float4 y = ly[k];
        float4 v;
        v.x = (y.x - st.mu) * st.rstd * w.x + b.x;
        v.y = (y.y - st.mu) * st.rstd * w.y + b.y;
        v.z = (y.z - st.mu) * st.rstd * w.z + b.z;
        v.w = (y.w - st.mu) * st.rstd * w.w + b.w;
        if (base != nullptr) { v.x += lx[k].x; v.y += lx[k].y; v.z += lx[k].z; v.w += lx[k].w; }
        *reinterpret_cast<float4*>(x_out + g) = v;
        *reinterpret_cast<float4*>(A + r * LDS + c4) = v;
      }
    }
    float acc[8][8];
    if (Pa != nullptr) {
      acc_zero(acc);
      gemm_rowA(A, WtA, H, acc, Ws);
      acc_store(acc, Pa + row0 * H, H);
      acc_zero(acc);
      gemm_rowA(A, WtB, H, acc, Ws);
      acc_store(acc, Pb + row0 * H, H);
    } else {
      __syncthreads();
    }
  }
}

// ------------------------------------------------------------------------------------
// K2 edge_step: one Processor step on a tile of 128 receiver-sorted edges
//   e_t      = e_{t-1} + LN(y2_{t-1})                       (lazy; written for step t+1 / backward)
//   G        = e_t We^T + b1
//   y1       = relu(relu(G + Pa[recv] + Pb[send]) W2^T + b2)   message   (models.py:233-238)
//   aggraw  += segment-sum of y1 over the receiver                        (PyG aggr="add")
//   y2       = relu(relu(G + Pa[send] + Pb[recv]) W2^T + b2)   edge update, swapped order (:219-222)
// LN partials of y1 -> slot LN1(t), of y2 -> slot LN2(t).
// ------------------------------------------------------------------------------------
constexpr size_t SMEM_EDGE = (size_t)(2 * TM * LDS + 2 * BK * H) * sizeof(float) + 2 * TM * sizeof(int) + 16 * sizeof(double) + 64 + 256;

__device__ __forceinline__ void gather_hidden(float (&acc)[8][8], const float* __restrict__ Gs, const float* __restrict__ P1,
                                              const int* __restrict__ idx1, const float* __restrict__ P2,
                                              const int* __restrict__ idx2) {
  // acc = relu(G + P1[idx1[row]] + P2[idx2[row]])
  const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int r = ty * 8 + i;
    const float* p1 = P1 + (size_t)idx1[r] * H + tx * 4;
    const float* p2 = P2 + (size_t)idx2[r] * H + tx * 4;
    const float4 a0 = __ldg(reinterpret_cast<const float4*>(p1));
    const float4 a1 = __ldg(reinterpret_cast<const float4*>(p1 + 64));
    const float4 c0 = __ldg(reinterpret_cast<const float4*>(p2));
    const float4 c1 = __ldg(reinterpret_cast<const float4*>(p2 + 64));
    const float4 g0 = *reinterpret_cast<const float4*>(Gs + r * LDS + tx * 4);
    const float4 g1 = *reinterpret_cast<const float4*>(Gs + r * LDS + 64 + tx * 4);
    acc[i][0] = fmaxf(g0.x + a0.x + c0.x, 0.f);
    acc[i][1] = fmaxf(g0.y + a0.y + c0.y, 0.f);
    acc[i][2] = fmaxf(g0.z + a0.z + c0.z, 0.f);
    acc[i][3] = fmaxf(g0.w + a0.w + c0.w, 0.f);
    acc[i][4] = fmaxf(g1.x + a1.x + c1.x, 0.f);
    acc[i][5] = fmaxf(g1.y + a1.y + c1.y, 0.f);
    acc[i][6] = fmaxf(g1.z + a1.z + c1.z, 0.f);
    acc[i][7] = fmaxf(g1.w + a1.w + c1.w, 0.f);
  }
}

template <bool INST>
__global__ void __launch_bounds__(NT, 1) k_edge_step(EdgeStepArgs a, size_t iws) {
  extern __shared__ __align__(16) float smem[];
  if constexpr (INST) {
    const size_t off = blockIdx.y * iws;
    a.base = copy_at(a.base, off);
    a.yprev = copy_at(a.yprev, off);
    a.prev_parts = copy_at(a.prev_parts, off);
    a.e_out = copy_at(a.e_out, off);
    a.Pa = copy_at(a.Pa, off);
    a.Pb = copy_at(a.Pb, off);
    a.y2_out = copy_at(a.y2_out, off);
    a.aggraw = copy_at(a.aggraw, off);
    a.parts1 = copy_at(a.parts1, off);
    a.parts2 = copy_at(a.parts2, off);
  }
  float* A = smem;
  float* Gs = A + TM * LDS;
  float* Ws = Gs + TM * LDS;
  int* recv_s = (int*)(Ws + 2 * BK * H);
  int* send_s = recv_s + TM;
  double* red = (double*)(send_s + TM);
  float* smf = (float*)(red + 16);
  unsigned* seg_masks = (unsigned*)(smf + 4);
  unsigned char* seg_row = (unsigned char*)(seg_masks + 4);  // [TM + 1]
  const int tid = threadIdx.x;
  const int c4 = (tid & 31) * 4;
  const LnStat st = ln_stat_block(a.prev_parts, a.prev_count, smf);
  const float4 w = *reinterpret_cast<const float4*>(a.prev_w + c4);
  const float4 b = *reinterpret_cast<const float4*>(a.prev_b + c4);
  float bias1[8], bias2[8];
  load_cols(bias1, a.b1);
  load_cols(bias2, a.b2);
  double t1s = 0, t1ss = 0, t2s = 0, t2ss = 0;
  for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const int row0 = tile * TM;
    const int nvalid = min(TM, a.E - row0);
    if (tid < TM) {
      recv_s[tid] = a.recv[row0 + tid];
      send_s[tid] = a.send[row0 + tid];
    }
    // ---- e_t tile (lazy LayerNorm + residual) ----
    // row loads in two batches of eight, every load of a batch in flight before its first use (with four rows in flight
    // this loop was 16 % of the kernel's stall samples, all long-scoreboard)
#pragma unroll
    for (int bt = 0; bt < 2; ++bt) {
      float4 ly[8], lx[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const size_t g = ((size_t)row0 + (tid >> 5) + (bt * 8 + k) * 8) * H + c4;
        ly[k] = *reinterpret_cast<const float4*>(a.yprev + g);
        lx[k] = a.base != nullptr ? *reinterpret_cast<const float4*>(a.base + g) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int r = (tid >> 5) + (bt * 8 + k) * 8;
        const size_t g = ((size_t)row0 + r) * H + c4;
        const float4 y = ly[k];
        float4 v;
        v.x = (y.x - st.mu) * st.rstd * w.x + b.x;
        v.y = (y.y - st.mu) * st.rstd * w.y + b.y;
        v.z = (y.z - st.mu) * st.rstd * w.z + b.z;
        v.w = (y.w - st.mu) * st.rstd * w.w + b.w;
        if (a.base != nullptr) { v.x += lx[k].x; v.y += lx[k].y; v.z += lx[k].z; v.w += lx[k].w; }
        if (a.e_out != nullptr) *reinterpret_cast<float4*>(a.e_out + g) = v;
        *reinterpret_cast<float4*>(A + r * LDS + c4) = v;
      }
    }
    __syncthreads();  // recv_s/send_s + A visible
    const int nseg = tile_segments(recv_s, nvalid, seg_row, seg_masks);  // receiver segments of the tile
    // ---- G = e_t We^T + b1 ----
    float acc[8][8];
    acc_zero(acc);
    gemm_rowA(A, a.WtE, H, acc, Ws);
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[i][j] += bias1[j];
    acc_store(acc, Gs, LDS);
    __syncthreads();
    // ---- message path ----
    gather_hidden(acc, Gs, a.Pa, recv_s, a.Pb, send_s);
    acc_store(acc, A, LDS);
    acc_zero(acc);
    gemm_rowA(A, a.Wt2, H, acc, Ws);
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[i][j] = fmaxf(acc[i][j] + bias2[j], 0.f);
    acc_store(acc, A, LDS);  // y1 tile (gemm_rowA ended with a barrier)
    __syncthreads();
    {
      // receiver-segment sums (warp per segment, rows added in row order) + LayerNorm partials of y1
      float s = 0.f, ss = 0.f;
      tile_segsum_warp<true>(A, recv_s, seg_row, nseg, a.rowptr, row0, nvalid, a.aggraw, s, ss);
      double ds = s, dss = ss;
      block_sum2(ds, dss, red);
      if (tid == 0) { t1s += ds; t1ss += dss; }
    }
    // ---- edge-update path (skipped on the last step: its result is never read) ----
    if (a.y2_out != nullptr) {
      __syncthreads();
      gather_hidden(acc, Gs, a.Pa, send_s, a.Pb, recv_s);
      acc_store(acc, A, LDS);
      acc_zero(acc);
      gemm_rowA(A, a.Wt2, H, acc, Ws);
      float s = 0, ss = 0;
      bias_relu_stats(acc, bias2, nvalid, s, ss);
      acc_store(acc, a.y2_out + (size_t)row0 * H, H);
      double ds = s, dss = ss;
      block_sum2(ds, dss, red);
      if (tid == 0) { t2s += ds; t2ss += dss; }
    }
    __syncthreads();
  }
  if (tid == 0) {
    a.parts1[2 * blockIdx.x] = t1s;
    a.parts1[2 * blockIdx.x + 1] = t1ss;
    if (a.parts2 != nullptr) {
      a.parts2[2 * blockIdx.x] = t2s;
      a.parts2[2 * blockIdx.x + 1] = t2ss;
    }
  }
}

// ------------------------------------------------------------------------------------
// K3 node_update: update() of models.py:240-243
//   agg = w_e/(sigma1+eps) * (aggraw - deg*mu1) + deg*b_e      (LN1 pushed through the sum)
//   y3  = relu(relu([agg, x_t] V1^T + c1) V2^T + c2)           RAW + partials (slot LN3)
// ------------------------------------------------------------------------------------
template <bool INST>
__global__ void __launch_bounds__(NT, 1)
k_node_update(const float* __restrict__ aggraw, const int32_t* __restrict__ rowptr, const double* __restrict__ parts1,
              double count1, const float* __restrict__ lnw_e, const float* __restrict__ lnb_e,
              const float* __restrict__ x_t, const float* __restrict__ WtA, const float* __restrict__ WtX,
              const float* __restrict__ c1, const float* __restrict__ Wt2, const float* __restrict__ c2,
              float* __restrict__ hq_out, float* __restrict__ y3_out, double* __restrict__ parts3, int N, int n_tiles,
              size_t iws) {
  extern __shared__ __align__(16) float smem[];
  if constexpr (INST) {
    const size_t off = blockIdx.y * iws;
    aggraw = copy_at(aggraw, off);
    parts1 = copy_at(parts1, off);
    x_t = copy_at(x_t, off);
    hq_out = copy_at(hq_out, off);
    y3_out = copy_at(y3_out, off);
    parts3 = copy_at(parts3, off);
  }
  float* A0 = smem;
  float* A1 = A0 + TM * LDS;
  float* Ws = A1 + TM * LDS;
  double* red = (double*)(Ws + 2 * BK * H);
  float* smf = (float*)(red + 16);
  const int tid = threadIdx.x;
  const int c4 = (tid & 31) * 4;
  const LnStat st = ln_stat_block(parts1, count1, smf);
  const float4 w = *reinterpret_cast<const float4*>(lnw_e + c4);
  const float4 b = *reinterpret_cast<const float4*>(lnb_e + c4);
  float bias1[8], bias2[8];
  load_cols(bias1, c1);
  load_cols(bias2, c2);
  double tot_s = 0, tot_ss = 0;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int row0 = tile * TM;
    const int nvalid = min(TM, N - row0);
#pragma unroll
    for (int it = 0; it < (TM * H / 4) / NT; ++it) {  // x_t rows straight into A1 (asynchronous, no registers)
      const int r = (tid >> 5) + it * 8;
      cp_async16(A1 + r * LDS + c4, x_t + ((size_t)row0 + r) * H + c4);
    }
    cp_async_commit();
#pragma unroll
    for (int bt = 0; bt < 2; ++bt) {  // aggregate rows in two batches of eight, all loads of a batch in flight
      float4 ls[8];
      float ldeg[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int row = row0 + (tid >> 5) + (bt * 8 + k) * 8;
        ldeg[k] = row < N ? (float)(rowptr[row + 1] - rowptr[row]) : 0.f;
        ls[k] = *reinterpret_cast<const float4*>(aggraw + (size_t)row * H + c4);
      }
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int r = (tid >> 5) + (bt * 8 + k) * 8;
        const float deg = ldeg[k];
        const float4 s4 = ls[k];
        const float dm = deg * st.mu;
        float4 v;
        v.x = (s4.x - dm) * st.rstd * w.x + deg * b.x;
        v.y = (s4.y - dm) * st.rstd * w.y + deg * b.y;
        v.z = (s4.z - dm) * st.rstd * w.z + deg * b.z;
        v.w = (s4.w - dm) * st.rstd * w.w + deg * b.w;
        *reinterpret_cast<float4*>(A0 + r * LDS + c4) = v;
      }
    }
    cp_async_wait<0>();  // gemm_rowA's first barrier makes A0 / A1 visible
    float acc[8][8];
    acc_zero(acc);
    gemm_rowA(A0, WtA, H, acc, Ws);
    gemm_rowA(A1, WtX, H, acc, Ws);
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[i][j] = fmaxf(acc[i][j] + bias1[j], 0.f);
    acc_store(acc, A0, LDS);
    if (hq_out != nullptr) acc_store(acc, hq_out + (size_t)row0 * H, H);
    acc_zero(acc);
    gemm_rowA(A0, Wt2, H, acc, Ws);
    float s = 0, ss = 0;
    bias_relu_stats(acc, bias2, nvalid, s, ss);
    acc_store(acc, y3_out + (size_t)row0 * H, H);
    double ds = s, dss = ss;
    block_sum2(ds, dss, red);
    if (tid == 0) { tot_s += ds; tot_ss += dss; }
  }
  if (tid == 0) { parts3[2 * blockIdx.x] = tot_s; parts3[2 * blockIdx.x + 1] = tot_ss; }
}

// ------------------------------------------------------------------------------------
// decoder: x_T = x_{T-1} + LN(y3_{T-1}); node_decoder (models.py:282-286, :316-321)
// ------------------------------------------------------------------------------------
template <bool INST>
__global__ void __launch_bounds__(NT, 1)
k_decoder(const float* __restrict__ base, const float* __restrict__ yprev, const double* __restrict__ prev_parts,
          double prev_count, const float* __restrict__ lnw, const float* __restrict__ lnb, float* __restrict__ x_out,
          const float* __restrict__ WtD, const float* __restrict__ d1, const float* __restrict__ D2,
          const float* __restrict__ d2, float* __restrict__ hd_out, float out_scale, float out_shift,
          float* __restrict__ out, const int* __restrict__ nzflag, int N, int n_tiles, size_t iws) {
  extern __shared__ __align__(16) float smem[];
  if constexpr (INST) {
    const size_t off = blockIdx.y * iws;
    base = copy_at(base, off);
    yprev = copy_at(yprev, off);
    prev_parts = copy_at(prev_parts, off);
    x_out = copy_at(x_out, off);
    hd_out = copy_at(hd_out, off);
    nzflag = copy_at(nzflag, off);
    out += (size_t)blockIdx.y * N * PDG_OUT;  // local_stress [K][N][3]
  }
  float* A = smem;
  float* Ws = A + TM * LDS;
  float* smf = Ws + 2 * BK * H;
  const int tid = threadIdx.x;
  const int c4 = (tid & 31) * 4;
  pdl_sync();
  const LnStat st = ln_stat_block(prev_parts, prev_count, smf);
  const float4 w = *reinterpret_cast<const float4*>(lnw + c4);
  const float4 b = *reinterpret_cast<const float4*>(lnb + c4);
  float bias1[8];
  load_cols(bias1, d1);
  const bool live = nzflag == nullptr || *nzflag != 0;  // all-zero load case: zeros, not even un-standardised (models.py:294-299)
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const size_t row0 = (size_t)tile * TM;
#pragma unroll 4
    for (int it = 0; it < (TM * H / 4) / NT; ++it) {
      const int r = (tid >> 5) + it * 8;
      const size_t g = (row0 + r) * H + c4;
      const float4 y = *reinterpret_cast<const float4*>(yprev + g);
      float4 v;
      v.x = (y.x - st.mu) * st.rstd * w.x + b.x;
      v.y = (y.y - st.mu) * st.rstd * w.y + b.y;
      v.z = (y.z - st.mu) * st.rstd * w.z + b.z;
      v.w = (y.w - st.mu) * st.rstd * w.w + b.w;
      if (base != nullptr) {
        const float4 x0 = *reinterpret_cast<const float4*>(base + g);
        v.x += x0.x; v.y += x0.y; v.z += x0.z; v.w += x0.w;
      }
      if (x_out != nullptr) *reinterpret_cast<float4*>(x_out + g) = v;
      *reinterpret_cast<float4*>(A + r * LDS + c4) = v;
    }
    float acc[8][8];
    acc_zero(acc);
    gemm_rowA(A, WtD, H, acc, Ws);
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[i][j] = fmaxf(acc[i][j] + bias1[j], 0.f);
    acc_store(acc, A, LDS);
    if (hd_out != nullptr) acc_store(acc, hd_out + row0 * H, H);
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
        out[row * PDG_OUT + o] = live ? (dsum + d2[o]) * out_scale + out_shift : 0.f;
      }
    }
    __syncthreads();
  }
}

// All weight packs of one forward in ONE launch: blockIdx.y = job.
//   kind 0: fp32 transpose  Wt[k][o] = W[o][col0 + k]                     (FFMA tiles, k-major B operand)
//   kind 1: fp16 pre-swizzled operand image (the exact smem bytes of a tcgen05 K-major B tile; fp16, not bf16: a
//           weight's rounding error is systematic -- same error in every row of every step -- see pdg_tc.cuh)
struct PackJob { const float* W; void* dst; int ld, col0, kind; };
constexpr int MAX_PACK_JOBS = 20;
struct PackJobs { PackJob j[MAX_PACK_JOBS]; };
__global__ void __launch_bounds__(256) k_pack_all(PackJobs jobs) {
  pdl_sync();
  const PackJob jb = jobs.j[blockIdx.y];
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (jb.kind == 0) {
    if (idx < H * H) {
      const int k = idx / H, o = idx % H;
      reinterpret_cast<float*>(jb.dst)[idx] = jb.W[(size_t)o * jb.ld + jb.col0 + k];
    }
  } else if (idx < 128 * 16) {  // one 16-byte chunk each: 128 rows x 16 chunks
    const int r = idx >> 4, ch = idx & 15;
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = jb.W[(size_t)r * jb.ld + jb.col0 + ch * 8 + j];
    *reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(jb.dst) + tc::sw128_chunk(r, ch)) = tc::pack8_f16(v);
  }
}
int pack_weights(const pdg_params_t* P, float* pack, uint8_t* img, bool images, cudaStream_t st) {
  PackJobs jobs;
  int n = 0;
  auto tr = [&](const float* W, int ld, int col0, int off) { jobs.j[n++] = PackJob{W, pack + off, ld, col0, 0}; };
  auto im = [&](int which, const float* W, int ld, int col0) {
    jobs.j[n++] = PackJob{W, img + (size_t)which * tc::TILE_BF16_BYTES, ld, col0, 1};
  };
  tr(P->p[NE_W2], H, 0, PackOffsets::NE_W2T);
  tr(P->p[EE_W2], H, 0, PackOffsets::EE_W2T);
  tr(P->p[PE_W0], 3 * H, 0, PackOffsets::PE_WAT);
  tr(P->p[PE_W0], 3 * H, H, PackOffsets::PE_WBT);
  tr(P->p[PE_W0], 3 * H, 2 * H, PackOffsets::PE_WET);
  tr(P->p[PE_W2], H, 0, PackOffsets::PE_W2T);
  tr(P->p[PN_W0], 2 * H, 0, PackOffsets::PN_WAT);
  tr(P->p[PN_W0], 2 * H, H, PackOffsets::PN_WXT);
  tr(P->p[PN_W2], H, 0, PackOffsets::PN_W2T);
  tr(P->p[ND_W0], H, 0, PackOffsets::ND_W0T);
  if (images) {
    im(IMG_PE_WE, P->p[PE_W0], 3 * H, 2 * H);
    im(IMG_PE_W2, P->p[PE_W2], H, 0);
    im(IMG_PE_WA, P->p[PE_W0], 3 * H, 0);
    im(IMG_PE_WB, P->p[PE_W0], 3 * H, H);
    im(IMG_PN_WA, P->p[PN_W0], 2 * H, 0);
    im(IMG_PN_WX, P->p[PN_W0], 2 * H, H);
    im(IMG_PN_W2, P->p[PN_W2], H, 0);
    im(IMG_EE_W2, P->p[EE_W2], H, 0);
    im(IMG_NE_W2, P->p[NE_W2], H, 0);
    im(IMG_ND_W0, P->p[ND_W0], H, 0);
  }
  PDG_CUDA_CHECK(launch_pdl(k_pack_all, dim3(H * H / 256, n), dim3(256), 0, st, jobs));
  PDG_LAUNCH_CHECK();
  return 0;
}

// Zeroes `bytes` at p in each of K instance workspaces, iws bytes apart: one memset for any K (a plain one for K = 1).
static cudaError_t memset_instances(void* p, size_t iws, size_t bytes, int K, cudaStream_t st) {
  return K == 1 ? cudaMemsetAsync(p, 0, bytes, st) : cudaMemset2DAsync(p, iws, 0, bytes, K, st);
}

// The fp32 (FFMA) forward of K instances of one graph.  Instance k's workspace is W moved by k * W.total bytes, its
// inputs start k * (element stride) after the given pointers, its output at local_stress + k * N * 3.  The weights are
// packed once, into instance 0's workspace, and every instance reads them there.  pdg_forward is K = 1 with INST off.
template <bool INST>
int forward_ffma(const pdg_params_t* params, const pdg_norm_t* norm, const float* mean_stress, int64_t ms_stride,
                 const float* pos, int64_t pos_stride, const int64_t* nodes_types, const float* edge_attr,
                 int64_t ea_stride, const void* plan, const FwdWs& W, int flags, int K, float* local_stress,
                 cudaStream_t st) {
  const size_t iws = W.total;
  const bool save = W.save;
  const int N = (int)W.N, E = (int)W.E, T = W.T;
  int32_t *perm, *recv, *send, *rowptr;
  pdg_plan_views(const_cast<void*>(plan), W.N, W.E, &perm, &recv, &send, &rowptr, nullptr, nullptr);
  const int nt_n = (int)(W.N_pad / TM), nt_e = (int)(W.E_pad / TM);
  int sms = num_sms();
  if (sms > MAXP) sms = MAXP;  // LayerNorm partials are kept per CTA in slots of MAXP entries (as in pdg_backward)
  const int grid_n = balanced_grid(nt_n, sms), grid_e = balanced_grid(nt_e, sms);
  const dim3 gn(grid_n, K), ge(grid_e, K);
  const double cnt_n = (double)N * H, cnt_e = (double)E * H;
  const size_t smem_enc = SMEM_1A + TM * 8 * sizeof(float);
  if (set_smem((const void*)k_node_encoder<INST>, smem_enc)) return -2;
  if (set_smem((const void*)k_edge_encoder<INST>, smem_enc)) return -2;
  if (set_smem((const void*)k_node_pre<INST>, SMEM_1A)) return -2;
  if (set_smem((const void*)k_edge_step<INST>, SMEM_EDGE)) return -2;
  if (set_smem((const void*)k_node_update<INST>, SMEM_2A)) return -2;
  if (set_smem((const void*)k_decoder<INST>, SMEM_1A)) return -2;

  // LayerNorm partials + the non-zero-load flag (contiguous) in one memset
  PDG_CUDA_CHECK(memset_instances(W.parts, iws, (size_t)((char*)W.nzflag - (char*)W.parts) + 256, K, st));
  int* nzflag = (flags & PDG_FLAG_ZERO_CHECK) ? W.nzflag : nullptr;
  {
    ScopedTimer tm_(KC_PACK, st);
    if (pack_weights(params, W.pack, W.img, false, st)) return -2;
  }
  const float* const* P = params->p;
  const float* pk = W.pack;
  const int scale_in = (flags & PDG_FLAG_SCALE_INPUT) ? 1 : 0;

  {
    ScopedTimer tm_(KC_NODE_ENC, st);
    PDG_CUDA_CHECK(launch_pdl(k_node_encoder<INST>, gn, dim3(NT), smem_enc, st, mean_stress, pos, nodes_types, *norm, scale_in,
                              P[NE_W0], P[NE_B0], pk + PackOffsets::NE_W2T, P[NE_B2], W.y_nenc, W.parts_slot(0), nzflag, N,
                              nt_n, ms_stride, pos_stride, iws));
  }
  PDG_LAUNCH_CHECK();
  {
    ScopedTimer tm_(KC_EDGE_ENC, st);
    k_edge_encoder<INST><<<ge, NT, smem_enc, st>>>(edge_attr, perm, *norm, scale_in, P[EE_W0], P[EE_B0],
                                                   pk + PackOffsets::EE_W2T, P[EE_B2], W.y_eenc, W.parts_slot(1), E, nt_e,
                                                   ea_stride, iws);
  }
  PDG_LAUNCH_CHECK();
  for (int t = 0; t < T; ++t) {
    const bool first = t == 0, last = t == T - 1;
    // K1
    {
      ScopedTimer tm_(KC_NODE_PRE, st);
      k_node_pre<INST><<<gn, NT, SMEM_1A, st>>>(first ? nullptr : W.x_[t - 1], first ? W.y_nenc : W.y3_[t - 1],
                                                W.parts_slot(first ? 0 : slot_ln3(t - 1)), cnt_n,
                                                first ? P[NE_LNW] : P[PN_LNW], first ? P[NE_LNB] : P[PN_LNB], W.x_[t],
                                                pk + PackOffsets::PE_WAT, pk + PackOffsets::PE_WBT, W.Pa_[t], W.Pb_[t], nt_n,
                                                iws);
    }
    PDG_LAUNCH_CHECK();
    // K2
    PDG_CUDA_CHECK(memset_instances(W.aggraw_[t], iws, (size_t)W.N_pad * H * sizeof(float), K, st));
    EdgeStepArgs a;
    a.base = first ? nullptr : W.e_[t - 1];
    a.yprev = first ? W.y_eenc : W.y2_[t - 1];
    a.prev_parts = W.parts_slot(first ? 1 : slot_ln2(t - 1));
    a.prev_count = cnt_e;
    a.prev_w = first ? P[EE_LNW] : P[PE_LNW];
    a.prev_b = first ? P[EE_LNB] : P[PE_LNB];
    a.e_out = (save || !last) ? W.e_[t] : nullptr;
    a.e_img = nullptr;
    a.Pa = W.Pa_[t];
    a.Pb = W.Pb_[t];
    a.recv = recv;
    a.send = send;
    a.rowptr = rowptr;
    a.WtE = pk + PackOffsets::PE_WET;
    a.b1 = P[PE_B0];
    a.Wt2 = pk + PackOffsets::PE_W2T;
    a.b2 = P[PE_B2];
    a.y2_out = last ? nullptr : W.y2_[t];
    a.aggraw = W.aggraw_[t];
    a.parts1 = W.parts_slot(slot_ln1(t));
    a.parts2 = last ? nullptr : W.parts_slot(slot_ln2(t));
    a.E = E;
    a.n_tiles = nt_e;
    {
      ScopedTimer tm_(KC_EDGE_STEP, st);
      k_edge_step<INST><<<ge, NT, SMEM_EDGE, st>>>(a, iws);
    }
    PDG_LAUNCH_CHECK();
    // K3
    {
      ScopedTimer tm_(KC_NODE_UPD, st);
      k_node_update<INST><<<gn, NT, SMEM_2A, st>>>(W.aggraw_[t], rowptr, W.parts_slot(slot_ln1(t)), cnt_e, P[PE_LNW],
                                                   P[PE_LNB], W.x_[t], pk + PackOffsets::PN_WAT, pk + PackOffsets::PN_WXT,
                                                   P[PN_B0], pk + PackOffsets::PN_W2T, P[PN_B2], save ? W.hq_[t] : nullptr,
                                                   W.y3_[t], W.parts_slot(slot_ln3(t)), N, nt_n, iws);
    }
    PDG_LAUNCH_CHECK();
  }
  const bool scale_out = (flags & PDG_FLAG_SCALE_OUTPUT) != 0;
  {
    ScopedTimer tm_(KC_DECODER, st);
    PDG_CUDA_CHECK(launch_pdl(k_decoder<INST>, gn, dim3(NT), SMEM_1A, st, W.x_[T - 1], W.y3_[T - 1], W.parts_slot(slot_ln3(T - 1)),
                              cnt_n, P[PN_LNW], P[PN_LNB], save ? W.x_[T] : nullptr, pk + PackOffsets::ND_W0T, P[ND_B0], P[ND_W2],
                              P[ND_B2], save ? W.hd : nullptr, scale_out ? norm->std_local_stress : 1.f,
                              scale_out ? norm->mean_local_stress : 0.f, local_stress, nzflag, N, nt_n, iws));
  }
  PDG_LAUNCH_CHECK();
  return 0;
}

}  // namespace pdg

using namespace pdg;

extern "C" size_t pdg_forward_ws_bytes(int64_t n_nodes, int64_t n_edges, int steps, int flags) {
  if (steps < 1 || steps > 62) return 0;
  const bool sv = (flags & PDG_FLAG_SAVE) != 0;  // one size for both precision modes (their layouts differ)
  const size_t a = FwdWs(n_nodes, n_edges, steps, sv, nullptr, false).total, b = FwdWs(n_nodes, n_edges, steps, sv, nullptr, true).total;
  return a > b ? a : b;
}

extern "C" int pdg_forward(const pdg_params_t* params, const pdg_norm_t* norm, const float* mean_stress,
                           const float* pos, const int64_t* nodes_types, const float* edge_attr, const void* plan,
                           int64_t n_nodes, int64_t n_edges, int steps, int flags, int precision, void* ws,
                           size_t ws_bytes, float* local_stress, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  if (steps < 1 || steps > 62) { set_error("pdg_forward: steps=%d unsupported", steps); return -1; }
  if (precision != PDG_PREC_FP32 && precision != PDG_PREC_BF16) { set_error("pdg_forward: unknown precision mode %d", precision); return -1; }
  if (n_nodes <= 0 || n_edges <= 0) { set_error("pdg_forward: empty graph"); return -1; }
  const bool tcm = precision == PDG_PREC_BF16;
  const bool save = (flags & PDG_FLAG_SAVE) != 0;
  FwdWs W(n_nodes, n_edges, steps, save, ws, tcm);
  if (ws_bytes < W.total) { set_error("pdg_forward: workspace %zu < %zu", ws_bytes, W.total); return -1; }
  if (!tcm) return forward_ffma<false>(params, norm, mean_stress, 0, pos, 0, nodes_types, edge_attr, 0, plan, W, flags, 1,
                                       local_stress, st);
  // 16-bit mode: tcgen05 tile kernels (pdg_tc_*.cu)
  const int N = (int)n_nodes, E = (int)n_edges, T = steps;
  int32_t *perm, *recv, *send, *rowptr;
  pdg_plan_views(const_cast<void*>(plan), n_nodes, n_edges, &perm, &recv, &send, &rowptr, nullptr, nullptr);
  const int nt_n = (int)(W.N_pad / TM), nt_e = (int)(W.E_pad / TM);
  int sms = num_sms();
  if (sms > MAXP) sms = MAXP;  // LayerNorm partials are kept per CTA in slots of MAXP entries (as in pdg_backward)
  const int grid_n = balanced_grid(nt_n, sms), grid_e = balanced_grid(nt_e, sms);
  const double cnt_n = (double)N * H, cnt_e = (double)E * H;

  // LayerNorm partials + the non-zero-load flag (contiguous) in one memset
  PDG_CUDA_CHECK(cudaMemsetAsync(W.parts, 0, (size_t)((char*)W.nzflag - (char*)W.parts) + 256, st));
  int* nzflag = (flags & PDG_FLAG_ZERO_CHECK) ? W.nzflag : nullptr;
  {
    ScopedTimer tm_(KC_PACK, st);
    if (pack_weights(params, W.pack, W.img, tcm, st)) return -2;
  }
  const float* const* P = params->p;
  const int scale_in = (flags & PDG_FLAG_SCALE_INPUT) ? 1 : 0;

  {
    ScopedTimer tm_(KC_NODE_ENC, st);
    if (launch_node_encoder_tc(mean_stress, pos, nodes_types, norm, scale_in, P[NE_W0], P[NE_B0], P[NE_B2], W.y_nenc,
                               W.parts_slot(0), nzflag, N, nt_n, grid_n, W.img, st)) return -2;
  }
  PDG_LAUNCH_CHECK();
  {
    ScopedTimer tm_(KC_EDGE_ENC, st);
    if (launch_edge_encoder_tc(edge_attr, perm, norm, scale_in, P[EE_W0], P[EE_B0], P[EE_B2], W.y_eenc, W.parts_slot(1), E,
                               nt_e, W.img, st)) return -2;
  }
  PDG_LAUNCH_CHECK();
  for (int t = 0; t < T; ++t) {
    const bool first = t == 0, last = t == T - 1;
    // K1
    {
      ScopedTimer tm_(KC_NODE_PRE, st);
      NodePreArgs np;
      np.base = first ? nullptr : W.x_[t - 1]; np.yprev = first ? W.y_nenc : W.y3_[t - 1];
      np.prev_parts = W.parts_slot(first ? 0 : slot_ln3(t - 1)); np.prev_count = cnt_n;
      np.lnw = first ? P[NE_LNW] : P[PN_LNW]; np.lnb = first ? P[NE_LNB] : P[PN_LNB];
      np.x_out = W.x_[t]; np.Pa = W.Pa_[t]; np.Pb = W.Pb_[t]; np.n_tiles = nt_n;
      np.aggraw_zero = W.aggraw_[t];  // zeroed here instead of a memset between the kernels (keeps the PDL chain)
      np.b1 = P[PE_B0];
      np.x_img = W.ximg(t);
      if (launch_node_pre_tc(np, W.img, nt_n, st)) return -2;
    }
    PDG_LAUNCH_CHECK();
    // K2
    EdgeStepArgs a;
    a.base = first ? nullptr : W.e_[t - 1];
    a.yprev = first ? W.y_eenc : W.y2_[t - 1];
    a.prev_parts = W.parts_slot(first ? 1 : slot_ln2(t - 1));
    a.prev_count = cnt_e;
    a.prev_w = first ? P[EE_LNW] : P[PE_LNW];
    a.prev_b = first ? P[EE_LNB] : P[PE_LNB];
    a.e_out = !last ? W.e_[t] : nullptr;  // the backward reads the fp16 image instead
    a.e_img = save ? W.eimg_[t] : nullptr;
    a.Pa = W.Pa_[t];
    a.Pb = W.Pb_[t];
    a.recv = recv;
    a.send = send;
    a.rowptr = rowptr;
    a.WtE = W.pack + PackOffsets::PE_WET;
    a.b1 = P[PE_B0];
    a.Wt2 = W.pack + PackOffsets::PE_W2T;
    a.b2 = P[PE_B2];
    a.y2_out = last ? nullptr : W.y2_[t];
    a.aggraw = W.aggraw_[t];
    a.parts1 = W.parts_slot(slot_ln1(t));
    a.parts2 = last ? nullptr : W.parts_slot(slot_ln2(t));
    a.E = E;
    a.n_tiles = nt_e;
    {
      ScopedTimer tm_(KC_EDGE_STEP, st);
      if (launch_edge_step_tc(a, W.img, grid_e, st)) return -2;
    }
    PDG_LAUNCH_CHECK();
    // K3
    {
      ScopedTimer tm_(KC_NODE_UPD, st);
      NodeUpdArgs nu;
      nu.aggraw = W.aggraw_[t]; nu.rowptr = rowptr; nu.parts1 = W.parts_slot(slot_ln1(t)); nu.count1 = cnt_e;
      nu.lnw_e = P[PE_LNW]; nu.lnb_e = P[PE_LNB]; nu.x_t = W.x_[t]; nu.c1 = P[PN_B0]; nu.c2 = P[PN_B2];
      nu.hq_out = save ? W.hq_[t] : nullptr; nu.y3_out = W.y3_[t]; nu.parts3 = W.parts_slot(slot_ln3(t));
      nu.N = N; nu.n_tiles = nt_n;
      nu.x_img = W.ximg(t); nu.hq_img = save ? W.hqimg(t) : nullptr; nu.agg_img = save ? W.aggimg(t) : nullptr;
      if (launch_node_update_tc(nu, W.img, grid_n, st)) return -2;
    }
    PDG_LAUNCH_CHECK();
  }
  const bool scale_out = (flags & PDG_FLAG_SCALE_OUTPUT) != 0;
  {
    ScopedTimer tm_(KC_DECODER, st);
    if (launch_decoder_tc(W.x_[T - 1], W.y3_[T - 1], W.parts_slot(slot_ln3(T - 1)), cnt_n, P[PN_LNW], P[PN_LNB],
                          save ? W.x_[T] : nullptr, P[ND_B0], P[ND_W2], P[ND_B2], save ? W.hd : nullptr,
                          scale_out ? norm->std_local_stress : 1.f, scale_out ? norm->mean_local_stress : 0.f, local_stress,
                          nzflag, N, nt_n, grid_n, W.img, st)) return -2;
  }
  PDG_LAUNCH_CHECK();
  return 0;
}

// K instances of one graph: the workspace holds K fp32 forward workspaces without saved state, one after another
// (each total is a multiple of 256 bytes, so every instance stays aligned).
extern "C" size_t pdg_forward_batched_ws_bytes(int64_t n_nodes, int64_t n_edges, int steps, int flags, int n_instances) {
  if (n_instances < 1 || n_instances > PDG_FWD_MAX_INSTANCES || steps < 1 || steps > 62) return 0;
  return (size_t)n_instances * FwdWs(n_nodes, n_edges, steps, (flags & PDG_FLAG_SAVE) != 0, nullptr, false).total;
}

extern "C" int pdg_forward_batched(const pdg_params_t* params, const pdg_norm_t* norm, const float* mean_stress,
                                   int64_t ms_stride, const float* pos, int64_t pos_stride, const int64_t* nodes_types,
                                   const float* edge_attr, int64_t ea_stride, const void* plan, int64_t n_nodes,
                                   int64_t n_edges, int steps, int flags, int precision, void* ws, size_t ws_bytes,
                                   int n_instances, float* local_stress, void* stream_) {
  const int K = n_instances;
  if (K < 1 || K > PDG_FWD_MAX_INSTANCES) {
    set_error("pdg_forward_batched: n_instances=%d outside 1..%d", K, PDG_FWD_MAX_INSTANCES);
    return -1;
  }
  if (precision != PDG_PREC_FP32) {
    set_error("pdg_forward_batched: only the fp32 mode (PDG_PREC_FP32) runs instances; the 16-bit mode's kernels are "
              "persistent, one CTA per SM");
    return -1;
  }
  if (flags & PDG_FLAG_SAVE) {
    set_error("pdg_forward_batched: PDG_FLAG_SAVE is not supported (the batched forward keeps no state for a backward)");
    return -1;
  }
  if (steps < 1 || steps > 62) { set_error("pdg_forward_batched: steps=%d unsupported", steps); return -1; }
  if (ms_stride < 0 || pos_stride < 0 || ea_stride < 0) {
    set_error("pdg_forward_batched: negative input stride (mean_stress %lld, pos %lld, edge_attr %lld)",
              (long long)ms_stride, (long long)pos_stride, (long long)ea_stride);
    return -1;
  }
  if (n_nodes <= 0 || n_edges <= 0) { set_error("pdg_forward_batched: empty graph"); return -1; }
  const FwdWs W(n_nodes, n_edges, steps, false, ws, false);
  if (ws_bytes < (size_t)K * W.total) {
    set_error("pdg_forward_batched: workspace %zu < %zu", ws_bytes, (size_t)K * W.total);
    return -1;
  }
  return forward_ffma<true>(params, norm, mean_stress, ms_stride, pos, pos_stride, nodes_types, edge_attr, ea_stride,
                            plan, W, flags, K, local_stress, (cudaStream_t)stream_);
}

// Test/debug helper: byte offset and element count of a saved tensor inside a forward
// workspace built with PDG_FLAG_SAVE.  what: 0 x_t, 1 e_t, 2 y2_t, 3 Pa_t, 4 Pb_t,
// 5 aggraw_t, 6 hq_t, 7 y3_t, 8 y_nenc, 9 y_eenc, 10 hd, 11 LN partials of slot t.
extern "C" int pdg_ws_offset(int64_t n_nodes, int64_t n_edges, int steps, int flags, int what, int t, size_t* offset,
                             size_t* elems) {
  if (steps < 1 || steps > 62 || t < 0 || t > steps + 3 * steps + 2) { set_error("pdg_ws_offset: bad args"); return -1; }
  FwdWs W(n_nodes, n_edges, steps, (flags & PDG_FLAG_SAVE) != 0, nullptr);
  const char* p = nullptr;
  size_t n = 0;
  const size_t nn = (size_t)W.N_pad * H, ne = (size_t)W.E_pad * H;
  switch (what) {
    case 0: p = (const char*)W.x_[t]; n = nn; break;
    case 1: p = (const char*)W.e_[t]; n = ne; break;
    case 2: p = (const char*)W.y2_[t]; n = ne; break;
    case 3: p = (const char*)W.Pa_[t]; n = nn; break;
    case 4: p = (const char*)W.Pb_[t]; n = nn; break;
    case 5: p = (const char*)W.aggraw_[t]; n = nn; break;
    case 6: p = (const char*)W.hq_[t]; n = nn; break;
    case 7: p = (const char*)W.y3_[t]; n = nn; break;
    case 8: p = (const char*)W.y_nenc; n = nn; break;
    case 9: p = (const char*)W.y_eenc; n = ne; break;
    case 10: p = (const char*)W.hd; n = nn; break;
    case 11: p = (const char*)W.parts_slot(t); n = (size_t)MAXP * 2; break;
    default: set_error("pdg_ws_offset: unknown tensor %d", what); return -1;
  }
  if (p == nullptr) { set_error("pdg_ws_offset: tensor not stored"); return -1; }
  *offset = (size_t)(p - (const char*)nullptr);
  *elems = n;
  return 0;
}
