// bf16 tensor-core versions of the two node-level "ends" of the model (PDG_PREC_BF16):
//   k_node_encoder_tc      format_node_features (models.py:140-152) + node_encoder MLP (:260-266): raw output + LN partials
//   k_node_encoder_bwd_tc  its backward (first-layer gradients from the six recomputed input features)
//   k_decoder_tc           x_T = x_{T-1} + LN(y3_{T-1}); node_decoder (models.py:282-286, :316-321)
//   k_decoder_bwd_tc       its backward, first producer of the node gradient gx
// Same conventions as the other pdg_tc_*.cu kernels: bf16 SWIZZLE_128B operand tiles, weight images staged by TMA
// bulk copies, fp32 accumulation in TMEM, weight-gradient accumulators resident in TMEM and flushed by TMA
// reduce-adds, programmatic dependent launch.  The 6 -> 128 input layer and the 128 -> 3 output layer stay on FMA.
#include "pdg_ws.cuh"
#include "pdg_tc_tile.cuh"

namespace pdg {

__device__ __forceinline__ uint32_t tc_setup_ends(uint64_t* bars, int nbars, uint32_t* tmem_slot, uint32_t ncols) {
  if (threadIdx.x == 0) {
    for (int i = 0; i < nbars; ++i) tc::mbar_init(&bars[i], 1);
    tc::mbar_init_fence();
  }
  if ((threadIdx.x >> 5) == 0) tc::tmem_alloc(tmem_slot, ncols);
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  return *tmem_slot;
}
// thread = (chunk of 8 channels = tid & 15, row group = tid >> 4): combine the 16 row groups; scr = [16][H] floats
__device__ __forceinline__ void chunk8_flush(const float (&v)[8], float* scr, float* dst, bool add) {
  const int chunk = threadIdx.x & 15, grp = threadIdx.x >> 4;
  __syncthreads();
  *reinterpret_cast<float4*>(scr + grp * H + chunk * 8) = make_float4(v[0], v[1], v[2], v[3]);
  *reinterpret_cast<float4*>(scr + grp * H + chunk * 8 + 4) = make_float4(v[4], v[5], v[6], v[7]);
  __syncthreads();
  if (threadIdx.x < H) {
    float s = 0.f;
#pragma unroll
    for (int g = 0; g < 16; ++g) s += scr[g * H + threadIdx.x];
    dst[threadIdx.x] = add ? dst[threadIdx.x] + s : s;
  }
}

// ------------------------------------------------------------------------------------------------
struct NodeEncArgs {
  const float* mean_stress;
  const float* pos;
  const int64_t* types;
  pdg_norm_t nrm;
  int scale_in;
  const float* W0;  // [128][6]
  const float* b0;
  const float* b2;
  float* y_out;
  double* parts;
  int* nzflag;
  int N, n_tiles;
};
constexpr int TC_SMEM_NODE_ENC = 2 * tc::TILE_BF16_BYTES + TM * 8 * 4 + H * 4 + 512 + 2048;

__global__ void __launch_bounds__(NT, 1)
k_node_encoder_tc(NodeEncArgs a, const uint8_t* __restrict__ imgW2) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* sm = tc_smem_base(smem_raw);
  uint8_t* sW2 = sm;
  uint8_t* tA = sW2 + tc::TILE_BF16_BYTES;
  float* feat = reinterpret_cast<float*>(tA + tc::TILE_BF16_BYTES);  // [TM][8]
  float* b2s = feat + TM * 8;
  double* red = reinterpret_cast<double*>(b2s + H);
  uint64_t* bars = reinterpret_cast<uint64_t*>(red + 16);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2);
  const TcThread t;
  if (t.tid < H) b2s[t.tid] = a.b2[t.tid];
  const uint32_t tmem = tc_setup_ends(bars, 2, tmem_slot, 128);
  const int ch = t.tid & 15;
  float w0[8][6], b0[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    b0[k] = a.b0[ch * 8 + k];
#pragma unroll
    for (int j = 0; j < 6; ++j) w0[k][j] = a.W0[(ch * 8 + k) * 6 + j];
  }
  pdl_sync();  // the weight image comes from k_pack_all, the previous launch
  if (t.tid == 0) {
    tc::mbar_expect_tx(&bars[0], tc::TILE_BF16_BYTES);
    tc::bulk_g2s(sW2, imgW2, tc::TILE_BF16_BYTES, &bars[0]);
  }
  double tot_s = 0, tot_ss = 0;
  uint32_t ph = 0;
  bool first = true;
  for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const int row0 = tile * TM;
    const int nvalid = min(TM, a.N - row0);
    if (t.tid < TM) {
      float f[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      bool nz = false;
      if (row0 + t.tid < a.N) node_features(a.mean_stress, a.pos, a.types, a.nrm, a.scale_in, row0 + t.tid, f, nz);
#pragma unroll
      for (int j = 0; j < 6; ++j) feat[t.tid * 8 + j] = f[j];
      if (a.nzflag != nullptr && __any_sync(0xffffffffu, nz) && (t.tid & 31) == 0) atomicOr(a.nzflag, 1);  // warps 0-3, whole
    }
    __syncthreads();
#pragma unroll 2
    for (int it = 0; it < 8; ++it) {
      const int r = (t.tid >> 4) + it * 16;
      const float4 f03 = *reinterpret_cast<const float4*>(feat + r * 8);
      const float2 f45 = *reinterpret_cast<const float2*>(feat + r * 8 + 4);
      const float f[6] = {f03.x, f03.y, f03.z, f03.w, f45.x, f45.y};
      float h[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        float v = b0[k];
#pragma unroll
        for (int j = 0; j < 6; ++j) v = fmaf(w0[k][j], f[j], v);
        h[k] = fmaxf(v, 0.f);
      }
      *reinterpret_cast<uint4*>(tA + tc::sw128_chunk(r, ch)) = tc::pack8_f16(h);
    }
    tc::fence_async_smem();
    __syncthreads();
    if (t.tid == 0) {
      if (first) tc::mbar_wait(&bars[0], 0);
      tc::fence_after_sync();
      tc::issue_gemm_kmajor(tmem, tc::smem_u32(tA), tc::smem_u32(sW2), H, false);
      tc::mma_commit(&bars[1]);
    }
    first = false;
    tc::mbar_wait(&bars[1], ph);
    tc::fence_after_sync();
    float s = 0.f, ss = 0.f;
    {
      const bool ok = t.row < nvalid;
      float* y = a.y_out + ((size_t)row0 + t.row) * H + t.half * 64;
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        float v[32];
        tc::tmem_ld32(tmem + t.lane_base + (uint32_t)(t.half * 64 + hh * 32), v);
        tc::tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          v[j] = fmaxf(v[j] + b2s[t.half * 64 + hh * 32 + j], 0.f);
          if (ok) { s += v[j]; ss = fmaf(v[j], v[j], ss); }
        }
        row_store_global32(y, v, hh);
      }
    }
    double ds = s, dss = ss;
    block_sum2(ds, dss, red);
    if (t.tid == 0) { tot_s += ds; tot_ss += dss; }
    ph ^= 1u;
    tc::fence_before_sync();
    __syncthreads();
  }
  if (t.tid == 0) { a.parts[2 * blockIdx.x] = tot_s; a.parts[2 * blockIdx.x + 1] = tot_ss; }
  if (t.warp == 0) tc::tmem_dealloc(tmem, 128);
}

// ------------------------------------------------------------------------------------------------
struct NodeEncBwdArgs {
  const float* g_in;   // d loss / d x_0
  const float* y_raw;  // raw encoder output
  const float* scal;   // {c1, c2, mu, rstd} of the encoder LayerNorm
  const float* lnw;
  const float* mean_stress;
  const float* pos;
  const int64_t* types;
  pdg_norm_t nrm;
  int scale_in;
  const float* W0;
  const float* b0;
  float* cta_grads;
  const float* gs;        // IG: device {S, 1/S} of k_grad_scale (the incoming gradient carries S)
  float* g_mean_stress;   // IG: d loss / d mean_stress [N,3] or null
  float* g_pos;           // IG: d loss / d pos [N,2] or null
  int N, n_tiles;
};
constexpr int TC_SMEM_NODE_ENC_BWD = 3 * tc::TILE_BF16_BYTES + TM * 8 * 4 + 4 * H * 4 + 512 + 2048;
constexpr int TC_SMEM_NODE_ENC_BWD_IG = TC_SMEM_NODE_ENC_BWD + H * 8 * 4;  // + W0 staged as [128][8] (features 0-4 used)

// IG: also write the input gradient dfeat = dh0 W0 (features 0-4, un-standardised, times 1/S), formed from the fp32 TMEM
// values of dh0.  Each thread owns 64 channels of one row; the half-1 thread hands its five partial sums to the half-0
// thread of the row through its own (then dead) 128 bytes of the h0 tile.  The <false> instance is unchanged.
template <bool IG>
__global__ void __launch_bounds__(NT, 1)
k_node_encoder_bwd_tc(NodeEncBwdArgs a, const uint8_t* __restrict__ imgW2) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* sm = tc_smem_base(smem_raw);
  uint8_t* sW2 = sm;
  uint8_t* T0 = sW2 + tc::TILE_BF16_BYTES;  // dy -> dh0
  uint8_t* T1 = T0 + tc::TILE_BF16_BYTES;   // h0
  float* feat = reinterpret_cast<float*>(T1 + tc::TILE_BF16_BYTES);  // [TM][8]
  float* comb = feat + TM * 8;  // [4][H]
  float* w0s = comb + 4 * H;    // IG: [H][8]
  uint64_t* bars = reinterpret_cast<uint64_t*>(w0s + (IG ? H * 8 : 0));
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2);
  const TcThread t;
  float* cg = a.cta_grads + (size_t)blockIdx.x * GRADP;
  if (IG && t.tid < H) {
#pragma unroll
    for (int j = 0; j < 8; ++j) w0s[t.tid * 8 + j] = j < 5 ? a.W0[t.tid * 6 + j] : 0.f;
  }
  const uint32_t tmem = tc_setup_ends(bars, 2, tmem_slot, 256);
  const uint32_t ACC = tmem, WORK = tmem + 128;
  if (t.tid == 0) {
    tc::mbar_expect_tx(&bars[0], tc::TILE_BF16_BYTES);
    tc::bulk_g2s(sW2, imgW2, tc::TILE_BF16_BYTES, &bars[0]);
  }
  const int ch = t.tid & 15;
  float w0[8][6], b0[8], lw[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    b0[k] = a.b0[ch * 8 + k];
    lw[k] = a.lnw[ch * 8 + k];
#pragma unroll
    for (int j = 0; j < 6; ++j) w0[k][j] = a.W0[(ch * 8 + k) * 6 + j];
  }
  pdl_sync();  // scal / g_in come from the preceding kernels
  const float c1 = a.scal[0], c2 = a.scal[1], mu = a.scal[2], rstd = a.scal[3];
  const float ims = IG ? a.gs[1] / (a.scale_in ? a.nrm.std_mean_stress : 1.f) : 0.f;
  const float ipos = IG ? a.gs[1] / (a.scale_in ? a.nrm.std_pos : 1.f) : 0.f;
  float db2[2] = {0.f, 0.f}, db0[2] = {0.f, 0.f}, dw0[6][2];
#pragma unroll
  for (int j = 0; j < 6; ++j) { dw0[j][0] = 0.f; dw0[j][1] = 0.f; }
  uint32_t ph = 0;
  bool first = true;
  for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const int row0 = tile * TM;
    const int nvalid = min(TM, a.N - row0);
    if (t.tid < TM) {
      float f[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      bool nz;
      if (row0 + t.tid < a.N) node_features(a.mean_stress, a.pos, a.types, a.nrm, a.scale_in, row0 + t.tid, f, nz);
#pragma unroll
      for (int j = 0; j < 6; ++j) feat[t.tid * 8 + j] = f[j];
    }
    __syncthreads();
#pragma unroll 2
    for (int it = 0; it < 8; ++it) {
      const int r = (t.tid >> 4) + it * 16;
      const size_t g = ((size_t)row0 + r) * H + ch * 8;
      float d[8] = {0, 0, 0, 0, 0, 0, 0, 0}, h[8];
      if (r < nvalid) {
        float gg[8], y[8];
        *reinterpret_cast<float4*>(gg) = *reinterpret_cast<const float4*>(a.g_in + g);
        *reinterpret_cast<float4*>(gg + 4) = *reinterpret_cast<const float4*>(a.g_in + g + 4);
        *reinterpret_cast<float4*>(y) = *reinterpret_cast<const float4*>(a.y_raw + g);
        *reinterpret_cast<float4*>(y + 4) = *reinterpret_cast<const float4*>(a.y_raw + g + 4);
#pragma unroll
        for (int k = 0; k < 8; ++k) d[k] = y[k] > 0.f ? rstd * gg[k] * lw[k] - c1 - c2 * (y[k] - mu) : 0.f;
      }
      const float4 f03 = *reinterpret_cast<const float4*>(feat + r * 8);
      const float2 f45 = *reinterpret_cast<const float2*>(feat + r * 8 + 4);
      const float f[6] = {f03.x, f03.y, f03.z, f03.w, f45.x, f45.y};
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        float v = b0[k];
#pragma unroll
        for (int j = 0; j < 6; ++j) v = fmaf(w0[k][j], f[j], v);
        h[k] = fmaxf(v, 0.f);
      }
      *reinterpret_cast<uint4*>(T0 + tc::sw128_chunk(r, ch)) = tc::pack8_f16(d);
      *reinterpret_cast<uint4*>(T1 + tc::sw128_chunk(r, ch)) = tc::pack8_f16(h);
    }
    tc::fence_async_smem();
    __syncthreads();
    if (t.tid == 0) {
      if (first) tc::mbar_wait(&bars[0], 0);
      tc::fence_after_sync();
      tc::issue_gemm_mnmajor(ACC, tc::smem_u32(T0), tc::smem_u32(T1), !first);   // dW2 += dy^T h0
      tc::issue_gemm_k_mn(WORK, tc::smem_u32(T0), tc::smem_u32(sW2), false);      // dh0_pre = dy W2
      tc::mma_commit(&bars[1]);
    }
    tile_colsum2_f16(T0, db2);
    tc::mbar_wait(&bars[1], ph);
    tc::fence_after_sync();
    __syncthreads();  // every column walker is done with dy before the epilogue overwrites T0 with dh0
    float gi[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int hh = 0; hh < 2; ++hh) {
      float v[32];
      tc::tmem_ld32(WORK + t.lane_base + (uint32_t)(t.half * 64 + hh * 32), v);
      tc::tmem_ld_wait();
#pragma unroll
      for (int c8 = 0; c8 < 4; ++c8) {
        float h[8], d[8];
        row_load8(T1, t.row, t.half, hh * 4 + c8, h);
#pragma unroll
        for (int j = 0; j < 8; ++j) d[j] = h[j] > 0.f ? v[c8 * 8 + j] : 0.f;
        row_store8(T0, t.row, t.half, hh * 4 + c8, d);
        if (IG) {
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float* w = w0s + (t.half * 64 + hh * 32 + c8 * 8 + j) * 8;  // warp-uniform: broadcast
            const float4 w03 = *reinterpret_cast<const float4*>(w);
            gi[0] = fmaf(d[j], w03.x, gi[0]); gi[1] = fmaf(d[j], w03.y, gi[1]); gi[2] = fmaf(d[j], w03.z, gi[2]);
            gi[3] = fmaf(d[j], w03.w, gi[3]); gi[4] = fmaf(d[j], w[4], gi[4]);
          }
        }
      }
    }
    if (IG && t.half == 1) {  // chunks 8-9 of this row of T1: read above by this thread only
      *reinterpret_cast<float4*>(T1 + tc::sw128_chunk(t.row, 8)) = make_float4(gi[0], gi[1], gi[2], gi[3]);
      *reinterpret_cast<float*>(T1 + tc::sw128_chunk(t.row, 9)) = gi[4];
    }
    tc::fence_before_sync();
    __syncthreads();
    if (IG && t.half == 0 && t.row < nvalid) {
      const float4 p03 = *reinterpret_cast<const float4*>(T1 + tc::sw128_chunk(t.row, 8));
      const float p4 = *reinterpret_cast<const float*>(T1 + tc::sw128_chunk(t.row, 9));
      const int row = row0 + t.row;
      if (a.g_mean_stress != nullptr) {
        a.g_mean_stress[row * 3 + 0] = (gi[0] + p03.x) * ims;
        a.g_mean_stress[row * 3 + 1] = (gi[1] + p03.y) * ims;
        a.g_mean_stress[row * 3 + 2] = (gi[2] + p03.z) * ims;
      }
      if (a.g_pos != nullptr) {
        a.g_pos[row * 2 + 0] = (gi[3] + p03.w) * ipos;
        a.g_pos[row * 2 + 1] = (gi[4] + p4) * ipos;
      }
    }
    {  // db0 = colsum(dh0), dW0[c][j] = sum_r dh0[r][c] * feat[r][j]   (thread = channel pair x 32-row quarter)
      const int cp = t.tid & 63, q = t.tid >> 6;
      float s0 = 0.f, s1 = 0.f, u[6][2];
#pragma unroll
      for (int j = 0; j < 6; ++j) { u[j][0] = 0.f; u[j][1] = 0.f; }
#pragma unroll 4
      for (int r = q * 32; r < q * 32 + 32; ++r) {
        const float2 v = __half22float2(*reinterpret_cast<const __half2*>(T0 + tc::sw128_off(r, 2 * cp)));
        const float4 f03 = *reinterpret_cast<const float4*>(feat + r * 8);
        const float2 f45 = *reinterpret_cast<const float2*>(feat + r * 8 + 4);
        const float f[6] = {f03.x, f03.y, f03.z, f03.w, f45.x, f45.y};
        s0 += v.x; s1 += v.y;
#pragma unroll
        for (int j = 0; j < 6; ++j) { u[j][0] = fmaf(v.x, f[j], u[j][0]); u[j][1] = fmaf(v.y, f[j], u[j][1]); }
      }
      db0[0] += s0; db0[1] += s1;
#pragma unroll
      for (int j = 0; j < 6; ++j) { dw0[j][0] += u[j][0]; dw0[j][1] += u[j][1]; }
    }
    ph ^= 1u;
    first = false;
    __syncthreads();
  }
  tmem_acc_flush(ACC, reinterpret_cast<float*>(T0), cg + param_offset(NE_W2), t.row, t.half, t.lane_base);  // T0 + T1 are dead
  colpart2_flush(db2, comb, cg + param_offset(NE_B2), true);
  colpart2_flush(db0, comb, cg + param_offset(NE_B0), true);
  {  // dW0 is [128][6] row-major: channel c, feature j at c * 6 + j
    const int cp = t.tid & 63, q = t.tid >> 6;
#pragma unroll
    for (int j = 0; j < 6; ++j) {
      __syncthreads();
      comb[q * H + 2 * cp] = dw0[j][0];
      comb[q * H + 2 * cp + 1] = dw0[j][1];
      __syncthreads();
      if (t.tid < H) cg[param_offset(NE_W0) + t.tid * 6 + j] += (comb[t.tid] + comb[H + t.tid]) + (comb[2 * H + t.tid] + comb[3 * H + t.tid]);
    }
  }
  if (t.tid < TM) tc::bulk_wait_all();
  tc::fence_before_sync();
  __syncthreads();
  if (t.warp == 0) tc::tmem_dealloc(tmem, 256);
}

// ------------------------------------------------------------------------------------------------
constexpr int TC_SMEM_DEC = 2 * tc::TILE_BF16_BYTES + 4 * H * 4 + 2 * TM * 4 * 4 + 512 + 2048;

__global__ void __launch_bounds__(NT, 1)
k_decoder_tc(DecArgs a, const uint8_t* __restrict__ imgD1) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* sm = tc_smem_base(smem_raw);
  uint8_t* sD1 = sm;
  uint8_t* tA = sD1 + tc::TILE_BF16_BYTES;
  float* d1s = reinterpret_cast<float*>(tA + tc::TILE_BF16_BYTES);  // [H]
  float* d2s = d1s + H;                                              // [3][H]
  float* part = d2s + 3 * H;                                         // [2][TM][4]
  float* smf = part + 2 * TM * 4;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smf + 4);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2);
  const TcThread t;
  if (t.tid < H) {
    d1s[t.tid] = a.d1[t.tid];
#pragma unroll
    for (int o = 0; o < 3; ++o) d2s[o * H + t.tid] = a.D2[o * H + t.tid];
  }
  const uint32_t tmem = tc_setup_ends(bars, 2, tmem_slot, 128);
  if (t.tid == 0) {
    tc::mbar_expect_tx(&bars[0], tc::TILE_BF16_BYTES);
    tc::bulk_g2s(sD1, imgD1, tc::TILE_BF16_BYTES, &bars[0]);
  }
  const int ch = t.tid & 15;
  float lw[8], lb[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { lw[j] = a.lnw[ch * 8 + j]; lb[j] = a.lnb[ch * 8 + j]; }
  pdl_sync();
  const LnStat st = ln_stat_block(a.prev_parts, a.prev_count, smf);
  const bool live = a.nzflag == nullptr || *a.nzflag != 0;  // all-zero load case: zeros, not even un-standardised (models.py:294-299)
  uint32_t ph = 0;
  bool first = true;
  for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const size_t row0 = (size_t)tile * TM;
#pragma unroll 2
    for (int it = 0; it < 8; ++it) {
      const int r = (t.tid >> 4) + it * 16;
      const size_t g = (row0 + r) * H + ch * 8;
      float v[8];
      *reinterpret_cast<float4*>(v) = *reinterpret_cast<const float4*>(a.yprev + g);
      *reinterpret_cast<float4*>(v + 4) = *reinterpret_cast<const float4*>(a.yprev + g + 4);
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = (v[j] - st.mu) * st.rstd * lw[j] + lb[j];
      if (a.base != nullptr) {
        const float4 x0 = *reinterpret_cast<const float4*>(a.base + g);
        const float4 x1 = *reinterpret_cast<const float4*>(a.base + g + 4);
        v[0] += x0.x; v[1] += x0.y; v[2] += x0.z; v[3] += x0.w;
        v[4] += x1.x; v[5] += x1.y; v[6] += x1.z; v[7] += x1.w;
      }
      if (a.x_out != nullptr) {
        *reinterpret_cast<float4*>(a.x_out + g) = make_float4(v[0], v[1], v[2], v[3]);
        *reinterpret_cast<float4*>(a.x_out + g + 4) = make_float4(v[4], v[5], v[6], v[7]);
      }
      *reinterpret_cast<uint4*>(tA + tc::sw128_chunk(r, ch)) = tc::pack8_f16(v);
    }
    tc::fence_async_smem();
    __syncthreads();
    if (t.tid == 0) {
      if (first) tc::mbar_wait(&bars[0], 0);
      tc::fence_after_sync();
      tc::issue_gemm_kmajor(tmem, tc::smem_u32(tA), tc::smem_u32(sD1), H, false);  // x_T D1^T
      tc::mma_commit(&bars[1]);
    }
    first = false;
    tc::mbar_wait(&bars[1], ph);
    tc::fence_after_sync();
    {
      float p0 = 0.f, p1 = 0.f, p2 = 0.f;
      float* hd = a.hd_out ? a.hd_out + (row0 + t.row) * H + t.half * 64 : nullptr;
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        float v[32];
        tc::tmem_ld32(tmem + t.lane_base + (uint32_t)(t.half * 64 + hh * 32), v);
        tc::tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const int c = t.half * 64 + hh * 32 + j;
          v[j] = fmaxf(v[j] + d1s[c], 0.f);
          p0 = fmaf(v[j], d2s[c], p0);
          p1 = fmaf(v[j], d2s[H + c], p1);
          p2 = fmaf(v[j], d2s[2 * H + c], p2);
        }
        if (hd) row_store_global32(hd, v, hh);
      }
      *reinterpret_cast<float4*>(part + (t.half * TM + t.row) * 4) = make_float4(p0, p1, p2, 0.f);
    }
    tc::fence_before_sync();
    __syncthreads();
    for (int idx = t.tid; idx < TM * PDG_OUT; idx += NT) {
      const int r = idx / PDG_OUT, o = idx - r * PDG_OUT;
      const size_t row = row0 + r;
      if (row < (size_t)a.N) {
        const float dsum = part[r * 4 + o] + part[(TM + r) * 4 + o];
        a.out[row * PDG_OUT + o] = live ? (dsum + a.d2[o]) * a.out_scale + a.out_shift : 0.f;
      }
    }
    ph ^= 1u;
    __syncthreads();
  }
  if (t.warp == 0) tc::tmem_dealloc(tmem, 128);
}

// ------------------------------------------------------------------------------------------------
struct DecBwdArgs {
  const float* g_out;  // [N][3]
  float gscale;
  const float* gs;     // device {S, 1/S}: power-of-two scale of the whole backward (k_grad_scale), multiplied in here
  const float* hd;
  const float* x_T;
  const float* y3_last;
  const double* parts_prev;
  double count_prev;
  const float* D2;  // [3][128]
  float* gx;
  float* cta_grads;
  float* cs3;
  const int* nzflag;
  int N, n_tiles;
};
constexpr int TC_SMEM_DEC_BWD = 3 * tc::TILE_BF16_BYTES + TM * 4 * 4 + 16 * H * 4 + 512 + 2048;

__global__ void __launch_bounds__(NT, 1)
k_decoder_bwd_tc(DecBwdArgs a, const uint8_t* __restrict__ imgD1) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* sm = tc_smem_base(smem_raw);
  uint8_t* sD1 = sm;
  uint8_t* T0 = sD1 + tc::TILE_BF16_BYTES;  // d hd
  uint8_t* T1 = T0 + tc::TILE_BF16_BYTES;   // x_T
  float* S32 = reinterpret_cast<float*>(T0);  // fp32 staging aliasing T0 + T1 once their GEMMs completed
  float* gd = reinterpret_cast<float*>(T1 + tc::TILE_BF16_BYTES);  // [TM][4]
  float* scr = gd + TM * 4;                                         // [16][H]
  float* smf = scr + 16 * H;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smf + 4);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2);
  const TcThread t;
  float* cg = a.cta_grads + (size_t)blockIdx.x * GRADP;
  const uint32_t tmem = tc_setup_ends(bars, 2, tmem_slot, 256);
  const uint32_t ACC = tmem, WORK = tmem + 128;
  if (t.tid == 0) {
    tc::mbar_expect_tx(&bars[0], tc::TILE_BF16_BYTES);
    tc::bulk_g2s(sD1, imgD1, tc::TILE_BF16_BYTES, &bars[0]);
  }
  const int ch = t.tid & 15;
  float d2w[3][8];
#pragma unroll
  for (int o = 0; o < 3; ++o)
#pragma unroll
    for (int k = 0; k < 8; ++k) d2w[o][k] = a.D2[o * H + ch * 8 + k];
  pdl_sync();
  const float mu_prev = ln_stat_block(a.parts_prev, a.count_prev, smf).mu;
  const bool live = a.nzflag == nullptr || *a.nzflag != 0;  // all-zero load case: the output was the constant 0
  const float gsc = a.gscale * (a.gs != nullptr ? a.gs[0] : 1.f);
  float dD2[3][8], dd1[8] = {0, 0, 0, 0, 0, 0, 0, 0}, dd2 = 0.f;
#pragma unroll
  for (int o = 0; o < 3; ++o)
#pragma unroll
    for (int k = 0; k < 8; ++k) dD2[o][k] = 0.f;
  float cgx8[8] = {0}, cgy8[8] = {0};  // chunk-mapped ({ch*4..+3, 64+ch*4..+3}) column partials of the LayerNorm feeding x_T
  uint32_t ph = 0;
  bool first = true;
  for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const int row0 = tile * TM;
    const int nvalid = min(TM, a.N - row0);
    if (t.tid < TM) {
      const int row = row0 + t.tid;
      float g3[3];
#pragma unroll
      for (int o = 0; o < 3; ++o) g3[o] = (row < a.N && live) ? a.g_out[row * 3 + o] * gsc : 0.f;
      *reinterpret_cast<float4*>(gd + t.tid * 4) = make_float4(g3[0], g3[1], g3[2], 0.f);
    }
    __syncthreads();
    if (t.tid < 3) {
      float s = 0.f;
      for (int r = 0; r < nvalid; ++r) s += gd[r * 4 + t.tid];
      dd2 += s;
    }
#pragma unroll 2
    for (int it = 0; it < 8; ++it) {
      const int r = (t.tid >> 4) + it * 16;
      const size_t g = ((size_t)row0 + r) * H + ch * 8;
      const float4 g4 = *reinterpret_cast<const float4*>(gd + r * 4);
      float h[8], x[8], d[8];
      *reinterpret_cast<float4*>(h) = *reinterpret_cast<const float4*>(a.hd + g);
      *reinterpret_cast<float4*>(h + 4) = *reinterpret_cast<const float4*>(a.hd + g + 4);
      *reinterpret_cast<float4*>(x) = *reinterpret_cast<const float4*>(a.x_T + g);
      *reinterpret_cast<float4*>(x + 4) = *reinterpret_cast<const float4*>(a.x_T + g + 4);
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        d[k] = h[k] > 0.f ? g4.x * d2w[0][k] + g4.y * d2w[1][k] + g4.z * d2w[2][k] : 0.f;  // rows >= nvalid: g4 = 0
        dd1[k] += d[k];
        if (r < nvalid) {
          dD2[0][k] = fmaf(g4.x, h[k], dD2[0][k]);
          dD2[1][k] = fmaf(g4.y, h[k], dD2[1][k]);
          dD2[2][k] = fmaf(g4.z, h[k], dD2[2][k]);
        }
      }
      *reinterpret_cast<uint4*>(T0 + tc::sw128_chunk(r, ch)) = tc::pack8_f16(d);
      *reinterpret_cast<uint4*>(T1 + tc::sw128_chunk(r, ch)) = tc::pack8_f16(x);
    }
    tc::fence_async_smem();
    __syncthreads();
    if (t.tid == 0) {
      if (first) tc::mbar_wait(&bars[0], 0);
      tc::fence_after_sync();
      tc::issue_gemm_mnmajor(ACC, tc::smem_u32(T0), tc::smem_u32(T1), !first);   // dD1 += dhd^T x_T
      tc::issue_gemm_k_mn(WORK, tc::smem_u32(T0), tc::smem_u32(sD1), false);      // gx_T = dhd D1
      tc::mma_commit(&bars[1]);
    }
    tc::mbar_wait(&bars[1], ph);
    tc::fence_after_sync();
    __syncthreads();  // T0 / T1 are dead for every thread: the staging may overwrite them
    tmem_to_s32(WORK, S32, t.row, t.half, t.lane_base);
    tc::fence_before_sync();
    __syncthreads();
#pragma unroll 4
    for (int it = 0; it < 8; ++it) {  // gx rows leave coalesced; column partials of the previous LayerNorm
      const int r = (t.tid >> 4) + it * 16;
      const size_t g = ((size_t)row0 + r) * H + ch * 4;
      const float4 d0 = *reinterpret_cast<const float4*>(s32_ptr(S32, r, ch * 4));
      const float4 d1 = *reinterpret_cast<const float4*>(s32_ptr(S32, r, 64 + ch * 4));
      const float4 y0 = *reinterpret_cast<const float4*>(a.y3_last + g);
      const float4 y1 = *reinterpret_cast<const float4*>(a.y3_last + g + 64);
      *reinterpret_cast<float4*>(a.gx + g) = d0;
      *reinterpret_cast<float4*>(a.gx + g + 64) = d1;
      cgx8[0] += d0.x; cgx8[1] += d0.y; cgx8[2] += d0.z; cgx8[3] += d0.w;
      cgx8[4] += d1.x; cgx8[5] += d1.y; cgx8[6] += d1.z; cgx8[7] += d1.w;
      cgy8[0] = fmaf(d0.x, y0.x - mu_prev, cgy8[0]); cgy8[1] = fmaf(d0.y, y0.y - mu_prev, cgy8[1]);
      cgy8[2] = fmaf(d0.z, y0.z - mu_prev, cgy8[2]); cgy8[3] = fmaf(d0.w, y0.w - mu_prev, cgy8[3]);
      cgy8[4] = fmaf(d1.x, y1.x - mu_prev, cgy8[4]); cgy8[5] = fmaf(d1.y, y1.y - mu_prev, cgy8[5]);
      cgy8[6] = fmaf(d1.z, y1.z - mu_prev, cgy8[6]); cgy8[7] = fmaf(d1.w, y1.w - mu_prev, cgy8[7]);
    }
    ph ^= 1u;
    first = false;
    tc::fence_before_sync();
    __syncthreads();
  }
  tmem_acc_flush(ACC, S32, cg + param_offset(ND_W0), t.row, t.half, t.lane_base);
  acc_reduce_drain();
  __syncthreads();
  chunk8_flush(dd1, scr, cg + param_offset(ND_B0), true);
#pragma unroll
  for (int o = 0; o < 3; ++o) chunk8_flush(dD2[o], scr, cg + param_offset(ND_W2) + o * H, true);
  if (t.tid < 3) cg[param_offset(ND_B2) + t.tid] += dd2;
  chunkpart_flush(cgx8, scr, a.cs3 + (size_t)blockIdx.x * 2 * H);
  chunkpart_flush(cgy8, scr, a.cs3 + (size_t)blockIdx.x * 2 * H + H);
  if (t.tid < TM) tc::bulk_wait_all();
  tc::fence_before_sync();
  __syncthreads();
  if (t.warp == 0) tc::tmem_dealloc(tmem, 256);
}

// ------------------------------------------------------------------------------------------------
int launch_node_encoder_tc(const float* mean_stress, const float* pos, const int64_t* types, const pdg_norm_t* nrm, int scale_in,
                           const float* W0, const float* b0, const float* b2, float* y_out, double* parts, int* nzflag, int N,
                           int n_tiles, int grid, const uint8_t* img, cudaStream_t st) {
  NodeEncArgs a{mean_stress, pos, types, *nrm, scale_in, W0, b0, b2, y_out, parts, nzflag, N, n_tiles};
  return launch_named("k_node_encoder_tc", true, k_node_encoder_tc, dim3(grid), dim3(NT), TC_SMEM_NODE_ENC, st, a,
                      weight_img(img, IMG_NE_W2));
}
int launch_node_encoder_bwd_tc(const float* g_in, const float* y_raw, const float* scal, const float* lnw, const float* mean_stress,
                               const float* pos, const int64_t* types, const pdg_norm_t* nrm, int scale_in, const float* W0,
                               const float* b0, float* cta_grads, const float* gs, float* grad_mean_stress, float* grad_pos, int N,
                               int n_tiles, int grid, const uint8_t* img, cudaStream_t st) {
  NodeEncBwdArgs a{g_in, y_raw, scal, lnw, mean_stress, pos, types, *nrm, scale_in, W0, b0, cta_grads, gs, grad_mean_stress, grad_pos,
                   N, n_tiles};
  const bool ig = grad_mean_stress != nullptr || grad_pos != nullptr;
  return launch_named("k_node_encoder_bwd_tc", true, ig ? k_node_encoder_bwd_tc<true> : k_node_encoder_bwd_tc<false>, dim3(grid),
                      dim3(NT), ig ? TC_SMEM_NODE_ENC_BWD_IG : TC_SMEM_NODE_ENC_BWD, st, a, weight_img(img, IMG_NE_W2));
}
int launch_decoder_tc(const DecArgs& a, const uint8_t* img, int grid, cudaStream_t st) {
  return launch_named("k_decoder_tc", true, k_decoder_tc, dim3(grid), dim3(NT), TC_SMEM_DEC, st, a, weight_img(img, IMG_ND_W0));
}
int launch_decoder_bwd_tc(const float* g_out, float gscale, const float* gs, const float* hd, const float* x_T, const float* y3_last,
                          const double* parts_prev, double count_prev, const float* D2, float* gx, float* cta_grads, float* cs3,
                          const int* nzflag, int N, int n_tiles, int grid, const uint8_t* img, cudaStream_t st) {
  DecBwdArgs a{g_out, gscale, gs, hd, x_T, y3_last, parts_prev, count_prev, D2, gx, cta_grads, cs3, nzflag, N, n_tiles};
  return launch_named("k_decoder_bwd_tc", true, k_decoder_bwd_tc, dim3(grid), dim3(NT), TC_SMEM_DEC_BWD, st, a,
                      weight_img(img, IMG_ND_W0));
}

}  // namespace pdg
