// bf16 tensor-core versions of the EDGE encoder (PDG_PREC_BF16): edge_encoder of models.py:268-274 on the
// standardised edge weight (models.py:154-162), forward and backward.  The node encoder stays on the FFMA
// path (N rows only).  Same conventions as the other pdg_tc_*.cu kernels.
#include "pdg_ws.cuh"
#include "pdg_tc_tile.cuh"

namespace pdg {

__device__ __forceinline__ uint32_t tc_setup_enc(uint64_t* bars, int nbars, uint32_t* tmem_slot, uint32_t ncols) {
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

struct EdgeEncArgs {
  const float* edge_attr;
  const int32_t* perm;
  float mean, std;
  int scale_in;
  const float* W0;  // [128][1]
  const float* b0;
  const float* b2;
  float* y_out;  // bf16 rows [E_pad][128]
  double* parts;
  int E, n_tiles;
};
constexpr int TC_SMEM_EDGE_ENC = 2 * tc::TILE_BF16_BYTES + TM * 4 + 3 * H * 4 + 512 + 2048;

__global__ void __launch_bounds__(NT, 2)
k_edge_encoder_tc(EdgeEncArgs a, const uint8_t* __restrict__ imgW2) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* sm = tc_smem_base(smem_raw);
  uint8_t* sW2 = sm;
  uint8_t* tA = sW2 + tc::TILE_BF16_BYTES;
  float* feat = reinterpret_cast<float*>(tA + tc::TILE_BF16_BYTES);
  float* b2s = feat + TM;
  double* red = reinterpret_cast<double*>(b2s + H);
  uint64_t* bars = reinterpret_cast<uint64_t*>(red + 16);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2);
  const TcThread t;
  if (t.tid < H) b2s[t.tid] = a.b2[t.tid];
  const uint32_t tmem = tc_setup_enc(bars, 2, tmem_slot, 128);
  if (t.tid == 0) {
    tc::mbar_expect_tx(&bars[0], tc::TILE_BF16_BYTES);
    tc::bulk_g2s(sW2, imgW2, tc::TILE_BF16_BYTES, &bars[0]);
  }
  const int ch = t.tid & 15;
  float w0[8], b0[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { w0[j] = a.W0[ch * 8 + j]; b0[j] = a.b0[ch * 8 + j]; }
  pdl_sync();  // keeps the dependency chain transitive (the next kernel waits for this one only)
  double tot_s = 0, tot_ss = 0;
  uint32_t ph = 0;
  bool first = true;
  for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const int row0 = tile * TM;
    const int nvalid = min(TM, a.E - row0);
    if (t.tid < TM) {
      float v = 0.f;
      if (row0 + t.tid < a.E) {
        v = a.edge_attr[a.perm[row0 + t.tid]];
        if (a.scale_in) v = (v - a.mean) / a.std;
      }
      feat[t.tid] = v;
    }
    __syncthreads();
#pragma unroll
    for (int it = 0; it < 8; ++it) {
      const int r = (t.tid >> 4) + it * 16;
      const float f = feat[r];
      float h[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) h[j] = fmaxf(fmaf(w0[j], f, b0[j]), 0.f);
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
      __half* y = reinterpret_cast<__half*>(a.y_out) + ((size_t)row0 + t.row) * H + t.half * 64;  // fp16 rows
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
        row_store_global32_f16(y, v, hh);
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

struct EdgeEncBwdArgs {
  const float* g_in;   // d loss / d e_0, receiver order
  const float* y_raw;  // raw encoder output (bf16 rows)
  const float* scal;   // {c1, c2, mu, rstd} of the encoder LayerNorm
  const float* lnw;
  const float* edge_attr;
  const int32_t* perm;
  float mean, std;
  int scale_in;
  const float* W0;
  const float* b0;
  float* cta_grads;
  const float* gs;        // IG: device {S, 1/S} of k_grad_scale (the incoming gradient carries S)
  float* g_edge_attr;     // IG: d loss / d edge_attr [E], PyG edge order
  int E, n_tiles;
};
constexpr int TC_SMEM_EDGE_ENC_BWD = 3 * tc::TILE_BF16_BYTES + TM * 4 + 4 * H * 4 + 512 + 2048;
constexpr int TC_SMEM_EDGE_ENC_BWD_IG = TC_SMEM_EDGE_ENC_BWD + H * 4;  // + W0 [128]

// IG: also write d loss / d edge_attr = (dh0 . W0) / std_edge_weight / S at perm[row], formed from the fp32 TMEM values of
// dh0; the half-1 thread of a row hands its partial sum to the half-0 thread through its own (then dead) bytes of the h0
// tile.  The <false> instance is unchanged.
template <bool IG>
__global__ void __launch_bounds__(NT, 1)
k_edge_encoder_bwd_tc(EdgeEncBwdArgs a, const uint8_t* __restrict__ imgW2) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* sm = tc_smem_base(smem_raw);
  uint8_t* sW2 = sm;
  uint8_t* T0 = sW2 + tc::TILE_BF16_BYTES;  // dy -> dh0
  uint8_t* T1 = T0 + tc::TILE_BF16_BYTES;   // h0
  float* feat = reinterpret_cast<float*>(T1 + tc::TILE_BF16_BYTES);
  float* comb = feat + TM;  // [4][H]
  float* w0s = comb + 4 * H;  // IG: [H]
  uint64_t* bars = reinterpret_cast<uint64_t*>(w0s + (IG ? H : 0));
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2);
  const TcThread t;
  float* cg = a.cta_grads + (size_t)blockIdx.x * GRADP;
  if (IG && t.tid < H) w0s[t.tid] = a.W0[t.tid];
  const uint32_t tmem = tc_setup_enc(bars, 2, tmem_slot, 256);
  const uint32_t ACC = tmem, WORK = tmem + 128;
  if (t.tid == 0) {
    tc::mbar_expect_tx(&bars[0], tc::TILE_BF16_BYTES);
    tc::bulk_g2s(sW2, imgW2, tc::TILE_BF16_BYTES, &bars[0]);
  }
  pdl_sync();  // scal / g_in / y_raw come from the preceding kernels
  const float c1 = a.scal[0], c2 = a.scal[1], mu = a.scal[2], rstd = a.scal[3];
  const float iea = IG ? a.gs[1] / (a.scale_in ? a.std : 1.f) : 0.f;
  const int ch = t.tid & 15;
  float w0[8], b0[8], lw[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { w0[j] = a.W0[ch * 8 + j]; b0[j] = a.b0[ch * 8 + j]; lw[j] = a.lnw[ch * 8 + j]; }
  float db2[2] = {0.f, 0.f}, db0[2] = {0.f, 0.f}, dw0[2] = {0.f, 0.f};
  uint32_t ph = 0;
  bool first = true;
  for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const int row0 = tile * TM;
    const int nvalid = min(TM, a.E - row0);
    if (t.tid < TM) {
      float v = 0.f;
      if (row0 + t.tid < a.E) {
        v = a.edge_attr[a.perm[row0 + t.tid]];
        if (a.scale_in) v = (v - a.mean) / a.std;
      }
      feat[t.tid] = v;
    }
    __syncthreads();
#pragma unroll 4
    for (int it = 0; it < 8; ++it) {
      const int r = (t.tid >> 4) + it * 16;
      const size_t g = ((size_t)row0 + r) * H + ch * 8;
      float d[8] = {0, 0, 0, 0, 0, 0, 0, 0}, h[8];
      if (r < nvalid) {
        float gg[8], y[8];
        *reinterpret_cast<float4*>(gg) = *reinterpret_cast<const float4*>(a.g_in + g);
        *reinterpret_cast<float4*>(gg + 4) = *reinterpret_cast<const float4*>(a.g_in + g + 4);
        unpack8_f16(*reinterpret_cast<const uint4*>(reinterpret_cast<const __half*>(a.y_raw) + g), y);  // fp16 rows
#pragma unroll
        for (int j = 0; j < 8; ++j) d[j] = y[j] > 0.f ? rstd * gg[j] * lw[j] - c1 - c2 * (y[j] - mu) : 0.f;
      }
      const float f = feat[r];
#pragma unroll
      for (int j = 0; j < 8; ++j) h[j] = fmaxf(fmaf(w0[j], f, b0[j]), 0.f);
      *reinterpret_cast<uint4*>(T0 + tc::sw128_chunk(r, ch)) = tc::pack8_f16(d);
      *reinterpret_cast<uint4*>(T1 + tc::sw128_chunk(r, ch)) = tc::pack8_f16(h);
    }
    tc::fence_async_smem();
    __syncthreads();
    if (t.tid == 0) {
      if (first) tc::mbar_wait(&bars[0], 0);
      tc::fence_after_sync();
      tc::issue_gemm_mnmajor(ACC, tc::smem_u32(T0), tc::smem_u32(T1), !first);       // dW2 += dy^T h0
      tc::issue_gemm_k_mn(WORK, tc::smem_u32(T0), tc::smem_u32(sW2), false);          // dh0_pre = dy W2
      tc::mma_commit(&bars[1]);
    }
    tile_colsum2_f16(T0, db2);
    tc::mbar_wait(&bars[1], ph);
    tc::fence_after_sync();
    __syncthreads();  // every column walker is done with dy before the epilogue overwrites T0 with dh0
    float gi = 0.f;
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
          const float* w = w0s + t.half * 64 + hh * 32 + c8 * 8;  // warp-uniform: broadcast
          const float4 wa = *reinterpret_cast<const float4*>(w), wb = *reinterpret_cast<const float4*>(w + 4);
          gi = fmaf(d[0], wa.x, gi); gi = fmaf(d[1], wa.y, gi); gi = fmaf(d[2], wa.z, gi); gi = fmaf(d[3], wa.w, gi);
          gi = fmaf(d[4], wb.x, gi); gi = fmaf(d[5], wb.y, gi); gi = fmaf(d[6], wb.z, gi); gi = fmaf(d[7], wb.w, gi);
        }
      }
    }
    if (IG && t.half == 1) *reinterpret_cast<float*>(T1 + tc::sw128_chunk(t.row, 8)) = gi;  // read above by this thread only
    tc::fence_before_sync();
    __syncthreads();
    if (IG && t.half == 0 && t.row < nvalid)
      a.g_edge_attr[a.perm[row0 + t.row]] = (gi + *reinterpret_cast<const float*>(T1 + tc::sw128_chunk(t.row, 8))) * iea;
    {  // db0 = colsum(dh0), dW0[c] = sum_r dh0[r][c] * feat[r]   (thread = channel pair x 32-row quarter)
      const int cp = t.tid & 63, q = t.tid >> 6;
      float s0 = 0.f, s1 = 0.f, u0 = 0.f, u1 = 0.f;
#pragma unroll 8
      for (int r = q * 32; r < q * 32 + 32; ++r) {
        const float2 v = __half22float2(*reinterpret_cast<const __half2*>(T0 + tc::sw128_off(r, 2 * cp)));
        const float f = feat[r];
        s0 += v.x; s1 += v.y;
        u0 = fmaf(v.x, f, u0); u1 = fmaf(v.y, f, u1);
      }
      db0[0] += s0; db0[1] += s1; dw0[0] += u0; dw0[1] += u1;
    }
    ph ^= 1u;
    first = false;
    __syncthreads();
  }
  tmem_acc_flush(ACC, reinterpret_cast<float*>(T0), cg + param_offset(EE_W2), t.row, t.half, t.lane_base);  // T0 + T1 are dead
  colpart2_flush(db2, comb, cg + param_offset(EE_B2), true);
  colpart2_flush(db0, comb, cg + param_offset(EE_B0), true);
  colpart2_flush(dw0, comb, cg + param_offset(EE_W0), true);
  if (t.tid < TM) tc::bulk_wait_all();
  tc::fence_before_sync();
  __syncthreads();
  if (t.warp == 0) tc::tmem_dealloc(tmem, 256);
}

int launch_edge_encoder_tc(const float* edge_attr, const int32_t* perm, const pdg_norm_t* nrm, int scale_in, const float* W0,
                           const float* b0, const float* b2, float* y_out, double* parts, int E, int n_tiles,
                           const uint8_t* img, cudaStream_t st) {
  cudaError_t e = cudaFuncSetAttribute((const void*)k_edge_encoder_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM_EDGE_ENC);
  if (e != cudaSuccess) { set_error("k_edge_encoder_tc smem attribute: %s", cudaGetErrorString(e)); return -2; }
  EdgeEncArgs a{edge_attr, perm, nrm->mean_edge_weight, nrm->std_edge_weight, scale_in, W0, b0, b2, y_out, parts, E, n_tiles};
  const int cap = 2 * num_sms() < MAXP ? 2 * num_sms() : MAXP;
  e = launch_pdl(k_edge_encoder_tc, dim3(n_tiles < cap ? n_tiles : cap), dim3(NT), TC_SMEM_EDGE_ENC, st, a,
                 img + (size_t)IMG_EE_W2 * tc::TILE_BF16_BYTES);
  if (e != cudaSuccess) { set_error("k_edge_encoder_tc launch: %s", cudaGetErrorString(e)); return -2; }
  return 0;
}
int launch_edge_encoder_bwd_tc(const float* g_in, const float* y_raw, const float* scal, const float* lnw, const float* edge_attr,
                               const int32_t* perm, const pdg_norm_t* nrm, int scale_in, const float* W0, const float* b0,
                               float* cta_grads, const float* gs, float* grad_edge_attr, int E, int n_tiles, int grid,
                               const uint8_t* img, cudaStream_t st) {
  const bool ig = grad_edge_attr != nullptr;
  const void* fn = ig ? (const void*)k_edge_encoder_bwd_tc<true> : (const void*)k_edge_encoder_bwd_tc<false>;
  const int smem = ig ? TC_SMEM_EDGE_ENC_BWD_IG : TC_SMEM_EDGE_ENC_BWD;
  cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e != cudaSuccess) { set_error("k_edge_encoder_bwd_tc smem attribute: %s", cudaGetErrorString(e)); return -2; }
  EdgeEncBwdArgs a{g_in, y_raw, scal, lnw, edge_attr, perm, nrm->mean_edge_weight, nrm->std_edge_weight, scale_in, W0, b0, cta_grads,
                   gs, grad_edge_attr, E, n_tiles};
  e = launch_pdl(ig ? k_edge_encoder_bwd_tc<true> : k_edge_encoder_bwd_tc<false>, dim3(grid), dim3(NT), smem, st, a,
                 img + (size_t)IMG_EE_W2 * tc::TILE_BF16_BYTES);
  if (e != cudaSuccess) { set_error("k_edge_encoder_bwd_tc launch: %s", cudaGetErrorString(e)); return -2; }
  return 0;
}

}  // namespace pdg
