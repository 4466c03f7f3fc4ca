// bf16 tensor-core (tcgen05 / TMEM) versions of the node-level kernels (PDG_PREC_BF16):
//   k_node_pre_tc          x_t = x + LN(y3);  Pa = x_t Wa^T, Pb = x_t Wb^T          (models.py:224, 233-238)
//   k_node_update_tc       agg affine; y3 = relu(relu([agg,x] V1^T + c1) V2^T + c2)  (models.py:240-243)
//   k_node_update_bwd_tc   backward of k_node_update (weight gradients in persistent TMEM accumulators)
//   k_node_pre_bwd_tc      sender gather of dhm/dhn + backward of the Pa/Pb projections
// Same conventions as pdg_tc_fwd.cu / pdg_tc_bwd3.cu: bf16 SWIZZLE_128B operand tiles, weights
// staged once per CTA by TMA bulk copies, fp32 accumulation / statistics / storage.
#include "pdg_ws.cuh"
#include "pdg_tc_tile.cuh"

// Tuning knobs (compile-time; defaults are the measured configuration).  Both trade registers for loads in flight:
//   PDG_NODE_BWD_ROWS   row iterations of k_node_update_bwd_tc's two load phases unrolled together (4 = two batches of
//                       loads per phase; 8 = one batch, 254 registers, no spills: 57.3 -> 55.7 us, step time unchanged)
//   PDG_PRE_BWD_GB      sender-gather batch of k_node_pre_bwd_tc (edges in flight per row)
#ifndef PDG_NODE_BWD_ROWS
#define PDG_NODE_BWD_ROWS 4
#endif
#ifndef PDG_PRE_BWD_GB
#define PDG_PRE_BWD_GB 8
#endif
#define PDG_PRAGMA_(x) _Pragma(#x)
#define PDG_UNROLL(n) PDG_PRAGMA_(unroll n)

namespace pdg {

#ifdef PDG_PHASE_TIMERS
__device__ unsigned long long g_phase_node[64];  // [0,16) node_update_bwd, [16,32) node_pre_bwd: first tile of the CTA; +32: later tiles
#define PHN(i) do { if (blockIdx.x == 0 && threadIdx.x == 0) { unsigned long long _t = clock64(); g_phase_node[(i) + _toff] += _t - _tl; _tl = _t; } } while (0)
#define PHN_INIT unsigned long long _tl = clock64(); int _toff = 0
#else
#define PHN(i) do {} while (0)
#define PHN_INIT do {} while (0)
#endif

// common prologue: barriers, TMEM, weight images.  nimg images are copied back to back into smem.
struct TcSetup {
  uint32_t tmem;
};
__device__ __forceinline__ uint32_t tc_setup(uint64_t* bars, int nbars, uint32_t* tmem_slot, uint32_t ncols) {
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

// A node tile is one contiguous 64 KB block of every [N_pad,128] fp32 array: thread 0 asks the copy engine to pull this
// CTA's blocks into L2 (cp.async.bulk.prefetch.L2) so the register-staged row loops below pay L2, not DRAM, latency.
// Arrays saved by the forward are requested BEFORE the dependent-launch wait (they are many launches old), the
// predecessors' outputs after it.
__device__ __forceinline__ void prefetch_node_tiles(const float* p, int n_tiles) {
  if (p != nullptr)
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) tc::bulk_prefetch_l2(p + (size_t)tile * TM * H, TM * H * 4);
}

// ------------------------------------------------------------------------------------------------
constexpr int TC_SMEM_NODE_PRE = 3 * tc::TILE_BF16_BYTES + H * 4 + 256 + 2048;

__global__ void __launch_bounds__(NT, 2)
k_node_pre_tc(NodePreArgs a, const uint8_t* __restrict__ imgWA, const uint8_t* __restrict__ imgWB) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* sm = tc_smem_base(smem_raw);
  uint8_t* sWA = sm;
  uint8_t* sWB = sWA + tc::TILE_BF16_BYTES;
  uint8_t* tA = sWB + tc::TILE_BF16_BYTES;
  float* b1s = reinterpret_cast<float*>(tA + tc::TILE_BF16_BYTES);  // [H]
  float* smf = b1s + H;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smf + 4);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2);
  const TcThread t;
  if (t.tid < H) b1s[t.tid] = a.b1[t.tid];
  const uint32_t tmem = tc_setup(bars, 2, tmem_slot, 256);
  if (t.tid == 0) {
    tc::mbar_expect_tx(&bars[0], 2 * tc::TILE_BF16_BYTES);
    tc::bulk_g2s(sWA, imgWA, tc::TILE_BF16_BYTES, &bars[0]);
    tc::bulk_g2s(sWB, imgWB, tc::TILE_BF16_BYTES, &bars[0]);
  }
  if (t.tid == 0) prefetch_node_tiles(a.base, a.n_tiles);  // x of the previous step: several launches old
  pdl_sync();
  if (t.tid == 0) prefetch_node_tiles(a.yprev, a.n_tiles);
  const LnStat st = ln_stat_block(a.prev_parts, a.prev_count, smf);
  const int ch = t.tid & 15;
  float lw[8], lb[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { lw[j] = a.lnw[ch * 8 + j]; lb[j] = a.lnb[ch * 8 + j]; }
  uint32_t ph = 0;
  bool first = true;
  for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const size_t row0 = (size_t)tile * TM;
#pragma unroll 4
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
      *reinterpret_cast<float4*>(a.x_out + g) = make_float4(v[0], v[1], v[2], v[3]);
      *reinterpret_cast<float4*>(a.x_out + g + 4) = make_float4(v[4], v[5], v[6], v[7]);
      if (a.aggraw_zero != nullptr) {  // the edge kernel's segment sums (stores + two-addend atomics) start from zero
        *reinterpret_cast<float4*>(a.aggraw_zero + g) = make_float4(0.f, 0.f, 0.f, 0.f);
        *reinterpret_cast<float4*>(a.aggraw_zero + g + 4) = make_float4(0.f, 0.f, 0.f, 0.f);
      }
      *reinterpret_cast<uint4*>(tA + tc::sw128_chunk(r, ch)) = tc::pack8_f16(v);
    }
    tc::fence_async_smem();
    __syncthreads();
    if (t.tid == 0) {
      if (first) tc::mbar_wait(&bars[0], 0);
      tc::fence_after_sync();
      // the finished operand tile is what k_node_update*_tc / k_node_pre_bwd_tc need of x_t: one 32 KB bulk store of the
      // swizzled image; the commit below is issued only after the copy engine has read the tile, so whoever waits for
      // the accumulators may overwrite tA
      if (a.x_img != nullptr) {
        tc::bulk_s2g(a.x_img + (size_t)tile * tc::TILE_BF16_BYTES, tA, tc::TILE_BF16_BYTES);
        tc::bulk_commit();
      }
      tc::issue_gemm_kmajor(tmem, tc::smem_u32(tA), tc::smem_u32(sWA), H, false);
      tc::issue_gemm_kmajor(tmem + 128, tc::smem_u32(tA), tc::smem_u32(sWB), H, false);
      if (a.x_img != nullptr) tc::bulk_wait_read();
      tc::mma_commit(&bars[1]);
    }
    first = false;
    tc::mbar_wait(&bars[1], ph);
    tc::fence_after_sync();
    // Pa / Pb leave as fp16 rows (256 B): they are only ever gathered as addends of the fp16 hidden tiles
    __half* pa = reinterpret_cast<__half*>(a.Pa) + (row0 + t.row) * H + t.half * 64;
    __half* pb = reinterpret_cast<__half*>(a.Pb) + (row0 + t.row) * H + t.half * 64;
#pragma unroll
    for (int hh = 0; hh < 2; ++hh) {
      float v[32];
      tc::tmem_ld32(tmem + t.lane_base + (uint32_t)(t.half * 64 + hh * 32), v);
      tc::tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] += b1s[t.half * 64 + hh * 32 + j];  // Pa rows carry the layer-1 bias of the edge MLP
#pragma unroll
      for (int c8 = 0; c8 < 4; c8 += 2) tc::stg256(pa + hh * 32 + c8 * 8, tc::pack8_f16(v + c8 * 8), tc::pack8_f16(v + c8 * 8 + 8));
      tc::tmem_ld32(tmem + 128 + t.lane_base + (uint32_t)(t.half * 64 + hh * 32), v);
      tc::tmem_ld_wait();
#pragma unroll
      for (int c8 = 0; c8 < 4; c8 += 2) tc::stg256(pb + hh * 32 + c8 * 8, tc::pack8_f16(v + c8 * 8), tc::pack8_f16(v + c8 * 8 + 8));
    }
    ph ^= 1u;
    tc::fence_before_sync();
    __syncthreads();
  }
  if (t.tid == 0) tc::bulk_wait_all();  // image stores have landed before the grid completes
  if (t.warp == 0) tc::tmem_dealloc(tmem, 256);
}

// ------------------------------------------------------------------------------------------------
constexpr int TC_SMEM_NODE_UPD = 5 * tc::TILE_BF16_BYTES + 2 * H * 4 + 512 + 2048;

__global__ void __launch_bounds__(NT, 1)
k_node_update_tc(NodeUpdArgs a, const uint8_t* __restrict__ imgVA, const uint8_t* __restrict__ imgVX,
                 const uint8_t* __restrict__ imgV2) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* sm = tc_smem_base(smem_raw);
  uint8_t* sVA = sm;
  uint8_t* sVX = sVA + tc::TILE_BF16_BYTES;
  uint8_t* sV2 = sVX + tc::TILE_BF16_BYTES;
  uint8_t* A0 = sV2 + tc::TILE_BF16_BYTES;
  uint8_t* A1 = A0 + tc::TILE_BF16_BYTES;
  float* c1s = reinterpret_cast<float*>(A1 + tc::TILE_BF16_BYTES);
  float* c2s = c1s + H;
  double* red = reinterpret_cast<double*>(c2s + H);
  float* smf = reinterpret_cast<float*>(red + 16);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smf + 4);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 4);
  const TcThread t;
  if (t.tid < H) { c1s[t.tid] = a.c1[t.tid]; c2s[t.tid] = a.c2[t.tid]; }
  const uint32_t tmem = tc_setup(bars, 4, tmem_slot, 256);
  const bool ximg = a.x_img != nullptr;  // x_t arrives as the operand image k_node_pre_tc wrote (bulk copy, no registers)
  if (t.tid == 0) {
    tc::mbar_expect_tx(&bars[0], 3 * tc::TILE_BF16_BYTES);
    tc::bulk_g2s(sVA, imgVA, tc::TILE_BF16_BYTES, &bars[0]);
    tc::bulk_g2s(sVX, imgVX, tc::TILE_BF16_BYTES, &bars[0]);
    tc::bulk_g2s(sV2, imgV2, tc::TILE_BF16_BYTES, &bars[0]);
  }
  if (t.tid == 0 && !ximg) prefetch_node_tiles(a.x_t, a.n_tiles);  // written two launches ago (k_node_pre_tc)
  if (t.tid == 0 && ximg && (int)blockIdx.x < a.n_tiles) {  // first tile's image: two launches old, fetched under the predecessor's tail
    tc::mbar_expect_tx(&bars[3], tc::TILE_BF16_BYTES);
    tc::bulk_g2s(A1, a.x_img + (size_t)blockIdx.x * tc::TILE_BF16_BYTES, tc::TILE_BF16_BYTES, &bars[3]);
  }
  pdl_sync();
  if (t.tid == 0) prefetch_node_tiles(a.aggraw, a.n_tiles);
  const LnStat st = ln_stat_block(a.parts1, a.count1, smf);
  const int ch = t.tid & 15;
  float we[8], be[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { we[j] = a.lnw_e[ch * 8 + j]; be[j] = a.lnb_e[ch * 8 + j]; }
  double tot_s = 0, tot_ss = 0;
  uint32_t ph = 0;
  bool first = true;
  for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const int row0 = tile * TM;
    const int nvalid = min(TM, a.N - row0);
#pragma unroll 4
    for (int it = 0; it < 8; ++it) {
      const int r = (t.tid >> 4) + it * 16;
      const int rw = row0 + r;
      const size_t g = (size_t)rw * H + ch * 8;
      const float deg = rw < a.N ? (float)(a.rowptr[rw + 1] - a.rowptr[rw]) : 0.f;
      const float dm = deg * st.mu;
      float v[8];
      *reinterpret_cast<float4*>(v) = *reinterpret_cast<const float4*>(a.aggraw + g);
      *reinterpret_cast<float4*>(v + 4) = *reinterpret_cast<const float4*>(a.aggraw + g + 4);
      if (!ximg) {
        float x[8];
        *reinterpret_cast<float4*>(x) = *reinterpret_cast<const float4*>(a.x_t + g);
        *reinterpret_cast<float4*>(x + 4) = *reinterpret_cast<const float4*>(a.x_t + g + 4);
        *reinterpret_cast<uint4*>(A1 + tc::sw128_chunk(r, ch)) = tc::pack8_f16(x);
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = (v[j] - dm) * st.rstd * we[j] + deg * be[j];
      *reinterpret_cast<uint4*>(A0 + tc::sw128_chunk(r, ch)) = tc::pack8_f16(v);
    }
    tc::fence_async_smem();
    __syncthreads();
    if (t.tid == 0) {
      if (first) tc::mbar_wait(&bars[0], 0);
      if (ximg) tc::mbar_wait(&bars[3], ph);
      tc::fence_after_sync();
      if (a.agg_img != nullptr) {  // training: the aggregate's operand tile is the backward's operand too
        tc::bulk_s2g(a.agg_img + (size_t)tile * tc::TILE_BF16_BYTES, A0, tc::TILE_BF16_BYTES);
        tc::bulk_commit();
      }
      tc::issue_gemm_kmajor(tmem, tc::smem_u32(A0), tc::smem_u32(sVA), H, false);
      tc::issue_gemm_kmajor(tmem, tc::smem_u32(A1), tc::smem_u32(sVX), H, true);
      if (a.agg_img != nullptr) tc::bulk_wait_read();  // A0 is overwritten by the hidden tile after the wait below
      tc::mma_commit(&bars[1]);
    }
    first = false;
    tc::mbar_wait(&bars[1], ph);
    tc::fence_after_sync();
    if (t.tid == 0 && ximg && tile + (int)gridDim.x < a.n_tiles) {  // A1 is free (its GEMM completed): next tile's x_t image
      tc::mbar_expect_tx(&bars[3], tc::TILE_BF16_BYTES);
      tc::bulk_g2s(A1, a.x_img + (size_t)(tile + gridDim.x) * tc::TILE_BF16_BYTES, tc::TILE_BF16_BYTES, &bars[3]);
    }
    {
      float* hq = (a.hq_out && a.hq_img == nullptr) ? a.hq_out + ((size_t)row0 + t.row) * H + t.half * 64 : nullptr;
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        float v[32];
        tc::tmem_ld32(tmem + t.lane_base + (uint32_t)(t.half * 64 + hh * 32), v);
        tc::tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j] + c1s[t.half * 64 + hh * 32 + j], 0.f);
        if (hq) row_store_global32(hq, v, hh);
#pragma unroll
        for (int c8 = 0; c8 < 4; ++c8) row_store8(A0, t.row, t.half, hh * 4 + c8, v + c8 * 8);
      }
    }
    tc::fence_before_sync();
    tc::fence_async_smem();
    __syncthreads();
    if (t.tid == 0) {
      tc::fence_after_sync();
      if (a.hq_img != nullptr) {  // the hidden activation leaves as its fp16 operand image (the backward needs nothing else of it)
        tc::bulk_s2g(a.hq_img + (size_t)tile * tc::TILE_BF16_BYTES, A0, tc::TILE_BF16_BYTES);
        tc::bulk_commit();
      }
      tc::issue_gemm_kmajor(tmem + 128, tc::smem_u32(A0), tc::smem_u32(sV2), H, false);
      if (a.hq_img != nullptr) tc::bulk_wait_read();
      tc::mma_commit(&bars[2]);
    }
    tc::mbar_wait(&bars[2], ph);
    tc::fence_after_sync();
    float s = 0.f, ss = 0.f;
    {
      const bool ok = t.row < nvalid;
      float* y3 = a.y3_out + ((size_t)row0 + t.row) * H + t.half * 64;
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        float v[32];
        tc::tmem_ld32(tmem + 128 + t.lane_base + (uint32_t)(t.half * 64 + hh * 32), v);
        tc::tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          v[j] = fmaxf(v[j] + c2s[t.half * 64 + hh * 32 + j], 0.f);
          if (ok) { s += v[j]; ss = fmaf(v[j], v[j], ss); }
        }
        row_store_global32(y3, v, hh);
      }
    }
    double ds = s, dss = ss;
    block_sum2(ds, dss, red);
    if (t.tid == 0) { tot_s += ds; tot_ss += dss; }
    ph ^= 1u;
    tc::fence_before_sync();
    __syncthreads();
  }
  if (t.tid == 0) { a.parts3[2 * blockIdx.x] = tot_s; a.parts3[2 * blockIdx.x + 1] = tot_ss; }
  if (t.tid == 0) tc::bulk_wait_all();  // image stores have landed before the grid completes
  if (t.warp == 0) tc::tmem_dealloc(tmem, 256);
}

// ------------------------------------------------------------------------------------------------
constexpr int TC_SMEM_NODE_UPD_BWD = 6 * tc::TILE_BF16_BYTES + 4 * H * 4 + 512 + 2048;

__global__ void __launch_bounds__(NT, 1)
k_node_update_bwd_tc(NodeUpdBwdArgs a, const uint8_t* __restrict__ imgVA, const uint8_t* __restrict__ imgVX,
                     const uint8_t* __restrict__ imgV2) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* sm = tc_smem_base(smem_raw);
  uint8_t* sVA = sm;
  uint8_t* sVX = sVA + tc::TILE_BF16_BYTES;
  uint8_t* sV2 = sVX + tc::TILE_BF16_BYTES;
  uint8_t* T0 = sV2 + tc::TILE_BF16_BYTES;  // dy3 -> dhq
  uint8_t* T1 = T0 + tc::TILE_BF16_BYTES;   // hq  -> agg
  uint8_t* T2 = T1 + tc::TILE_BF16_BYTES;   // x_t
  float* S32 = reinterpret_cast<float*>(T1);  // fp32 staging aliasing T1 + T2 once both are dead
  float* comb = reinterpret_cast<float*>(T2 + tc::TILE_BF16_BYTES);  // [2][H]
  float* smf = comb + 2 * H;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smf + 4);  // 0 weights, 1..3 MMA groups, 4 x_t + hq images, 5 aggregate image
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 6);
  const TcThread t;
  float* cg = a.cta_grads + (size_t)blockIdx.x * GRADP;
  const uint32_t tmem = tc_setup(bars, 6, tmem_slot, 512);
  const uint32_t ACC_V2 = tmem, ACC_VA = tmem + 128, ACC_VX = tmem + 256, WORK = tmem + 384;
  // The forward left hq, the aggregate and x_t as fp16 OPERAND-TILE IMAGES (32 KB per tile): they are bulk-copied straight
  // into T1 / T2 by the copy engine while the dy3 tile is built -- half the bytes of the fp32 rows, no register staging
  // and no second rounding (the backward multiplies exactly the tiles the forward multiplied).
  const bool imgs = a.hq_img != nullptr;
  auto prefetch_img = [&](const uint8_t* p) {
    if (p != nullptr)
      for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) tc::bulk_prefetch_l2(p + (size_t)tile * tc::TILE_BF16_BYTES, tc::TILE_BF16_BYTES);
  };
  if (t.tid == 0) {
    tc::mbar_expect_tx(&bars[0], 3 * tc::TILE_BF16_BYTES);
    tc::bulk_g2s(sVA, imgVA, tc::TILE_BF16_BYTES, &bars[0]);
    tc::bulk_g2s(sVX, imgVX, tc::TILE_BF16_BYTES, &bars[0]);
    tc::bulk_g2s(sV2, imgV2, tc::TILE_BF16_BYTES, &bars[0]);
  }
  if (t.tid == 0) {  // forward-saved state of this step
    prefetch_node_tiles(a.y3, a.n_tiles);
    if (imgs) {
      if ((int)blockIdx.x < a.n_tiles) {  // first tile: images straight into the operand buffers, under the predecessor's tail
        tc::mbar_expect_tx(&bars[4], 2 * tc::TILE_BF16_BYTES);
        tc::bulk_g2s(T2, a.x_img + (size_t)blockIdx.x * tc::TILE_BF16_BYTES, tc::TILE_BF16_BYTES, &bars[4]);
        tc::bulk_g2s(T1, a.hq_img + (size_t)blockIdx.x * tc::TILE_BF16_BYTES, tc::TILE_BF16_BYTES, &bars[4]);
      }
      prefetch_img(a.agg_img);
      if ((int)(blockIdx.x + gridDim.x) < a.n_tiles) { prefetch_img(a.x_img); prefetch_img(a.hq_img); }
    } else {
      prefetch_node_tiles(a.hq, a.n_tiles);
      prefetch_node_tiles(a.x_t, a.n_tiles);
    }
    prefetch_node_tiles(a.aggraw, a.n_tiles);
  }
  pdl_sync();
  if (t.tid == 0) prefetch_node_tiles(a.gx, a.n_tiles);
  const LnStat st1 = ln_stat_block(a.parts1, a.count1, smf);
  const float c1 = a.scal3[0], c2 = a.scal3[1], mu3 = a.scal3[2], rstd3 = a.scal3[3];
  const int ch = t.tid & 15;
  float wn[8], we[8], be[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { wn[j] = a.lnw_n[ch * 8 + j]; we[j] = a.lnw_e[ch * 8 + j]; be[j] = a.lnb_e[ch * 8 + j]; }
  float dc2 = 0.f, dc1 = 0.f;
  float cg8[8] = {0}, cgy8[8] = {0};  // chunk-mapped LN1 column partials
  float4 sw0 = *reinterpret_cast<const float4*>(a.lnw_e + ch * 4), sw1 = *reinterpret_cast<const float4*>(a.lnw_e + 64 + ch * 4);
  sw0.x *= st1.rstd; sw0.y *= st1.rstd; sw0.z *= st1.rstd; sw0.w *= st1.rstd;
  sw1.x *= st1.rstd; sw1.y *= st1.rstd; sw1.z *= st1.rstd; sw1.w *= st1.rstd;
  uint32_t ph = 0;
  bool first = true;
  const uint32_t s0 = tc::smem_u32(T0), s1 = tc::smem_u32(T1), s2 = tc::smem_u32(T2);
  PHN_INIT;
  for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const int row0 = tile * TM;
    const int nvalid = min(TM, a.N - row0);
    const size_t grow = ((size_t)row0 + t.row) * H + t.half * 64;
    PHN(0);
    if (imgs && !first && t.tid == 0) {  // T1 / T2 held the previous tile's fp32 staging (generic accesses, fenced below the loop)
      tc::mbar_expect_tx(&bars[4], 2 * tc::TILE_BF16_BYTES);
      tc::bulk_g2s(T2, a.x_img + (size_t)tile * tc::TILE_BF16_BYTES, tc::TILE_BF16_BYTES, &bars[4]);
      tc::bulk_g2s(T1, a.hq_img + (size_t)tile * tc::TILE_BF16_BYTES, tc::TILE_BF16_BYTES, &bars[4]);
    }
    // dy3 -> T0 ; hq -> T1
    PDG_UNROLL(PDG_NODE_BWD_ROWS)
    for (int it = 0; it < 8; ++it) {
      const int r = (t.tid >> 4) + it * 16;
      const size_t g = ((size_t)row0 + r) * H + ch * 8;
      float d[8] = {0, 0, 0, 0, 0, 0, 0, 0};
      if (r < nvalid) {
        float gg[8], y[8];
        *reinterpret_cast<float4*>(gg) = *reinterpret_cast<const float4*>(a.gx + g);
        *reinterpret_cast<float4*>(gg + 4) = *reinterpret_cast<const float4*>(a.gx + g + 4);
        *reinterpret_cast<float4*>(y) = *reinterpret_cast<const float4*>(a.y3 + g);
        *reinterpret_cast<float4*>(y + 4) = *reinterpret_cast<const float4*>(a.y3 + g + 4);
#pragma unroll
        for (int j = 0; j < 8; ++j) d[j] = y[j] > 0.f ? rstd3 * gg[j] * wn[j] - c1 - c2 * (y[j] - mu3) : 0.f;
      }
      *reinterpret_cast<uint4*>(T0 + tc::sw128_chunk(r, ch)) = tc::pack8_f16(d);
      if (!imgs) {
        float hq[8];
        *reinterpret_cast<float4*>(hq) = *reinterpret_cast<const float4*>(a.hq + g);
        *reinterpret_cast<float4*>(hq + 4) = *reinterpret_cast<const float4*>(a.hq + g + 4);
        *reinterpret_cast<uint4*>(T1 + tc::sw128_chunk(r, ch)) = tc::pack8_f16(hq);
      }
    }
    tc::fence_async_smem();
    __syncthreads();
    PHN(1);
    if (t.tid == 0) {
      if (first) tc::mbar_wait(&bars[0], 0);
      if (imgs) tc::mbar_wait(&bars[4], ph);
      tc::fence_after_sync();
      tc::issue_gemm_mnmajor(ACC_V2, s0, s1, !first);          // dV2 += dy3^T hq
      tc::issue_gemm_k_mn(WORK, s0, tc::smem_u32(sV2), false);  // dhq_pre = dy3 V2
      tc::mma_commit(&bars[1]);
    }
    dc2 += tile_colsum_f16(T0);
    tc::mbar_wait(&bars[1], ph);
    tc::fence_after_sync();
    if (imgs) tc::mbar_wait(&bars[4], ph);  // every thread: the hq image (read below through the generic proxy) has landed
    __syncthreads();  // every column walker is done with dy3 before the epilogue overwrites T0 with dhq
    PHN(2);
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
      }
    }
    tc::fence_before_sync();
    tc::fence_async_smem();  // dhq tile (T0) -> tensor core; the generic reads of hq (T1) before the copy engine overwrites it
    __syncthreads();  // hq (T1) no longer needed by anyone
    PHN(3);
    if (imgs) {
      // aggregate image -> T1 by the copy engine (pulled into L2 by the prologue); the GEMMs that do not need it go first
      if (t.tid == 0) {
        tc::mbar_expect_tx(&bars[5], tc::TILE_BF16_BYTES);
        tc::bulk_g2s(T1, a.agg_img + (size_t)tile * tc::TILE_BF16_BYTES, tc::TILE_BF16_BYTES, &bars[5]);
        tc::fence_after_sync();
        tc::issue_gemm_mnmajor(ACC_VX, s0, s2, !first);           // dV1[:, 128:] += dhq^T x_t
        tc::issue_gemm_k_mn(WORK, s0, tc::smem_u32(sVA), false);  // g_agg = dhq V1[:, :128]
        tc::mbar_wait(&bars[5], ph);
        tc::issue_gemm_mnmajor(ACC_VA, s0, s1, !first);           // dV1[:, :128] += dhq^T agg
        tc::mma_commit(&bars[2]);
      }
      PHN(4);
    } else {
      // agg -> T1 ; x_t -> T2
      PDG_UNROLL(PDG_NODE_BWD_ROWS)
      for (int it = 0; it < 8; ++it) {
        const int r = (t.tid >> 4) + it * 16;
        const int rw = row0 + r;
        const size_t g = (size_t)rw * H + ch * 8;
        const float deg = rw < a.N ? (float)(a.rowptr[rw + 1] - a.rowptr[rw]) : 0.f;
        const float dm = deg * st1.mu;
        float v[8], x[8];
        *reinterpret_cast<float4*>(v) = *reinterpret_cast<const float4*>(a.aggraw + g);
        *reinterpret_cast<float4*>(v + 4) = *reinterpret_cast<const float4*>(a.aggraw + g + 4);
        *reinterpret_cast<float4*>(x) = *reinterpret_cast<const float4*>(a.x_t + g);
        *reinterpret_cast<float4*>(x + 4) = *reinterpret_cast<const float4*>(a.x_t + g + 4);
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = (v[j] - dm) * st1.rstd * we[j] + deg * be[j];
        *reinterpret_cast<uint4*>(T1 + tc::sw128_chunk(r, ch)) = tc::pack8_f16(v);
        *reinterpret_cast<uint4*>(T2 + tc::sw128_chunk(r, ch)) = tc::pack8_f16(x);
      }
      tc::fence_async_smem();
      __syncthreads();
      PHN(4);
      if (t.tid == 0) {
        tc::fence_after_sync();
        tc::issue_gemm_mnmajor(ACC_VA, s0, s1, !first);           // dV1[:, :128] += dhq^T agg
        tc::issue_gemm_mnmajor(ACC_VX, s0, s2, !first);           // dV1[:, 128:] += dhq^T x_t
        tc::issue_gemm_k_mn(WORK, s0, tc::smem_u32(sVA), false);  // g_agg = dhq V1[:, :128]
        tc::mma_commit(&bars[2]);
      }
    }
    dc1 += tile_colsum_f16(T0);
    tc::mbar_wait(&bars[2], ph);
    tc::fence_after_sync();
    PHN(5);
    // g_agg: TMEM -> fp32 staging (T1/T2 are dead: their GEMMs completed) -> coalesced pass
    tmem_to_s32(WORK, S32, t.row, t.half, t.lane_base);
    tc::fence_before_sync();
    __syncthreads();  // WORK drained by every thread
    PHN(6);
    if (t.tid == 0) {
      tc::fence_after_sync();
      tc::issue_gemm_k_mn(WORK, s0, tc::smem_u32(sVX), false);  // direct path: dhq V1[:, 128:]
      tc::mma_commit(&bars[3]);
    }
    // g_agg rows leave as bf16 (only consumer: the dy1 gather); LN1 column sums (g is constant over a receiver
    // segment): cg = sum deg*g_agg, cgy = sum g_agg*(aggraw - deg*mu)
#pragma unroll 4
    for (int it = 0; it < 8; ++it) {
      const int r = (t.tid >> 4) + it * 16;
      const int rw = row0 + r;
      const size_t g = (size_t)rw * H + ch * 4;
      const float deg = rw < a.N ? (float)(a.rowptr[rw + 1] - a.rowptr[rw]) : 0.f;
      const float dm = deg * st1.mu;
      const float4 g0 = *reinterpret_cast<const float4*>(s32_ptr(S32, r, ch * 4));
      const float4 g1 = *reinterpret_cast<const float4*>(s32_ptr(S32, r, 64 + ch * 4));
      const float4 a0 = *reinterpret_cast<const float4*>(a.aggraw + g);
      const float4 a1 = *reinterpret_cast<const float4*>(a.aggraw + g + 64);
      __half* gq = reinterpret_cast<__half*>(a.gagg) + g;
      // stored pre-multiplied by rstd1 * lnw (the only consumer, dy1 of the edge kernel, needs exactly that product)
      uint2 u0, u1;
      u0.x = tc::pack2_f16(g0.x * sw0.x, g0.y * sw0.y); u0.y = tc::pack2_f16(g0.z * sw0.z, g0.w * sw0.w);
      u1.x = tc::pack2_f16(g1.x * sw1.x, g1.y * sw1.y); u1.y = tc::pack2_f16(g1.z * sw1.z, g1.w * sw1.w);
      *reinterpret_cast<uint2*>(gq) = u0;
      *reinterpret_cast<uint2*>(gq + 64) = u1;
      cg8[0] = fmaf(deg, g0.x, cg8[0]); cg8[1] = fmaf(deg, g0.y, cg8[1]); cg8[2] = fmaf(deg, g0.z, cg8[2]); cg8[3] = fmaf(deg, g0.w, cg8[3]);
      cg8[4] = fmaf(deg, g1.x, cg8[4]); cg8[5] = fmaf(deg, g1.y, cg8[5]); cg8[6] = fmaf(deg, g1.z, cg8[6]); cg8[7] = fmaf(deg, g1.w, cg8[7]);
      cgy8[0] = fmaf(g0.x, a0.x - dm, cgy8[0]); cgy8[1] = fmaf(g0.y, a0.y - dm, cgy8[1]);
      cgy8[2] = fmaf(g0.z, a0.z - dm, cgy8[2]); cgy8[3] = fmaf(g0.w, a0.w - dm, cgy8[3]);
      cgy8[4] = fmaf(g1.x, a1.x - dm, cgy8[4]); cgy8[5] = fmaf(g1.y, a1.y - dm, cgy8[5]);
      cgy8[6] = fmaf(g1.z, a1.z - dm, cgy8[6]); cgy8[7] = fmaf(g1.w, a1.w - dm, cgy8[7]);
    }
    PHN(7);
    tc::mbar_wait(&bars[3], ph);
    tc::fence_after_sync();
    __syncthreads();  // staging tile free again
    tmem_to_s32(WORK, S32, t.row, t.half, t.lane_base);
    tc::fence_before_sync();
    __syncthreads();
    PHN(8);
#pragma unroll 4
    for (int it = 0; it < 8; ++it) {  // gx_t (partial) = gx_{t+1} + dhq V1[:, 128:], coalesced read-modify-write
      const int r = (t.tid >> 4) + it * 16;
      const size_t g = ((size_t)row0 + r) * H + ch * 4;
      float4 d0 = *reinterpret_cast<const float4*>(s32_ptr(S32, r, ch * 4));
      float4 d1 = *reinterpret_cast<const float4*>(s32_ptr(S32, r, 64 + ch * 4));
      const float4 x0 = *reinterpret_cast<const float4*>(a.gx + g);
      const float4 x1 = *reinterpret_cast<const float4*>(a.gx + g + 64);
      d0.x += x0.x; d0.y += x0.y; d0.z += x0.z; d0.w += x0.w;
      d1.x += x1.x; d1.y += x1.y; d1.z += x1.z; d1.w += x1.w;
      *reinterpret_cast<float4*>(a.gx + g) = d0;
      *reinterpret_cast<float4*>(a.gx + g + 64) = d1;
    }
    ph ^= 1u;
    first = false;
    tc::fence_before_sync();
    tc::fence_async_smem();  // generic accesses of the staging (T1 + T2) before the next tile's bulk copies land there
    __syncthreads();
    PHN(9);
#ifdef PDG_PHASE_TIMERS
    _toff = 32;
#endif
  }
  // weight-gradient accumulators -> this CTA's gradient slice (coalesced through the fp32 staging tile)
  {  // every buffer is dead (all MMAs completed, staging consumed): the three accumulators are staged side by side in
     // the six 32 KB buffers and leave with six bulk reduce-adds -- no drain between them
    float* F = reinterpret_cast<float*>(sm);
    constexpr int HB = 64 * H;  // floats of a 32 KB half block
    acc_stage(ACC_V2, F, F + HB, t.row, t.half, t.lane_base);
    acc_stage(ACC_VA, F + 2 * HB, F + 3 * HB, t.row, t.half, t.lane_base);
    acc_stage(ACC_VX, F + 4 * HB, F + 5 * HB, t.row, t.half, t.lane_base);
    tc::fence_async_smem();
    __syncthreads();
    if (t.tid == 0) {
      acc_reduce_issue(F, F + HB, cg + param_offset(PN_W2));
      acc_reduce_issue(F + 2 * HB, F + 3 * HB, cg + param_offset(PN_W0));            // block 0: columns [0, 128) (aggregate)
      acc_reduce_issue(F + 4 * HB, F + 5 * HB, cg + param_offset(PN_W0) + H * H);    // block 1: columns [128, 256) (x_t)
      acc_reduce_drain();
    }
    __syncthreads();  // comb / T0 scratch below
  }
  colpart_flush(dc2, comb, cg + param_offset(PN_B2), true);
  colpart_flush(dc1, comb, cg + param_offset(PN_B0), true);
  chunkpart_flush(cg8, reinterpret_cast<float*>(T0), a.cs1 + (size_t)blockIdx.x * 2 * H);
  chunkpart_flush(cgy8, reinterpret_cast<float*>(T0), a.cs1 + (size_t)blockIdx.x * 2 * H + H);
  if (t.tid == 0) tc::bulk_wait_all();
  tc::fence_before_sync();
  __syncthreads();
  PHN(10);
  if (t.warp == 0) tc::tmem_dealloc(tmem, 512);
}

// ------------------------------------------------------------------------------------------------
constexpr int SL_CAP = 2048;  // sender-list entries of one node tile staged in smem
constexpr int TC_SMEM_NODE_PRE_BWD = 5 * tc::TILE_BF16_BYTES + 2 * H * 4 + (SL_CAP + TM + 8) * 4 + 512 + 2048;

__global__ void __launch_bounds__(NT, 1)
k_node_pre_bwd_tc(NodePreBwdArgs a, const uint8_t* __restrict__ imgWA, const uint8_t* __restrict__ imgWB) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* sm = tc_smem_base(smem_raw);
  uint8_t* sWA = sm;
  uint8_t* sWB = sWA + tc::TILE_BF16_BYTES;
  uint8_t* T0 = sWB + tc::TILE_BF16_BYTES;  // dPa
  uint8_t* T1 = T0 + tc::TILE_BF16_BYTES;   // dPb
  uint8_t* T2 = T1 + tc::TILE_BF16_BYTES;   // x_t
  float* S32 = reinterpret_cast<float*>(T0);  // aliases T0 + T1 after their GEMMs completed
  float* comb = reinterpret_cast<float*>(T2 + tc::TILE_BF16_BYTES);
  float* smf = comb + 2 * H;
  int* s_ptr = reinterpret_cast<int*>(smf + 4);  // [TM + 1] sender-CSR offsets of the tile's nodes
  int* s_list = s_ptr + TM + 4;                  // [SL_CAP] edge positions (receiver order) grouped by sender
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_list + SL_CAP);  // 0 weights, 1 MMA group, 2 x_t image
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 4);
  const TcThread t;
  float* cg = a.cta_grads + (size_t)blockIdx.x * GRADP;
  const uint32_t tmem = tc_setup(bars, 3, tmem_slot, 512);
  const bool ximg = a.x_img != nullptr;  // x_t arrives as the fp16 operand image of k_node_pre_tc (bulk copy into T2)
  const uint32_t ACC_WA = tmem, ACC_WB = tmem + 128, WORK = tmem + 256;
  if (t.tid == 0) {
    tc::mbar_expect_tx(&bars[0], 2 * tc::TILE_BF16_BYTES);
    tc::bulk_g2s(sWA, imgWA, tc::TILE_BF16_BYTES, &bars[0]);
    tc::bulk_g2s(sWB, imgWB, tc::TILE_BF16_BYTES, &bars[0]);
  }
  if (t.tid == 0) {  // forward-saved state of this step
    if (ximg) {
      if ((int)blockIdx.x < a.n_tiles) {
        tc::mbar_expect_tx(&bars[2], tc::TILE_BF16_BYTES);
        tc::bulk_g2s(T2, a.x_img + (size_t)blockIdx.x * tc::TILE_BF16_BYTES, tc::TILE_BF16_BYTES, &bars[2]);
      }
      for (int tile = blockIdx.x + gridDim.x; tile < a.n_tiles; tile += gridDim.x)
        tc::bulk_prefetch_l2(a.x_img + (size_t)tile * tc::TILE_BF16_BYTES, tc::TILE_BF16_BYTES);
    } else {
      prefetch_node_tiles(a.x_t, a.n_tiles);
    }
    prefetch_node_tiles(a.yprev, a.n_tiles);
  }
  pdl_sync();
  if (t.tid == 0) {
    prefetch_node_tiles(a.RA, a.n_tiles);
    prefetch_node_tiles(a.RB, a.n_tiles);
    prefetch_node_tiles(a.gx, a.n_tiles);
  }
  const float mu_prev = ln_stat_block(a.parts_prev, a.count_prev, smf).mu;
  const int ch = t.tid & 15;
  float cgx8[8] = {0}, cgy8[8] = {0};  // chunk-mapped column partials
  uint32_t ph = 0;
  bool first = true;
  const uint32_t s0 = tc::smem_u32(T0), s1 = tc::smem_u32(T1), s2 = tc::smem_u32(T2);
  PHN_INIT;
  for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const int row0 = tile * TM;
    const size_t grow = ((size_t)row0 + t.row) * H + t.half * 64;
    PHN(16);
    // dPa = RA + sum_{send = n} dhn ; dPb = RB + sum_{send = n} dhm.
    // The tile's sender lists are one contiguous range of send_list: staged in smem first, so the row loads
    // below carry no dependent index loads.  Half-warp per row (16 lanes x 8 channels), GB edges in flight (a mesh
    // node sends to 6-7 edges: one batch per row).
    if (t.tid <= TM) s_ptr[t.tid] = a.sptr[min(row0 + t.tid, a.N)];
    __syncthreads();
    const int k_lo = s_ptr[0], cnt = s_ptr[TM] - s_ptr[0];
    const bool staged = cnt <= SL_CAP;
    if (staged)
      for (int i = t.tid; i < cnt; i += NT) s_list[i] = a.slist[k_lo + i];
    __syncthreads();
    PHN(17);
    {
      const int hw = t.tid >> 4, l16 = t.tid & 15;
      const __half* dhm = reinterpret_cast<const __half*>(a.DHM) + l16 * 8;
      const __half* dhn = a.DHN ? reinterpret_cast<const __half*>(a.DHN) + l16 * 8 : nullptr;
      for (int rr = 0; rr < 8; ++rr) {
        const int r = hw * 8 + rr;
        const int n = row0 + r;
        float pa[8] = {0, 0, 0, 0, 0, 0, 0, 0}, pb[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        if (n < a.N) {
          *reinterpret_cast<float4*>(pa) = *reinterpret_cast<const float4*>(a.RA + (size_t)n * H + l16 * 8);
          *reinterpret_cast<float4*>(pa + 4) = *reinterpret_cast<const float4*>(a.RA + (size_t)n * H + l16 * 8 + 4);
          if (a.RB) {
            *reinterpret_cast<float4*>(pb) = *reinterpret_cast<const float4*>(a.RB + (size_t)n * H + l16 * 8);
            *reinterpret_cast<float4*>(pb + 4) = *reinterpret_cast<const float4*>(a.RB + (size_t)n * H + l16 * 8 + 4);
          }
          const int k1 = s_ptr[r + 1];
          constexpr int GB = PDG_PRE_BWD_GB;
          for (int k = s_ptr[r]; k < k1; k += GB) {
            uint4 um[GB], uq[GB];
#pragma unroll
            for (int j = 0; j < GB; ++j) {
              um[j] = make_uint4(0u, 0u, 0u, 0u);
              uq[j] = um[j];
              if (k + j < k1) {
                const size_t p = (size_t)(staged ? s_list[k + j - k_lo] : a.slist[k + j]) * H;
                um[j] = *reinterpret_cast<const uint4*>(dhm + p);
                if (dhn) uq[j] = *reinterpret_cast<const uint4*>(dhn + p);
              }
            }
#pragma unroll
            for (int j = 0; j < GB; ++j) {  // fixed order k, k+1, ... => deterministic sums (bf16 zeros add nothing)
              const uint32_t* wm = reinterpret_cast<const uint32_t*>(&um[j]);
              const uint32_t* wq = reinterpret_cast<const uint32_t*>(&uq[j]);
#pragma unroll
              for (int h2 = 0; h2 < 4; ++h2) {
                const float2 fm = __half22float2(*reinterpret_cast<const __half2*>(&wm[h2]));
                const float2 fq = __half22float2(*reinterpret_cast<const __half2*>(&wq[h2]));
                pb[2 * h2] += fm.x; pb[2 * h2 + 1] += fm.y;
                pa[2 * h2] += fq.x; pa[2 * h2 + 1] += fq.y;
              }
            }
          }
        }
        *reinterpret_cast<uint4*>(T0 + tc::sw128_chunk(r, l16)) = tc::pack8_f16(pa);
        *reinterpret_cast<uint4*>(T1 + tc::sw128_chunk(r, l16)) = tc::pack8_f16(pb);
      }
    }
    PHN(18);
    if (!ximg) {
#pragma unroll 8
      for (int it = 0; it < 8; ++it) {
        const int r = (t.tid >> 4) + it * 16;
        const size_t g = ((size_t)row0 + r) * H + ch * 8;
        float x[8];
        *reinterpret_cast<float4*>(x) = *reinterpret_cast<const float4*>(a.x_t + g);
        *reinterpret_cast<float4*>(x + 4) = *reinterpret_cast<const float4*>(a.x_t + g + 4);
        *reinterpret_cast<uint4*>(T2 + tc::sw128_chunk(r, ch)) = tc::pack8_f16(x);
      }
    }
    tc::fence_async_smem();
    __syncthreads();
    PHN(19);
    if (t.tid == 0) {
      if (first) tc::mbar_wait(&bars[0], 0);
      if (ximg) tc::mbar_wait(&bars[2], ph);
      tc::fence_after_sync();
      tc::issue_gemm_mnmajor(ACC_WA, s0, s2, !first);           // dWa += dPa^T x_t
      tc::issue_gemm_mnmajor(ACC_WB, s1, s2, !first);           // dWb += dPb^T x_t
      tc::issue_gemm_k_mn(WORK, s0, tc::smem_u32(sWA), false);  // dPa Wa
      tc::issue_gemm_k_mn(WORK, s1, tc::smem_u32(sWB), true);   // + dPb Wb
      tc::mma_commit(&bars[1]);
    }
    tc::mbar_wait(&bars[1], ph);
    tc::fence_after_sync();
    if (ximg && t.tid == 0 && tile + (int)gridDim.x < a.n_tiles) {  // T2 is free (its GEMMs completed): next tile's x_t image
      tc::mbar_expect_tx(&bars[2], tc::TILE_BF16_BYTES);
      tc::bulk_g2s(T2, a.x_img + (size_t)(tile + gridDim.x) * tc::TILE_BF16_BYTES, tc::TILE_BF16_BYTES, &bars[2]);
    }
    // gx_t = partial + dPa Wa + dPb Wb: TMEM -> fp32 staging (T0/T1 dead) -> coalesced read-modify-write, plus the
    // column sums for the LayerNorm that produced x_t's increment
    PHN(20);
    tmem_to_s32(WORK, S32, t.row, t.half, t.lane_base);
    tc::fence_before_sync();
    __syncthreads();
    PHN(21);
    // two batches of four row groups: every global load of a batch is issued before the batch's first store (the stores
    // of a read-modify-write loop cannot be overtaken by the next iteration's loads -- possible aliasing -- so the
    // one-row-group-at-a-time loop paid eight dependent round trips per tile)
#pragma unroll
    for (int bt = 0; bt < 2; ++bt) {
      float4 lx0[4], lx1[4], ly0[4], ly1[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const size_t g = ((size_t)row0 + (t.tid >> 4) + (bt * 4 + k) * 16) * H + ch * 4;
        lx0[k] = *reinterpret_cast<const float4*>(a.gx + g);
        lx1[k] = *reinterpret_cast<const float4*>(a.gx + g + 64);
        ly0[k] = *reinterpret_cast<const float4*>(a.yprev + g);
        ly1[k] = *reinterpret_cast<const float4*>(a.yprev + g + 64);
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int r = (t.tid >> 4) + (bt * 4 + k) * 16;
        const size_t g = ((size_t)row0 + r) * H + ch * 4;
        float4 d0 = *reinterpret_cast<const float4*>(s32_ptr(S32, r, ch * 4));
        float4 d1 = *reinterpret_cast<const float4*>(s32_ptr(S32, r, 64 + ch * 4));
        const float4 x0 = lx0[k], x1 = lx1[k], y0 = ly0[k], y1 = ly1[k];
        d0.x += x0.x; d0.y += x0.y; d0.z += x0.z; d0.w += x0.w;
        d1.x += x1.x; d1.y += x1.y; d1.z += x1.z; d1.w += x1.w;
        *reinterpret_cast<float4*>(a.gx + g) = d0;
        *reinterpret_cast<float4*>(a.gx + g + 64) = d1;
        {  // RA / RB rows of this tile were consumed above: re-zero them for the next step's segment sums
          const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
          *reinterpret_cast<float4*>(a.RA + g) = z4;
          *reinterpret_cast<float4*>(a.RA + g + 64) = z4;
          if (a.RB) {
            *reinterpret_cast<float4*>(a.RB + g) = z4;
            *reinterpret_cast<float4*>(a.RB + g + 64) = z4;
          }
        }
        cgx8[0] += d0.x; cgx8[1] += d0.y; cgx8[2] += d0.z; cgx8[3] += d0.w;
        cgx8[4] += d1.x; cgx8[5] += d1.y; cgx8[6] += d1.z; cgx8[7] += d1.w;
        cgy8[0] = fmaf(d0.x, y0.x - mu_prev, cgy8[0]); cgy8[1] = fmaf(d0.y, y0.y - mu_prev, cgy8[1]);
        cgy8[2] = fmaf(d0.z, y0.z - mu_prev, cgy8[2]); cgy8[3] = fmaf(d0.w, y0.w - mu_prev, cgy8[3]);
        cgy8[4] = fmaf(d1.x, y1.x - mu_prev, cgy8[4]); cgy8[5] = fmaf(d1.y, y1.y - mu_prev, cgy8[5]);
        cgy8[6] = fmaf(d1.z, y1.z - mu_prev, cgy8[6]); cgy8[7] = fmaf(d1.w, y1.w - mu_prev, cgy8[7]);
      }
    }
    ph ^= 1u;
    first = false;
    tc::fence_before_sync();
    __syncthreads();
    PHN(22);
#ifdef PDG_PHASE_TIMERS
    _toff = 32;
#endif
  }
  {  // weight images and T0 / T1 are dead: both accumulators are staged side by side, four bulk reduce-adds
    float* F = reinterpret_cast<float*>(sm);
    constexpr int HB = 64 * H;
    acc_stage(ACC_WA, F, F + HB, t.row, t.half, t.lane_base);
    acc_stage(ACC_WB, F + 2 * HB, F + 3 * HB, t.row, t.half, t.lane_base);
    tc::fence_async_smem();
    __syncthreads();
    if (t.tid == 0) {
      acc_reduce_issue(F, F + HB, cg + param_offset(PE_W0));                       // block 0: columns [0, 128)   (Wa)
      acc_reduce_issue(F + 2 * HB, F + 3 * HB, cg + param_offset(PE_W0) + H * H);  // block 1: columns [128, 256) (Wb)
    }
  }
  chunkpart_flush(cgx8, reinterpret_cast<float*>(T2), a.cs3 + (size_t)blockIdx.x * 2 * H);
  chunkpart_flush(cgy8, reinterpret_cast<float*>(T2), a.cs3 + (size_t)blockIdx.x * 2 * H + H);
  if (t.tid == 0) tc::bulk_wait_all();
  tc::fence_before_sync();
  __syncthreads();
  PHN(23);
  if (t.warp == 0) tc::tmem_dealloc(tmem, 512);
}

#ifdef PDG_PHASE_TIMERS
extern "C" int pdg_phase_read_node(unsigned long long* out64) {
  return cudaMemcpyFromSymbol(out64, g_phase_node, sizeof(unsigned long long) * 64) == cudaSuccess ? 0 : -1;
}
#endif

// ------------------------------------------------------------------------------------------------
int launch_node_pre_tc(const NodePreArgs& a, const uint8_t* img, int n_tiles, cudaStream_t st) {
  const int cap = 2 * num_sms();
  return launch_named("k_node_pre_tc", true, k_node_pre_tc, dim3(n_tiles < cap ? n_tiles : cap), dim3(NT), TC_SMEM_NODE_PRE, st, a,
                      weight_img(img, IMG_PE_WA), weight_img(img, IMG_PE_WB));
}
int launch_node_update_tc(const NodeUpdArgs& a, const uint8_t* img, int grid, cudaStream_t st) {
  return launch_named("k_node_update_tc", true, k_node_update_tc, dim3(grid), dim3(NT), TC_SMEM_NODE_UPD, st, a,
                      weight_img(img, IMG_PN_WA), weight_img(img, IMG_PN_WX), weight_img(img, IMG_PN_W2));
}
int launch_node_update_bwd_tc(const NodeUpdBwdArgs& a, const uint8_t* img, int grid, cudaStream_t st) {
  return launch_named("k_node_update_bwd_tc", true, k_node_update_bwd_tc, dim3(grid), dim3(NT), TC_SMEM_NODE_UPD_BWD, st, a,
                      weight_img(img, IMG_PN_WA), weight_img(img, IMG_PN_WX), weight_img(img, IMG_PN_W2));
}
int launch_node_pre_bwd_tc(const NodePreBwdArgs& a, const uint8_t* img, int grid, cudaStream_t st) {
  return launch_named("k_node_pre_bwd_tc", true, k_node_pre_bwd_tc, dim3(grid), dim3(NT), TC_SMEM_NODE_PRE_BWD, st, a,
                      weight_img(img, IMG_PE_WA), weight_img(img, IMG_PE_WB));
}

}  // namespace pdg
