// Warp-specialised bf16 tensor-core backward edge kernel (PDG_PREC_BF16), third generation.
//
// Same math as the FFMA kernel k_edge_step_bwd (pdg_backward.cu).  Structure:
//   * 8 consumer warps run the MMAs + TMEM epilogues; a producer warpgroup (4 warps) runs the two
//     HBM-streaming phases of a tile concurrently with them:
//       fill_tile(j)   e_t operand tile E[j & 1] = one 32 KB bulk copy of the bf16 image the forward wrote
//       fill_ids(j)    ids / segment codes of tile j
//       dy2_build(j)   dy2 (LayerNorm backward of the edge update, from y2_t and ge_{t+1}) -> DY operand tile
//       final_pass(j)  ge_t = ge_{t+1} + de (coalesced read-modify-write), y_prev read and the
//                      LayerNorm-backward column partials, from the fp32 staging of de
//     hand-off by mbarriers: full[buf] (producers -> consumers), sfull (consumers -> producers,
//     "de of this tile is staged"), sfree (producers -> consumers, "staging is free again").
//   * the message path and the edge-update path run one after the other and share ONE hidden tile H:
//       G = E We^T -> hm -> H ; y1 = H W2^T -> dy1 -> DY ; dW2 += DY^T H ; dhm = (DY W2)*[H>0] -> H
//       de  = H We ; dWe += H^T E ;  G again -> hn -> H ; dy2 -> DY ; dW2 += DY^T H ; dhn -> H
//       de += H We ; dWe += H^T E
//     (one more G GEMM, two accumulating de / dWe GEMMs instead of a dG tile) which frees the
//     shared memory for the second E buffer.  The fp32 staging of de aliases E[buf] (rows 0-63)
//     and DY (rows 64-127), both dead by then.
// TMEM: [0,128) dW2 and [128,256) dWe persistent accumulators, [256,384) WORK0 (G, dhm, G, dhn),
// [384,512) WORK1 (y1, then de).
#include "pdg_ws.cuh"
#include "pdg_tc_tile.cuh"

namespace pdg {

constexpr int NT_B3 = 384;
constexpr int NC_B3 = 256;
constexpr int DB = 8;  // dy2_build rows per batch (bytes in flight per SM = 128 threads x 3*DB x 16 B)

#ifdef PDG_PHASE_TIMERS
__device__ unsigned long long g_phase3[32];
#define PH3(i) do { if (blockIdx.x == 0 && threadIdx.x == 0) { unsigned long long _t = clock64(); g_phase3[i] += _t - _tl; _tl = _t; } } while (0)
// producer-side phases (producer thread 0 of CTA 0): slots 16..
#define PP3(i) do { if (blockIdx.x == 0 && threadIdx.x == NC_B3) { unsigned long long _t = clock64(); g_phase3[16 + (i)] += _t - _tp; _tp = _t; } } while (0)
#define PP3_INIT unsigned long long _tp = clock64()
#else
#define PH3(i) do {} while (0)
#define PP3(i) do {} while (0)
#define PP3_INIT do {} while (0)
#endif

constexpr int TC_SMEM_EDGE_BWD3 = 6 * tc::TILE_BF16_BYTES   // We, W2, E[2], H, DY
                                  + 2 * 2 * TM * 4          // recv / send, double buffered
                                  + 3 * H * 4               // b1, b2, ln weight
                                  + 16 * H * 4              // consumer column-sum combine scratch [16 row groups][H]
                                  + 8 * H * 4               // producer column-sum combine scratch
                                  + 1024 + 2048;

__device__ __forceinline__ void b3_csync() { asm volatile("bar.sync 1, 256;" ::: "memory"); }
__device__ __forceinline__ void b3_psync() { asm volatile("bar.sync 2, 128;" ::: "memory"); }
__device__ __forceinline__ void b3_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tc::smem_u32(bar)) : "memory");
}
// fp32 staging of a [128][128] tile split over two 32 KB regions (rows 0-63 / 64-127), float4 chunks XOR-swizzled
__device__ __forceinline__ float* b3_s32(float* Sa, float* Sb, int r, int c) {
  float* base = r < 64 ? Sa + r * H : Sb + (r - 64) * H;
  return base + ((((c >> 2) ^ (r & 31)) << 2) | (c & 3));
}
// consumer-side flush of chunk-mapped column partials (thread = (chunk = tid & 15, group = tid >> 4)); comb = [16][H]
__device__ __forceinline__ void b3_chunk_flush(const float (&v)[8], float* comb, float* dst) {
  b3_csync();
  const int chunk = threadIdx.x & 15, grp = threadIdx.x >> 4;
  *reinterpret_cast<float4*>(comb + grp * H + chunk * 8) = make_float4(v[0], v[1], v[2], v[3]);
  *reinterpret_cast<float4*>(comb + grp * H + chunk * 8 + 4) = make_float4(v[4], v[5], v[6], v[7]);
  b3_csync();
  if (threadIdx.x < H) {
    float s = 0.f;
#pragma unroll
    for (int g = 0; g < 16; ++g) s += comb[g * H + threadIdx.x];
    dst[threadIdx.x] += s;
  }
}
// producer: receiver segments of the tile (see tile_segsum_items in pdg_tc_tile.cuh).  128 producer threads, r = row.
// lo / hi = rowptr[recv[r]], rowptr[recv[r] + 1], fetched a tile ahead by the caller.
__device__ __forceinline__ void b3_segments(int r, const int* recv_s, int lo, int hi, int row0, int nvalid,
                                            unsigned char* seg_row, unsigned char* seg_cut, int* nseg, unsigned* masks) {
  const bool first = r < nvalid && (r == 0 || recv_s[r] != recv_s[r - 1]);
  const unsigned m = __ballot_sync(0xffffffffu, first);
  if ((r & 31) == 0) masks[r >> 5] = m;
  b3_psync();
  if (first) {
    int idx = __popc(m & ((1u << (r & 31)) - 1u));
    for (int w = 0; w < (r >> 5); ++w) idx += __popc(masks[w]);
    seg_row[idx] = (unsigned char)r;
    seg_cut[idx] = (lo >= row0 && hi <= row0 + nvalid) ? 1 : 2;
  }
  if (r == 0) {
    const int n = __popc(masks[0]) + __popc(masks[1]) + __popc(masks[2]) + __popc(masks[3]);
    *nseg = n;
    seg_row[n] = (unsigned char)nvalid;
  }
}

__global__ void __launch_bounds__(NT_B3, 1)
k_edge_step_bwd_tc3(EdgeBwdArgs a, const uint8_t* __restrict__ imgWe, const uint8_t* __restrict__ imgW2) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* sm = tc_smem_base(smem_raw);
  uint8_t* sWe = sm;
  uint8_t* sW2 = sWe + tc::TILE_BF16_BYTES;
  uint8_t* tEb = sW2 + tc::TILE_BF16_BYTES;  // [2]
  uint8_t* tH = tEb + 2 * tc::TILE_BF16_BYTES;
  uint8_t* tDY = tH + tc::TILE_BF16_BYTES;
  int* recv_b = reinterpret_cast<int*>(tDY + tc::TILE_BF16_BYTES);  // [2][TM]
  int* send_b = recv_b + 2 * TM;
  float* b1s = reinterpret_cast<float*>(send_b + 2 * TM);
  float* b2s = b1s + H;
  float* lws = b2s + H;
  float* comb = lws + H;        // [16][H] consumers
  float* pcomb = comb + 16 * H;  // [8][H] producers
  float* smf = pcomb + 8 * H;
  int* nseg_b = reinterpret_cast<int*>(smf + 4);  // [2] (+2 pad)
  unsigned* masks = reinterpret_cast<unsigned*>(nseg_b + 4);
  unsigned char* seg_row_b = reinterpret_cast<unsigned char*>(masks + 4);  // [2][TM + 8]: first row of each receiver segment
  unsigned char* seg_cut_b = seg_row_b + 2 * (TM + 8);                      // [2][TM]: 1 whole / 2 cut by a tile boundary
  uint64_t* bars = reinterpret_cast<uint64_t*>(seg_cut_b + 2 * TM);  // 0 weights, 1..6 MMA groups, 7,8 full, 9 sfull, 10 sfree, 11 dyfree, 12 dyfull
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 14);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) {
    for (int i = 0; i < 7; ++i) tc::mbar_init(&bars[i], 1);
    tc::mbar_init(&bars[7], NT_B3 - NC_B3);
    tc::mbar_init(&bars[8], NT_B3 - NC_B3);
    tc::mbar_init(&bars[9], 1);
    tc::mbar_init(&bars[10], NT_B3 - NC_B3);
    tc::mbar_init(&bars[11], 1);                 // xfree: consumers -> producers (the dy2 tile in E[(j+1)&1] is consumed: refill it)
    tc::mbar_init(&bars[12], NT_B3 - NC_B3);     // dyfull: producers -> consumers (dy2 tile written)
    tc::mbar_init_fence();
  }
  if (warp == 0) tc::tmem_alloc(tmem_slot, 512);
  if (tid < H) { b2s[tid] = a.b2[tid]; lws[tid] = a.lnw[tid]; }
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem = *tmem_slot;
  if (tid == 0) {
    tc::mbar_expect_tx(&bars[0], 2 * tc::TILE_BF16_BYTES);
    tc::bulk_g2s(sWe, imgWe, tc::TILE_BF16_BYTES, &bars[0]);
    tc::bulk_g2s(sW2, imgW2, tc::TILE_BF16_BYTES, &bars[0]);
  }
  pdl_sync();  // parameters / packed weights above, predecessor data (LN partials, scalars, gradients) below
  const float mu_prev = ln_stat_block(a.parts_prev, a.count_prev, smf).mu;  // all 384 threads
  const int n_my = (a.n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;  // tiles of this CTA

  if (tid >= NC_B3) {
    // ================================ PRODUCER warpgroup ================================
    const int ptid = tid - NC_B3;
    PP3_INIT;
    const int ch = ptid & 15, rg = ptid >> 4;  // 8 row groups
    float cge8[8] = {0}, cgye8[8] = {0};
    float c1n = 0.f, c2n = 0.f, mu2 = 0.f, rstd2 = 0.f;
    if (!a.last) { c1n = a.scal2[0]; c2n = a.scal2[1]; mu2 = a.scal2[2]; rstd2 = a.scal2[3]; }
    float rw8[8];  // rstd2 * ln weight of this thread's 8 channels; dy2 = rw * ge - c1 - c2 (y - mu) = fma(rw, ge, fma(-c2, y, k0))
#pragma unroll
    for (int q = 0; q < 8; ++q) rw8[q] = rstd2 * lws[ch * 8 + q];
    const float k0n = c2n * mu2 - c1n;
    // ids and receiver row pointers of a tile are fetched a tile ahead into registers
    int nrv = 0, nsv = 0, nlo = 0, nhi = 0;
    auto ids_load = [&](int j) {
      if (j < n_my) {
        const int g = (blockIdx.x + j * gridDim.x) * TM + ptid;
        nrv = a.recv[g];
        nsv = a.send[g];
      }
    };
    auto ptr_load = [&](int j) {
      if (j < n_my && (int)(blockIdx.x + j * gridDim.x) * TM + ptid < a.E) { nlo = a.rowptr[nrv]; nhi = a.rowptr[nrv + 1]; }
    };
    // dy2 of tile j (edge-update path), elementwise, coalesced: 16 lanes per row.  It is written into the OTHER e_t
    // buffer E[(j+1)&1] -- free from the end of final_pass(j-1) until the bulk copy of tile j+1 -- so that it can be
    // built long before the consumers need it instead of waiting for DY (which holds dy1 until mid-tile).
    auto dy2_build = [&](int j) {
      const int row0 = (blockIdx.x + j * gridDim.x) * TM;
      const int nvalid = min(TM, a.E - row0);
      uint8_t* tX = tEb + ((j + 1) & 1) * tc::TILE_BF16_BYTES;
      PP3(0);
      const __half* y2b = reinterpret_cast<const __half*>(a.y2_t);  // raw y2 rows are fp16
      for (int bt = 0; bt < TM / 8 / DB; ++bt) {
        uint4 ly[DB];
        float4 lg[2 * DB];
#pragma unroll
        for (int k = 0; k < DB; ++k) {
          const size_t g = ((size_t)row0 + rg + (bt * DB + k) * 8) * H + ch * 8;
          ly[k] = tc::ldcg128(y2b + g);
          tc::ldcg256(a.ge + g, lg[2 * k], lg[2 * k + 1]);
        }
#pragma unroll
        for (int k = 0; k < DB; ++k) {
          const int r = rg + (bt * DB + k) * 8;
          float y[8];
          unpack8_f16(ly[k], y);
          const float gg[8] = {lg[2 * k].x, lg[2 * k].y, lg[2 * k].z, lg[2 * k].w, lg[2 * k + 1].x, lg[2 * k + 1].y, lg[2 * k + 1].z, lg[2 * k + 1].w};
          float d[8];
#pragma unroll
          for (int q = 0; q < 8; ++q)
            d[q] = (r < nvalid && y[q] > 0.f) ? fmaf(rw8[q], gg[q], fmaf(-c2n, y[q], k0n)) : 0.f;
          *reinterpret_cast<uint4*>(tX + tc::sw128_chunk(r, ch)) = tc::pack8_f16(d);
        }
      }
      tc::fence_async_smem();
      b3_arrive(&bars[12]);
      PP3(2);
    };
    // e_t operand tile of tile j: ONE 32 KB bulk copy of the swizzled bf16 image the forward wrote (no registers, no
    // shared-memory stores); its bytes complete on the same full barrier the id / segment-code arrivals go to
    // The expect-tx must reach the barrier before the phase can complete, i.e. before producer thread 0's arrival:
    // either the copy is issued before fill_ids (expect only), or thread 0 skips its arrival in fill_ids and
    // arrives here together with the expect-tx (arrive0).
    auto fill_tile = [&](int j, bool arrive0) {
      if (ptid == 0) {
        const int buf = j & 1;
        if (arrive0) tc::mbar_expect_tx(&bars[7 + buf], tc::TILE_BF16_BYTES);
        else tc::mbar_expect_tx_only(&bars[7 + buf], tc::TILE_BF16_BYTES);
        tc::bulk_g2s(tEb + buf * tc::TILE_BF16_BYTES, a.e_img + (size_t)(blockIdx.x + j * gridDim.x) * tc::TILE_BF16_BYTES,
                     tc::TILE_BF16_BYTES, &bars[7 + buf]);
      }
    };
    auto fill_ids = [&](int j, bool arrive0) {
      const int buf = j & 1;
      const int row0 = (blockIdx.x + j * gridDim.x) * TM;
      int* recv_s = recv_b + buf * TM;
      recv_s[ptid] = nrv;
      send_b[buf * TM + ptid] = nsv;
      b3_psync();
      b3_segments(ptid, recv_s, nlo, nhi, row0, min(TM, a.E - row0), seg_row_b + buf * (TM + 8), seg_cut_b + buf * TM, nseg_b + buf, masks);
      if (ptid != 0 || arrive0) b3_arrive(&bars[7 + buf]);
      ids_load(j + 1);  // the row pointers follow at the top of the next producer iteration (ptr_load)
    };
    auto final_pass = [&](int j) {
      const int buf = j & 1;
      const int row0 = (blockIdx.x + j * gridDim.x) * TM;
      float* Sa = reinterpret_cast<float*>(tEb + buf * tc::TILE_BF16_BYTES);
      float* Sb = reinterpret_cast<float*>(tDY);
      PP3(3);
      const __half* ypb = reinterpret_cast<const __half*>(a.yprev);  // raw y rows are fp16
      constexpr int FB = 8;  // rows per batch: two batches per tile, the first one's loads fly under the wait below
#pragma unroll 1
      for (int bt = 0; bt < 16 / FB; ++bt) {
        float4 lg[2 * FB];
        uint2 ly[2 * FB];
#pragma unroll
        for (int k = 0; k < FB; ++k) {
          const size_t g = ((size_t)row0 + rg + (bt * FB + k) * 8) * H + ch * 4;
          if (!a.last) {
            lg[2 * k] = *reinterpret_cast<const float4*>(a.ge + g);
            lg[2 * k + 1] = *reinterpret_cast<const float4*>(a.ge + g + 64);
          } else {
            lg[2 * k] = make_float4(0.f, 0.f, 0.f, 0.f);
            lg[2 * k + 1] = lg[2 * k];
          }
          ly[2 * k] = *reinterpret_cast<const uint2*>(ypb + g);
          ly[2 * k + 1] = *reinterpret_cast<const uint2*>(ypb + g + 64);
        }
        if (bt == 0) {
          tc::mbar_wait(&bars[9], j & 1);  // de of tile j staged by the consumers
          PP3(4);
        }
#pragma unroll
        for (int k = 0; k < FB; ++k) {
          const int r = rg + (bt * FB + k) * 8;
          const size_t g = ((size_t)row0 + r) * H + ch * 4;
          float4 d0 = *reinterpret_cast<const float4*>(b3_s32(Sa, Sb, r, ch * 4));
          float4 d1 = *reinterpret_cast<const float4*>(b3_s32(Sa, Sb, r, 64 + ch * 4));
          d0.x += lg[2 * k].x; d0.y += lg[2 * k].y; d0.z += lg[2 * k].z; d0.w += lg[2 * k].w;
          d1.x += lg[2 * k + 1].x; d1.y += lg[2 * k + 1].y; d1.z += lg[2 * k + 1].z; d1.w += lg[2 * k + 1].w;
          *reinterpret_cast<float4*>(a.ge + g) = d0;
          *reinterpret_cast<float4*>(a.ge + g + 64) = d1;
          const float4 y0 = unpack4_f16(ly[2 * k]), y1 = unpack4_f16(ly[2 * k + 1]);
          cge8[0] += d0.x; cge8[1] += d0.y; cge8[2] += d0.z; cge8[3] += d0.w;
          cge8[4] += d1.x; cge8[5] += d1.y; cge8[6] += d1.z; cge8[7] += d1.w;
          cgye8[0] = fmaf(d0.x, y0.x - mu_prev, cgye8[0]); cgye8[1] = fmaf(d0.y, y0.y - mu_prev, cgye8[1]);
          cgye8[2] = fmaf(d0.z, y0.z - mu_prev, cgye8[2]); cgye8[3] = fmaf(d0.w, y0.w - mu_prev, cgye8[3]);
          cgye8[4] = fmaf(d1.x, y1.x - mu_prev, cgye8[4]); cgye8[5] = fmaf(d1.y, y1.y - mu_prev, cgye8[5]);
          cgye8[6] = fmaf(d1.z, y1.z - mu_prev, cgye8[6]); cgye8[7] = fmaf(d1.w, y1.w - mu_prev, cgye8[7]);
        }
      }
      tc::fence_async_smem();  // the next writer of E[buf] is the copy engine (fill_tile)
      b3_arrive(&bars[10]);    // staging (E[buf] rows + DY) free again
      PP3(5);
    };
    // duties in the order the consumers need them: per consumer tile j: [final_pass(j-1), bulk copy of tile j+1] dy2(j) ids(j+1)
    // the streaming passes are latency-bound batch loops: pull the rows of tile j into L2 ahead of them
    auto prefetch_rows = [&](int j) {
      if (ptid == 0) {
        const size_t row0 = (size_t)(blockIdx.x + j * gridDim.x) * TM;
        tc::bulk_prefetch_l2(a.e_img + (row0 / TM) * tc::TILE_BF16_BYTES, tc::TILE_BF16_BYTES);
        if (!a.last) {
          tc::bulk_prefetch_l2(reinterpret_cast<const __half*>(a.y2_t) + row0 * H, TM * H * 2);
          tc::bulk_prefetch_l2(a.ge + row0 * H, TM * H * 4);
        }
        tc::bulk_prefetch_l2(reinterpret_cast<const __half*>(a.yprev) + row0 * H, TM * H * 2);
      }
    };
    fill_tile(0, false);
    prefetch_rows(0);
    ids_load(0);
    ptr_load(0);
    fill_ids(0, true);
    if (a.last && n_my > 1) fill_tile(1, false);
    for (int j = 0; j < n_my; ++j) {
      ptr_load(j + 1);
      if (j + 1 < n_my) prefetch_rows(j + 1);
      if (j > 0) {
        final_pass(j - 1);
        b3_psync();  // staging (E[(j-1)&1] rows + DY) fully consumed by every producer thread
      }
      if (a.last) {
        if (j > 0 && j + 1 < n_my) fill_tile(j + 1, false);  // into E[(j+1)&1]: its previous tenant (tile j-1) was staged and consumed above
      } else {
        dy2_build(j);  // into E[(j+1)&1]
      }
      if (j + 1 < n_my) {
        fill_ids(j + 1, a.last != 0);
        if (!a.last) {
          PP3(1);
          tc::mbar_wait(&bars[11], j & 1);  // dy2 tile consumed (MMAs + column sums): E[(j+1)&1] takes the next e_t tile
          PP3(6);
          fill_tile(j + 1, true);
        }
      }
    }
    final_pass(n_my - 1);
    // flush the column partials of this CTA: 8 row groups x columns {ch*4..+3, 64+ch*4..+3}
    auto pflush = [&](const float (&v)[8], float* dst) {
      b3_psync();
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        pcomb[rg * H + ch * 4 + q] = v[q];
        pcomb[rg * H + 64 + ch * 4 + q] = v[4 + q];
      }
      b3_psync();
      float s = 0.f;
#pragma unroll
      for (int g2 = 0; g2 < 8; ++g2) s += pcomb[g2 * H + ptid];
      dst[ptid] = s;
    };
    pflush(cge8, a.cs2 + (size_t)blockIdx.x * 2 * H);
    pflush(cgye8, a.cs2 + (size_t)blockIdx.x * 2 * H + H);
    return;
  }

  // ================================== CONSUMER warps ==================================
  const int row = 32 * (warp & 3) + lane, half = warp >> 2;
  const uint32_t lane_base = (uint32_t)(32 * (warp & 3)) << 16;
  const uint32_t ACC_W2 = tmem, ACC_WE = tmem + 128, WORK0 = tmem + 256, WORK1 = tmem + 384;
  float* cg = a.cta_grads + (size_t)blockIdx.x * GRADP;
  const float c1m = a.scal1[0], c2m = a.scal1[1], mu1 = a.scal1[2];
  float db2[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, db1[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};  // chunk-mapped column sums
  const uint32_t sH = tc::smem_u32(tH), sDY = tc::smem_u32(tDY), aWe = tc::smem_u32(sWe), aW2 = tc::smem_u32(sW2);
  uint32_t ph = 0;

  // hidden activation of one edge-MLP evaluation -> H: relu(G + b1 + Pa[ia] + Pb[ib]).  The row gathers are issued
  // (hidden_gather) before the wait for the G GEMM / before the segment walk, so their L2 latency is hidden; sync_first: barrier between the wait and the
  // first write of H (its previous readers).
  uint4 ga[2][4], gb[2][4];  // gathered Pa / Pb row pieces of this thread (64 channels each)
  auto hidden_gather = [&](const int ia, const int ib) {
    const __half* pa = reinterpret_cast<const __half*>(a.Pa) + (size_t)ia * H + half * 64;
    const __half* pb = reinterpret_cast<const __half*>(a.Pb) + (size_t)ib * H + half * 64;
#pragma unroll
    for (int hh = 0; hh < 2; ++hh)
#pragma unroll
      for (int c8 = 0; c8 < 4; c8 += 2) {
        tc::ldg256(pa + hh * 32 + c8 * 8, ga[hh][c8], ga[hh][c8 + 1]);
        tc::ldg256(pb + hh * 32 + c8 * 8, gb[hh][c8], gb[hh][c8 + 1]);
      }
  };
  auto hidden = [&](uint64_t* bar, const bool sync_first) {
    tc::mbar_wait(bar, ph);
    tc::fence_after_sync();
    if (sync_first) b3_csync();
#pragma unroll
    for (int hh = 0; hh < 2; ++hh) {
      float gacc[32];
      tc::tmem_ld32(WORK0 + lane_base + (uint32_t)(half * 64 + hh * 32), gacc);
      tc::tmem_ld_wait();
#pragma unroll
      for (int c8 = 0; c8 < 4; ++c8) {
        float p[8], q[8], h[8];
        unpack8_f16(ga[hh][c8], p);
        unpack8_f16(gb[hh][c8], q);
#pragma unroll
        for (int k = 0; k < 8; ++k) h[k] = fmaxf(gacc[c8 * 8 + k] + p[k] + q[k], 0.f);  // layer-1 bias: inside the Pa rows
        row_store8(tH, row, half, hh * 4 + c8, h);
      }
    }
  };
  // d(hidden) = WORK0 * [H > 0] -> H (own chunks) + bf16 rows to global
  auto dhidden = [&](float* out_rows, size_t grow) {
    __half* dh = reinterpret_cast<__half*>(out_rows) + grow;
#pragma unroll
    for (int hh = 0; hh < 2; ++hh) {
      float v[32];
      tc::tmem_ld32(WORK0 + lane_base + (uint32_t)(half * 64 + hh * 32), v);
      tc::tmem_ld_wait();
      uint4 pk[4];
#pragma unroll
      for (int c8 = 0; c8 < 4; ++c8) {
        float h[8], d[8];
        row_load8(tH, row, half, hh * 4 + c8, h);
#pragma unroll
        for (int k = 0; k < 8; ++k) d[k] = h[k] > 0.f ? v[c8 * 8 + k] : 0.f;
        pk[c8] = tc::pack8_f16(d);
        *reinterpret_cast<uint4*>(tH + tc::sw128_chunk(row, half * 8 + hh * 4 + c8)) = pk[c8];
      }
      tc::stg256(dh + hh * 32, pk[0], pk[1]);
      tc::stg256(dh + hh * 32 + 16, pk[2], pk[3]);
    }
  };

#ifdef PDG_PHASE_TIMERS
  unsigned long long _tl = clock64();
#endif
  for (int i = 0; i < n_my; ++i) {
    const int buf = i & 1;
    const int row0 = (blockIdx.x + i * gridDim.x) * TM;
    const int nvalid = min(TM, a.E - row0);
    const bool ok = row < nvalid;
    const bool first = i == 0;
    const size_t grow = ((size_t)row0 + row) * H + half * 64;
    const uint32_t sE = tc::smem_u32(tEb + buf * tc::TILE_BF16_BYTES);
    const int* recv_s = recv_b + buf * TM;
    const int* send_s = send_b + buf * TM;
    const unsigned char* seg_row = seg_row_b + buf * (TM + 8);
    const unsigned char* seg_cut = seg_cut_b + buf * TM;
    tc::mbar_wait(&bars[7 + buf], (i >> 1) & 1);  // E tile, ids, codes of this tile are ready
    PH3(0);
    if (tid == 0) {
      if (first) tc::mbar_wait(&bars[0], 0);
      tc::fence_after_sync();
      tc::issue_gemm_kmajor(WORK0, sE, aWe, H, false);  // G
      tc::mma_commit(&bars[1]);
    }
    const int rc = recv_s[row], sd = send_s[row];
    PH3(1);
    hidden_gather(rc, sd);  // message: x_i = x[recv] -> Pa, x_j = x[send] -> Pb
    hidden(&bars[1], false);
    PH3(2);
    tc::fence_before_sync();
    tc::fence_async_smem();
    b3_csync();
    if (tid == 0) {
      tc::fence_after_sync();
      tc::issue_gemm_kmajor(WORK1, sH, aW2, H, false);  // y1 pre-activation
      tc::mma_commit(&bars[2]);
    }
    {  // dy1 -> DY (the g_agg row gathers fly while the y1 GEMM completes)
      const __half* gp = reinterpret_cast<const __half*>(a.gagg) + (size_t)rc * H + half * 64;
      uint4 gqq[2][4];
#pragma unroll
      for (int hh = 0; hh < 2; ++hh)
#pragma unroll
        for (int c8 = 0; c8 < 4; c8 += 2) tc::ldg256(gp + hh * 32 + c8 * 8, gqq[hh][c8], gqq[hh][c8 + 1]);
      if (i > 0) tc::mbar_wait(&bars[10], (i - 1) & 1);  // previous tile's staging (aliases DY) consumed
      tc::mbar_wait(&bars[2], ph);
      tc::fence_after_sync();
      PH3(3);
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        const uint4* gq = gqq[hh];
        float v[32];
        tc::tmem_ld32(WORK1 + lane_base + (uint32_t)(half * 64 + hh * 32), v);
        tc::tmem_ld_wait();
#pragma unroll
        for (int c8 = 0; c8 < 4; ++c8) {
          float gg[8], d[8];
          unpack8_f16(gq[c8], gg);
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            const int c = half * 64 + hh * 32 + c8 * 8 + k;
            const float y = fmaxf(v[c8 * 8 + k] + b2s[c], 0.f);
            d[k] = (ok && y > 0.f) ? gg[k] - c1m - c2m * (y - mu1) : 0.f;  // gagg rows arrive pre-multiplied by rstd1 * lnw
          }
          row_store8(tDY, row, half, hh * 4 + c8, d);
        }
      }
    }
    PH3(4);
    tc::fence_before_sync();
    tc::fence_async_smem();
    b3_csync();
    if (tid == 0) {
      tc::fence_after_sync();
      tc::issue_gemm_mnmajor(ACC_W2, sDY, sH, !first);  // dW2 += dy1^T hm
      tc::issue_gemm_k_mn(WORK0, sDY, aW2, false);      // dhm_pre = dy1 W2
      tc::mma_commit(&bars[3]);
    }
    tile_colsum_chunks(tDY, db2);
    tc::mbar_wait(&bars[3], ph);
    tc::fence_after_sync();
    PH3(5);
    dhidden(a.DHM, grow);
    PH3(6);
    tc::fence_before_sync();
    tc::fence_async_smem();
    b3_csync();
    if (tid == 0) {
      tc::fence_after_sync();
      tc::issue_gemm_k_mn(WORK1, sH, aWe, false);         // de  = dhm We
      tc::issue_gemm_mnmajor(ACC_WE, sH, sE, !first);     // dWe += dhm^T e_t
      if (!a.last) tc::issue_gemm_kmajor(WORK0, sE, aWe, H, false);  // G again for the edge-update path
      tc::mma_commit(&bars[4]);
    }
    if (!a.last) hidden_gather(sd, rc);  // rows of the edge-update evaluation: in flight under the segment walk
    tile_segsum_items(tH, recv_s, seg_row, seg_cut, nseg_b[buf], a.RA, db1);  // RA segment sums + db1 column sums
    if (a.last) {
      tc::mbar_wait(&bars[4], ph);
      tc::fence_after_sync();
    }
    PH3(7);
    if (!a.last) {
      // edge update: x[row] = x[send] -> Pa, x[col] = x[recv] -> Pb (swapped order); waits for the MMA group, then
      // for every segment walker to be done with H
      hidden(&bars[4], true);
      PH3(8);
      tc::mbar_wait(&bars[12], ph);  // dy2 tile written by the producers (into the other e_t buffer)
      uint8_t* tX = tEb + ((i + 1) & 1) * tc::TILE_BF16_BYTES;
      const uint32_t sX = tc::smem_u32(tX);
      PH3(9);
      tc::fence_before_sync();
      tc::fence_async_smem();
      b3_csync();
      if (tid == 0) {
        tc::fence_after_sync();
        tc::issue_gemm_mnmajor(ACC_W2, sX, sH, true);  // dW2 += dy2^T hn
        tc::issue_gemm_k_mn(WORK0, sX, aW2, false);    // dhn_pre = dy2 W2
        tc::mma_commit(&bars[5]);
      }
      tile_colsum_chunks(tX, db2);
      tc::mbar_wait(&bars[5], ph);
      tc::fence_after_sync();
      PH3(10);
      dhidden(a.DHN, grow);
      PH3(11);
      tc::fence_before_sync();
      tc::fence_async_smem();
      b3_csync();
      if (tid == 0) {
        b3_arrive(&bars[11]);  // dy2 tile consumed by its MMAs (bars[5]) and by every column-sum walker (barrier above)
        tc::fence_after_sync();
        tc::issue_gemm_k_mn(WORK1, sH, aWe, true);       // de  += dhn We
        tc::issue_gemm_mnmajor(ACC_WE, sH, sE, true);    // dWe += dhn^T e_t
        tc::mma_commit(&bars[6]);
      }
      tile_segsum_items(tH, recv_s, seg_row, seg_cut, nseg_b[buf], a.RB, db1);
      tc::mbar_wait(&bars[6], ph);
      tc::fence_after_sync();
      PH3(12);
    }
    // de -> fp32 staging (rows 0-63 over E[buf], rows 64-127 over DY; both dead: every MMA reading them completed)
    {
      float* Sa = reinterpret_cast<float*>(tEb + buf * tc::TILE_BF16_BYTES);
      float* Sb = reinterpret_cast<float*>(tDY);
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        float v[32];
        tc::tmem_ld32(WORK1 + lane_base + (uint32_t)(half * 64 + hh * 32), v);
        tc::tmem_ld_wait();
#pragma unroll
        for (int k = 0; k < 32; k += 4)
          *reinterpret_cast<float4*>(b3_s32(Sa, Sb, row, half * 64 + hh * 32 + k)) = make_float4(v[k], v[k + 1], v[k + 2], v[k + 3]);
      }
    }
    ph ^= 1u;
    tc::fence_before_sync();
    b3_csync();
    if (tid == 0) b3_arrive(&bars[9]);  // producers: run the ge / y_prev pass of this tile
    PH3(13);
  }
  // ---- flush: TMEM weight-gradient accumulators -> this CTA's gradient slice ----
  // through fp32 staging: rows 0-63 over the E buffer the last tile did not use (its last
  // tenant, tile n_my-2, was consumed before this CTA's last y1 stage), rows 64-127 over H (dead: every MMA and
  // walker of the last tile is done).  DY / E[last buf] still belong to the producers' final pass.
  // dW2 is staged over the E buffer the last tile did not use + H, dWe over the two weight images (dead: every MMA of
  // this CTA has completed); four 32 KB bulk reduce-adds, no drain in between.
  {
    float* Fa = reinterpret_cast<float*>(tEb + (n_my & 1) * tc::TILE_BF16_BYTES);
    float* Fb = reinterpret_cast<float*>(tH);
    float* Ga = reinterpret_cast<float*>(sWe);
    float* Gb = reinterpret_cast<float*>(sW2);
    acc_stage(ACC_W2, Fa, Fb, row, half, lane_base);
    acc_stage(ACC_WE, Ga, Gb, row, half, lane_base);
    tc::fence_async_smem();
    b3_csync();
    if (tid == 0) {
      acc_reduce_issue(Fa, Fb, cg + param_offset(PE_W2));
      acc_reduce_issue(Ga, Gb, cg + param_offset(PE_W0) + 2 * H * H);  // block 2 of edge_net.0.weight: columns [256, 384) (We)
    }
  }
  b3_chunk_flush(db2, comb, cg + param_offset(PE_B2));
  b3_chunk_flush(db1, comb, cg + param_offset(PE_B0));
  if (tid == 0) tc::bulk_wait_all();  // the reduce-adds have landed before the grid completes
  tc::fence_before_sync();
  b3_csync();
  if (warp == 0) tc::tmem_dealloc(tmem, 512);
}

#ifdef PDG_PHASE_TIMERS
extern "C" int pdg_phase_read3(unsigned long long* out32) {
  return cudaMemcpyFromSymbol(out32, g_phase3, sizeof(unsigned long long) * 32) == cudaSuccess ? 0 : -1;
}
#endif

int launch_edge_step_bwd_tc3(const EdgeBwdArgs& a, const uint8_t* img, int grid, cudaStream_t st) {
  return launch_named("k_edge_step_bwd_tc3", true, k_edge_step_bwd_tc3, dim3(grid), dim3(NT_B3), TC_SMEM_EDGE_BWD3, st, a,
                      weight_img(img, IMG_PE_WE), weight_img(img, IMG_PE_W2));
}

}  // namespace pdg
