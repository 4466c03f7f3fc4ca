// bf16 tensor-core (tcgen05 / TMEM) version of the forward edge kernel (PDG_PREC_BF16).
//
// Same math and data flow as k_edge_step (pdg_forward.cu; reference models.py:215-238), but
//   * the three 128x128x128 GEMMs of a tile run on the 5th-gen tensor cores: bf16 operands in
//     SWIZZLE_128B shared-memory tiles (weights staged once per CTA by 1-D TMA bulk copies of
//     pre-swizzled images), fp32 accumulation in TMEM (3 x 128 columns);
//   * the CTA is WARP-SPECIALISED: warps 8-11 (producer warpgroup) stream the next
//     tile's rows from HBM -- lazy LayerNorm + residual, fp32 e_t back to HBM, bf16 operand tile
//     into a double-buffered A0 -- while warps 0-7 (consumers) run the MMAs and the
//     TMEM epilogues of the current tile.  Hand-off through mbarriers: full[buf] (128 producer
//     arrivals) / empty[buf] (tcgen05.commit of the last MMA that reads the buffer).  The
//     HBM-bound phase (one third of a tile's time) is thereby hidden under the epilogues.
//     The producers' rows arrive through a ring of landing slots filled by bulk copies issued four chunks ahead.
//   * epilogues read TMEM with tcgen05.ld (thread = one edge row x 64 channels): bias, gathered
//     bf16 node projections (256-bit loads, issued before the GEMM wait), ReLU in fp32; the messages y1 go
//     into the dead hidden tile as bf16 and are summed per receiver segment from there, the raw edge-update
//     output y2 leaves as bf16 rows straight from the registers (256-bit stores); LayerNorm partials from fp32.
// Latent storage, LayerNorm and all reductions stay fp32; tolerance of this mode: 2e-2.
#include "pdg_ws.cuh"
#include "pdg_tc_tile.cuh"

namespace pdg {

#ifdef PDG_PHASE_TIMERS
__device__ unsigned long long g_phase_fwd[32];
#define PHF(i) do { if (blockIdx.x == 0 && threadIdx.x == 0) { unsigned long long _t = clock64(); g_phase_fwd[i] += _t - _tl; _tl = _t; } } while (0)
#else
#define PHF(i) do {} while (0)
#endif

constexpr int NT_FWD = 384;   // 8 consumer warps + 4 producer warps
constexpr int NCONS = 256;
constexpr int RING_ROWS = 16;                      // rows per landing slot (8 chunks per tile)
constexpr int RING_Y = RING_ROWS * H * 2;          // bf16 raw y rows
constexpr int RING_BYTES = RING_Y + RING_ROWS * H * 4;  // + fp32 residual rows = 12 KB
constexpr int RING_SLOTS = 4;                      // 48 KB of loads in flight per SM
constexpr int TC_SMEM_EDGE = 2 * tc::TILE_BF16_BYTES      // weight images We, W2
                             + 3 * tc::TILE_BF16_BYTES    // A0[2] (e_t / hn, double buffered), A1 (hm)
                             + RING_SLOTS * RING_BYTES    // landing ring of the producers' bulk row copies
                             + 3 * 2 * TM * 4             // recv / send (three slots)
                             + 2 * H * 4                  // b1, b2
                             + 2048 + 2048;               // scalars, segment codes (x3), barriers, alignment slack

__device__ __forceinline__ void csync() { asm volatile("bar.sync 1, 256;" ::: "memory"); }  // consumer warps only
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tc::smem_u32(bar)) : "memory");
}
// consumer-only block sum of two doubles (result valid in thread 0)
__device__ __forceinline__ void block_sum2_c(double& a, double& b, double* red) {
  a = warp_sum(a);
  b = warp_sum(b);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  csync();
  if (l == 0) { red[2 * w] = a; red[2 * w + 1] = b; }
  csync();
  if (threadIdx.x == 0) {
    double sa = 0, sb = 0;
#pragma unroll
    for (int i = 0; i < NCONS / 32; ++i) { sa += red[2 * i]; sb += red[2 * i + 1]; }
    a = sa; b = sb;
  }
}
__device__ __forceinline__ void psync() { asm volatile("bar.sync 2, 128;" ::: "memory"); }  // producer warps only
// producer: receiver segments of the tile (see tile_segsum_items in pdg_tc_tile.cuh).  128 producer threads, r = row.
__device__ __forceinline__ void tile_segments_p(int r, const int* recv_s, const int32_t* __restrict__ rowptr, int row0, int nvalid,
                                                unsigned char* seg_row, unsigned char* seg_cut, int* nseg, unsigned* masks) {
  const bool first = r < nvalid && (r == 0 || recv_s[r] != recv_s[r - 1]);
  const unsigned m = __ballot_sync(0xffffffffu, first);
  if ((r & 31) == 0) masks[r >> 5] = m;
  psync();
  if (first) {
    int idx = __popc(m & ((1u << (r & 31)) - 1u));
    for (int w = 0; w < (r >> 5); ++w) idx += __popc(masks[w]);
    seg_row[idx] = (unsigned char)r;
    const int c = recv_s[r];
    seg_cut[idx] = (rowptr[c] >= row0 && rowptr[c + 1] <= row0 + nvalid) ? 1 : 2;
  }
  if (r == 0) {
    const int n = __popc(masks[0]) + __popc(masks[1]) + __popc(masks[2]) + __popc(masks[3]);
    *nseg = n;
    seg_row[n] = (unsigned char)nvalid;
  }
}

__global__ void __launch_bounds__(NT_FWD, 1)
k_edge_step_tc(EdgeStepArgs a, const uint8_t* __restrict__ imgWe, const uint8_t* __restrict__ imgW2) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* sm = tc_smem_base(smem_raw);
  uint8_t* sWe = sm;
  uint8_t* sW2 = sWe + tc::TILE_BF16_BYTES;
  uint8_t* A0b = sW2 + tc::TILE_BF16_BYTES;  // [2] tiles
  uint8_t* A1 = A0b + 2 * tc::TILE_BF16_BYTES;
  uint8_t* ring = A1 + tc::TILE_BF16_BYTES;  // [RING_SLOTS][RING_BYTES]
  int* recv_b = reinterpret_cast<int*>(ring + RING_SLOTS * RING_BYTES);  // [3][TM]: ids / segment tables live in THREE slots (tile % 3) so that
                                                      // the producers may refill A0[buf] as soon as its last MMA has read it
  int* send_b = recv_b + 3 * TM;                      // [3][TM]
  float* b1s = reinterpret_cast<float*>(send_b + 3 * TM);
  float* b2s = b1s + H;
  double* red = reinterpret_cast<double*>(b2s + H);
  float* smf = reinterpret_cast<float*>(red + 16);
  int* nseg_b = reinterpret_cast<int*>(smf + 4);  // [3] (+1 pad)
  unsigned* masks = reinterpret_cast<unsigned*>(nseg_b + 4);
  unsigned char* seg_row_b = reinterpret_cast<unsigned char*>(masks + 4);  // [3][TM + 8]: first row of each receiver segment
  unsigned char* seg_cut_b = seg_row_b + 3 * (TM + 8);                      // [3][TM]: 1 whole / 2 cut by a tile boundary
  uint64_t* bars = reinterpret_cast<uint64_t*>(seg_cut_b + 3 * TM);  // [0] weights, [1..3] accumulators, [4,5] full, [6,7] empty
  uint64_t* lfull = bars + 8;  // [RING_SLOTS] landing slot filled (tx bytes)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 8 + RING_SLOTS);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) {
    tc::mbar_init(&bars[0], 1);
    tc::mbar_init(&bars[1], 1);
    tc::mbar_init(&bars[2], 1);
    tc::mbar_init(&bars[3], 1);
    tc::mbar_init(&bars[4], NT_FWD - NCONS);
    tc::mbar_init(&bars[5], NT_FWD - NCONS);
    tc::mbar_init(&bars[6], 1);  // empty[buf]: the last MMA reading A0[buf] (tcgen05.commit)
    tc::mbar_init(&bars[7], 1);
    for (int i = 0; i < RING_SLOTS; ++i) tc::mbar_init(&lfull[i], 1);
    tc::mbar_init_fence();
  }
  if (warp == 0) tc::tmem_alloc(tmem_slot, 512);
  if (tid < H) b2s[tid] = a.b2[tid];
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem = *tmem_slot;
  if (tid == 0) {
    tc::mbar_expect_tx(&bars[0], 2 * tc::TILE_BF16_BYTES);
    tc::bulk_g2s(sWe, imgWe, tc::TILE_BF16_BYTES, &bars[0]);
    tc::bulk_g2s(sW2, imgW2, tc::TILE_BF16_BYTES, &bars[0]);
  }
  pdl_sync();  // everything above touched parameters / packed weights only; activations of the predecessor from here on
  const LnStat st = ln_stat_block(a.prev_parts, a.prev_count, smf);  // all 384 threads (uses __syncthreads)
  const bool last_step = a.y2_out == nullptr;

  if (tid >= NCONS) {
    // =========================== PRODUCER warpgroup ===========================
    const int ptid = tid - NCONS;
    const int ch = ptid & 15;
    float lw[8], lb[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { lw[j] = a.prev_w[ch * 8 + j]; lb[j] = a.prev_b[ch * 8 + j]; }
    // The rows of this CTA's tiles arrive through a ring of landing slots filled by bulk copies (16 rows each: bf16 raw
    // y rows + fp32 residual rows), issued RING_SLOTS chunks ahead -- across tile boundaries and while A0 is still
    // busy -- so 48 KB of loads are in flight per SM without holding a register.
    const __half* yb = reinterpret_cast<const __half*>(a.yprev);  // raw y rows are fp16
    const int n_my = (a.n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
    const int n_chunks = n_my * (TM / RING_ROWS);
    auto issue_chunk = [&](const int c) {  // producer thread 0
      const size_t r0 = (size_t)(blockIdx.x + (c >> 3) * gridDim.x) * TM + (size_t)(c & 7) * RING_ROWS;
      uint8_t* slot = ring + (c & (RING_SLOTS - 1)) * RING_BYTES;
      uint64_t* bar = &lfull[c & (RING_SLOTS - 1)];
      tc::mbar_expect_tx(bar, a.base != nullptr ? RING_BYTES : RING_Y);
      tc::bulk_g2s(slot, yb + r0 * H, RING_Y, bar);
      if (a.base != nullptr) tc::bulk_g2s(slot + RING_Y, a.base + r0 * H, RING_BYTES - RING_Y, bar);
    };
    if (ptid == 0)
      for (int c = 0; c < RING_SLOTS && c < n_chunks; ++c) issue_chunk(c);
    int j = 0, c = 0;
    for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x, ++j) {
      const int buf = j & 1;
      uint8_t* A0 = A0b + buf * tc::TILE_BF16_BYTES;
      tc::mbar_wait(&bars[6 + buf], ((j >> 1) & 1) ^ 1);  // buffer free (first use passes immediately)
      const int row0 = tile * TM;
      {  // receiver / sender ids and segment bookkeeping of this tile (consumed two buffers later at the earliest)
        const int sl = j % 3;  // its previous tenant (tile j - 3) was finished before the MMA that freed A0[buf] was issued
        int* recv_s = recv_b + sl * TM;
        recv_s[ptid] = a.recv[row0 + ptid];
        send_b[sl * TM + ptid] = a.send[row0 + ptid];
        psync();
        tile_segments_p(ptid, recv_s, a.rowptr, row0, min(TM, a.E - row0), seg_row_b + sl * (TM + 8), seg_cut_b + sl * TM, nseg_b + sl, masks);
      }
      for (int cc = 0; cc < TM / RING_ROWS; ++cc, ++c) {
        const uint8_t* slot = ring + (c & (RING_SLOTS - 1)) * RING_BYTES;
        tc::mbar_wait(&lfull[c & (RING_SLOTS - 1)], (c / RING_SLOTS) & 1);
#pragma unroll
        for (int k = 0; k < RING_ROWS / 8; ++k) {
          const int rs = (ptid >> 4) + k * 8;  // row inside the slot
          const int r = cc * RING_ROWS + rs;   // row inside the tile
          const size_t g = ((size_t)row0 + r) * H + ch * 8;
          float yv[8];
          unpack8_f16(*reinterpret_cast<const uint4*>(slot + rs * (H * 2) + ch * 16), yv);
          float4 x0 = make_float4(0.f, 0.f, 0.f, 0.f), x1 = x0;
          if (a.base != nullptr) {
            x0 = *reinterpret_cast<const float4*>(slot + RING_Y + rs * (H * 4) + ch * 32);
            x1 = *reinterpret_cast<const float4*>(slot + RING_Y + rs * (H * 4) + ch * 32 + 16);
          }
          const float xv[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
          float v[8];
#pragma unroll
          for (int q = 0; q < 8; ++q) v[q] = (yv[q] - st.mu) * st.rstd * lw[q] + lb[q] + xv[q];
          if (a.e_out != nullptr) {
            *reinterpret_cast<float4*>(a.e_out + g) = make_float4(v[0], v[1], v[2], v[3]);
            *reinterpret_cast<float4*>(a.e_out + g + 4) = make_float4(v[4], v[5], v[6], v[7]);
          }
          *reinterpret_cast<uint4*>(A0 + tc::sw128_chunk(r, ch)) = tc::pack8_f16(v);
        }
        tc::fence_async_smem();  // generic reads of the slot (and the A0 writes) before the next asynchronous write
        psync();                 // every producer thread is done with the slot
        if (ptid == 0 && c + RING_SLOTS < n_chunks) issue_chunk(c + RING_SLOTS);
      }
      if (a.e_img != nullptr) {
        // training: the finished operand tile is also the backward's e_t operand -> one 32 KB bulk store of the
        // swizzled image.  The consumers overwrite A0 with the edge-update hidden tile, so the full barrier
        // completes only after the copy engine has read the buffer (thread 0 arrives last).
        if (ptid == 0) {
          tc::bulk_s2g(a.e_img + (size_t)tile * tc::TILE_BF16_BYTES, A0, tc::TILE_BF16_BYTES);
          tc::bulk_commit();
          tc::bulk_wait_read();
        }
      }
      mbar_arrive(&bars[4 + buf]);
    }
    if (ptid == 0) tc::bulk_wait_all();  // image stores have landed before the grid completes
    return;
  }

  // ============================= CONSUMER warps =============================
  const int row = 32 * (warp & 3) + lane, half = warp >> 2;
  const uint32_t lane_base = (uint32_t)(32 * (warp & 3)) << 16;
  const int ch = tid & 15;
  double t1s = 0, t1ss = 0, t2s = 0, t2ss = 0;
  uint32_t ph = 0;
  int i = 0;
#ifdef PDG_PHASE_TIMERS
  unsigned long long _tl = clock64();
#endif
  for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x, ++i) {
    const int buf = i & 1;
    uint8_t* A0 = A0b + buf * tc::TILE_BF16_BYTES;
    const int row0 = tile * TM;
    const int nvalid = min(TM, a.E - row0);
    const int sl = i % 3;
    const int* recv_s = recv_b + sl * TM;
    const int* send_s = send_b + sl * TM;
    const unsigned char* seg_row = seg_row_b + sl * (TM + 8);
    const unsigned char* seg_cut = seg_cut_b + sl * TM;
    if (tid == 0) {
      if (i == 0) tc::mbar_wait(&bars[0], 0);
      tc::mbar_wait(&bars[4 + buf], (i >> 1) & 1);  // e_t operand tile written by the producers
      tc::fence_after_sync();
      tc::issue_gemm_kmajor(tmem, tc::smem_u32(A0), tc::smem_u32(sWe), H, false);  // G = e_t We^T
      tc::mma_commit(&bars[1]);
      if (last_step) tc::mma_commit(&bars[6 + buf]);  // nothing else reads A0 on the last step
    }
    tc::mbar_wait(&bars[4 + buf], (i >> 1) & 1);  // every consumer: ids / segments of this tile are visible
    const int nseg = nseg_b[sl];
    PHF(0);
    // ---- hidden activations of both edge-MLP evaluations -> A1 (message), A0 (edge update) ----
    {
      const int rc = recv_s[row], sd = send_s[row];
      const __half* par = reinterpret_cast<const __half*>(a.Pa) + (size_t)rc * H + half * 64;
      const __half* pbs = reinterpret_cast<const __half*>(a.Pb) + (size_t)sd * H + half * 64;
      const __half* pas = reinterpret_cast<const __half*>(a.Pa) + (size_t)sd * H + half * 64;
      const __half* pbr = reinterpret_cast<const __half*>(a.Pb) + (size_t)rc * H + half * 64;
      uint4 gp[4][4];
      auto gather = [&](const int hh) {  // 256-bit loads: 8 instructions for this thread's four 64-byte row pieces
#pragma unroll
        for (int c8 = 0; c8 < 4; c8 += 2) {
          const int co = hh * 32 + c8 * 8;
          tc::ldg256(par + co, gp[c8][0], gp[c8 + 1][0]);
          tc::ldg256(pbs + co, gp[c8][1], gp[c8 + 1][1]);
          tc::ldg256(pas + co, gp[c8][2], gp[c8 + 1][2]);
          tc::ldg256(pbr + co, gp[c8][3], gp[c8 + 1][3]);
        }
      };
      gather(0);  // in flight while the G GEMM completes
      tc::mbar_wait(&bars[1], ph);
      tc::fence_after_sync();
      PHF(1);
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        if (hh) gather(hh);
        float gacc[32];
        tc::tmem_ld32(tmem + lane_base + (uint32_t)(half * 64 + hh * 32), gacc);
        tc::tmem_ld_wait();
#pragma unroll
        for (int c8 = 0; c8 < 4; ++c8) {
          const int co = hh * 32 + c8 * 8;  // column offset inside this thread's 64
          float pr[8], ps[8], qs8[8], qr[8];
          unpack8_f16(gp[c8][0], pr);
          unpack8_f16(gp[c8][1], ps);
          unpack8_f16(gp[c8][2], qs8);
          unpack8_f16(gp[c8][3], qr);
          float hm[8], hn[8];
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            const float g = gacc[c8 * 8 + q];  // the layer-1 bias rides in the Pa rows (k_node_pre_tc)
            hm[q] = fmaxf(g + pr[q] + ps[q], 0.f);
            hn[q] = fmaxf(g + qs8[q] + qr[q], 0.f);
          }
          const int chunk = half * 8 + hh * 4 + c8;
          *reinterpret_cast<uint4*>(A1 + tc::sw128_chunk(row, chunk)) = tc::pack8_f16(hm);
          if (!last_step) *reinterpret_cast<uint4*>(A0 + tc::sw128_chunk(row, chunk)) = tc::pack8_f16(hn);
        }
      }
    }
    PHF(2);
    tc::fence_before_sync();
    tc::fence_async_smem();
    csync();
    if (tid == 0) {
      tc::fence_after_sync();
      tc::issue_gemm_kmajor(tmem + 128, tc::smem_u32(A1), tc::smem_u32(sW2), H, false);  // message layer 2
      tc::mma_commit(&bars[2]);
      if (!last_step) {
        tc::issue_gemm_kmajor(tmem + 256, tc::smem_u32(A0), tc::smem_u32(sW2), H, false);  // edge-update layer 2
        tc::mma_commit(&bars[3]);
        tc::mma_commit(&bars[6 + buf]);  // A0[buf] may be refilled once this MMA has read it
      }
    }
    // ---- message: y1 = relu(acc1 + b2) -> bf16 tile in A1 (hm is dead: its GEMM completed) -> receiver-segment sums.
    //      LN1 partials come from the fp32 registers; the aggregated messages carry one bf16 rounding (the node MLP
    //      rounds the aggregate to a bf16 operand anyway).  One barrier, 128-bit shared-memory reads of 8 channels.
    tc::mbar_wait(&bars[2], ph);
    tc::fence_after_sync();
    PHF(3);
    {
      float s = 0.f, ss = 0.f;
      const bool ok = row < nvalid;
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        float v[32];
        tc::tmem_ld32(tmem + 128 + lane_base + (uint32_t)(half * 64 + hh * 32), v);
        tc::tmem_ld_wait();
#pragma unroll
        for (int q = 0; q < 32; q += 8) {
          const int c = half * 64 + hh * 32 + q;
          float o[8];
#pragma unroll
          for (int k = 0; k < 8; ++k) o[k] = fmaxf(v[q + k] + b2s[c + k], 0.f);
          if (ok) {
#pragma unroll
            for (int k = 0; k < 8; ++k) { s += o[k]; ss = fmaf(o[k], o[k], ss); }
          }
          *reinterpret_cast<uint4*>(A1 + tc::sw128_chunk(row, half * 8 + hh * 4 + (q >> 3))) = tc::pack8_f16(o);
        }
      }
      csync();
      float unused[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      tile_segsum_items(A1, recv_s, seg_row, seg_cut, nseg, a.aggraw, unused);
      double ds = s, dss = ss;
      block_sum2_c(ds, dss, red);
      if (tid == 0) { t1s += ds; t1ss += dss; }
    }
    PHF(4);
    // ---- edge update: y2 = relu(acc2 + b2): LN2 partials from registers, rows leave coalesced ----
    if (!last_step) {
      tc::mbar_wait(&bars[3], ph);
      tc::fence_after_sync();
      float s = 0.f, ss = 0.f;
      const bool ok = row < nvalid;
      // raw y2 rows are stored as bf16, straight from the accumulator registers: this thread's 64 channels are one
      // 128-byte line, written with four 256-bit stores (no staging tile, no barrier)
      __half* y2r = reinterpret_cast<__half*>(a.y2_out) + ((size_t)row0 + row) * H + half * 64;
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        float v[32];
        tc::tmem_ld32(tmem + 256 + lane_base + (uint32_t)(half * 64 + hh * 32), v);
        tc::tmem_ld_wait();
        uint4 pk[4];
#pragma unroll
        for (int q = 0; q < 32; q += 8) {
          const int c = half * 64 + hh * 32 + q;
          float o[8];
#pragma unroll
          for (int k = 0; k < 8; ++k) o[k] = fmaxf(v[q + k] + b2s[c + k], 0.f);
          if (ok) {
#pragma unroll
            for (int k = 0; k < 8; ++k) { s += o[k]; ss = fmaf(o[k], o[k], ss); }
          }
          pk[q >> 3] = tc::pack8_f16(o);
        }
        tc::stg256(y2r + hh * 32, pk[0], pk[1]);
        tc::stg256(y2r + hh * 32 + 16, pk[2], pk[3]);
      }
      double ds = s, dss = ss;
      block_sum2_c(ds, dss, red);
      if (tid == 0) { t2s += ds; t2ss += dss; }
    }
    PHF(5);
    ph ^= 1u;
    tc::fence_before_sync();
    csync();
    PHF(6);
  }
  if (tid == 0) {
    a.parts1[2 * blockIdx.x] = t1s;
    a.parts1[2 * blockIdx.x + 1] = t1ss;
    if (a.parts2 != nullptr) {
      a.parts2[2 * blockIdx.x] = t2s;
      a.parts2[2 * blockIdx.x + 1] = t2ss;
    }
  }
  if (warp == 0) tc::tmem_dealloc(tmem, 512);
}

#ifdef PDG_PHASE_TIMERS
extern "C" int pdg_phase_read_fwd(unsigned long long* out32) {
  return cudaMemcpyFromSymbol(out32, g_phase_fwd, sizeof(unsigned long long) * 32) == cudaSuccess ? 0 : -1;
}
#endif

int launch_edge_step_tc(const EdgeStepArgs& a, const uint8_t* img, int grid, cudaStream_t st) {
  return launch_named("k_edge_step_tc", true, k_edge_step_tc, dim3(grid), dim3(NT_FWD), TC_SMEM_EDGE, st, a,
                      weight_img(img, IMG_PE_WE), weight_img(img, IMG_PE_W2));
}

}  // namespace pdg
