// tcgen05 / TMEM / mbarrier / bulk-copy helpers for the 16-bit tensor-core tile engine (sm_100a).
//
// Operand format: fp16 everywhere (kind::f16 with both operand formats F16; the hardware rejects mixed bf16 x fp16
// operands with an illegal-instruction fault, tried).  fp16 has 11 significand bits against bf16's 8:
//   * weights: a weight image is rounded ONCE and then used by every row of every step, so its rounding is a
//     systematic perturbation of the model that no sum averages out -- with bf16 weights the gradients sat
//     1.5e-2 .. 2.5e-2 from the fp64 oracle whatever the batch size (DESIGN.md section 4b);
//   * forward-valued tiles / rows (latents, hidden activations, raw MLP outputs, Pa / Pb) are O(1e-2) .. O(1e2):
//     well inside fp16's range; every conversion saturates (cvt.rn.satfinite) so nothing can become inf;
//   * gradient-valued tiles / rows (dy, d-hidden, g_agg, dhm / dhn) span ~6 decades along the backward chain and are
//     tiny in absolute terms (1e-3 .. 1e-9): pdg_backward multiplies d loss / d local_stress by a power of two S chosen
//     on the device so that the largest element of the decoder's first gradient tile, g * gscale (gscale =
//     std_local_stress with scale_output), sits at 2^8 (k_grad_scale), the whole -- linear -- backward runs on
//     scaled values (fp32 streams included) and k_grad_reduce multiplies the weight gradients by 1/S.  That is the
//     GradScaler of the reference train loop (gnn_train.py:111,204-207) moved inside the operator, with no host sync.
//     Values down to 2^-15 of the scaled stream keep at least bf16's relative precision, smaller ones an absolute
//     error of 6e-8; the headroom above is 2^8.
// Operand tile = [128 rows][128 cols] of 16-bit elements stored as TWO column blocks of [128 rows][64 cols]
// (128-byte rows, 16 KB per block), each in the canonical SWIZZLE_128B layout (16-byte chunk
// index XOR (row & 7)).  The SAME bytes serve two roles:
//   * K-major operand  (row = M/N index, col = K):  D = A . B^T         (forward / dgrad GEMMs)
//   * MN-major operand (row = K index,  col = M/N): D = A^T . B         (weight-gradient GEMMs)
// so an activation tile written once by an epilogue feeds both the next dgrad and its wgrad.
// Descriptor fields follow cute/arch/mma_sm100_desc.hpp (SmemDescriptor, InstrDescriptor).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>

namespace pdg {
namespace tc {

constexpr int TILE_BF16_BYTES = 128 * 128 * 2;  // 32 KB
constexpr int BLOCK_BF16_BYTES = 128 * 64 * 2;  // 16 KB (one 64-column block)

// byte offset of element (r, c) inside a tile
__host__ __device__ __forceinline__ uint32_t sw128_off(int r, int c) {
  return (uint32_t)((c >> 6) * BLOCK_BF16_BYTES + r * 128 + (((((c & 63) >> 3) ^ (r & 7))) << 4) + (c & 7) * 2);
}
// byte offset of the 16-byte chunk holding columns [8*ch, 8*ch+8) of row r  (ch in 0..15)
__host__ __device__ __forceinline__ uint32_t sw128_chunk(int r, int ch) {
  return (uint32_t)((ch >> 3) * BLOCK_BF16_BYTES + r * 128 + (((ch & 7) ^ (r & 7)) << 4));
}

#ifdef __CUDACC__
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- shared-memory matrix descriptors (version 1 = Blackwell, SWIZZLE_128B = 2) ---------------
__device__ __forceinline__ uint64_t desc_base(uint32_t lbo16, uint32_t sbo16) {
  return ((uint64_t)(lbo16 & 0x3FFF) << 16) | ((uint64_t)(sbo16 & 0x3FFF) << 32) | (1ull << 46) | (2ull << 61);
}
// K-major: rows 128 B apart, 8-row groups 1024 B apart (SBO = 64), LBO unused (= 1)
__device__ __forceinline__ uint64_t desc_kmajor(uint32_t saddr) { return desc_base(1, 64) | (uint64_t)((saddr >> 4) & 0x3FFF); }
// MN-major: 64-column blocks 16 KB apart (LBO = 1024), 8-row (K) groups 1024 B apart (SBO = 64)
__device__ __forceinline__ uint64_t desc_mnmajor(uint32_t saddr) { return desc_base(1024, 64) | (uint64_t)((saddr >> 4) & 0x3FFF); }

// instruction descriptor: D fp32, M = 128, N = n; a_fmt / b_fmt: 0 = fp16, 1 = bf16 (cute::UMMA::F16F32Format)
constexpr uint32_t FMT_F16 = 0, FMT_BF16 = 1;
__host__ __device__ constexpr uint32_t idesc_16(int n, int a_mn, int b_mn, uint32_t a_fmt, uint32_t b_fmt) {
  return (1u << 4) | (a_fmt << 7) | (b_fmt << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) | ((uint32_t)(n >> 3) << 17) |
         ((uint32_t)(128 >> 4) << 24);
}

__device__ __forceinline__ void mma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[128 x n] (+)= A[128 x 128] . B[n x 128]^T ; both tiles K-major.  One thread issues 8 MMAs.
// Forward shape: A = forward-valued activation tile, B = weight image.
__device__ __forceinline__ void issue_gemm_kmajor(uint32_t tmem_d, uint32_t a_saddr, uint32_t b_saddr, int n, bool accumulate) {
  const uint32_t id = idesc_16(n, 0, 0, FMT_F16, FMT_F16);
#pragma unroll
  for (int kb = 0; kb < 2; ++kb)
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      const uint32_t off = kb * BLOCK_BF16_BYTES + ks * 32;
      mma_bf16(tmem_d, desc_kmajor(a_saddr + off), desc_kmajor(b_saddr + off), id, (accumulate || kb || ks) ? 1u : 0u);
    }
}
// D[128 x 128] (+)= A^T . B with A, B = [128 rows (K)][128 cols] tiles (MN-major operands)
// Weight-gradient shape: A = gradient tile, B = forward-valued activation tile.
__device__ __forceinline__ void issue_gemm_mnmajor(uint32_t tmem_d, uint32_t a_saddr, uint32_t b_saddr, bool accumulate) {
  const uint32_t id = idesc_16(128, 1, 1, FMT_F16, FMT_F16);
#pragma unroll
  for (int ks = 0; ks < 8; ++ks) {
    const uint32_t off = ks * 16 * 128;  // 16 K-rows
    mma_bf16(tmem_d, desc_mnmajor(a_saddr + off), desc_mnmajor(b_saddr + off), id, (accumulate || ks) ? 1u : 0u);
  }
}
// D[128 x 128] (+)= A . B with A = [128 rows (M)][128 cols (K)] K-major and B = [128 rows (K)][128 cols (N)]
// MN-major: the data-gradient shape dX = dY . W for an nn.Linear weight image W[out = K][in = N].
// A = gradient tile, B = weight image.
__device__ __forceinline__ void issue_gemm_k_mn(uint32_t tmem_d, uint32_t a_saddr, uint32_t b_saddr, bool accumulate) {
  const uint32_t id = idesc_16(128, 0, 1, FMT_F16, FMT_F16);
#pragma unroll
  for (int kk = 0; kk < 8; ++kk) {
    const uint32_t aoff = (kk >> 2) * BLOCK_BF16_BYTES + (kk & 3) * 32;
    const uint32_t boff = kk * 16 * 128;
    mma_bf16(tmem_d, desc_kmajor(a_saddr + aoff), desc_mnmajor(b_saddr + boff), id, (accumulate || kk) ? 1u : 0u);
  }
}
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// generic-proxy smem writes -> visible to the async proxy (tensor core / bulk copies)
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- TMEM --------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* slot, uint32_t ncols) {  // one full warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t ncols) {  // same warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(ncols) : "memory");
}
// 32 consecutive fp32 columns of this thread's lane (lane = 32*(warp%4) + laneid)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t* u = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
      : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]), "=r"(u[8]),
        "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15]), "=r"(u[16]),
        "=r"(u[17]), "=r"(u[18]), "=r"(u[19]), "=r"(u[20]), "=r"(u[21]), "=r"(u[22]), "=r"(u[23]), "=r"(u[24]),
        "=r"(u[25]), "=r"(u[26]), "=r"(u[27]), "=r"(u[28]), "=r"(u[29]), "=r"(u[30]), "=r"(u[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---- mbarrier + 1-D bulk copy (TMA engine, SASS UBLKCP) --------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// expect-tx WITHOUT an arrival (the thread arrives later, after its generic-proxy writes)
__device__ __forceinline__ void mbar_expect_tx_only(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t done;
  do {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}\n"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  } while (!done);
}
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(smem_dst)),
               "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// TMA reduce: global[i] += smem[i] over a contiguous range, performed by the copy engine at L2 (no loads, no
// registers, asynchronous).  bytes % 16 == 0, both addresses 16-byte aligned.  Bulk-group completion.
__device__ __forceinline__ void bulk_reduce_add_f32(float* gmem_dst, const float* smem_src, uint32_t bytes) {
  asm volatile("cp.reduce.async.bulk.global.shared::cta.bulk_group.add.f32 [%0], [%1], %2;" ::"l"(gmem_dst),
               "r"(smem_u32(smem_src)), "r"(bytes)
               : "memory");
}
// plain bulk store shared -> global (bulk-group completion)
__device__ __forceinline__ void bulk_s2g(void* gmem_dst, const void* smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gmem_dst), "r"(smem_u32(smem_src)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }  // smem reusable
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }         // writes done

// 256-bit read-only global load (SASS LDG.E.256): two 16-byte chunks per instruction.  The row gathers of the
// edge kernels are bound by L1 tag-stage cycles (one per distinct line per instruction), so half the instructions
// is half the cost.  p must be 32-byte aligned.
__device__ __forceinline__ void ldg256(const void* p, uint4& a, uint4& b) {
  asm volatile("ld.global.nc.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(a.x), "=r"(a.y), "=r"(a.z), "=r"(a.w), "=r"(b.x), "=r"(b.y), "=r"(b.z), "=r"(b.w)
               : "l"(p));
}
// streaming loads that do not allocate in L1 (the L1 left beside >200 KB of shared memory is tiny; rows that are
// read once should not compete with the gathers for its lines / miss tracking)
__device__ __forceinline__ uint4 ldcg128(const void* p) {
  uint4 a;
  asm volatile("ld.global.cg.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(a.x), "=r"(a.y), "=r"(a.z), "=r"(a.w) : "l"(p));
  return a;
}
__device__ __forceinline__ void ldcg256(const void* p, float4& a, float4& b) {
  asm volatile("ld.global.cg.v8.f32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w), "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w)
               : "l"(p));
}
// 256-bit global store (SASS STG.E.256): row-per-thread stores pay one L1 tag-stage cycle per line per instruction
__device__ __forceinline__ void stg256(void* p, const uint4& a, const uint4& b) {
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "r"(a.x), "r"(a.y), "r"(a.z), "r"(a.w),
               "r"(b.x), "r"(b.y), "r"(b.z), "r"(b.w)
               : "memory");
}
// L2 prefetch of a contiguous range by the copy engine (one instruction; bytes % 16 == 0)
__device__ __forceinline__ void bulk_prefetch_l2(const void* p, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}
// L2 prefetch of one 128-byte line (used to pull the NEXT tile's rows in while this tile computes)
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// pack 8 floats -> 8 fp16 (one 16-byte chunk), round to nearest, saturating to +-65504 (SASS F2FP.SATFINITE.F16.F32.PACK_AB):
// forward-valued tiles / rows and weight images
__device__ __forceinline__ uint32_t pack2_f16(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ uint4 pack8_f16(const float* v) {
  return make_uint4(pack2_f16(v[0], v[1]), pack2_f16(v[2], v[3]), pack2_f16(v[4], v[5]), pack2_f16(v[6], v[7]));
}
#endif  // __CUDACC__

}  // namespace tc
}  // namespace pdg
