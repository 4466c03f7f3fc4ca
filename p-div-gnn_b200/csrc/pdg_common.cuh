// Shared device/host helpers for libpdivgnn (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/pdg.h"

namespace pdg {

constexpr int H = PDG_H;        // latent width
constexpr int TM = PDG_TILE;    // rows per tile
constexpr int LDS = H + 4;      // smem row pitch (floats): rows stay 16B aligned
constexpr int NT = 256;         // threads per CTA of every tile kernel
constexpr int BK = 32;          // k-chunk of the streamed weight operand
constexpr int MAXP = 296;       // max CTAs whose LayerNorm partials are kept (2 x 148)
// Persistent tile kernels: the smallest grid that needs no more rounds than `cap` CTAs would (1 516 tiles on 148 SMs are
// 11 rounds either way: 138 CTAs do them as well as 148).  The SMs left over take the side stream's batch-building
// kernels, which otherwise wait for a kernel boundary each (the training kernels fill every SM).
inline int balanced_grid(int n_tiles, int cap) {
  if (n_tiles <= cap) return n_tiles;
  const int rounds = (n_tiles + cap - 1) / cap;
  return (n_tiles + rounds - 1) / rounds;
}
constexpr float LN_EPS = 1e-5f; // torch_geometric.nn.LayerNorm eps

// ---- error reporting ---------------------------------------------------------------
void set_error(const char* fmt, ...);
// a kernel's dynamic shared-memory limit (cudaFuncAttributeMaxDynamicSharedMemorySize); -2 with the error set on failure
int set_smem(const void* fn, size_t bytes);
int num_sms();
#define PDG_CUDA_CHECK(expr)                                                          \
  do {                                                                                \
    cudaError_t _e = (expr);                                                          \
    if (_e != cudaSuccess) {                                                          \
      pdg::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return -2;                                                                      \
    }                                                                                 \
  } while (0)
void count_launches(int n);
#define PDG_LAUNCH_CHECK()              \
  do {                                  \
    pdg::count_launches(1);             \
    PDG_CUDA_CHECK(cudaGetLastError()); \
  } while (0)

// kernel classes for the optional CUDA-event timers (pdg_timing_enable / _collect)
enum KClass {
  KC_PACK = 0, KC_NODE_ENC, KC_EDGE_ENC, KC_NODE_PRE, KC_EDGE_STEP, KC_NODE_UPD, KC_DECODER,
  KC_DEC_BWD, KC_NODE_UPD_BWD, KC_EDGE_STEP_BWD, KC_NODE_PRE_BWD, KC_ENC_BWD, KC_LN_FIN, KC_GRAD_REDUCE,
  KC_LOSS, KC_LOSS_BWD,
  KC_JVP_NODE_ENC, KC_JVP_EDGE_ENC, KC_JVP_NODE_PRE, KC_JVP_EDGE_STEP, KC_JVP_NODE_UPD, KC_JVP_DECODER,
  KC_VJP_DECODER, KC_VJP_NODE_UPD, KC_VJP_EDGE_STEP, KC_VJP_NODE_PRE, KC_VJP_ENC, KC_VJP_LN_FIN, KC_COUNT
};
void timing_begin(int cls, cudaStream_t st);
void timing_end(cudaStream_t st);
struct ScopedTimer {
  cudaStream_t st;
  ScopedTimer(int cls, cudaStream_t s) : st(s) { timing_begin(cls, s); }
  ~ScopedTimer() { timing_end(st); }
};

static inline int64_t round_up(int64_t v, int64_t m) { return (v + m - 1) / m * m; }

// ---- programmatic dependent launch (PDL) ------------------------------------------------------------------
// The hot path is a serial chain of ~120 kernels per training step.  Kernels launched with launch_pdl() may be
// scheduled while their predecessor is still draining: their CTAs start on SMs the predecessor has left, run the
// part of their prologue that touches no activation data (barrier init, TMEM allocation, TMA load of the weight
// images, biases) and then block in pdl_wait() until the predecessor grid has completed and its writes are
// visible.  pdl_trigger() right after the wait lets the NEXT kernel start launching; because it comes after the
// wait, a kernel's pre-wait prologue may read anything written two or more launches earlier (the packed weights).
// Every kernel launched with launch_pdl() MUST call pdl_wait() before its first read of predecessor data.
// Without the launch attribute both instructions are no-ops.  PDG_NO_PDL=1 in the environment disables it.
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_sync() { pdl_wait(); pdl_trigger(); }
bool pdl_enabled();
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = pdl_enabled() ? 1 : 0;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}
#endif

// ---- parameter indices (state_dict order) ------------------------------------------
enum ParamIdx {
  NE_W0 = 0, NE_B0, NE_W2, NE_B2, NE_LNW, NE_LNB,
  EE_W0, EE_B0, EE_W2, EE_B2, EE_LNW, EE_LNB,
  PE_W0, PE_B0, PE_W2, PE_B2, PE_LNW, PE_LNB,
  PN_W0, PN_B0, PN_W2, PN_B2, PN_LNW, PN_LNB,
  ND_W0, ND_B0, ND_W2, ND_B2
};
// element offsets of each tensor inside the flat [PDG_PARAM_ELEMS] gradient buffer
__host__ __device__ constexpr int param_size(int i) {
  return i == NE_W0 ? H * 6 : i == EE_W0 ? H : i == PE_W0 ? H * 3 * H : i == PN_W0 ? H * 2 * H
       : (i == NE_W2 || i == EE_W2 || i == PE_W2 || i == PN_W2 || i == ND_W0) ? H * H
       : i == ND_W2 ? 3 * H : i == ND_B2 ? 3 : H;
}
__host__ __device__ constexpr int param_offset(int i) {
  int o = 0;
  for (int j = 0; j < i; ++j) o += param_size(j);
  return o;
}
static_assert(param_offset(PDG_NUM_PARAMS) == PDG_PARAM_ELEMS, "parameter layout");

// ---- transposed weight pack ([K][128] row-major so k-chunks stream contiguously) ----
struct PackOffsets {
  // float offsets inside the pack buffer
  static constexpr int NE_W2T = 0;                 // [128][128]
  static constexpr int EE_W2T = NE_W2T + H * H;
  static constexpr int PE_WAT = EE_W2T + H * H;    // edge_net.0.weight[:, 0:128]^T   (x_i = x[col])
  static constexpr int PE_WBT = PE_WAT + H * H;    // edge_net.0.weight[:, 128:256]^T (x_j = x[row])
  static constexpr int PE_WET = PE_WBT + H * H;    // edge_net.0.weight[:, 256:384]^T (edge_attr)
  static constexpr int PE_W2T = PE_WET + H * H;
  static constexpr int PN_WAT = PE_W2T + H * H;    // node_net.0.weight[:, 0:128]^T   (aggr)
  static constexpr int PN_WXT = PN_WAT + H * H;    // node_net.0.weight[:, 128:256]^T (x)
  static constexpr int PN_W2T = PN_WXT + H * H;
  static constexpr int ND_W0T = PN_W2T + H * H;
  static constexpr int TOTAL = ND_W0T + H * H;
};

// ---- device helpers ----------------------------------------------------------------
#ifdef __CUDACC__

// tangent or cotangent k's copy of a workspace buffer (or of an output): p + off bytes, off = k * (bytes between
// consecutive copies); nullptr stays nullptr
template <class T>
__device__ __forceinline__ T* copy_at(T* p, size_t off) {
  return p == nullptr ? p : reinterpret_cast<T*>(reinterpret_cast<uintptr_t>(p) + off);
}

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Block-wide sum of two doubles (all NT threads call; result valid in thread 0).
// red: smem scratch of >= 2*NT/32 doubles.
__device__ __forceinline__ void block_sum2(double& a, double& b, double* red) {
  a = warp_sum(a);
  b = warp_sum(b);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();
  if (l == 0) { red[2 * w] = a; red[2 * w + 1] = b; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double sa = 0, sb = 0;
#pragma unroll
    for (int i = 0; i < NT / 32; ++i) { sa += red[2 * i]; sb += red[2 * i + 1]; }
    a = sa; b = sb;
  }
}

// Graph-mode LayerNorm statistics from per-CTA partial sums {sum, sumsq} (doubles).
// Fixed-order reduction => every CTA derives bit-identical (mu, 1/(sigma+eps)).
struct LnStat { float mu, rstd, sigma; };
__device__ __forceinline__ LnStat ln_stat_from_parts(const double* __restrict__ parts, double count) {
  double s = 0, ss = 0;
  for (int i = 0; i < MAXP; ++i) { s += parts[2 * i]; ss += parts[2 * i + 1]; }
  const double mu = s / count;
  double var = ss / count - mu * mu;
  var = var > 0 ? var : 0;
  const double sigma = sqrt(var);
  LnStat r;
  r.mu = (float)mu;
  r.sigma = (float)sigma;
  r.rstd = (float)(1.0 / ((double)(float)sigma + (double)LN_EPS));
  return r;
}
// CTA-wide: warp 0 reduces the partials (lane-strided, then a fixed shuffle tree),
// broadcasts through smem.  sm: >= 3 floats.
__device__ __forceinline__ LnStat ln_stat_block(const double* __restrict__ parts, double count, float* sm) {
  if (threadIdx.x < 32) {
    // all loads issued before the first add (one L2 round trip, not a dependent chain); same summation order
    constexpr int K = (MAXP + 31) / 32;
    double2 v[K];
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const int i = threadIdx.x + 32 * k;
      v[k] = i < MAXP ? reinterpret_cast<const double2*>(parts)[i] : make_double2(0.0, 0.0);
    }
    double s = 0, ss = 0;
#pragma unroll
    for (int k = 0; k < K; ++k) { s += v[k].x; ss += v[k].y; }
    s = warp_sum(s);
    ss = warp_sum(ss);
    if (threadIdx.x == 0) {
      const double mu = s / count;
      double var = ss / count - mu * mu;
      var = var > 0 ? var : 0;
      const double sigma = sqrt(var);
      sm[0] = (float)mu;
      sm[1] = (float)(1.0 / ((double)(float)sigma + (double)LN_EPS));
      sm[2] = (float)sigma;
    }
  }
  __syncthreads();
  LnStat r;
  r.mu = sm[0];
  r.rstd = sm[1];
  r.sigma = sm[2];
  __syncthreads();
  return r;
}

// ---- receiver segments of a 128-row edge tile (fp32 tile kernels, NT = 256 threads) ---------------------
// seg_row[0..nseg]: first row of every run of equal receiver ids (seg_row[nseg] = nvalid); returns nseg.  All NT threads
// call; contains two __syncthreads().  seg_row: TM + 1 bytes, masks: 4 words.
__device__ __forceinline__ int tile_segments(const int* recv_s, int nvalid, unsigned char* seg_row, unsigned* masks) {
  const int r = threadIdx.x;
  const bool first = r < nvalid && (r == 0 || recv_s[r] != recv_s[r - 1]);
  const unsigned m = __ballot_sync(0xffffffffu, first);
  if (r < TM && (r & 31) == 0) masks[r >> 5] = m;
  __syncthreads();
  if (first) {
    int idx = __popc(m & ((1u << (r & 31)) - 1u));
    for (int w = 0; w < (r >> 5); ++w) idx += __popc(masks[w]);
    seg_row[idx] = (unsigned char)r;
  }
  const int n = __popc(masks[0]) + __popc(masks[1]) + __popc(masks[2]) + __popc(masks[3]);
  if (r == 0) seg_row[n] = (unsigned char)nvalid;
  __syncthreads();
  return n;
}
// Receiver-segment sums of an fp32 smem tile T[128][LDS] into dst[N][128]: one WARP per segment, lane = float4 chunk of the
// row (one 128-bit shared-memory load per row instead of a 64-row column walk per thread with a branch per row).  Rows are
// added in row order => the same bits as the column walk.  A segment that lies wholly inside the tile is a plain store;
// one cut by a tile boundary meets exactly one other partial sum: atomicAdd onto a zeroed row (order-free).  When STATS,
// s / ss accumulate the sum and the sum of squares of every element the lane touched (LayerNorm partials).
template <bool STATS>
__device__ __forceinline__ void tile_segsum_warp(const float* T, const int* recv_s, const unsigned char* seg_row, int nseg,
                                                 const int32_t* __restrict__ rowptr, int row0, int nvalid,
                                                 float* __restrict__ dst, float& s, float& ss) {
  const int lane = threadIdx.x & 31;
  for (int sg = threadIdx.x >> 5; sg < nseg; sg += NT / 32) {
    const int r0 = seg_row[sg], r1 = seg_row[sg + 1];
    const int c = recv_s[r0];
    const int lo = rowptr[c], hi = rowptr[c + 1];
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int r = r0; r < r1; ++r) {
      const float4 v = *reinterpret_cast<const float4*>(T + r * LDS + lane * 4);
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
      if (STATS) {
        s += (v.x + v.y) + (v.z + v.w);
        ss = fmaf(v.x, v.x, ss); ss = fmaf(v.y, v.y, ss); ss = fmaf(v.z, v.z, ss); ss = fmaf(v.w, v.w, ss);
      }
    }
    float* d = dst + (size_t)c * H + lane * 4;
    if (lo >= row0 && hi <= row0 + nvalid) {
      *reinterpret_cast<float4*>(d) = acc;
    } else {
      atomicAdd(d, acc.x); atomicAdd(d + 1, acc.y); atomicAdd(d + 2, acc.z); atomicAdd(d + 3, acc.w);
    }
  }
}

// ---- 128x128 register-tiled FFMA GEMM engine -----------------------------------------
// One micro-tile row update  acc[0..7] += a * {b0, b1}  as FOUR packed FFMA2 (fma.rn.f32x2, sm_100: two IEEE fp32 FMAs per
// instruction, scalar-broadcast first operand -- SASS `FFMA2 Rd, Ra.F32, Rb.F32x2.HI_LO, Rc.F32x2.HI_LO`).  The 3-register
// FFMA issues every other cycle per scheduler on Blackwell, so the scalar form tops out at half the fp32 peak; the packed
// form does the same arithmetic (each lane is a plain round-to-nearest fma: results bit-identical to fmaf) in half
// the instructions.  PDG_NO_FFMA2 keeps the scalar form for A/B measurements.
__device__ __forceinline__ void fma_row8(float (&acc)[8], float a, const float4& b0, const float4& b1) {
#ifndef PDG_NO_FFMA2
  const float2 a2 = make_float2(a, a);
  const float2 r0 = __ffma2_rn(a2, make_float2(b0.x, b0.y), make_float2(acc[0], acc[1]));
  const float2 r1 = __ffma2_rn(a2, make_float2(b0.z, b0.w), make_float2(acc[2], acc[3]));
  const float2 r2 = __ffma2_rn(a2, make_float2(b1.x, b1.y), make_float2(acc[4], acc[5]));
  const float2 r3 = __ffma2_rn(a2, make_float2(b1.z, b1.w), make_float2(acc[6], acc[7]));
  acc[0] = r0.x; acc[1] = r0.y; acc[2] = r1.x; acc[3] = r1.y;
  acc[4] = r2.x; acc[5] = r2.y; acc[6] = r3.x; acc[7] = r3.y;
#else
  acc[0] = fmaf(a, b0.x, acc[0]); acc[1] = fmaf(a, b0.y, acc[1]); acc[2] = fmaf(a, b0.z, acc[2]); acc[3] = fmaf(a, b0.w, acc[3]);
  acc[4] = fmaf(a, b1.x, acc[4]); acc[5] = fmaf(a, b1.y, acc[5]); acc[6] = fmaf(a, b1.z, acc[6]); acc[7] = fmaf(a, b1.w, acc[7]);
#endif
}
// acc[i][j] (+)= sum_k As[row_i][k] * Wt[k][col_j]
//   rows  row_i = ty*8 + i            (ty = tid / 16)
//   cols  col_j = tx*4 + j (j<4) , 64 + tx*4 + (j-4) (j>=4)   (tx = tid % 16)
// As: smem [128][LDS] fp32;  Wt: global [K][128] fp32 (k-major, i.e. W^T of nn.Linear);
// Ws: smem double buffer [2][BKT][128]; ldw: row pitch of Wt in floats (column blocks of
// a wider matrix are addressed by offsetting Wt).
// All NT threads must call.  Contains the __syncthreads() that make prior smem writes to
// As visible, and ends with one so the caller may overwrite As right after.
template <int BKT = BK>
__device__ __forceinline__ void gemm_rowA(const float* __restrict__ As, const float* __restrict__ Wt, int K,
                                          float (&acc)[8][8], float* __restrict__ Ws, int ldw = H) {
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  const int nch = K / BKT;
  auto load_chunk = [&](int c, int buf) {
    const float* src = Wt + (size_t)c * BKT * ldw;
    float* dst = Ws + buf * BKT * H;
#pragma unroll
    for (int i = 0; i < (BKT * H / 4) / NT; ++i) {
      const int idx = tid + i * NT;
      cp_async16(dst + idx * 4, src + (size_t)(idx >> 5) * ldw + (idx & 31) * 4);
    }
    cp_async_commit();
  };
  load_chunk(0, 0);
  for (int c = 0; c < nch; ++c) {
    // ONE barrier per chunk: it makes chunk c (and, for c = 0, the caller's writes to As) visible and tells that every
    // thread is done with chunk c - 1, whose buffer then takes chunk c + 1 while chunk c is multiplied
    cp_async_wait<0>();
    __syncthreads();
    if (c + 1 < nch) load_chunk(c + 1, (c + 1) & 1);
    const float* Wb = Ws + (c & 1) * BKT * H;
    const float* Ab = As + (ty * 8) * LDS + c * BKT;
#pragma unroll
    for (int kk = 0; kk < BKT; kk += 4) {
      float4 a[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) a[i] = *reinterpret_cast<const float4*>(Ab + i * LDS + kk);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float4 b0 = *reinterpret_cast<const float4*>(Wb + (kk + q) * H + tx * 4);
        const float4 b1 = *reinterpret_cast<const float4*>(Wb + (kk + q) * H + 64 + tx * 4);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float av = q == 0 ? a[i].x : q == 1 ? a[i].y : q == 2 ? a[i].z : a[i].w;
          fma_row8(acc[i], av, b0, b1);
        }
      }
    }
  }
  __syncthreads();
}

// acc[i][j] += sum_r A[r][row_i] * B[r][col_j]   (weight-gradient shape: reduction over
// the tile's rows r < nrows).  A, B: smem [128][LDS].  Same (i, j) -> (row, col) mapping
// as gemm_rowA with row_i = ty*8+i indexing A's COLUMNS.  Caller syncs before/after.
__device__ __forceinline__ void gemm_colA(const float* __restrict__ A, const float* __restrict__ B, int nrows,
                                          float (&acc)[8][8]) {
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
#pragma unroll 4
  for (int r = 0; r < nrows; ++r) {
    const float4 a0 = *reinterpret_cast<const float4*>(A + r * LDS + ty * 8);
    const float4 a1 = *reinterpret_cast<const float4*>(A + r * LDS + ty * 8 + 4);
    const float4 b0 = *reinterpret_cast<const float4*>(B + r * LDS + tx * 4);
    const float4 b1 = *reinterpret_cast<const float4*>(B + r * LDS + 64 + tx * 4);
    const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
#pragma unroll
    for (int i = 0; i < 8; ++i) fma_row8(acc[i], av[i], b0, b1);
  }
}

__device__ __forceinline__ void acc_zero(float (&acc)[8][8]) {
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
}
// micro-tile <-> smem / global (row-major, pitch ld floats)
__device__ __forceinline__ void acc_store(const float (&acc)[8][8], float* dst, int ld) {
  const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    float* p = dst + (size_t)(ty * 8 + i) * ld + tx * 4;
    *reinterpret_cast<float4*>(p) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
    *reinterpret_cast<float4*>(p + 64) = make_float4(acc[i][4], acc[i][5], acc[i][6], acc[i][7]);
  }
}
__device__ __forceinline__ void acc_load(float (&acc)[8][8], const float* src, int ld) {
  const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const float* p = src + (size_t)(ty * 8 + i) * ld + tx * 4;
    const float4 u = *reinterpret_cast<const float4*>(p);
    const float4 v = *reinterpret_cast<const float4*>(p + 64);
    acc[i][0] = u.x; acc[i][1] = u.y; acc[i][2] = u.z; acc[i][3] = u.w;
    acc[i][4] = v.x; acc[i][5] = v.y; acc[i][6] = v.z; acc[i][7] = v.w;
  }
}
// per-thread column constants (bias etc.): cols tx*4..+3 and 64+tx*4..+3
__device__ __forceinline__ void load_cols(float (&v)[8], const float* __restrict__ vec) {
  const int tx = threadIdx.x & 15;
  const float4 u = *reinterpret_cast<const float4*>(vec + tx * 4);
  const float4 w = *reinterpret_cast<const float4*>(vec + 64 + tx * 4);
  v[0] = u.x; v[1] = u.y; v[2] = u.z; v[3] = u.w;
  v[4] = w.x; v[5] = w.y; v[6] = w.z; v[7] = w.w;
}
#endif  // __CUDACC__

}  // namespace pdg
