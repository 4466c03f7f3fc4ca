// Fused training loss: per-graph NMSE + divergence-of-stress regulariser.
//
// Replaces the per-graph Python loop of the reference train() (gnn_train.py:162-202):
//   normalized_mse_loss_single   gnn_train.py:41-57
//   compute_divergence           gnn_train.py:60-92   (densify + slice + dense mm per graph)
//   slice_batch_gt_and_predictions / standardize      data_utils.py:25-33, 46-51
// The divergence is a batched CSR SpMM with 2 right-hand sides over the row-stacked
// operator exactly as PyG collation leaves it (graph-local column ids, SURVEY 2.3d); its
// backward is the CSC gather of the same operator (no atomics, fixed summation order).
#include <cub/cub.cuh>

#include "pdg_common.cuh"

namespace pdg {

struct OpPlanLayout {
  size_t off_rowptr, off_col, off_tptr, off_tidx, off_trow, total;
  __host__ OpPlanLayout(int64_t N, int64_t nnz) {
    size_t o = 0;
    auto take = [&](size_t elems) { size_t r = o; o += (size_t)round_up((int64_t)(elems * 4), 256); return r; };
    off_rowptr = take(N + 1);
    off_col = take(nnz);
    off_tptr = take(2 * N + 1);
    off_tidx = take(nnz);
    off_trow = take(nnz);
    total = o;
  }
};

__global__ void k_op_keys(const int64_t* __restrict__ coo_row, const int64_t* __restrict__ coo_col, int64_t nnz,
                          const int64_t* __restrict__ gptr, int B, int64_t N, int32_t* __restrict__ row32,
                          int32_t* __restrict__ col32, int32_t* __restrict__ skey, int32_t* __restrict__ iota) {
  const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (k < nnz) {
    const int64_t r = coo_row[k];
    int lo = 0, hi = B;  // graph g with gptr[g] <= r < gptr[g+1]
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (gptr[mid] <= r) lo = mid; else hi = mid;
    }
    // PyG stacks the per-graph operators along rows only, so the batch operator is as wide as the LARGEST graph's
    // 2 N_i; the reference slices the columns of graph i back to [0, 2 N_i) (`to_dense()[:, :shape[0]*2]`,
    // gnn_train.py:73-76).  Entries beyond that (or negative) are dropped here the same way: col32 = -1 is skipped
    // by the forward, key 2N sorts behind every stacked-stress row of the transpose.
    const int64_t c = coo_col[k];
    const int64_t ni = gptr[lo + 1] - gptr[lo];
    const bool keep = c >= 0 && c < 2 * ni;
    row32[k] = (int32_t)r;
    col32[k] = keep ? (int32_t)c : -1;
    skey[k] = keep ? (int32_t)(2 * gptr[lo] + c) : (int32_t)(2 * N);  // stacked-stress row, batch-global
    iota[k] = (int32_t)k;
  }
}
__global__ void k_lower_bound32(const int32_t* __restrict__ key, int64_t n, int64_t nrows, int32_t* __restrict__ ptr) {
  const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (r <= nrows) {
    int64_t lo = 0, hi = n;
    while (lo < hi) {
      const int64_t mid = (lo + hi) >> 1;
      if (key[mid] < (int32_t)r) lo = mid + 1; else hi = mid;
    }
    ptr[r] = (int32_t)lo;
  }
}
__global__ void k_gather32(const int32_t* __restrict__ src, const int32_t* __restrict__ idx, int64_t n,
                           int32_t* __restrict__ dst) {
  const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (k < n) dst[k] = src[idx[k]];
}

// ---- forward: one CTA per graph --------------------------------------------------------
// ws_graph[i] = {nmse_i, div_i, 1/norm_0, 1/norm_1, 1/norm_2} (stride 8); gdiv [N][2] masked divergence
constexpr int LOSS_NT = 256;
__device__ __forceinline__ double block_sum_d(double v, double* red) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double s = 0;
  for (int i = 0; i < LOSS_NT / 32; ++i) s += red[i];
  return s;  // every thread gets the same value (fixed order)
}

__global__ void __launch_bounds__(LOSS_NT)
k_loss_graph(const float* __restrict__ pred, const float* __restrict__ ls, float mean_ls, float std_ls,
             const int64_t* __restrict__ gptr, const int64_t* __restrict__ labels, const int32_t* __restrict__ rowptr,
             const int32_t* __restrict__ col, const float* __restrict__ val, int use_div, float* __restrict__ ws_graph,
             float* __restrict__ gdiv) {
  __shared__ double red[LOSS_NT / 32];
  const int g = blockIdx.x;
  const int n0 = (int)gptr[g], n1 = (int)gptr[g + 1], ni = n1 - n0;
  const int tid = threadIdx.x;
  double m[3] = {0, 0, 0};
  for (int n = n0 + tid; n < n1; n += LOSS_NT)
#pragma unroll
    for (int c = 0; c < 3; ++c) m[c] += (double)((ls[n * 3 + c] - mean_ls) / std_ls);
  float mean_gt[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) mean_gt[c] = (float)(block_sum_d(m[c], red) / ni);
  double mse[3] = {0, 0, 0}, nrm[3] = {0, 0, 0};
  for (int n = n0 + tid; n < n1; n += LOSS_NT)
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float gt = (ls[n * 3 + c] - mean_ls) / std_ls;
      const float d = gt - pred[n * 3 + c];
      const float e = gt - mean_gt[c];
      mse[c] += (double)(d * d);
      nrm[c] += (double)(e * e);
    }
  double nmse = 0;
  float inv_norm[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const double a = block_sum_d(mse[c], red), b = block_sum_d(nrm[c], red);
    nmse += (double)((float)a / (float)b);
    inv_norm[c] = 1.0f / (float)b;
  }
  nmse /= 3.0;
  double dv = 0;
  if (use_div) {
    double d2[2] = {0, 0};
    for (int n = n0 + tid; n < n1; n += LOSS_NT) {
      float d0 = 0.f, d1 = 0.f;
      // the reference zeroes the rows labelled 1 or -1 (gnn_train.py:88-89) and keeps every other label
      if (labels[n] != 1 && labels[n] != -1) {
        for (int k = rowptr[n]; k < rowptr[n + 1]; ++k) {
          const int j = col[k];
          if (j < 0) continue;  // column outside [0, 2 N_i): sliced away by the reference
          const float v = val[k];
          // S[j] = j < N_i ? (sxx, sxy)[j] : (sxy, syy)[j - N_i]     (gnn_train.py:68-70)
          const float s0 = j < ni ? pred[(n0 + j) * 3 + 0] : pred[(n0 + j - ni) * 3 + 2];
          const float s1 = j < ni ? pred[(n0 + j) * 3 + 2] : pred[(n0 + j - ni) * 3 + 1];
          d0 = fmaf(v, s0, d0);
          d1 = fmaf(v, s1, d1);
        }
      }
      gdiv[n * 2 + 0] = d0;
      gdiv[n * 2 + 1] = d1;
      d2[0] += (double)(d0 * d0);
      d2[1] += (double)(d1 * d1);
    }
    const double a = block_sum_d(d2[0], red), b = block_sum_d(d2[1], red);
    dv = (double)((float)a / (float)ni) + (double)((float)b / (float)ni);
  }
  if (tid == 0) {
    float* w = ws_graph + g * 8;
    w[0] = (float)nmse;
    w[1] = (float)dv;
    w[2] = inv_norm[0];
    w[3] = inv_norm[1];
    w[4] = inv_norm[2];
  }
}

__global__ void k_loss_finish(const float* __restrict__ ws_graph, int B, float penalty, int use_div,
                              float* __restrict__ out2) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    float a = 0.f, d = 0.f;  // sequential, like the reference's Python accumulation
    for (int g = 0; g < B; ++g) {
      a += ws_graph[g * 8 + 0];
      d += ws_graph[g * 8 + 1] * penalty;
    }
    out2[0] = a / (float)B;
    out2[1] = use_div ? d / (float)B : 0.f;
  }
}

// ---- backward: thread per node -----------------------------------------------------------
__global__ void k_loss_backward(const float* __restrict__ pred, const float* __restrict__ ls, float mean_ls,
                                float std_ls, const int64_t* __restrict__ gptr, int B, int N,
                                const float* __restrict__ ws_graph, const float* __restrict__ gdiv,
                                const int32_t* __restrict__ tptr, const int32_t* __restrict__ tidx,
                                const int32_t* __restrict__ trow, const float* __restrict__ val, int use_div,
                                float penalty, const float* __restrict__ upstream2, float* __restrict__ grad) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  int lo = 0, hi = B;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (gptr[mid] <= n) lo = mid; else hi = mid;
  }
  const float* w = ws_graph + lo * 8;
  const float up0 = upstream2 ? upstream2[0] : 1.f, up1 = upstream2 ? upstream2[1] : 1.f;
  float gr[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float gt = (ls[n * 3 + c] - mean_ls) / std_ls;
    gr[c] = up0 * (2.f * (pred[n * 3 + c] - gt) * w[2 + c]) / (3.f * (float)B);
  }
  if (use_div) {
    const int n0 = (int)gptr[lo];
    const int ni = (int)gptr[lo + 1] - n0;  // exact: a float holds N_i only up to 2^24
    const int ml = n - n0;
    float a0 = 0, a1 = 0, b0 = 0, b1 = 0;  // dS[ml][0], dS[ml][1], dS[ni+ml][0], dS[ni+ml][1]
    const int s1 = 2 * n0 + ml, s2 = 2 * n0 + ni + ml;
    for (int k = tptr[s1]; k < tptr[s1 + 1]; ++k) {
      const float v = val[tidx[k]];
      const int r = trow[k];
      a0 = fmaf(v, gdiv[r * 2 + 0], a0);
      a1 = fmaf(v, gdiv[r * 2 + 1], a1);
    }
    for (int k = tptr[s2]; k < tptr[s2 + 1]; ++k) {
      const float v = val[tidx[k]];
      const int r = trow[k];
      b0 = fmaf(v, gdiv[r * 2 + 0], b0);
      b1 = fmaf(v, gdiv[r * 2 + 1], b1);
    }
    const float coef = up1 * penalty * 2.f / ((float)ni * (float)B);
    gr[0] += coef * a0;         // sxx  = S[ml][0]
    gr[1] += coef * b1;         // syy  = S[ni+ml][1]
    gr[2] += coef * (b0 + a1);  // sxy  = S[ni+ml][0] and S[ml][1]
  }
  grad[n * 3 + 0] = gr[0];
  grad[n * 3 + 1] = gr[1];
  grad[n * 3 + 2] = gr[2];
}

static size_t sort_tmp_bytes32(int64_t n) {
  size_t b = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, b, (const int32_t*)nullptr, (int32_t*)nullptr, (const int32_t*)nullptr,
                                  (int32_t*)nullptr, (int)n);
  return b;
}

}  // namespace pdg

using namespace pdg;

extern "C" size_t pdg_opdiv_plan_bytes(int64_t n_nodes, int64_t nnz) { return OpPlanLayout(n_nodes, nnz).total; }
extern "C" size_t pdg_opdiv_tmp_bytes(int64_t n_nodes, int64_t nnz) {
  return (size_t)round_up((int64_t)sort_tmp_bytes32(nnz), 256) + 4 * (size_t)round_up(nnz * 4, 256);
}

extern "C" int pdg_opdiv_plan_build(const int64_t* coo_row, const int64_t* coo_col, int64_t nnz,
                                    const int64_t* graph_ptr, int64_t n_graphs, int64_t n_nodes, void* plan, void* tmp,
                                    size_t tmp_bytes, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  if (nnz < 0 || nnz >= 0x7fffffff || n_nodes * 2 >= 0x7fffffff) { set_error("pdg_opdiv_plan_build: sizes out of range"); return -1; }
  if (tmp_bytes < pdg_opdiv_tmp_bytes(n_nodes, nnz)) { set_error("pdg_opdiv_plan_build: tmp too small"); return -1; }
  OpPlanLayout L(n_nodes, nnz);
  char* pb = (char*)plan;
  int32_t* rowptr = (int32_t*)(pb + L.off_rowptr);
  int32_t* col32 = (int32_t*)(pb + L.off_col);
  int32_t* tptr = (int32_t*)(pb + L.off_tptr);
  int32_t* tidx = (int32_t*)(pb + L.off_tidx);
  int32_t* trow = (int32_t*)(pb + L.off_trow);
  const size_t sb = sort_tmp_bytes32(nnz);
  char* t = (char*)tmp;
  void* sort_tmp = t;
  t += round_up((int64_t)sb, 256);
  int32_t* row32 = (int32_t*)t; t += round_up(nnz * 4, 256);
  int32_t* skey = (int32_t*)t; t += round_up(nnz * 4, 256);
  int32_t* iota = (int32_t*)t; t += round_up(nnz * 4, 256);
  int32_t* skey_sorted = (int32_t*)t;
  const int TB = 256, gb = (int)((nnz + TB - 1) / TB);
  // nnz == 0 (an empty operator): no keys to make or sort; both pointer arrays come out all 0
  if (nnz > 0) {
    k_op_keys<<<gb, TB, 0, st>>>(coo_row, coo_col, nnz, graph_ptr, (int)n_graphs, n_nodes, row32, col32, skey, iota);
    PDG_LAUNCH_CHECK();
  }
  // CSR: coalesced COO is already row-sorted (torch .coalesce())
  k_lower_bound32<<<(int)((n_nodes + 1 + TB - 1) / TB), TB, 0, st>>>(row32, nnz, n_nodes, rowptr);
  PDG_LAUNCH_CHECK();
  int bits = 1;
  while ((1ll << bits) <= 2 * n_nodes && bits < 31) ++bits;
  if (nnz > 0)
    PDG_CUDA_CHECK(cub::DeviceRadixSort::SortPairs(sort_tmp, const_cast<size_t&>(sb), skey, skey_sorted, iota, tidx,
                                                   (int)nnz, 0, bits, st));
  k_lower_bound32<<<(int)((2 * n_nodes + 1 + TB - 1) / TB), TB, 0, st>>>(skey_sorted, nnz, 2 * n_nodes, tptr);
  PDG_LAUNCH_CHECK();
  if (nnz > 0) {
    k_gather32<<<gb, TB, 0, st>>>(row32, tidx, nnz, trow);
    PDG_LAUNCH_CHECK();
  }
  return 0;
}

extern "C" size_t pdg_loss_ws_bytes(int64_t n_nodes, int64_t n_graphs) {
  return (size_t)round_up(n_graphs * 8 * 4, 256) + (size_t)round_up(n_nodes * 2 * 4, 256);
}

extern "C" int pdg_loss(const float* pred, const float* local_stress, const pdg_norm_t* norm, const int64_t* graph_ptr,
                        int64_t n_graphs, int64_t n_nodes, const int64_t* labels, const void* opdiv_plan,
                        const float* op_val, int64_t nnz, int use_divergence, float penalty, void* ws, float* out2,
                        void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  if (n_graphs <= 0 || n_nodes <= 0) { set_error("pdg_loss: empty batch"); return -1; }
  if (use_divergence && (opdiv_plan == nullptr || (op_val == nullptr && nnz > 0) || labels == nullptr)) {
    set_error("pdg_loss: divergence requested without operator/labels");
    return -1;
  }
  float* ws_graph = (float*)ws;
  float* gdiv = (float*)((char*)ws + round_up(n_graphs * 8 * 4, 256));
  const int32_t *rowptr = nullptr, *col = nullptr;
  if (use_divergence) {
    OpPlanLayout L(n_nodes, nnz);
    rowptr = (const int32_t*)((const char*)opdiv_plan + L.off_rowptr);
    col = (const int32_t*)((const char*)opdiv_plan + L.off_col);
  }
  {
    ScopedTimer tm_(KC_LOSS, st);
    k_loss_graph<<<(int)n_graphs, LOSS_NT, 0, st>>>(pred, local_stress, norm->mean_local_stress, norm->std_local_stress,
                                                    graph_ptr, labels, rowptr, col, op_val, use_divergence, ws_graph, gdiv);
  }
  PDG_LAUNCH_CHECK();
  k_loss_finish<<<1, 32, 0, st>>>(ws_graph, (int)n_graphs, penalty, use_divergence, out2);
  PDG_LAUNCH_CHECK();
  return 0;
}

extern "C" int pdg_loss_backward(const float* pred, const float* local_stress, const pdg_norm_t* norm,
                                 const int64_t* graph_ptr, int64_t n_graphs, int64_t n_nodes, const void* opdiv_plan,
                                 const float* op_val, int64_t nnz, int use_divergence, float penalty, const void* ws,
                                 const float* upstream2, float* grad_pred, void* stream_) {
  cudaStream_t st = (cudaStream_t)stream_;
  const float* ws_graph = (const float*)ws;
  const float* gdiv = (const float*)((const char*)ws + round_up(n_graphs * 8 * 4, 256));
  const int32_t *tptr = nullptr, *tidx = nullptr, *trow = nullptr;
  if (use_divergence) {
    OpPlanLayout L(n_nodes, nnz);
    tptr = (const int32_t*)((const char*)opdiv_plan + L.off_tptr);
    tidx = (const int32_t*)((const char*)opdiv_plan + L.off_tidx);
    trow = (const int32_t*)((const char*)opdiv_plan + L.off_trow);
  }
  const int TB = 128;
  {
    ScopedTimer tm_(KC_LOSS_BWD, st);
    k_loss_backward<<<(int)((n_nodes + TB - 1) / TB), TB, 0, st>>>(pred, local_stress, norm->mean_local_stress,
                                                                   norm->std_local_stress, graph_ptr, (int)n_graphs,
                                                                   (int)n_nodes, ws_graph, gdiv, tptr, tidx, trow, op_val,
                                                                   use_divergence, penalty, upstream2, grad_pred);
  }
  PDG_LAUNCH_CHECK();
  return 0;
}
