// Workspace layouts shared by forward and backward (host side).
#pragma once
#include "pdg_common.cuh"

namespace pdg {

// LayerNorm instances ("slots") of one forward pass: 2 + 3T  (SURVEY a7: 32 at T=10)
//   0 node_encoder.4   1 edge_encoder.4   2+3t edge_net.4 on the message (LN1)
//   3+3t edge_net.4 on the edge update (LN2)   4+3t node_net.4 (LN3)
static inline int slot_ln1(int t) { return 2 + 3 * t; }
static inline int slot_ln2(int t) { return 3 + 3 * t; }
static inline int slot_ln3(int t) { return 4 + 3 * t; }

// fp16 operand images kept in the forward workspace (tcgen05 path)
enum ImgIdx { IMG_PE_WE = 0, IMG_PE_W2, IMG_PE_WA, IMG_PE_WB, IMG_PN_WA, IMG_PN_WX, IMG_PN_W2, IMG_EE_W2, IMG_NE_W2, IMG_ND_W0, IMG_COUNT };

struct EdgeStepArgs {
  const float* base;
  const float* yprev;
  const double* prev_parts;
  double prev_count;
  const float* prev_w;
  const float* prev_b;
  float* e_out;
  uint8_t* e_img;  // tcgen05 path, training: bf16 SWIZZLE_128B operand-tile image of e_t ([n_tiles][32 KB]) for the backward
  const float* Pa;
  const float* Pb;
  const int32_t* recv;
  const int32_t* send;
  const int32_t* rowptr;
  const float* WtE;
  const float* b1;
  const float* Wt2;
  const float* b2;
  float* y2_out;  // tcgen05 path: yprev / y2_out (raw edge-MLP outputs) hold fp16 rows
  float* aggraw;
  double* parts1;
  double* parts2;
  int E;
  int n_tiles;
};
int launch_edge_step_tc(const EdgeStepArgs& a, const uint8_t* img, int grid, cudaStream_t st);  // pdg_tc_fwd.cu

constexpr int GRADP = (PDG_PARAM_ELEMS + 63) / 64 * 64;  // floats per CTA gradient slice

struct EdgeBwdArgs {
  const float* e_t;      // FFMA path: fp32 rows
  const uint8_t* e_img;  // tcgen05 path: fp16 operand-tile images written by the forward

  const float* Pa;
  const float* Pb;
  const float* gagg;
  float* ge;
  const float* y2_t;
  const float* yprev;
  const double* parts_prev;
  double count_prev;
  const int32_t* recv;
  const int32_t* send;
  const int32_t* rowptr;
  const float* WtE;
  const float* b1;
  const float* Wt2;
  const float* b2;
  const float* W0;
  const float* W2;
  const float* lnw;
  const float* scal1;
  const float* scal2;
  float* DHM;
  float* DHN;
  float* RA;
  float* RB;
  float* cta_grads;
  float* cs2;
  int E, n_tiles, last;
};
int launch_edge_step_bwd_tc3(const EdgeBwdArgs& a, const uint8_t* img, int grid, cudaStream_t st);  // pdg_tc_bwd3.cu (warp-specialised)

struct NodeUpdBwdArgs {
  float* gx;
  const float* y3;
  const float* hq;
  const float* aggraw;
  const float* x_t;
  const int32_t* rowptr;
  const float* scal3;
  const float* lnw_n;
  const double* parts1;
  double count1;
  const float* lnw_e;
  const float* lnb_e;
  const float* V1;
  const float* V2;
  float* gagg;
  float* cta_grads;
  float* cs1;
  int N, n_tiles;
  // tcgen05 path: fp16 operand-tile images written by the forward node kernels ([n_tiles][32 KB]); bulk-copied straight
  // into the operand buffers instead of re-reading and re-rounding the fp32 rows of hq / aggraw / x_t
  const uint8_t* x_img;
  const uint8_t* hq_img;
  const uint8_t* agg_img;
};
struct NodePreBwdArgs {
  float* gx;
  float* RA;  // read, then re-zeroed row by row (next step's segment sums start from zero)
  float* RB;
  const float* DHM;
  const float* DHN;
  const int32_t* sptr;
  const int32_t* slist;
  const float* x_t;
  const float* yprev;
  const double* parts_prev;
  double count_prev;
  const float* W0;
  float* cta_grads;
  float* cs3;
  int N, n_tiles;
  const uint8_t* x_img;  // tcgen05 path: fp16 operand-tile image of x_t (k_node_pre_tc)
};
// forward node kernels (tensor-core variants take the same data as the FFMA ones)
struct NodePreArgs {
  const float* base;
  const float* yprev;
  const double* prev_parts;
  double prev_count;
  const float* lnw;
  const float* lnb;
  float* x_out;
  float* Pa;
  float* Pb;
  float* aggraw_zero;  // [N_pad][H] segment-sum target of the following edge kernel: zeroed tile by tile
  const float* b1;     // edge-MLP layer-1 bias, folded into the Pa rows (every hidden evaluation adds exactly one Pa row)
  int n_tiles;
  uint8_t* x_img;      // tcgen05 path: the fp16 operand tile of x_t also leaves as a 32 KB image per tile (k_node_update*_tc, k_node_pre_bwd_tc)
};
struct NodeUpdArgs {
  const float* aggraw;
  const int32_t* rowptr;
  const double* parts1;
  double count1;
  const float* lnw_e;
  const float* lnb_e;
  const float* x_t;
  const float* c1;
  const float* c2;
  float* hq_out;
  float* y3_out;
  double* parts3;
  int N, n_tiles;
  const uint8_t* x_img;  // tcgen05 path: x_t operand image written by k_node_pre_tc (read instead of the fp32 rows)
  uint8_t* hq_img;       // tcgen05 path, training: operand images of the hidden activation and of the aggregate for the backward
  uint8_t* agg_img;
};
// pdg_tc_ends.cu: node encoder and decoder on the tensor cores
int launch_node_encoder_tc(const float* mean_stress, const float* pos, const int64_t* types, const pdg_norm_t* nrm, int scale_in,
                           const float* W0, const float* b0, const float* b2, float* y_out, double* parts, int* nzflag, int N,
                           int n_tiles, int grid, const uint8_t* img, cudaStream_t st);
int launch_node_encoder_bwd_tc(const float* g_in, const float* y_raw, const float* scal, const float* lnw, const float* mean_stress,
                               const float* pos, const int64_t* types, const pdg_norm_t* nrm, int scale_in, const float* W0,
                               const float* b0, float* cta_grads, const float* gs, float* grad_mean_stress, float* grad_pos, int N,
                               int n_tiles, int grid, const uint8_t* img, cudaStream_t st);
int launch_decoder_tc(const float* base, const float* yprev, const double* prev_parts, double prev_count, const float* lnw,
                      const float* lnb, float* x_out, const float* d1, const float* D2, const float* d2, float* hd_out,
                      float out_scale, float out_shift, float* out, const int* nzflag, int N, int n_tiles, int grid,
                      const uint8_t* img, cudaStream_t st);
int launch_decoder_bwd_tc(const float* g_out, float gscale, const float* gs, const float* hd, const float* x_T, const float* y3_last,
                          const double* parts_prev, double count_prev, const float* D2, float* gx, float* cta_grads, float* cs3,
                          const int* nzflag, int N, int n_tiles, int grid, const uint8_t* img, cudaStream_t st);
int launch_edge_encoder_tc(const float* edge_attr, const int32_t* perm, const pdg_norm_t* nrm, int scale_in, const float* W0,
                           const float* b0, const float* b2, float* y_out, double* parts, int E, int n_tiles,
                           const uint8_t* img, cudaStream_t st);  // pdg_tc_enc.cu
int launch_edge_encoder_bwd_tc(const float* g_in, const float* y_raw, const float* scal, const float* lnw, const float* edge_attr,
                               const int32_t* perm, const pdg_norm_t* nrm, int scale_in, const float* W0, const float* b0,
                               float* cta_grads, const float* gs, float* grad_edge_attr, int E, int n_tiles, int grid,
                               const uint8_t* img, cudaStream_t st);
int launch_node_pre_tc(const NodePreArgs& a, const uint8_t* img, int n_tiles, cudaStream_t st);          // pdg_tc_node.cu
int launch_node_update_tc(const NodeUpdArgs& a, const uint8_t* img, int grid, cudaStream_t st);
int launch_node_update_bwd_tc(const NodeUpdBwdArgs& a, const uint8_t* img, int grid, cudaStream_t st);
int launch_node_pre_bwd_tc(const NodePreBwdArgs& a, const uint8_t* img, int grid, cudaStream_t st);

struct FwdWs {
  int64_t N, E, N_pad, E_pad;
  int T;
  bool save;
  char* base;
  size_t total;
  // sections
  float* pack;
  uint8_t* img;   // [IMG_COUNT][32 KB] fp16 swizzled weight images (tcgen05 path)
  double* parts;  // [2+3T][MAXP][2]
  int* nzflag;    // [64] word 0: != 0 when mean_stress has a non-zero entry (PDG_FLAG_ZERO_CHECK); directly after parts
  float* y_nenc;  // raw node-encoder output [N_pad][H]
  float* y_eenc;  // raw edge-encoder output [E_pad][H]
  float* hd;      // decoder hidden [N_pad][H]
  // per-step arrays (index t); without `save` every t aliases the same buffer
  float* x_[64];      // x_t, t = 0..T   (x_T feeds the decoder)
  float* Pa_[64];     // t = 0..T-1
  float* Pb_[64];
  float* aggraw_[64];
  float* hq_[64];
  float* y3_[64];
  float* e_[64];      // e_t, t = 0..T-1
  float* y2_[64];     // raw edge-update MLP output of step t, t = 0..T-2
  uint8_t* eimg_[64];  // tcgen05 path with `save`: fp16 operand-tile image of e_t
  // tcgen05 path: node-level operand images.  They live in space the fp16 rows leave free inside buffers that keep their
  // fp32 size: x_img in the second half of Pa_[t] (Pa rows are fp16 there), hq_img / agg_img in hq_[t] (replaces the fp32 rows)
  uint8_t* ximg(int t) const { return (uint8_t*)Pa_[t] + (size_t)N_pad * H * 2; }
  uint8_t* hqimg(int t) const { return hq_[t] ? (uint8_t*)hq_[t] : nullptr; }
  uint8_t* aggimg(int t) const { return hq_[t] ? (uint8_t*)hq_[t] + (size_t)N_pad * H * 2 : nullptr; }

  // tcm = tcgen05 / bf16 path: raw edge-MLP outputs (y_eenc, y2_t) are stored as fp16 rows, and with `save` the
  // fp32 e_t stream is ONE buffer updated in place (as in inference) while the backward reads per-step fp16
  // operand-tile images.  Its total never exceeds the fp32 layout's, which pdg_forward_ws_bytes reports.
  FwdWs(int64_t n, int64_t e, int steps, bool save_, void* ws, bool tcm = false) : N(n), E(e), T(steps), save(save_), base((char*)ws) {
    N_pad = round_up(n, TM);
    E_pad = round_up(e, TM);
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t r = o; o += (size_t)round_up((int64_t)bytes, 256); return base + r; };
    const size_t nb = (size_t)N_pad * H * sizeof(float), eb = (size_t)E_pad * H * sizeof(float);
    const size_t eh = (size_t)E_pad * H * 2;  // fp16 rows / operand-tile images
    for (int t = 0; t < 64; ++t) eimg_[t] = nullptr;
    pack = (float*)take(PackOffsets::TOTAL * sizeof(float));
    img = (uint8_t*)take((size_t)IMG_COUNT * 32768);
    parts = (double*)take((size_t)(2 + 3 * T) * MAXP * 2 * sizeof(double));
    nzflag = (int*)take(256);
    y_nenc = (float*)take(nb);
    y_eenc = (float*)take(tcm ? eh : eb);
    hd = (float*)take(nb);
    if (save) {
      float* e_inplace = tcm ? (float*)take(eb) : nullptr;
      for (int t = 0; t <= T; ++t) x_[t] = (float*)take(nb);
      for (int t = 0; t < T; ++t) {
        Pa_[t] = (float*)take(nb);
        Pb_[t] = (float*)take(nb);
        aggraw_[t] = (float*)take(nb);
        hq_[t] = (float*)take(nb);
        y3_[t] = (float*)take(nb);
        if (tcm) {
          e_[t] = e_inplace;
          eimg_[t] = (uint8_t*)take(eh);
          y2_[t] = t < T - 1 ? (float*)take(eh) : nullptr;
        } else {
          e_[t] = (float*)take(eb);
          y2_[t] = t < T - 1 ? (float*)take(eb) : nullptr;
        }
      }
    } else {
      float* xa = (float*)take(nb);
      float* xb = (float*)take(nb);
      float* pa = (float*)take(nb);
      float* pb = (float*)take(nb);
      float* ag = (float*)take(nb);
      float* y3 = (float*)take(nb);
      float* eb_ = (float*)take(eb);
      (void)eh;
      for (int t = 0; t <= T; ++t) x_[t] = (t & 1) ? xb : xa;
      for (int t = 0; t < T; ++t) {
        Pa_[t] = pa; Pb_[t] = pb; aggraw_[t] = ag; hq_[t] = nullptr; y3_[t] = y3;
        e_[t] = eb_;          // e_t overwrites e_{t-1} tile by tile (same rows read then written)
        y2_[t] = y_eenc;      // raw y2_t overwrites the raw tensor it was derived from
      }
    }
    total = o;
  }
  double* parts_slot(int s) const { return parts + (size_t)s * MAXP * 2; }
};

}  // namespace pdg
