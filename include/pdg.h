/*
 * pdg.h -- C ABI of libpdivgnn.so: the B200-native (sm_100a) P-DivGNN hot path.
 *
 * Drop-in boundary for the reference's message-passing processor and loss
 * (ricardo0115/p-div-gnn).  Every entry point cites the reference interface it
 * replaces (file:line relative to the reference checkout).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *   - the caller owns every buffer, including workspaces (sizes from the *_bytes
 *     queries); the library never allocates device memory and never synchronises;
 *   - kernels are enqueued on `stream` (a cudaStream_t passed as void*);
 *   - return value 0 = success, negative = error (text via pdg_last_error());
 *   - latent size is fixed at PDG_H = 128 (every shipped config,
 *     scripts/configs_train, line 10 of each yml), node/edge/output feature sizes at 6 / 1 / 3
 *     (scripts/gnn_train.py:395-402); message-passing steps T is a run-time value.
 *   - no torch types.  Every buffer that crosses the boundary (inputs, parameters, outputs, gradients) is fp32 / int64
 *     as in the reference (its autocast(float32) is a no-op); with PDG_PREC_BF16 (the 16-bit tile mode: fp16 operand
 *     tiles since round 2) the MLP-tile operands and some saved activations INSIDE the caller-owned workspace are
 *     16-bit (DESIGN.md sections 3 and 4b), nothing else changes.
 */
#ifndef PDG_H_
#define PDG_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PDG_H 128          /* latent_size */
#define PDG_NODE_IN 6      /* input_nodes_features_size */
#define PDG_EDGE_IN 1      /* input_edges_features_size */
#define PDG_OUT 3          /* output_nodes_features_size */
#define PDG_TILE 128       /* rows per CTA tile; node/edge arrays are padded to it */
#define PDG_NUM_PARAMS 28  /* state_dict tensors */
#define PDG_PARAM_ELEMS 167299

/* Parameter tensors in state_dict order (models.py:260-286, 194-208):
 *  0..5   node_encoder.{0.weight[128,6],0.bias,2.weight[128,128],2.bias,4.weight,4.bias}
 *  6..11  edge_encoder.{0.weight[128,1],0.bias,2.weight,2.bias,4.weight,4.bias}
 * 12..17  processor.edge_net.{0.weight[128,384],0.bias,2.weight,2.bias,4.weight,4.bias}
 * 18..23  processor.node_net.{0.weight[128,256],0.bias,2.weight,2.bias,4.weight,4.bias}
 * 24..27  node_decoder.{0.weight[128,128],0.bias,2.weight[3,128],2.bias[3]}
 * nn.Linear layout: weight is [out,in] row-major. */
typedef struct pdg_params {
  const float* p[PDG_NUM_PARAMS];
} pdg_params_t;

/* The 8 scalar dataset statistics (models.py:98-139; datasets.py:283-291). */
typedef struct pdg_norm {
  float mean_pos, std_pos;
  float mean_mean_stress, std_mean_stress;
  float mean_local_stress, std_local_stress;
  float mean_edge_weight, std_edge_weight;
} pdg_norm_t;

enum {
  PDG_FLAG_SCALE_INPUT = 1,   /* forward(scale_input=True)  models.py:140-162 */
  PDG_FLAG_SCALE_OUTPUT = 2,  /* forward(scale_output=True) models.py:318-321 */
  PDG_FLAG_SAVE = 4,          /* keep per-step state for pdg_backward           */
  PDG_FLAG_ZERO_CHECK = 8     /* device-predicated form of the all-zero mean_stress early exit (models.py:294-299):
                                 local_stress (and, in pdg_backward, every gradient) is exactly 0 when mean_stress is
                                 all zero -- same result as the reference's host-side `torch.any`, without its sync */
};

enum { PDG_PREC_FP32 = 0, PDG_PREC_BF16 = 1 };

const char* pdg_last_error(void);
int pdg_version(void);
/* number of SMs the library sizes its persistent grids for (queried once) */
int pdg_num_sms(void);
/* grid a persistent tile kernel is launched with for n_tiles 128-row tiles on `sms` SMs: the smallest grid that needs
 * no more rounds than `sms` CTAs would (1 516 tiles: 138 instead of 148, 11 rounds either way); host arithmetic only */
int pdg_persistent_grid(int n_tiles, int sms);

/* ---- measurement hooks (bench.py) ------------------------------------------------------
 * pdg_launch_count: kernels this library launched so far (reset != 0 clears the counter).
 * pdg_timing_*: when enabled, every kernel class is bracketed by CUDA events on its launch
 * stream; pdg_timing_collect sums elapsed ms / launch counts per class (arrays of
 * pdg_timing_classes() entries), synchronising on the recorded events, and clears the log. */
long long pdg_launch_count(int reset);
int pdg_timing_enable(int on);
int pdg_timing_classes(void);
const char* pdg_timing_class_name(int cls);
int pdg_timing_collect(double* ms_per_class, long long* count_per_class);

/* self-test of the tcgen05 bf16 tile engine on one [128,128] tile pair (A, B fp32, rounded to bf16 inside; img = 32 KB
 * device scratch): mode 0  D = A.B^T  (both operands K-major: forward / data-gradient of the previous layer's output),
 * mode 1  D = A^T.B  (both MN-major: weight gradients), mode 2  D = A.B  (A K-major, B MN-major: dX = dY.W). */
int pdg_tc_selftest(int mode, const float* A, const float* B, float* D, void* img, void* stream);

/* ---- graph plan: receiver-sorted CSR + sender CSR of a batched edge_index ----------
 * Replaces the per-call gather/scatter bookkeeping of PyG MessagePassing.propagate
 * (models.py:215-217) and is the device half of the batcher (SURVEY 8 a12/a13).
 * edge_index is the PyG [2,E] int64 tensor (row = source, col = target). */
size_t pdg_plan_bytes(int64_t n_nodes, int64_t n_edges);
size_t pdg_plan_tmp_bytes(int64_t n_nodes, int64_t n_edges);
int pdg_plan_build(const int64_t* edge_index, int64_t n_nodes, int64_t n_edges, void* plan, void* tmp,
                   size_t tmp_bytes, void* stream);
/* Node ids of edge_index outside [0, n_nodes) -- the reference raises an IndexError in x[col] (models.py:233-238) --
 * are CLAMPED into range by pdg_plan_build (every later kernel stays memory-safe) and recorded in a status word inside
 * the plan.  pdg_plan_status is the optional check, and the one call of this family that synchronises `stream`: it
 * copies the word to *status_host and returns -3 (text in pdg_last_error()) when it is non-zero, 0 otherwise. */
int pdg_plan_status(const void* plan, int64_t n_nodes, int64_t n_edges, int32_t* status_host, void* stream);
/* views into a built plan (device pointers; int32): perm[E_pad] (sorted position ->
 * input edge id), recv[E_pad], send[E_pad], rowptr[N+1] */
int pdg_plan_views(void* plan, int64_t n_nodes, int64_t n_edges, int32_t** perm, int32_t** recv, int32_t** send,
                   int32_t** rowptr, int32_t** send_ptr, int32_t** send_list);

/* ---- model forward: EncodeProcessDecode.forward (models.py:288-326) -----------------
 * mean_stress [N,3], pos [N,2], nodes_types [N] int64, edge_attr [E] (PyG edge order),
 * out local_stress [N,3].  The all-zero mean_stress early exit (models.py:294-299) is either
 * the caller's host-visible decision or, with PDG_FLAG_ZERO_CHECK, predicated on the device.  With PDG_FLAG_SAVE the workspace afterwards
 * holds everything pdg_backward needs. */
size_t pdg_forward_ws_bytes(int64_t n_nodes, int64_t n_edges, int steps, int flags);
int pdg_forward(const pdg_params_t* params, const pdg_norm_t* norm, const float* mean_stress, const float* pos,
                const int64_t* nodes_types, const float* edge_attr, const void* plan, int64_t n_nodes,
                int64_t n_edges, int steps, int flags, int precision, void* ws, size_t ws_bytes,
                float* local_stress, void* stream);

/* Batched forward: n_instances (1..PDG_FWD_MAX_INSTANCES) instances K of one graph in one pass.  All instances share
 * the plan, nodes_types, the parameters and the statistics; instance k has its own inputs, its own graph-LayerNorm
 * statistics and its own output.  Instance k's input x starts at x + k * x_stride (elements; each instance contiguous in
 * the layout of pdg_forward); stride 0 gives every k the same input.  local_stress [K][N][3].  ws:
 * pdg_forward_batched_ws_bytes (K forward workspaces of the fp32 mode, one after another); 0 for K or steps out of
 * range.  Row k has the bits of pdg_forward on instance k's inputs with the same flags; with PDG_FLAG_ZERO_CHECK an
 * instance whose mean_stress is all zeros gives zeros whatever the others hold.  Launches the kernels and memsets of
 * one pdg_forward for any K.  Returns -1 for K outside 1..PDG_FWD_MAX_INSTANCES, precision != PDG_PREC_FP32,
 * PDG_FLAG_SAVE (no derivative follows a batched forward), steps outside 1..62, a negative stride, a workspace that is
 * too small and an empty graph.  Replaces torch.func.vmap over the inputs of models.py:288-326. */
#define PDG_FWD_MAX_INSTANCES 64
size_t pdg_forward_batched_ws_bytes(int64_t n_nodes, int64_t n_edges, int steps, int flags, int n_instances);
int pdg_forward_batched(const pdg_params_t* params, const pdg_norm_t* norm, const float* mean_stress, int64_t ms_stride,
                        const float* pos, int64_t pos_stride, const int64_t* nodes_types, const float* edge_attr,
                        int64_t ea_stride, const void* plan, int64_t n_nodes, int64_t n_edges, int steps, int flags,
                        int precision, void* ws, size_t ws_bytes, int n_instances, float* local_stress, void* stream);

/* test/debug: byte offset + element count of a saved tensor in a PDG_FLAG_SAVE workspace.
 * what: 0 x_t, 1 e_t, 2 y2_t, 3 Pa_t, 4 Pb_t, 5 aggraw_t, 6 hq_t, 7 y3_t, 8 y_nenc,
 * 9 y_eenc, 10 hd (fp32), 11 LayerNorm partials of slot t (doubles). Edge tensors are in
 * receiver-sorted order (row p <-> input edge perm[p]). */
int pdg_ws_offset(int64_t n_nodes, int64_t n_edges, int steps, int flags, int what, int t, size_t* offset,
                  size_t* elems);

/* ---- model backward: d loss / d params given d loss / d local_stress [N,3] ----------
 * grads_flat: PDG_PARAM_ELEMS floats, state_dict order, overwritten (not accumulated).
 * pdg_backward differentiates the parameters only; pdg_backward_inputs, with the same arguments, also writes the
 * gradients of the differentiable inputs of models.py:140-162 into each non-NULL output (overwritten, not
 * accumulated; the parameter gradients are the same bits either way):
 *   grad_mean_stress [N,3], grad_pos [N,2], grad_edge_attr [E] in the caller's (PyG) edge order.
 * nodes_types is an integer input and has no gradient.  pdg_backward is pdg_backward_inputs with three NULLs.
 * Replaces torch autograd through models.py:288-326. */
size_t pdg_backward_ws_bytes(int64_t n_nodes, int64_t n_edges, int steps);
int pdg_backward(const pdg_params_t* params, const pdg_norm_t* norm, const float* mean_stress, const float* pos,
                 const int64_t* nodes_types, const float* edge_attr, const void* plan, int64_t n_nodes,
                 int64_t n_edges, int steps, int flags, int precision, void* fwd_ws, void* bwd_ws, size_t bwd_ws_bytes,
                 const float* grad_local_stress, float* grads_flat, void* stream);
int pdg_backward_inputs(const pdg_params_t* params, const pdg_norm_t* norm, const float* mean_stress, const float* pos,
                        const int64_t* nodes_types, const float* edge_attr, const void* plan, int64_t n_nodes,
                        int64_t n_edges, int steps, int flags, int precision, void* fwd_ws, void* bwd_ws,
                        size_t bwd_ws_bytes, const float* grad_local_stress, float* grads_flat,
                        float* grad_mean_stress, float* grad_pos, float* grad_edge_attr, void* stream);

/* ---- model forward-mode derivative (Jacobian-vector product) ---------------------------
 * tan_local_stress [N,3] (overwritten) = d local_stress / d (mean_stress, pos, edge_attr) applied to the tangents
 * tan_mean_stress [N,3], tan_pos [N,2], tan_edge_attr [E] (caller's PyG edge order); a NULL tangent is a zero tangent.
 * nodes_types is an integer input and has no tangent.  fwd_ws is the workspace of a pdg_forward with PDG_FLAG_SAVE
 * and the same arguments (flags included); it is only read, so a pdg_backward may follow.  jvp_ws: the tangent
 * workspace, pdg_jvp_ws_bytes.  Returns -1 for precision != PDG_PREC_FP32 (the 16-bit mode has no forward-mode
 * derivative), flags without PDG_FLAG_SAVE, steps outside 1..62 or a workspace that is too small.
 * Replaces torch forward-mode AD (torch.func.jvp, torch.autograd.forward_ad) through models.py:288-326. */
size_t pdg_jvp_ws_bytes(int64_t n_nodes, int64_t n_edges, int steps);
int pdg_jvp(const pdg_params_t* params, const pdg_norm_t* norm, const float* mean_stress, const float* pos,
            const int64_t* nodes_types, const float* edge_attr, const void* plan, int64_t n_nodes, int64_t n_edges,
            int steps, int flags, int precision, const void* fwd_ws, void* jvp_ws, size_t jvp_ws_bytes,
            const float* tan_mean_stress, const float* tan_pos, const float* tan_edge_attr, float* tan_local_stress,
            void* stream);

/* Batched tangents: one tangent pass carries n_tangents (1..PDG_JVP_MAX_TANGENTS) tangents K.  Tangent k of an input is
 * contiguous in the layout of pdg_jvp and starts at tan_x + k * x_stride (elements); stride 0 gives every k the same
 * tangent, NULL a zero tangent.  tan_local_stress [K][N][3].  jvp_ws: pdg_jvp_batched_ws_bytes (K tangent workspaces
 * of pdg_jvp_ws_bytes each); 0 for K or steps out of range.  Column k has the bits of a pdg_jvp call on tangent k.
 * Launches the kernels of one pdg_jvp for any K.  Returns -1 for K outside 1..PDG_JVP_MAX_TANGENTS and for every
 * refusal of pdg_jvp.  pdg_jvp is this call with K = 1. */
#define PDG_JVP_MAX_TANGENTS 64
size_t pdg_jvp_batched_ws_bytes(int64_t n_nodes, int64_t n_edges, int steps, int n_tangents);
int pdg_jvp_batched(const pdg_params_t* params, const pdg_norm_t* norm, const float* mean_stress, const float* pos,
                    const int64_t* nodes_types, const float* edge_attr, const void* plan, int64_t n_nodes,
                    int64_t n_edges, int steps, int flags, int precision, const void* fwd_ws, void* jvp_ws,
                    size_t jvp_ws_bytes, int n_tangents, const float* tan_mean_stress, int64_t ms_stride,
                    const float* tan_pos, int64_t pos_stride, const float* tan_edge_attr, int64_t ea_stride,
                    float* tan_local_stress, void* stream);

/* ---- batched reverse-mode derivative (vector-Jacobian products) of the inputs -----------------------
 * For n_cotangents (1..PDG_VJP_MAX_COTANGENTS) cotangents K of local_stress, grad_local_stress [K][N][3], writes
 * d <u_k, local_stress> / d (mean_stress, pos, edge_attr) into each non-NULL output (overwritten, not accumulated):
 * grad_mean_stress [K][N][3], grad_pos [K][N][2], grad_edge_attr [K][E] in the caller's (PyG) edge order.  No parameter
 * gradient is formed.  fwd_ws is the workspace of a pdg_forward with PDG_FLAG_SAVE and the same arguments (flags
 * included); it is only read, so a pdg_backward may follow.  vjp_ws: pdg_vjp_batched_ws_bytes (K cotangent workspaces
 * of the data-gradient buffers of the backward; 0 for K or steps out of range).  Column k has the bits of the input
 * gradients of pdg_backward_inputs with cotangent k, the same flags and PDG_PREC_FP32.  Launches the same kernels for
 * any K.  Returns -1 for K outside 1..PDG_VJP_MAX_COTANGENTS, precision != PDG_PREC_FP32, flags without PDG_FLAG_SAVE,
 * steps outside 1..62, a workspace that is too small, three NULL outputs and an empty graph.
 * Replaces torch.func.jacrev / torch.func.vmap over torch.func.vjp through models.py:288-326. */
#define PDG_VJP_MAX_COTANGENTS 64
size_t pdg_vjp_batched_ws_bytes(int64_t n_nodes, int64_t n_edges, int steps, int n_cotangents);
int pdg_vjp_batched(const pdg_params_t* params, const pdg_norm_t* norm, const float* mean_stress, const float* pos,
                    const int64_t* nodes_types, const float* edge_attr, const void* plan, int64_t n_nodes,
                    int64_t n_edges, int steps, int flags, int precision, const void* fwd_ws, void* vjp_ws,
                    size_t vjp_ws_bytes, int n_cotangents, const float* grad_local_stress, float* grad_mean_stress,
                    float* grad_pos, float* grad_edge_attr, void* stream);

/* ---- loss: per-graph NMSE + divergence regulariser, batch means ---------------------
 * Replaces the per-graph Python loop of train() (gnn_train.py:162-202):
 * normalized_mse_loss_single (:41-57), compute_divergence (:60-92),
 * data_utils.slice_batch_gt_and_predictions (data_utils.py:25-33) and
 * data_utils.standardize (:46-51).
 *   pred [N,3] standardised prediction; local_stress [N,3] raw ground truth
 *   (standardised inside with norm->mean/std_local_stress); graph_ptr [B+1] int64;
 *   labels [N] int64 (NodeType); op_div given as a plan (below) over batch rows with
 *   graph-LOCAL columns in [0, 2*N_i) exactly as PyG collation leaves them (SURVEY 2.3d).
 *   out[0] = sum_i NMSE_i / B ; out[1] = penalty * sum_i div_i / B   (device floats) */
/* op_div plan: CSR (by batch row) + CSC (by stacked-stress row 2*n0_i + j) of the
 * row-stacked operator, from the coalesced COO triplets torch holds
 * (datasets.py:191-213 + SURVEY 2.3d).  coo_row/coo_col int64 [nnz], values stay in the
 * caller's buffer and are indexed by the plan. */
size_t pdg_opdiv_plan_bytes(int64_t n_nodes, int64_t nnz);
size_t pdg_opdiv_tmp_bytes(int64_t n_nodes, int64_t nnz);
int pdg_opdiv_plan_build(const int64_t* coo_row, const int64_t* coo_col, int64_t nnz, const int64_t* graph_ptr,
                         int64_t n_graphs, int64_t n_nodes, void* plan, void* tmp, size_t tmp_bytes, void* stream);
size_t pdg_loss_ws_bytes(int64_t n_nodes, int64_t n_graphs);
int pdg_loss(const float* pred, const float* local_stress, const pdg_norm_t* norm, const int64_t* graph_ptr,
             int64_t n_graphs, int64_t n_nodes, const int64_t* labels, const void* opdiv_plan, const float* op_val,
             int64_t nnz, int use_divergence, float penalty, void* ws, float* out2, void* stream);
/* grad_pred [N,3] = upstream2[0] * d out[0]/d pred + upstream2[1] * d out[1]/d pred
 * (upstream2: 2 device floats, NULL = ones); ws is the buffer pdg_loss filled. */
int pdg_loss_backward(const float* pred, const float* local_stress, const pdg_norm_t* norm, const int64_t* graph_ptr,
                      int64_t n_graphs, int64_t n_nodes, const void* opdiv_plan, const float* op_val, int64_t nnz,
                      int use_divergence, float penalty, const void* ws, const float* upstream2, float* grad_pred,
                      void* stream);

/* ---- fused Adam + non-finite check over the 28 parameter tensors (SURVEY 8f rank 3) ------
 * Replaces `scaler.step(optimizer)` with torch.optim.Adam (scripts/gnn_train.py:111,118,204-207) by ONE launch:
 *   g' = g * inv_scale + weight_decay * p;  m = m + (1-beta1)(g'-m);  v = beta2 v + (1-beta2) g'^2
 *   p -= lr/(1-beta1^step) * m / (sqrt(v)/sqrt(1-beta2^step) + eps)        (amsgrad = False, maximize = False)
 * params / grads: host arrays of PDG_NUM_PARAMS DEVICE pointers in state_dict order; exp_avg / exp_avg_sq: flat
 * [PDG_PARAM_ELEMS] device buffers owned by the caller (zero before the first step); step counts from 1.
 * found_inf (device int, may be NULL): GradScaler semantics -- the step is skipped when *found_inf != 0;
 * pdg_grads_check_finite ORs 1 into *found_inf when any gradient element is inf / nan. */
typedef struct pdg_adam {
  double lr, beta1, beta2, eps, weight_decay, inv_scale; /* Python-float hyper-parameters: derived scalars (1-beta,
                                                           bias corrections) are formed in double, like torch */
  int step;
} pdg_adam_t;
int pdg_grads_check_finite(const float* const* grads, int* found_inf, void* stream);
int pdg_adam_step(float* const* params, const float* const* grads, float* exp_avg, float* exp_avg_sq,
                  const pdg_adam_t* cfg, const int* found_inf, void* stream);
/* Same update with the step count kept on the DEVICE: *step_count = number of updates applied so far (0 before the
 * first); the bias corrections use *step_count + 1 (cfg->step is ignored) and the count advances only when the update
 * is applied.  A step skipped through found_inf therefore leaves the count -- and the next step's bias corrections --
 * exactly where GradScaler.step leaves torch.optim.Adam's (it does not call optimizer.step() on overflow,
 * scripts/gnn_train.py:205-207), still without a host sync. */
int pdg_adam_step_counted(float* const* params, const float* const* grads, float* exp_avg, float* exp_avg_sq,
                          const pdg_adam_t* cfg, const int* found_inf, int* step_count, void* stream);

/* ---- device graph batcher (SURVEY 8 a12/a13) ----------------------------------------
 * Builds, for B meshes concatenated along nodes (node_ptr [B+1]) and faces
 * (face_ptr [B+1], faces [nodes_per_face,F] int64 with graph-local node ids; nodes_per_face = 3
 * triangles or 4 quads, one cell type per batch like the reference's "single element-type meshes"),
 * the PyG-ordered, coalesced edge_index [2,E] (batch-global ids) and fp32 edge_attr [E]:
 *   mesh_to_graph/FaceToEdge + to_undirected   convert_utils.py:47-60 (triangles)
 *   _quad_face_to_edge + to_undirected         convert_utils.py:62-81 (quads: sides 01,12,23,03)
 *   |pos_r - pos_c|                            datasets.py:182-188 (float64 -> fp32)
 *   compute_periodic_graph + coalesce          datasets.py:39-119 (periodic != 0)
 *   Batch.from_data_list index offsets         SURVEY 2.3d
 * pos is [N,2] float64.  Two-phase: count (returns E through *n_edges_host after a
 * stream sync inside pdg_batch_count only) then fill. */
size_t pdg_batch_tmp_bytes(int64_t n_nodes, int64_t n_faces, int nodes_per_face, int64_t n_graphs);
int pdg_batch_count(const double* pos, const int64_t* faces, const int64_t* node_ptr, const int64_t* face_ptr,
                    int64_t n_graphs, int64_t n_nodes, int64_t n_faces, int nodes_per_face, int periodic, void* tmp,
                    size_t tmp_bytes, int64_t* n_edges_host, void* stream);
int pdg_batch_fill(const double* pos, int64_t n_nodes, int64_t n_faces, int nodes_per_face, int64_t n_graphs,
                   int64_t n_edges, void* tmp, int64_t* edge_index, float* edge_attr, void* stream);

/* ---- device node labelling (SURVEY 8f rank 4) ------------------------------------------
 * Replaces datasets.compute_node_labels (datasets.py:133-179; VTK extract_feature_edges + connectivity on the
 * host): an edge used by exactly one cell (triangle or quad) is a boundary edge, the boundary loops are the regions, the
 * region touching the mesh bounding box is the external boundary.  labels [N] int64 = NodeType
 * (datasets.py:33-36): -1 internal boundary (hole), 0 internal, 1 external boundary; n_regions [B] int32 is
 * the number of boundary loops of each mesh (the reference asserts 2).  pos [N,2] float64, faces
 * [nodes_per_face,F] int64 graph-local ids (3 = triangles, 4 = quads), node_ptr / face_ptr [B+1] int64. */
size_t pdg_labels_tmp_bytes(int64_t n_nodes, int64_t n_faces, int nodes_per_face, int64_t n_graphs);
int pdg_node_labels(const double* pos, const int64_t* faces, const int64_t* node_ptr, const int64_t* face_ptr,
                    int64_t n_graphs, int64_t n_nodes, int64_t n_faces, int nodes_per_face, void* tmp, size_t tmp_bytes,
                    int64_t* labels, int32_t* n_regions, void* stream);

/* ---- device periodicity check (SURVEY 8f rank 4) -------------------------------------------
 * Replaces microgen.mesh.is_periodic / microgen.remesh.is_periodic, asserted by the reference on the host for every mesh
 * it generates or benchmarks (generate_dataset.py:191, generate_dataset_hyperelast.py:160,237,
 * benchmark_gnn_fem.py:195; in-plane [N,2] coordinates, tol = 1e-8): the nodes within tol of the bounding-box minimum /
 * maximum of an axis are its two opposite sides; each side is sorted along the other axis; periodic[g] = 1 when the
 * opposite sides of mesh g hold the same number of nodes and no sorted coordinate of the max side exceeds its partner
 * on the min side by more than tol (one-sided, as published), else 0.  pos [N,2] float64, node_ptr [B+1] int64,
 * periodic [B] int32.  Whole batch in one pass (two stable radix sorts), no host sync. */
size_t pdg_periodic_tmp_bytes(int64_t n_nodes, int64_t n_graphs);
int pdg_is_periodic(const double* pos, const int64_t* node_ptr, int64_t n_graphs, int64_t n_nodes, double tol, void* tmp,
                    size_t tmp_bytes, int32_t* periodic, void* stream);

/* ---- batch gather from a device-resident dataset (SURVEY 8f rank 1) ------------------------------
 * The collate step of the reference's DataLoader (gnn_train.py:387-394) for a dataset that lives in HBM as concatenated
 * per-sample arrays: one launch copies the B sample ranges of the node rows, face columns and operator triplets into
 * contiguous batch arrays (operator rows re-based to the batch's node numbering) and writes the PyG `batch` vector.
 * meta (device, int64): [node_ptr B+1 | face_ptr B+1 | nnz_ptr B+1 | node_src B | face_src B | nnz_src B] = destination
 * prefix sums and source offsets of every sample.  faces [nodes_per_face][faces_total]; o_op_idx [2][n_nnz]. */
int pdg_resident_gather(const double* pos64, const float* mean_stress, const float* local_stress, const int64_t* labels,
                        const int64_t* faces, int64_t faces_total, int nodes_per_face, const int64_t* op_row,
                        const int64_t* op_col, const float* op_val, const int64_t* meta, int n_graphs, int64_t n_nodes,
                        int64_t n_faces, int64_t n_nnz, double* o_pos64, float* o_pos32, float* o_mean_stress,
                        float* o_local_stress, int64_t* o_labels, int64_t* o_batch, int64_t* o_faces, int64_t* o_op_idx,
                        float* o_op_val, void* stream);

/* ---- data-parallel gradient exchange over NVLink peer memory (SURVEY 8e) ---------------------
 * The reference is single-device; the B200 path shards batches of graphs over GPUs and averages ONE flat gradient
 * buffer per step (what torch DistributedDataParallel would do around gnn_train.py:154-207).  At 669 KB the exchange
 * is latency, so instead of a ring collective every rank pushes its buffer into a slot of every peer's exchange area
 * (CUDA IPC mapping over NVLink / NVSwitch, posted stores), raises a flag there and sums the slots it holds in rank
 * order: one kernel, bit-identical means on every rank.
 *   pdg_peer_alloc   cudaMalloc's the exchange area for n_floats x world ranks (the ONE allocation this library makes:
 *                    IPC needs an allocation base) and returns its 64-byte IPC handle; pdg_peer_open maps a peer's;
 *   pdg_allreduce_mean(flat, n, bufs, rank, world, seq, status, stream): in place mean of `flat` over the ranks.
 *                    bufs = HOST array of `world` device pointers (own area at index rank, peers' mapped areas),
 *                    seq = 1, 2, 3, ... the same on every rank for the same step; *status (device int, may be NULL)
 *                    is set to 1 if a peer did not arrive within ~3 s (results undefined, nothing hangs).
 *                    `flat` must be 16-byte aligned. */
size_t pdg_peer_bytes(int64_t n_floats, int world);
int pdg_peer_alloc(int64_t n_floats, int world, void** dev_ptr, void* handle64);
int pdg_peer_open(const void* handle64, void** dev_ptr);
int pdg_peer_close(void* dev_ptr);
int pdg_peer_free(void* dev_ptr);
int pdg_allreduce_mean(float* flat, int64_t n_floats, void* const* peer_bufs_host, int rank, int world, int64_t seq, int* status,
                       void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PDG_H_ */
