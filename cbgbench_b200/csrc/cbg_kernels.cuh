// Internal launcher declarations (one per kernel family).  Not part of the C-ABI.
#pragma once
#include "cbg_common.cuh"

#define CBG_MODE_KNN 0
#define CBG_MODE_RADIUS 1

// graph.cu
// static_only != 0: neighbour search restricted to nodes without the generate bit (centres with
// the bit get an empty row) - the static-only kNN lists behind the R-cache
// snbr (optional): static-only lists of the same graphs -> incremental search for non-moving centres
int cbg_launch_knn(const float4* x4, const int* graph_ptr, int n_graphs, int max_graph_nodes, int mode,
                   int k, float r_max, int static_only, const int* snbr, int* nbr, cudaStream_t st);
// ew_static (optional): gates of the static-only neighbour lists, reused for static edges
// glist (optional, with ew_static): scratch of 64 + 32*n_nodes ints; the moving edges are compacted into it
// and their gates computed by a second, dense launch
// full_static (optional, with ew_static): per node, 1 when all 32 slots hold static edges (fast path of edge_setup)
int cbg_launch_edge_gate(const float* blob_global, const float4* x4, const int* nbr, long long n_nodes,
                         const float* ew_static, int* glist, float* ew, cudaStream_t st,
                         unsigned char* full_static = nullptr);

// Receptive-field pruning (sampling path): depth[i] = last layer whose X2H output of node i can still
// influence a generated / classified atom (-2: never).  order[] lists nodes by decreasing depth,
// cnt_ge[l + 1] = number of nodes with depth >= l for l = -1 .. num_layers-1.
int cbg_launch_depth(const int* nbr, const int* graph_ptr, int n_graphs, int max_graph_nodes, long long n_nodes,
                     const int* seed_idx, int n_seed, const int* cls_idx, int n_cls, int num_layers,
                     int* depth, int* order, int* cnt_ge, cudaStream_t st);

// node_gemm.cu
struct NodeGemmArgs {
  const float* a;        // [*,128] input rows (h)
  const int* row_idx;    // optional gather list (node ids); nullptr = identity
  int n_rows;            // rows to process
  const float* wt;       // Wt[k][ldw] (k-major), already offset to the first plane's column
  const float* bias;     // [n_planes*128], already offset
  int ldw;               // row stride of wt in floats
  int n_planes;          // planes computed by this launch (the last one is q_hidden if has_q)
  float* out[CBG_NPLANES];  // destination plane per computed plane ([N,128], indexed by node id)
  int has_q;             // 1: last plane goes LN->ReLU->W1T GEMM -> out_q instead of global
  const float* q_ln;     // gamma[128], beta[128]
  const float* q_w1t;    // [128][128] k-major
  const float* q_b1;     // [128]
  float* out_q;          // [N,128]
  // tensor-core path only: pre-split weight planes of the sub-layer (layout: cbg_layout.h *_NODE_TC)
  const int* n_rows_dev;   // optional: rows to process is min(n_rows, *n_rows_dev) (device-side list length)
  const float* tc_planes;  // plane 0 of the sub-layer
  int tc_first_plane;      // index of this launch's first plane (q second Linear is always plane 5)
  const float* tch_planes; // f16 (hi | lo) images of the same six planes (node_gemm_f16.cu)
  // f16 kernel only: merged launch - planes >= CBG_NODE_SRC_PLANES (destination planes Pi, q) are computed for the first
  // min(n_rows, *n_dst_dev) rows of the list only, the source planes Pj for all n_rows (nullptr = no second limit)
  const int* n_dst_dev;
  long long* trace;        // debug: globaltimer stamps of CTA 0 (cbg_debug_node_gemm_trace)
};
int cbg_launch_node_gemm(const NodeGemmArgs& a, cudaStream_t st);      // fp32 SIMT
// tcgen05 3xTF32; cluster = 1/2/4 CTAs sharing weight chunks by multicast, 0 = default (env CBG_GEMM_CLUSTER)
int cbg_launch_node_gemm_tc(const NodeGemmArgs& a, cudaStream_t st, int cluster = 0);
// tcgen05 kind::f16 with the (hi, lo) split: default
int cbg_launch_node_gemm_f16(const NodeGemmArgs& a, cudaStream_t st);
void cbg_node_gemm_f16_set_trace(long long* buf_dev);

// edge.cu
struct EdgeArgs {
  const float4* x4;      // [N] xyz + flags
  const int* nbr;        // [N,32]
  const float* ew;       // [N,32]
  const float* pj_k;     // planes [N,128]
  const float* pj_v;
  const float* pi_k;
  const float* pi_v;
  const float* q;        // [N,128] (already scaled by 1/sqrt(8))
  const float* layer;    // base of this layer's weight block
  float* w;              // [N,32,16] scratch: alpha * e_w
  float* h;              // [N,128] in/out (x2h_v residual update)
  const int* node_idx;   // h2x: list of generated nodes
  int n_nodes;           // x2h: N ; h2x: number of generated nodes
  float* dx;             // h2x: [n_nodes,4] coordinate deltas (compact, same order as node_idx)
  const int* n_nodes_dev; // optional device-side length of node_idx (x2h with a pruned node list)
  const float* rc_k;     // x2h: R-cache of this layer's hk / hv MLP ([N][32][128]) or nullptr
  const float* rc_v;
  int* ticket;           // x2h: optional work counter (zeroed by the caller) for dynamic node scheduling; k uses ticket[0], v ticket[1]
  const unsigned char* fstat;  // x2h with an R-cache: 1 = all 32 in-edges of the node are static (nbr row == its static list)
  long long* trace;      // x2h_tc debugging: per-tile SM-clock stamps of CTA 0 ([tile][16 events]) or nullptr
  int trace_tiles;
  int w_compact;         // x2h_tc: 1 = w is indexed by the position in node_idx ([n_nodes,32,16], H2X), 0 = by node id
};
int cbg_launch_rcache(const float* layers, int num_layers, const float4* x4, const int* snbr, int n_nodes,
                      float* rcache, cudaStream_t st);
int cbg_launch_x2h(const EdgeArgs& a, cudaStream_t st);
// x2h_tc.cu: both X2H kernels on tcgen05 (A operands in TMEM, f16 hi/lo split); edge order of w = neighbour-table order
int cbg_launch_x2h_tc(const EdgeArgs& a, cudaStream_t st);
// hardware self-test of the tcgen05 operand conventions (tests): d[128][128] = a[128][32] * b[128][32]^T, f16 inputs
// debugging: x2h_tc kernels of later launches stamp CTA 0's pipeline events into buf ([max_tiles][16] int64; nullptr = off)
void cbg_x2h_tc_set_trace(long long* buf, int max_tiles);
// H2X on the same tcgen05 kernel (generated nodes only): a.w = compact [n_nodes,32,16] scratch, a.dx = [n_nodes,4] out
int cbg_launch_h2x_tc(const EdgeArgs& a, cudaStream_t st);
int cbg_launch_umma_selftest(const void* a, const void* b, float* d, int a_from_smem, cudaStream_t st);
int cbg_launch_h2x(const EdgeArgs& a, cudaStream_t st);
int cbg_edge_init(void);  // sets max-dynamic-smem attributes once
int cbg_edge_set_impl(int impl, int warps);  // X2H implementation switch (cbg_set_edge_impl)

// misc.cu
int cbg_launch_pack_x4(const float* x, const unsigned char* lig_flag, const unsigned char* gen_flag,
                       long long n, float4* x4, cudaStream_t st);
int cbg_launch_unpack_x(const float4* x4, long long n, float* x, cudaStream_t st);
int cbg_launch_gather_x(const float4* x4, const int* idx, int n, float* out /*[n,3]*/, cudaStream_t st);
int cbg_launch_apply_dx(float4* x4, const int* node_idx, const float* dx, int n, cudaStream_t st);
int cbg_launch_classifier(const float* blob_global, const float* h, const int* row_idx, int n_rows,
                          int num_classes, float* logits, cudaStream_t st);
int cbg_launch_step_init(const float* x_lig, const float* c_lig, const int* lig_node, int n_lig,
                         int num_classes, const float* emb_wt, const float* h_lig_bias,
                         const float* h_static, long long n_nodes, float4* x4, float* h, cudaStream_t st);
struct ReverseArgs {
  const float* x0;         // denoiser output coordinates (x0 prediction), row stride x0_stride floats
  int x0_stride;           // 4 when reading the packed node array, 3 for a plain [n,3] tensor
  const int* x0_idx;       // optional row index per ligand atom (lig_node); nullptr = identity
  const float* logits;     // [n_lig, K]
  const float* x_t;        // [n_lig,3]
  const float* c_t;        // [n_lig,K]
  const unsigned char* gen;  // [n_lig]
  const float* pos_noise;  // [n_lig,3]
  const float* type_u;     // [n_lig,K]
  float c0, ct;            // posterior_mean_c0_coef[t], posterior_mean_ct_coef[t]
  float lac_prev, l1mac_prev, la, l1ma;  // type tables at t-1 (clamped) and t
  int n_lig, num_classes;
  float* x_next;           // [n_lig,3]
  float* c_next;           // [n_lig,K]
  long long* v_next;       // [n_lig]
};
// logvar = posterior_logvar[t]; nonzero = 0 at t == 0 else 1
int cbg_launch_reverse(const ReverseArgs& a, float logvar, float nonzero, cudaStream_t st);

// Per-step inputs / outputs of the TargetDiff step in DEVICE memory: what changes from step to step when the step is
// replayed from a CUDA graph (cbg_sample_step_graph_f32): the graph's kernels read these through one pointer.
struct StepIO {
  const float* x_t;
  const float* c_t;
  const float* pos_noise;
  const float* type_u;
  float* x_next;
  float* c_next;
  long long* v_next;
  float c0, ct, lac_prev, l1mac_prev, la, l1ma, logvar, nonzero;
};
int cbg_launch_step_init_io(const StepIO* io, const int* lig_node, int n_lig, int num_classes, const float* emb_wt,
                            const float* h_lig_bias, const float* h_static, long long n_nodes, float4* x4, float* h,
                            cudaStream_t st);
// the step-invariant members of `a` are used, the per-step ones (x_t, c_t, noise, outputs, coefficients) come from *io
int cbg_launch_reverse_io(const ReverseArgs& a, const StepIO* io, cudaStream_t st);

// DiffSBDD reverse step (SURVEY.md section 8 row f2): one CTA per graph.
//   mode 0  zs = z_t / a - b * eps_pred + s * noise              (sample_p_zs_given_zt, diffusion_scheduler.py:1005-1039)
//   mode 1  zs = a * (z_t - b * eps_pred) + s * noise            (sample_p_xh_given_z0, diffsbdd.py:323-360; a = 1/alpha_0)
// for the coordinates (eps_pred = the denoiser's output coordinates of the ligand atoms, read from x4) followed by
// the COM projection remove_mean_batch (diffusion_scheduler.py:706-710): the mean of zs over the graph's ligand
// atoms is subtracted from zs AND from the pocket atoms of the graph (x4 rows without the ligand bit).
// Types: mode 0 the same update without projection (eps_pred = logits), mode 1 c_next = 4 * c_t.
struct SbddArgs {
  float4* x4;               // [N] node coordinates + flags (pocket rows are shifted in place)
  const int* graph_ptr;     // [B+1]
  const int* lig_node;      // [n_lig] ascending composed index of every ligand atom
  int n_lig, num_classes, n_graphs;
  const float* logits;      // [n_lig,K]
  const float* x_t;         // [n_lig,3]
  const float* c_t;         // [n_lig,K]
  const float* x_noise;     // [n_lig,3]
  const float* c_noise;     // [n_lig,K]
  float a, b, s;
  int mode;
  float* x_next;            // [n_lig,3]
  float* c_next;            // [n_lig,K]
};
int cbg_launch_sbdd_reverse(const SbddArgs& a, cudaStream_t st);

// DiffBP (row f2).  x4[idx[a]].xyz = x[a] (flags kept): puts the step's INPUT ligand coordinates back before the
// CoM head runs on them (diffbp.py:80-97 works on x_composed, not on the denoiser's output)
int cbg_launch_scatter_x(const float* x /*[n,3]*/, const int* idx, int n, float4* x4, cudaStream_t st);
// edge gate of the listed rows only (the CoM head needs it for the generated atoms' edges)
int cbg_launch_edge_gate_rows(const float* blob_global, const float4* x4, const int* nbr, const int* row_idx,
                              int n_rows, float* ew, cudaStream_t st);
// Fused DiffBP reverse step, one CTA per graph:
//   eps  = (x_pred - x_t) - mean_g(x_pred - x_t) + mean_g(x_com - x_t)          CoMPredictor.forward diffbp.py:80-101
//   x_s  = (x_t + beta * (-eps / sqrt(1 - abar))) / sqrt(1 - beta) + nonzero * sqrt(beta) * noise, gen-masked
//                                                  CTNVPScheduler.backward_remove_noise('score') diffusion_scheduler.py:144-165
//   v_s  = (u < prob) & gen & (v_t == 0) ? argmax softmax(logits) : v_t   MaskTypeSchedule.backward_remove_noise :474-498
struct BpArgs {
  const float4* x4;         // ligand rows hold x_com (output of the CoM head's H2X stack)
  const int* graph_ptr;
  const int* lig_node;
  int n_lig, num_classes, n_graphs;
  const float* x_pred;      // [n_lig,3] denoiser output coordinates
  const float* logits;      // [n_lig,K]
  const float* x_t;         // [n_lig,3]
  const float* c_t;         // [n_lig,K]
  const unsigned char* gen; // [n_lig]
  const float* pos_noise;   // [n_lig,3]
  const float* type_u;      // [n_lig]
  float abar, beta, nonzero, prob;
  float* x_next;            // [n_lig,3]
  float* c_next;            // [n_lig,K]
  long long* v_next;        // [n_lig]
  float* eps_out;           // optional [n_lig,3]
};
int cbg_launch_bp_reverse(const BpArgs& a, cudaStream_t st);

// batch.cu (row f3: device-side batch construction)
int cbg_launch_pocket_stats(const float* prot_pos, const int* prot_ptr, int n_pockets, const float* ctx_pos,
                            const int* ctx_ptr, int centre_mode, float* space_size, float* centre, cudaStream_t st);
int cbg_launch_ligand_sizes(const double* bounds, int n_bounds, const int* bin_ptr, const int* values, const double* cdf,
                            const float* space_size, int n_pockets, int repeat, const double* u, const int* ctx_ptr,
                            const int* extra, int* n_lig, int* lig_ptr, cudaStream_t st);
int cbg_launch_build_batch(const float* prot_pos, const int* prot_element, const unsigned char* prot_backbone,
                           const int* prot_aa, const int* prot_ptr, int n_pockets, int repeat, const float* centre,
                           const float* ctx_pos, const int* ctx_type, const int* ctx_ptr, const int* lig_ptr,
                           const float* pos_noise, const float* type_u, int num_classes, int type_dist, int pos_dist,
                           float* o_prot_pos, float* o_prot_feat, long long* o_prot_aa, long long* o_prot_batch,
                           float* o_prot_tr, float* o_lig_pos, long long* o_lig_type, long long* o_lig_batch,
                           unsigned char* o_lig_ctx, unsigned char* o_lig_gen, cudaStream_t st);

// ipa.cu (row f4: D3FG encoder).  The head block has its own class bound: D3FG's fg_only mode has 28 FG types, while the
// denoiser blob (cbg_layout.h) keeps CBG_MAXCLS.
#define CBG_IPA_MAXCLS 32
// h_out == h_in: the layers update h in place (no copy); ws: cbg_ipa_workspace_bytes(n_nodes, hidden), 256-byte aligned
int cbg_launch_ipa_forward(const float* blob, int hidden, int num_sublayers, int num_blocks, int num_classes, const float* x,
                           const float* o, const float* h_in, const int* graph_ptr, int n_graphs, int max_graph_nodes,
                           const unsigned char* lig_flag, const unsigned char* gen_flag, int n_nodes, int k, float* eps_pos,
                           float* h_out, float* o_next, float* r_next, float* logits, char* ws, cudaStream_t st);
