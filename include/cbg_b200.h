/* cbg_b200 - C-ABI of the B200-native CBGBench diffusion-sampling hot path.
 *
 * The reference (EDAPINENUT/CBGBench @ 983fca2, /root/reference) is 100 % Python/PyTorch and
 * has NO FFI / plugin / operator boundary of its own (SURVEY.md section 8b): its seam is the Python
 * factory get_e3_gnn() (repo/modules/e3nn/__init__.py:5-18) returning an nn.Module whose
 * forward(x, h, batch_idx, lig_flag, gen_flag) -> (x, h, c) is repo/modules/e3nn/unitransformer.py:102-123,
 * iterated by TargetDiff.sample (repo/models/diffusion/targetdiff.py:127-184).  The entry points
 * below are what a ctypes binding for that seam needs; each one cites the reference code it
 * replaces.  INTEGRATION.md shows the reference-side stub.
 *
 * Conventions
 *   - plain C, no C++ types or exceptions across the boundary;
 *   - every pointer is a DEVICE pointer owned by the caller unless the name ends in _host;
 *   - fp32 data, int32 indices, uint8 flags; row-major contiguous;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); calls only
 *     enqueue work (no host synchronisation) unless the name ends in _host;
 *   - return 0 on success; non-zero = error, message from cbg_last_error() (thread-local);
 *   - graphs are contiguous node ranges: graph g owns nodes graph_ptr[g] .. graph_ptr[g+1]-1
 *     (the reference's sorted PyG `batch` vector, repo/modules/common.py:189-214);
 *   - neighbour tables have fixed width CBG_NBR_WIDTH = 32 (k <= 32), nearest first,
 *     padded with -1 (graphs with fewer than k+1 atoms, radius mode).
 */
#ifndef CBG_B200_H_
#define CBG_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CBG_NBR_WIDTH 32
#define CBG_HIDDEN 128
#define CBG_N_HEADS 16
#define CBG_MAX_CLASSES 16

#define CBG_CUTOFF_KNN 0     /* reference default, unitransformer.py:27-28,78-80 */
#define CBG_CUTOFF_RADIUS 1  /* defined in SURVEY.md section 8c (reference branch is dead code, unitransformer.py:76-77) */

int32_t cbg_version(void);
const char* cbg_last_error(void);
/* number of CUDA kernels this library has launched in the calling process (bench.py gpu_launches) */
int64_t cbg_launch_count(void);

/* Optional per-kernel profile: while enabled every kernel launch of the library is bracketed by
 * CUDA events on the launching stream; cbg_profile_collect synchronises and returns the summed
 * device time (ms) and launch count per kernel family (bench.py roofline block). */
int32_t cbg_profile_num_families(void);
const char* cbg_profile_family_name(int32_t i);
int32_t cbg_profile_enable(int32_t on);
int32_t cbg_profile_collect(double* ms_per_family, int64_t* launches_per_family);

/* TESTING hook (process-wide, not thread-safe; production code never calls it): implementation of the fused X2H / H2X
 * edge kernels.  impl 6 (default): the tcgen05 tile kernel (csrc/x2h_tc.cu: A operands in tensor memory, f16 hi/lo split);
 * impl 0: the fp32 SIMT kernels (csrc/edge.cu), kept as an independent implementation for the parity tests - the only
 * consumer of the optional R-cache.  warps = CTA size of the SIMT kernels (8, 12, 16; 0 keeps the current value).
 * Also env CBG_EDGE_IMPL / CBG_EDGE_WARPS.  Needs a current CUDA device. */
int32_t cbg_set_edge_impl(int32_t impl, int32_t warps);
/* Hardware self-test of the tcgen05 operand conventions the X2H kernels rely on (tests only):
 * d[128][128] (fp32) = a[128][32] * b[128][32]^T with f16 row-major device inputs; a_from_smem = 0 feeds A from
 * tensor memory (tcgen05.st, two K-consecutive f16 per column), 1 from shared memory (canonical K-major layout). */
int32_t cbg_selftest_umma_f16(const void* a, const void* b, float* d, int32_t a_from_smem, void* stream);
/* Debugging: the next launch of the tcgen05 attention-weight kernel (max_tiles > 0) or aggregation kernel (max_tiles < 0,
 * |max_tiles| rows) stamps the pipeline events of CTA 0 (SM clock) into buf_dev[|max_tiles| + 1][16] (int64, device memory;
 * the last row takes kernel entry / end of prologue / exit); NULL turns it off.  Process-wide, one-shot. */
int32_t cbg_debug_x2h_trace(int64_t* buf_dev, int32_t max_tiles);
/* debug: %globaltimer stamps (ns) of CTA 0 of every following f16 node-GEMM launch into buf_dev[32] (NULL = off):
 * [0] start, [1] A tile staged, [2+g] accumulator g complete, [10+g] epilogue of g done, [20] end */
int32_t cbg_debug_node_gemm_trace(int64_t* buf_dev);
/* Other TESTING switches of the SIMT kernels (process-wide): "static_fast" = 1 (default; env CBG_STATIC_FAST) lets them
 * skip the coordinate gathers / RBF set-up of nodes whose 32 in-edges are all served from the R-cache (bit-identical);
 * "dyn_sched" = 1 (default; env CBG_DYN_SCHED): their warps draw the next node from a work counter instead of a static
 * round-robin (bit-identical). */
int32_t cbg_set_option(const char* key, int32_t value);

/* ---- packed weight blob layout (single source of truth: csrc/cbg_layout.h) -------------------
 * blob = [global section][layer 0][layer 1]...; section 0 = global, 1 = per-layer.
 * Replaces the nn.Module parameter tree of UniTransformer (state-dict keys in SURVEY.md section 8b). */
int64_t cbg_blob_global_floats(void);
int64_t cbg_blob_layer_floats(void);
int32_t cbg_blob_num_fields(int32_t section);
const char* cbg_blob_field_name(int32_t section, int32_t idx);
int64_t cbg_blob_field_offset(int32_t section, int32_t idx);
int64_t cbg_blob_field_size(int32_t section, int32_t idx);

/* bytes of the optional R-cache of a sampling plan: 2 * num_layers * n_nodes * 32 * 128 floats */
int64_t cbg_rcache_bytes(int64_t n_nodes, int32_t num_layers);

/* scratch bytes needed by the calls below for n_nodes nodes of which n_gen carry gen_flag */
int64_t cbg_workspace_bytes(int64_t n_nodes, int64_t n_gen);

/* Neighbour lists on device.
 * Replaces torch_geometric.nn.knn_graph(x, k, batch, flow='source_to_target')
 * (call site unitransformer.py:79-80; third-party torch_cluster kernel).  nbr[i, s] = global index
 * of the s-th nearest j != i of i's graph (ties -> lower index), -1 padded.  The reference's
 * edge_index is [nbr[i,s] ; i] for all valid slots, grouped by i. */
int32_t cbg_build_neighbors_f32(const float* x /*[N,3]*/, const int32_t* graph_ptr /*[B+1]*/,
                                int32_t n_graphs, int64_t n_nodes, int32_t max_graph_nodes,
                                int32_t mode, int32_t k, float r_max,
                                int32_t* nbr /*[N,32] out*/,
                                void* workspace, size_t workspace_bytes, void* stream);

/* Global edge gate e_w = sigmoid(dist_emb(|x_i - x_j|)) (unitransformer.py:109-112,
 * embs/dist_emb.py:6-14).  ew[i, s] for slot s of node i (0 for padded slots). */
int32_t cbg_edge_gate_f32(const float* blob, const float* x /*[N,3]*/, const int32_t* nbr /*[N,32]*/,
                          int64_t n_nodes, float* ew /*[N,32] out*/,
                          void* workspace, size_t workspace_bytes, void* stream);

/* One full denoiser forward = UniTransformer.forward (unitransformer.py:102-123): graph build,
 * edge gate, num_layers x (X2HAttention, H2XAttention, masked coordinate update), classifier.
 * Inputs are not modified.  gen_idx lists the nodes with gen_flag set (any order);
 * cls_idx = NULL computes logits for all nodes (logits_out [N,K]) else only for the listed
 * rows (logits_out [n_cls,K]).  stop_after_layers < 0 runs all layers (testing hook: run
 * only the first stop_after_layers layers, then the classifier). */
int32_t cbg_denoiser_forward_f32(const float* blob, int32_t num_layers, int32_t num_classes,
                                 const float* x /*[N,3]*/, const float* h /*[N,128]*/,
                                 const int32_t* graph_ptr, int32_t n_graphs, int32_t max_graph_nodes,
                                 const uint8_t* lig_flag /*[N]*/, const uint8_t* gen_flag /*[N]*/,
                                 const int32_t* gen_idx, int32_t n_gen,
                                 const int32_t* cls_idx, int32_t n_cls,
                                 int64_t n_nodes, int32_t mode, int32_t k, float r_max,
                                 int32_t stop_after_layers,
                                 float* x_out /*[N,3]*/, float* h_out /*[N,128]*/, float* logits_out,
                                 void* workspace, size_t workspace_bytes, void* stream);

/* Same call with HOST buffers (pageable or pinned): copies inputs to the device, runs the
 * forward, copies x_out/h_out/logits_out back and synchronises.  Device scratch is cached
 * inside the library.  blob_host holds the packed weights; it is re-uploaded when
 * blob_version changes. */
int32_t cbg_denoiser_forward_host_f32(const float* blob_host, int64_t blob_floats, int64_t blob_version,
                                      int32_t num_layers, int32_t num_classes,
                                      const float* x_host, const float* h_host,
                                      const int32_t* graph_ptr_host, int32_t n_graphs,
                                      const uint8_t* lig_flag_host, const uint8_t* gen_flag_host,
                                      int64_t n_nodes, int32_t mode, int32_t k, float r_max,
                                      float* x_out_host, float* h_out_host, float* logits_out_host);

/* Node projections of one attention sub-layer alone (testing / integration hook): the five planes
 * [Pj_k, Pj_v, Pi_k, Pi_v, q] of sub-layer `sublayer` (0 = X2H, 1 = H2X) for the listed rows
 * (row_idx NULL = rows 0..n_rows-1), planes = [5][n_nodes][128].  impl 0 = fp32 SIMT kernel,
 * 1 = tcgen05 3xTF32 kernel (warp-specialised, default), 11 = single-issuer variant, 12 / 14 = that variant
 * with weight chunks multicast over clusters of 2 / 4 CTAs.  blob_layer points at the layer's block inside the packed blob.
 * Replaces the h-dependent part of MLP.net[0] and hq_func/xq_func (x2h_attention.py:58-83). */
int32_t cbg_node_proj_f32(const float* blob_layer, int32_t sublayer, int32_t impl, const float* h,
                          const int32_t* row_idx, int32_t n_rows, int64_t n_nodes, float* planes, void* stream);

/* ---- fused sampling step: embed -> denoiser -> reverse diffusion step -------------------------
 * One iteration of the loop body of TargetDiff.sample (targetdiff.py:150-182):
 *   PLContextEmbedder.forward (context_emb.py:179-231), compose_context (common.py:189-214,
 *   hoisted: the permutation is step-invariant), denoiser, then
 *   CTNVPScheduler.backward_remove_noise(type='denoise') (diffusion_scheduler.py:144-165) and
 *   TypeVPScheduler.backward_remove_noise (diffusion_scheduler.py:367-378).
 * Random numbers stay with the caller (torch.randn_like / rand_like order of the reference). */
typedef struct cbg_sample_plan {
  const float* blob;            /* packed denoiser weights */
  int32_t num_layers;
  int32_t num_classes;
  const float* emb_wt;          /* [K,128] context_embedder.ligand_atom_emb.weight^T */
  const float* h_lig_bias;      /* [n_lig,128] ligand_atom_emb.bias + ligand_indicator(lig_flag) */
  const float* h_static;        /* [N,128] step-invariant node features (protein rows) */
  const int32_t* graph_ptr;     /* [B+1] over composed nodes ([protein | ligand] per graph) */
  int32_t n_graphs;
  int32_t max_graph_nodes;
  int64_t n_nodes;
  const int32_t* lig_node;      /* [n_lig] composed node index of every ligand atom */
  int32_t n_lig;
  const uint8_t* gen_lig;       /* [n_lig] ligand_gen_flag */
  const int32_t* gen_node;      /* [n_gen] composed node indices with gen_flag */
  int32_t n_gen;
  int32_t mode;                 /* CBG_CUTOFF_* */
  int32_t k;
  float r_max;
  void* workspace;
  size_t workspace_bytes;
  float* rcache;                /* optional (NULL = off): cbg_rcache_bytes() of scratch for the step-invariant
                                   first-Linear terms of edges between non-generated atoms (SURVEY.md App. B);
                                   filled by cbg_sample_begin_f32, streamed by the fused X2H kernels */
  size_t rcache_bytes;
  int32_t prune;                /* 1: receptive-field pruning - layer l only updates the nodes that can still
                                   influence a generated / ligand atom through the remaining layers (exact for
                                   everything cbg_sample_step_f32 returns; intermediate h of other nodes is skipped) */
  int32_t static_lists;         /* 1: atoms without gen_flag never move, so cbg_sample_begin_f32 builds their static-only
                                   neighbour lists and edge gates once per batch; every step's neighbour search is then
                                   incremental and static edges reuse their gate (exact).  Implied by rcache != NULL.
                                   Must be 0 for samplers that move the pocket (DiffSBDD). */
} cbg_sample_plan;

typedef struct cbg_step_coef {  /* scheduler table entries of the current step (host scalars) */
  float pos_c0;                 /* pos_scheduler.posterior_mean_c0_coef[t] */
  float pos_ct;                 /* pos_scheduler.posterior_mean_ct_coef[t] */
  float pos_logvar;             /* pos_scheduler.posterior_logvar[t] */
  float pos_nonzero;            /* 0 if t == 0 else 1 */
  float log_alphas_cumprod_prev;          /* type_scheduler.log_alphas_cumprod_v[max(t-1,0)] */
  float log_one_minus_alphas_cumprod_prev;/* type_scheduler.log_one_minus_alphas_cumprod_v[max(t-1,0)] */
  float log_alpha;              /* type_scheduler.log_alphas_v[t] */
  float log_one_minus_alpha;    /* type_scheduler.log_one_minus_alphas_v[t] */
} cbg_step_coef;

/* writes the static part of the node state (all coordinates + flags) into the plan workspace */
int32_t cbg_sample_begin_f32(const cbg_sample_plan* plan, const float* x_nodes /*[N,3]*/,
                             const uint8_t* lig_flag /*[N]*/, const uint8_t* gen_flag /*[N]*/, void* stream);

/* Measurement hook (bench.py roofline): node counts of the receptive-field pruning of the LAST step run on this plan,
 * counts_host[l + 1] = nodes whose X2H output of layer l is still needed (= rows the X2H kernels of layer l process),
 * counts_host[0] = nodes needed at all; num_layers + 1 entries.  Copies to host memory and synchronises the stream. */
int32_t cbg_sample_prune_counts_host(const cbg_sample_plan* plan, int32_t* counts_host /*[num_layers+1]*/, void* stream);

int32_t cbg_sample_step_f32(const cbg_sample_plan* plan, const cbg_step_coef* coef,
                            const float* x_t /*[n_lig,3]*/, const float* c_t /*[n_lig,K]*/,
                            const float* pos_noise /*[n_lig,3]*/, const float* type_uniform /*[n_lig,K]*/,
                            float* x_next /*[n_lig,3]*/, float* c_next /*[n_lig,K]*/, int64_t* v_next /*[n_lig]*/,
                            float* x0_pred /*[n_lig,3] or NULL*/, float* logits /*[n_lig,K] or NULL*/,
                            void* stream);

/* cbg_sample_step_f32 replayed from a CUDA graph: the first call for a plan runs eagerly, the second captures the step
 * (its ~85 kernel launches, fork/join events and memsets) on `stream`, later calls cost one small H2D copy of the per-step
 * pointers / schedule coefficients plus one cudaGraphLaunch.  Results are bit-identical to cbg_sample_step_f32 (same
 * kernels, same order).  The plan must be unchanged between calls (same contents); x0_pred / logits outputs are not
 * available on this path.  cbg_sample_step_graph_nodes: kernel launches inside the captured graph (0: not captured yet). */
int32_t cbg_sample_step_graph_f32(const cbg_sample_plan* plan, const cbg_step_coef* coef,
                                  const float* x_t, const float* c_t, const float* pos_noise, const float* type_uniform,
                                  float* x_next, float* c_next, int64_t* v_next, void* stream);
int64_t cbg_sample_step_graph_nodes(const cbg_sample_plan* plan, void* stream);

/* the reverse step alone (testing / integration hook) */
int32_t cbg_reverse_step_f32(const cbg_step_coef* coef, const float* x0_pred /*[n,3]*/, const float* logits /*[n,K]*/,
                             const float* x_t, const float* c_t, const uint8_t* gen /*[n]*/,
                             const float* pos_noise, const float* type_uniform,
                             int32_t n, int32_t num_classes,
                             float* x_next, float* c_next, int64_t* v_next, void* stream);

/* ---- SURVEY.md section 8 row f2: the other diffusion samplers that drive the same denoiser -------------------
 *
 * DiffSBDD (diffsbdd.py:240-321): every step is embed -> denoiser -> sample_p_zs_given_zt
 * (diffusion_scheduler.py:1005-1039) for coordinates and (continuous) type features, with the COM projection
 * remove_mean_batch (:706-710) that also translates the pocket.  All graphs share (s, t), so the schedule enters as
 * three host scalars.  mode 1 is the final stage sample_p_xh_given_z0 (diffsbdd.py:323-360).
 * The plan is the one of cbg_sample_begin_f32 WITHOUT an R-cache (the pocket is not static here). */
typedef struct cbg_sbdd_coef {
  float a;       /* mode 0: alpha_t|s                      mode 1: 1 / alpha_0            */
  float b;       /* mode 0: sigma2_t|s / alpha_t|s / sigma_t   mode 1: sigma_0            */
  float s;       /* mode 0: sigma_t|s * sigma_s / sigma_t  mode 1: exp(0.5 * gamma_0)     */
  int32_t mode;  /* 0: z_s = z_t / a - b * eps + s * noise;  1: z = a * (z_t - b * eps) + s * noise, c_next = 4 c_t */
} cbg_sbdd_coef;

int32_t cbg_sbdd_step_f32(const cbg_sample_plan* plan, const cbg_sbdd_coef* coef,
                          const float* x_t /*[n_lig,3]*/, const float* c_t /*[n_lig,K]*/,
                          const float* x_noise /*[n_lig,3]*/, const float* c_noise /*[n_lig,K]*/,
                          float* x_next /*[n_lig,3]*/, float* c_next /*[n_lig,K]*/,
                          float* x_pred /*[n_lig,3] or NULL*/, float* logits /*[n_lig,K] or NULL*/, void* stream);

/* DiffBP (diffbp.py:240-299): embed -> denoiser -> CoM head (CoMPredictor, diffbp.py:30-101: the step's kNN graph,
 * its own edge gate, com_layers x H2X on the denoiser's final h starting from the step's input coordinates) ->
 * CTNVPScheduler.backward_remove_noise(type='score') (diffusion_scheduler.py:144-165) on eps + eps_com and
 * MaskTypeSchedule.backward_remove_noise (:474-498).  com_blob packs the CoM head in the denoiser's blob layout
 * (gate fields of the global block, H2X fields of com_layers layer blocks).  type_uniform is [n_lig]. */
typedef struct cbg_bp_coef {
  float alpha_cumprod;   /* pos_scheduler.alphas_cumprod[t] */
  float beta;            /* pos_scheduler.betas[t] */
  float nonzero;         /* 0 if t == 0 else 1 */
  float change_prob;     /* clamp((T - t) / T, 0, 1) */
} cbg_bp_coef;

int32_t cbg_bp_step_f32(const cbg_sample_plan* plan, const float* com_blob, int32_t com_layers,
                        const cbg_bp_coef* coef, const float* x_t /*[n_lig,3]*/, const float* c_t /*[n_lig,K]*/,
                        const float* pos_noise /*[n_lig,3]*/, const float* type_uniform /*[n_lig]*/,
                        float* x_next /*[n_lig,3]*/, float* c_next /*[n_lig,K]*/, int64_t* v_next /*[n_lig]*/,
                        float* eps_out /*[n_lig,3] or NULL: eps + eps_com*/, float* logits /*[n_lig,K] or NULL*/,
                        void* stream);

/* ---- SURVEY.md section 8 row f3: sampling-time transforms + batch construction on the device ------------------
 *
 * The reference builds a sampling batch by evaluating dataset[i] num_samples times (sample.py:177), i.e. by running
 * the Python transform list of configs/<task>/test/<model>.yml once per sample, and collating with PyG.  The three calls
 * below produce the same flat batch from the raw pocket arrays on the device.  Pockets are ragged ranges
 * (prot_ptr[n_pockets+1]); every pocket is sampled `repeat` times; sample s belongs to pocket s / repeat.
 * Random numbers are the caller's (numpy / torch order of the reference: one uniform per sample for the size prior,
 * optionally one randint(1, 8), then rand [n, K] for the types and randn [n, 3] for the positions). */

/* Pocket centre and "space size".
 *   centre_mode 0: centre = mean of the pocket atoms (center_pos(center_flag=protein), translation.py:11-24, and
 *                  center_whole_pos without a ligand, :36-50); space size measured on the centred coordinates
 *   centre_mode 1: centre = mean of the pocket's context ligand atoms, 0 if it has none (center_pos(ligand,
 *                  mask_flag=ctx_flag)); space size measured on the raw coordinates (assign_gensize runs first)
 * space_size = median of the 10 largest pairwise atom distances (AssignMolSize.get_space_size, init_lig.py:247-250). */
int32_t cbg_pocket_stats_f32(const float* prot_pos /*[n_atoms,3]*/, const int32_t* prot_ptr /*[n_pockets+1]*/,
                             int32_t n_pockets, const float* ctx_pos /*[n_ctx,3] or NULL*/,
                             const int32_t* ctx_ptr /*[n_pockets+1] or NULL*/, int32_t centre_mode,
                             float* space_size /*[n_pockets] out*/, float* centre /*[n_pockets,3] out*/, void* stream);

/* Size prior (repo/datasets/transforms/_atom_num_dist.npy) as flat device arrays: bin b (b = 0..n_bounds) is chosen by
 * the first bound greater than the space size (init_lig.py:47-52) and holds values[bin_ptr[b]:bin_ptr[b+1]] with the
 * cumulative distribution cdf[...] = cumsum(p) / sum(p) that numpy's legacy choice(values, p=p) searches
 * (side='right') with its uniform draw (sample_atom_num, init_lig.py:27-31). */
typedef struct cbg_size_prior {
  const double* bounds;
  int32_t n_bounds;
  const int32_t* bin_ptr;   /* [n_bounds + 2] */
  const int32_t* values;
  const double* cdf;
} cbg_size_prior;

/* Ligand atom counts of the n_pockets * repeat samples and their exclusive prefix sum.  With ctx_ptr (context tasks,
 * AssignGenSize init_lig.py:253-296) a draw that does not exceed the pocket's context atom count is replaced by
 * context + extra[s] (the reference's torch.randint(1, 8)). */
int32_t cbg_sample_ligand_sizes(const cbg_size_prior* prior, const float* space_size /*[n_pockets]*/, int32_t n_pockets,
                                int32_t repeat, const double* u /*[S]*/, const int32_t* ctx_ptr /*or NULL*/,
                                const int32_t* extra /*[S] or NULL*/, int32_t* n_lig /*[S] out*/,
                                int32_t* lig_ptr /*[S+1] out*/, void* stream);

#define CBG_TYPE_UNIFORM 0    /* assign_atomtype / assign_genatomtype 'uniform': Gumbel arg-max over zero logits (init_lig.py:22-26) */
#define CBG_TYPE_ABSORBING 1  /* 'absorbing' (state 0); also used for 'zeros' (the caller allocates the [n,K] zero features) */
#define CBG_POS_GAUSSIAN 0            /* assign_molpos / assign_genpos 'gaussian' (init_lig.py:404-457) */
#define CBG_POS_ZERO_MEAN_GAUSSIAN 1  /* 'zero_mean_gaussian': the sample's mean is removed (de-novo only) */

typedef struct cbg_batch_spec {
  /* raw pockets (protein_featurizer.py:19-30 runs on the device) */
  const float* prot_pos;          /* [n_atoms,3] */
  const int32_t* prot_element;    /* [n_atoms] atomic numbers */
  const uint8_t* prot_backbone;   /* [n_atoms] is_backbone */
  const int32_t* prot_aa;         /* [n_atoms] atom_to_aa_type */
  const int32_t* prot_ptr;        /* [n_pockets+1] */
  int32_t n_pockets;
  int32_t repeat;
  const float* centre;            /* [n_pockets,3] from cbg_pocket_stats_f32 */
  /* context ligand atoms per pocket (NULL / NULL / NULL for de-novo): they come first in every sample, are centred like
   * the pocket, keep their types and get ctx_flag = 1, gen_flag = 0 */
  const float* ctx_pos;
  const int32_t* ctx_type;
  const int32_t* ctx_ptr;
  const int32_t* lig_ptr;         /* [S+1] from cbg_sample_ligand_sizes */
  const float* pos_noise;         /* [n_lig_total,3] standard normal (rows of context atoms are ignored) */
  const float* type_u;            /* [n_lig_total,K] uniform(0,1) or NULL unless type_dist == CBG_TYPE_UNIFORM */
  int32_t num_classes;
  int32_t type_dist;
  int32_t pos_dist;
  /* outputs = the flat batch of SURVEY.md section 8b (graph id = sample index) */
  float* protein_pos;             /* [S_atoms,3] centred */
  float* protein_atom_feature;    /* [S_atoms,7] */
  int64_t* protein_aa_type;       /* [S_atoms] */
  int64_t* protein_element_batch; /* [S_atoms] */
  float* protein_translation;     /* [S_atoms,3] the centre, per atom (translation.py:19) */
  float* ligand_pos;              /* [n_lig_total,3] */
  int64_t* ligand_atom_type;      /* [n_lig_total] */
  int64_t* ligand_element_batch;  /* [n_lig_total] */
  uint8_t* ligand_ctx_flag;       /* [n_lig_total] or NULL */
  uint8_t* ligand_gen_flag;       /* [n_lig_total] or NULL */
} cbg_batch_spec;

int32_t cbg_build_batch_f32(const cbg_batch_spec* spec, void* stream);

/* ---- SURVEY.md section 8 row f4: D3FG encoder `IPATransformer` (repo/modules/e3nn/itatransformer.py:14-145) --------------
 * X2H-only encoder (InvAttentionLayer :147-188, coordinates fixed) at hidden width 128 or 256 (configs/denovo/train/
 * d3fg_fg.yml:5: 256), then the rotation / translation / type heads and the SO(3) update (:127-145):
 *   eps_pos [N,3], h [N,H], o_next [N,3] (so3 vector), R_next [N,3,3], logits [N,K]
 * = IPATransformer.forward(x, o, h, batch_idx, lig_flag, gen_flag).  Weights: one blob = the global block of the denoiser
 * layout (edge-gate fields) | head block | num_sublayers layer blocks; the field table below is the single source of
 * truth the Python packer queries (cbgbench_b200/ipatransformer.py). */
int64_t cbg_ipa_head_floats(int32_t hidden);
int64_t cbg_ipa_layer_floats(int32_t hidden);
int32_t cbg_ipa_head_fields(void);
int32_t cbg_ipa_layer_fields(void);
const char* cbg_ipa_head_field_name(int32_t field);
const char* cbg_ipa_layer_field_name(int32_t field);
int64_t cbg_ipa_head_field_offset(int32_t hidden, int32_t field);
int64_t cbg_ipa_head_field_size(int32_t hidden, int32_t field);
int64_t cbg_ipa_layer_field_offset(int32_t hidden, int32_t field);
int64_t cbg_ipa_layer_field_size(int32_t hidden, int32_t field);
int64_t cbg_ipa_workspace_bytes(int64_t n_nodes, int32_t hidden);
int32_t cbg_ipa_forward_f32(const float* blob, int32_t hidden, int32_t num_sublayers /* num_layers * num_x2h */,
                            int32_t num_blocks, int32_t num_classes, const float* x /*[N,3]*/, const float* o /*[N,3]*/,
                            const float* h /*[N,hidden]*/, const int32_t* graph_ptr /*[B+1]*/, int32_t n_graphs,
                            int32_t max_graph_nodes, const uint8_t* lig_flag, const uint8_t* gen_flag, int64_t n_nodes,
                            int32_t k, float* eps_pos, float* h_out, float* o_next, float* r_next, float* logits,
                            void* workspace, int64_t workspace_bytes, void* stream);

/* ---- D3FG sampler: one reverse step of D3FG.sample (repo/models/diffusion/difffg.py:174-246) per call ------------------
 * num_classes <= 32 (fg_only mode: 28 FG types).  Per call, on `stream`:
 *   step-init kernel   composed rows of the ligand FGs: x = x_t, o = o_t and
 *                        h = (ligand_fg_emb.weight[:, argmax(c_t)] + ligand_fg_emb.bias) + ligand_indicator(1)
 *                      (argmax = first maximum, like torch.argmax: FGContextEmbedder re-one-hots the 28-wide c_t into its
 *                      49-wide input, context_emb.py:95-102).  The protein rows of x and o are written once by the caller
 *                      and never rewritten; those of h are copied from h_static (the layers update h in place).
 *   IPA encoder        cbg_ipa_forward_f32 on the plan's workspace -> eps_pos, o_pred (gen-masked), logits on every row
 *   d3fg_reverse       one warp per FG (lane = class), gen_flag-masked (rows without it keep x_t, o_t, argmax(c_t)):
 *     position  CTNVPScheduler.backward_remove_noise(type='score'):
 *               x' = (x_t + beta * (-eps / sqrt(1 - alpha_cumprod))) / sqrt(1 - beta) + pos_nonzero * sqrt(beta) * pos_noise
 *     rotation  RotVPScheduler.backward_remove_noise: e = normalize(rot_dir) * theta if t > 1 else 0,
 *               o' = log(exp(e) exp(o_pred)) with so3.py's 1e-8 guards and min_cos = -1 (sampling runs without grad);
 *               theta ~ ApproxAngularDistribution(inverse sigmas) at t:  stddev <= 0.1: |2 sd + sd * rot_gauss| mod pi,
 *               otherwise X[t, bin] + rot_in_u * (X[t, bin + 1] - X[t, bin]) with the bin drawn below
 *     type      TypeVPScheduler.backward_remove_noise: log_softmax(logits), the q_v_posterior log-add-exp, Gumbel argmax
 *               of type_u (categorical.py:26-37)
 *
 * Multinomial draw.  The reference draws the histogram bin with torch.multinomial(Y[t, :-1]), whose internal draw cannot
 * be passed in.  Here a draw is an inverse CDF: with rot_cdf[t] = cumsum(Y[t, :-1]) in float64 (n_bins = 8191 entries
 * per row, computed once on the host), bin = the first index with rot_cdf[t][bin] > (double)rot_bin_u * rot_cdf[t][n_bins-1].
 * A bin of zero weight is never chosen, so the distribution is torch.multinomial's; the device searches the same float64
 * table, so a given uniform selects the same bin as the host definition (oracle/diffusion_fg.py). */
typedef struct cbg_d3fg_plan {
  const float* blob;          /* IPA blob (cbg_ipa_* field table) */
  int32_t hidden;             /* 128 or 256 */
  int32_t num_sublayers;      /* num_layers * num_x2h */
  int32_t num_blocks;
  int32_t num_classes;        /* K <= 32 */
  int32_t k;                  /* kNN neighbours */
  const int32_t* graph_ptr;   /* [n_graphs + 1] composed rows */
  int32_t n_graphs;
  int32_t max_graph_nodes;
  int64_t n_nodes;
  const uint8_t* lig_flag;    /* [n_nodes] composed */
  const uint8_t* gen_flag;    /* [n_nodes] composed */
  const int32_t* lig_node;    /* [n_lig] composed row of FG a, increasing */
  int32_t n_lig;
  const uint8_t* gen_lig;     /* [n_lig] */
  const float* fg_wt;         /* [K, hidden] = ligand_fg_emb.weight[:, :K]^T */
  const float* fg_b;          /* [hidden] ligand_fg_emb.bias */
  const float* lig_bias;      /* [hidden] ligand_indicator(1) */
  const float* h_static;      /* [n_nodes, hidden]: the protein rows (h_rec); ligand rows are not read */
  float* x;                   /* [n_nodes, 3] composed coordinates */
  float* o;                   /* [n_nodes, 3] composed so3 vectors */
  const double* rot_cdf;      /* [T, n_bins] */
  const float* rot_x;         /* [T, n_bins + 1] bin edges (angular_distrib_inv.X) */
  int32_t n_bins;
  void* workspace;            /* cbg_d3fg_workspace_bytes, 256-byte aligned */
  int64_t workspace_bytes;
} cbg_d3fg_plan;

typedef struct cbg_d3fg_coef {  /* scheduler table entries of step t (host scalars) */
  float alpha_cumprod;          /* pos_scheduler.alphas_cumprod[t] */
  float beta;                   /* pos_scheduler.betas[t] */
  float pos_nonzero;            /* t > 0 */
  float rot_stddev;             /* rot_scheduler.angular_distrib_inv.stddevs[t] */
  int32_t rot_approx;           /* angular_distrib_inv.approx_flag[t] */
  float rot_nonzero;            /* t > 1 */
  int32_t rot_row;              /* row of rot_cdf / rot_x (= t) */
  float log_alphas_cumprod_prev;            /* type_scheduler tables at max(t - 1, 0) ... */
  float log_one_minus_alphas_cumprod_prev;
  float log_alpha;                          /* ... and at t */
  float log_one_minus_alpha;
} cbg_d3fg_coef;

int64_t cbg_d3fg_workspace_bytes(int64_t n_nodes, int32_t hidden, int32_t num_classes);
int32_t cbg_d3fg_step_f32(const cbg_d3fg_plan* plan, const cbg_d3fg_coef* coef, const float* x_t /*[n_lig,3]*/,
                          const float* c_t /*[n_lig,K]*/, const float* o_t /*[n_lig,3]*/, const float* pos_noise /*[n_lig,3]*/,
                          const float* rot_dir /*[n_lig,3]*/, const float* rot_bin_u /*[n_lig]*/,
                          const float* rot_in_u /*[n_lig]*/, const float* rot_gauss /*[n_lig]*/,
                          const float* type_u /*[n_lig,K]*/, float* x_next, float* c_next, float* o_next,
                          int64_t* v_next /*[n_lig]*/, float* eps_pos_out /*[n_lig,3] or NULL*/,
                          float* logits_out /*[n_lig,K] or NULL*/, float* o_pred_out /*[n_lig,3] or NULL*/, void* stream);
/* The reverse step alone (test hook, like cbg_reverse_step_f32): eps / logits / o_pred are per-FG rows; bin_out receives
 * the histogram bin of every row (drawn whether or not the Gaussian branch is taken), or NULL. */
int32_t cbg_d3fg_reverse_f32(const cbg_d3fg_coef* coef, const double* rot_cdf, const float* rot_x, int32_t n_bins,
                             const float* eps /*[n,3]*/, const float* logits /*[n,K]*/, const float* o_pred /*[n,3]*/,
                             const float* x_t, const float* c_t, const float* o_t, const uint8_t* gen,
                             const float* pos_noise, const float* rot_dir, const float* rot_bin_u, const float* rot_in_u,
                             const float* rot_gauss, const float* type_u, int32_t n, int32_t num_classes, float* x_next,
                             float* c_next, float* o_next, int64_t* v_next, int32_t* bin_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CBG_B200_H_ */
