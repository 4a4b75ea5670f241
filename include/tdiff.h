/* tdiff.h -- C-ABI of libtdiff.so: the B200 (sm_100a) engine for targetdiff's denoising-sampling hot path.
 *
 * This is the drop-in boundary (SURVEY.md section 8(b)).  The reference is pure Python; the "FFI" a maintainer
 * binds is ctypes (see INTEGRATION.md).  Each entry point names the reference interface it replaces
 * (paths relative to the reference tree).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no torch types.
 *   - `d_` arguments are DEVICE pointers owned by the caller; `h_` arguments are HOST pointers.
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream).  Calls are asynchronous on it
 *     unless stated otherwise.
 *   - every function returns 0 on success or a negative TDIFF_E* code; tdiff_last_error() gives the text.
 *     Nothing throws across the ABI.  One engine per device; an engine is not thread-safe.
 *   - there is NO CPU fallback: without a CUDA device tdiff_create fails with TDIFF_ECUDA.
 *   - node order everywhere is the reference's `compose_context` order (models/common.py:120-137):
 *     per graph, protein atoms (input order) then ligand atoms (input order).  `batch_protein`/`batch_ligand`
 *     must be sorted ascending (they are in scripts/sample_diffusion.py:42,50), expressed here as per-graph counts.
 */
#ifndef TDIFF_H_
#define TDIFF_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define TDIFF_API __attribute__((visibility("default")))
#else
#define TDIFF_API
#endif

#define TDIFF_OK 0
#define TDIFF_EINVAL (-1)   /* bad argument / unsupported configuration */
#define TDIFF_ECUDA (-2)    /* CUDA runtime error (no device, launch failure, out of memory) */
#define TDIFF_ESTATE (-3)   /* call order violated (e.g. forward before bind_batch) */
#define TDIFF_EWEIGHT (-4)  /* missing / mis-shaped state_dict entry */

typedef struct tdiff_engine tdiff_engine;

/* Model hyper-parameters: the keys of reference configs/training.yml:9-42 that shape the network
 * (read at models/molopt_score_model.py:13-33,205-305).  Unsupported values are rejected with TDIFF_EINVAL. */
typedef struct tdiff_config {
  int32_t hidden_dim;        /* 128 (only value supported by the kernels) */
  int32_t n_heads;           /* 16 */
  int32_t num_layers;        /* 9 (any >= 1) */
  int32_t knn;               /* k of the k-NN graph, 1..64 (32 default, 48 stress) */
  int32_t num_r_gaussian;    /* 20 (the reference's fixed offsets, models/common.py:15) */
  int32_t num_classes;       /* ligand_atom_feature_dim, 13 */
  int32_t protein_feat_dim;  /* protein_atom_feature_dim, 27 */
  int32_t num_timesteps;     /* num_diffusion_timesteps, 1000 */
  int32_t model_mean_type;   /* 0 = 'C0' (network predicts x0), 1 = 'noise' (x0 from the predicted displacement,
                              * reference models/molopt_score_model.py:419-422,663-666) */
  int32_t num_blocks;        /* 0 or 1: one block; n > 1: the k-NN graph is rebuilt from the updated coordinates and the SAME layers run
                              * again, n times in total (models/uni_transformer.py:306-321) */
  int32_t ew_net_type;       /* edge gate: 0 'global' (one MLP gate per forward, :312-316), 1 'r' (per sub-layer Linear(r_feat) -> sigmoid,
                              * :58-59,121-122), 2 'm' (x2h: Linear(value) -> sigmoid, h2x: 1, :60-61,123-124), 3 'none' (1) */
  int32_t x2h_out_fc;        /* 1: node_output MLP on [aggregate | h] before the residual (:39-40,80-81) */
  int32_t time_emb;          /* 0: time_emb_dim = 0; 1: time_emb_mode 'simple', one extra ligand input column time_step / T
                              * (models/molopt_score_model.py:319-324); 'sin' cannot run in the reference itself (:325-326) */
  int32_t cutoff_mode;       /* 0 'knn' (models/uni_transformer.py:279-280); 1 'hybrid' (:281-283 -> models/common.py:165-212, add_p_index):
                              * a ligand destination gets every other ligand atom of its graph + its knn nearest protein atoms, protein
                              * destinations keep the k-NN over all atoms.  Needs knn + max ligand atoms per graph - 1 <= 64 slots and
                              * >= knn protein atoms per graph (checked at tdiff_bind_batch).  'radius' is a dead path in the reference */
  int32_t reserved[2];       /* must be 0 */
} tdiff_config;

/* One state_dict entry (reference key name, fp32, host memory).  SURVEY.md Appendix D lists the 384 keys. */
typedef struct tdiff_tensor {
  const char* name;
  const float* data;
  int64_t numel;
} tdiff_tensor;

/* ---- engine life cycle ------------------------------------------------------------------------------
 * Replaces: ScorePosNet3D.__init__ + load_state_dict (models/molopt_score_model.py:200-311,
 * scripts/sample_diffusion.py:158-163).  Copies and re-packs the weights for the kernels (first-layer split of the
 * [128,340] edge-MLP matrices into type / gaussian / h_dst / h_src blocks, transposes for the GEMM B operand). */
TDIFF_API int tdiff_create(const tdiff_config* cfg, const tdiff_tensor* h_state_dict, int n_entries, int device, tdiff_engine** out);
TDIFF_API void tdiff_destroy(tdiff_engine* e);
TDIFF_API const char* tdiff_last_error(void);
TDIFF_API const char* tdiff_version(void);

/* ---- batch binding -----------------------------------------------------------------------------------
 * Replaces: Batch.from_data_list(...).to(device) + center_pos + the step-invariant half of forward
 * (scripts/sample_diffusion.py:42, models/molopt_score_model.py:110-120,333-347).
 * h_protein_counts / h_ligand_counts: atoms per graph [n_graphs].  d_protein_pos [Np,3], d_protein_feat [Np,F] fp32.
 * center_mode: 0 'none', 1 'protein' (subtract the per-graph protein centroid; scatter_mean semantics). */
TDIFF_API int tdiff_bind_batch(tdiff_engine* e, int n_graphs, const int32_t* h_protein_counts, const int32_t* h_ligand_counts,
                     const float* d_protein_pos, const float* d_protein_feat, int center_mode, void* stream);

/* Set the ligand state.  d_ligand_pos [Nl,3] fp32 (lab frame if apply_center!=0, already centred otherwise),
 * d_ligand_v [Nl] int64 class indices (checked < num_classes like models/molopt_score_model.py:125). */
TDIFF_API int tdiff_set_ligand(tdiff_engine* e, const float* d_ligand_pos, const int64_t* d_ligand_v, int apply_center, void* stream);
/* Read the ligand state back; add_offset!=0 adds the pocket centroid (models/molopt_score_model.py:695). */
TDIFF_API int tdiff_get_ligand(tdiff_engine* e, float* d_ligand_pos, int64_t* d_ligand_v, int add_offset, void* stream);
/* Per-graph centring offset [n_graphs,3] (zeros for center_mode 0). */
TDIFF_API int tdiff_get_offset(tdiff_engine* e, float* d_offset, void* stream);

/* Time step of every graph for the next tdiff_forward, as time_step / num_timesteps (fp32, device, [n_graphs]); only read when the
 * engine was created with time_emb = 1 (models/molopt_score_model.py:319-324).  tdiff_sample sets it itself every step. */
TDIFF_API int tdiff_set_time(tdiff_engine* e, const float* d_time_norm, void* stream);

/* ---- one network evaluation ----------------------------------------------------------------------------
 * Replaces: ScorePosNet3D.forward (models/molopt_score_model.py:313-368) for time_emb_dim=0 on the bound batch and
 * current ligand state.  Outputs (any may be NULL): d_pred_pos [Nl,3] (centred frame), d_pred_logits [Nl,K],
 * d_final_h [N,128] (composed node order).  fix_x!=0 freezes coordinates (fetch_embedding, :619-631).
 * Does not modify the ligand state. */
TDIFF_API int tdiff_forward(tdiff_engine* e, float* d_pred_pos, float* d_pred_logits, float* d_final_h, int fix_x, void* stream);

/* Graph of the most recent forward: number of edges, and edge_index as int64 [2,E] (row 0 = src/neighbour,
 * row 1 = dst/query), bit-compatible with PyG knn_graph(flow='source_to_target') (models/uni_transformer.py:280).
 * tdiff_num_edges synchronises the stream. */
TDIFF_API int64_t tdiff_num_edges(tdiff_engine* e, void* stream);
TDIFF_API int tdiff_get_edge_index(tdiff_engine* e, int64_t* d_edge_index, void* stream);
/* Intermediate state of the most recent forward for parity tests: x after layer `layer` ([N,3]); e_w per edge
 * (compacted, [E]). */
TDIFF_API int tdiff_get_edge_weight(tdiff_engine* e, float* d_e_w, void* stream);
TDIFF_API int tdiff_get_node_pos(tdiff_engine* e, float* d_x, void* stream);

/* ---- the sampling loop ---------------------------------------------------------------------------------
 * Replaces: ScorePosNet3D.sample_diffusion's loop body x num_steps (models/molopt_score_model.py:649-693), C0 mode.
 * Time sequence t = T-1 ... T-num_steps (:649).  Noise: if d_pos_noise/d_v_uniform are non-NULL they are the tape
 * ([num_steps,Nl,3] / [num_steps,Nl,K], reference draw order randn_like then rand_like); otherwise counter-based
 * Philox4x32-10 keyed by `seed`.  Trajectory outputs (each may be NULL), written on device, zero host syncs:
 *   d_pos_traj [S,Nl,3] fp32 (lab frame, :691-692), d_v_traj [S,Nl] int64 (:693),
 *   d_v0_traj [S,Nl,K] (log_softmax of logits, :687), d_vt_traj [S,Nl,K] (log posterior, :688).
 * pos_only!=0 keeps atom types fixed (:681).  The ligand state is advanced in place (read it with tdiff_get_ligand).
 * The whole step is captured once into a CUDA graph and replayed. */
TDIFF_API int tdiff_sample(tdiff_engine* e, int num_steps, const float* d_pos_noise, const float* d_v_uniform, uint64_t seed,
                 float* d_pos_traj, int64_t* d_v_traj, float* d_v0_traj, float* d_vt_traj, int pos_only, void* stream);

/* Same loop through HOST buffers (the end-to-end path: H2D of the inputs, the chain, D2H of the results, all on
 * `stream`, synchronised before returning).  Equivalent of the device-facing part of sample_diffusion_ligand
 * (scripts/sample_diffusion.py:42-112) for one batch.  h_out_* may be NULL. */
TDIFF_API int tdiff_sample_host(tdiff_engine* e, int n_graphs, const int32_t* h_protein_counts, const int32_t* h_ligand_counts,
                      const float* h_protein_pos, const float* h_protein_feat, const float* h_ligand_pos,
                      const int64_t* h_ligand_v, int center_mode, int num_steps, const float* h_pos_noise,
                      const float* h_v_uniform, uint64_t seed, float* h_out_pos, int64_t* h_out_v, float* h_pos_traj,
                      int64_t* h_v_traj, float* h_v0_traj, float* h_vt_traj, int pos_only, void* stream);

/* ---- stand-alone graph / scatter operators (the reference's native seam, SURVEY.md 8(b)) ----------------
 * tdiff_knn_graph replaces torch_geometric.nn.knn_graph(x, k, batch, flow='source_to_target')
 * (models/uni_transformer.py:280): d_x [N,3], h_graph_counts [n_graphs] nodes per graph (batch sorted).
 * Outputs: d_src_slots [N*k] int32 (neighbour of node i in slots i*k.., ascending (d2,index), -1 padded when the graph
 * has <= k nodes), d_edge_index int64 [2, *n_edges] compacted (may be NULL).  h_n_edges receives E (synchronises). */
TDIFF_API int tdiff_knn_graph(const float* d_x, int n_nodes, const int32_t* h_graph_counts, int n_graphs, int k,
                    int32_t* d_src_slots, int64_t* d_edge_index, int64_t* h_n_edges, void* stream);

/* Fused scatter_softmax -> scatter_sum over a dst-sorted fixed-degree neighbour list (replaces
 * models/uni_transformer.py:73-83): logits[e,h] = sum_d (q[dst,h,d]*k[e,h,d]/sqrt(8)); alpha = softmax over the
 * edges of dst; out[dst] = h_in[dst] + sum_e alpha*v[e]*e_w[e].   d_k,d_v [N*kk,128], d_q,d_h_in,d_h_out [N,128],
 * d_src_slots [N*kk] (-1 = absent edge), d_e_w [N*kk]. */
TDIFF_API int tdiff_attn_aggregate_h(const float* d_k, const float* d_v, const float* d_e_w, const int32_t* d_src_slots,
                           const float* d_q, const float* d_h_in, float* d_h_out, int n_nodes, int kk, void* stream);
/* Coordinate variant (replaces models/uni_transformer.py:131-140 and :205-206): v [N*kk,16] per-head scalars,
 * message alpha*v*e_w*(x[dst]-x[src]), mean over heads, x_out = x + delta*mask.  d_x, d_x_out [N,3]; d_mask [N] uint8. */
TDIFF_API int tdiff_attn_aggregate_x(const float* d_k, const float* d_v16, const float* d_e_w, const int32_t* d_src_slots,
                           const float* d_q, const float* d_x, const uint8_t* d_mask, float* d_x_out, int n_nodes, int kk,
                           void* stream);
/* scatter_mean(src [M,3], index [M] sorted, dim=0) given per-segment counts (models/molopt_score_model.py:115). */
TDIFF_API int tdiff_scatter_mean3(const float* d_src, const int32_t* h_counts, int n_segments, float* d_out, void* stream);

/* Bond-count stability screen of generated molecules (the step after the sampling path: utils/evaluation/analyze.py:106-143
 * `check_stability`, called per molecule by scripts/evaluate_diffusion.py:78-84).  d_pos [n_atoms,3] fp32, d_atomic_num [n_atoms] int32
 * (atomic numbers, utils/transforms.py `get_atomic_number_from_index`), h_counts [n_mol] atoms per molecule.  Outputs (device):
 * d_nr_bonds [n_atoms] summed bond orders (may be NULL), d_stable_atoms [n_mol], d_mol_stable [n_mol] (1 = every atom stable).
 * hs != 0 requires bonds == valence instead of 0 < bonds <= valence.  An atomic number outside the reference's table -> TDIFF_EINVAL
 * (KeyError in the reference).  Synchronises the stream. */
TDIFF_API int tdiff_check_stability(const float* d_pos, const int32_t* d_atomic_num, const int32_t* h_counts, int n_mol, int hs,
                                    int32_t* d_nr_bonds, int32_t* d_stable_atoms, uint8_t* d_mol_stable, void* stream);

/* ---- binding-affinity regressor ---------------------------------------------------------------------------
 * Replaces: PropPredNet / PropPredNetEnc with the EnEquiEncoder (models/property_pred/prop_model.py:27-165,
 * models/property_pred/prop_egnn.py:8-83), inference only (scripts/property_prediction/inference.py).
 * Kernels are built for hidden_dim 256, act_fn 'relu', norm False, edge_dim 0, num_r_gaussian 2..64, knn 1..64. */
typedef struct tdiff_prop tdiff_prop;

typedef struct tdiff_prop_config {
  int32_t hidden_dim;        /* hidden_channels == encoder.hidden_dim, 256 (only value supported by the kernels) */
  int32_t num_layers;        /* encoder.num_layers, >= 1 (6 in both published configs) */
  int32_t knn;               /* encoder.knn, 1..64 (48) */
  int32_t num_r_gaussian;    /* encoder.num_r_gaussian, 2..64 (64); centres come from encoder.distance_expansion.offset */
  int32_t edge_dim;          /* encoder.edge_dim, must be 0 */
  int32_t norm;              /* encoder.norm, must be 0 */
  int32_t protein_feat_dim;  /* protein_atom_feature_dim (27) */
  int32_t ligand_feat_dim;   /* ligand_atom_feature_dim: width of ligand_atom_feature_full, from the checkpoint */
  int32_t enc_ligand_dim;    /* PropPredNetEnc: columns appended to the ligand features (0 for PropPredNet) */
  int32_t enc_node_dim;      /* PropPredNetEnc: width of enc_node_feature; > 0 adds enc_node_layer */
  int32_t enc_graph_dim;     /* PropPredNetEnc: columns appended to the pooled vector */
  int32_t output_dim;        /* 3 (PropPredNet) or 1 (PropPredNetEnc) */
  int32_t reserved[4];       /* must be 0 */
} tdiff_prop_config;

/* Copies and re-packs the weights (reference key names, fp32 host tensors; the per-layer r_expansion.offset buffers are
 * accepted and ignored, as the reference never reads them).  Without a CUDA device: TDIFF_ECUDA. */
TDIFF_API int tdiff_prop_create(const tdiff_prop_config* cfg, const tdiff_tensor* h_state_dict, int n_entries, int device, tdiff_prop** out);
TDIFF_API void tdiff_prop_destroy(tdiff_prop* p);
/* One forward.  h_protein_counts / h_ligand_counts: atoms per graph [n_graphs] (batch vectors sorted ascending).  Device inputs:
 * d_protein_pos [Np,3], d_protein_feat [Np,protein_feat_dim], d_ligand_pos [Nl,3], d_ligand_feat [Nl,ligand_feat_dim] fp32;
 * nullable like the reference's None: d_enc_ligand [Nl,enc_ligand_dim], d_enc_node [N,enc_node_dim] (composed node order: per graph,
 * protein atoms then ligand atoms, = ScorePosNet3D.fetch_embedding's final_h order), d_enc_graph [n_graphs,enc_graph_dim],
 * d_kind [n_graphs] int64 in 1..output_dim (output_kind; NULL returns every column).  Outputs: d_out [n_graphs,1] with d_kind,
 * [n_graphs,output_dim] without; d_h_out [N,256] the encoder output in composed order (may be NULL).  Deterministic (no atomics).
 * Synchronises the stream (a kind outside 1..output_dim is reported as TDIFF_EINVAL). */
TDIFF_API int tdiff_prop_forward(tdiff_prop* p, int n_graphs, const int32_t* h_protein_counts, const int32_t* h_ligand_counts,
                                 const float* d_protein_pos, const float* d_protein_feat, const float* d_ligand_pos, const float* d_ligand_feat,
                                 const float* d_enc_ligand, const float* d_enc_node, const float* d_enc_graph, const int64_t* d_kind,
                                 float* d_out, float* d_h_out, void* stream);
/* Time (ms, CUDA events) and count of the encoder edge-kernel launches accumulated while profiling is on (enable != 0 resets). */
TDIFF_API int tdiff_prop_profile(tdiff_prop* p, int enable);
TDIFF_API int tdiff_prop_profile_read(tdiff_prop* p, double* ms_edge, int64_t* n_edge_launches, int64_t* n_edge_rows);

/* ---- instrumentation ------------------------------------------------------------------------------------
 * Number of kernel launches issued by this engine since creation (graph replays count their nodes). */
TDIFF_API int64_t tdiff_launch_count(tdiff_engine* e);
/* Edge-MLP execution mode of this engine (env TDIFF_EDGE_MLP at creation): 0 FP32 FFMA ("simt"), 2 tcgen05 bf16x2 split with keys in HBM
 * ("tc3v2"), 3 tcgen05 bf16x3 split ("tc6"), 5 tcgen05 bf16x2 split, gaussian block on the tensor core and attention logits fused into the
 * key-MLP epilogue (default, "tc3"). */
TDIFF_API int tdiff_edge_mlp_mode(tdiff_engine* e);
/* Time (ms, CUDA events on `stream`) and count of the attention-aggregate launches accumulated while profiling is on. */
TDIFF_API int tdiff_profile(tdiff_engine* e, int enable);
TDIFF_API int tdiff_profile_read(tdiff_engine* e, double* ms_aggregate_h, int64_t* n_aggregate_h, double* ms_aggregate_x,
                       int64_t* n_aggregate_x, double* ms_edge_mlp, int64_t* n_edge_mlp, double* ms_total);

#ifdef __cplusplus
}
#endif
#endif /* TDIFF_H_ */
