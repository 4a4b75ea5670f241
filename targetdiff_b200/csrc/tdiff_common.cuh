// tdiff_common.cuh -- shared definitions for the sm_100a kernels of libtdiff.so.
//
// Vocabulary follows the reference: nodes = protein + ligand atoms in `compose_context` order
// (reference models/common.py:120-137), edges = dst-sorted k-NN slots (node i owns slots [i*K, (i+1)*K),
// neighbour index in `src`, -1 = absent), x2h / h2x = the two attention sub-layers
// (reference models/uni_transformer.py:11-140).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define TD_H 128        // hidden_dim
#define TD_HEADS 16     // n_heads
#define TD_HD 8         // head dim
#define TD_NG 20        // num_r_gaussian
#define TD_TAB 21       // per edge type: 20 gaussian rows + 1 constant row (type column + bias)
#define TD_KMAX 64      // max k of the k-NN graph
#define TD_NPROJ 640    // node projection width: [A_k | A_v | B_k | B_v | q_pre]
#define TD_CMAX 24      // max number of ligand classes held in registers by the step epilogue (ligand_atom_mode 'full' has 23)

// One 2-layer edge/node MLP after the exact first-layer split (SURVEY.md Appendix B):
//   pre = P[dst, offA:] + P[src, offB:] + tab[type][20] + sum_j g_j * tab[type][j]      (edge MLPs)
//   hid = relu(LN(pre) * ln_g + ln_b);  out = hid . w2t + b2
struct TdMlp {
  const float* tab;    // [4][TD_TAB][128] (edge MLPs only)
  const float* ln_g;   // [128]
  const float* ln_b;   // [128]
  const float* w2t;    // [128][nout]  (second Linear, transposed: k-major rows)
  const float* b2;     // [nout]
  int nout;            // 128 or 16
  int offA, offB;      // column offsets into the node projection P
  const unsigned char* w2_img;   // nout==128 edge MLPs: second Linear as 3 bf16 pieces in the UMMA K-major SWIZZLE_128B image
  const unsigned char* tabcls_img;   // gaussian/type blocks per destination class: 2 x [128 x 64] in two bf16 pieces, K-major SWIZZLE_128B
                                     // (class 0 = protein destination: types 3 | 1, class 1 = ligand destination: types 2 | 0)
};

// ew_net_type 'r': per-layer gate parameters of both sub-layers and the per-slot outputs (all NULL when unused)
struct TdEwR {
  const float* w_x2h;      // [80] Linear(r_feat -> 1) of the x2h sub-layer (type-major: 20 type + j)
  const float* w_h2x;      // [80] same for h2x
  float b_x2h, b_h2x;
  const float* offsets;    // [20] gaussian centres of the layer
  float coeff;
  float* out_x2h;          // [N*k] gates
  float* out_h2x;
};

struct TdSubLayer {       // x2h or h2x
  const float* wn_t;      // [128][TD_NPROJ] node projection weights (transposed)
  const float* bn;        // [TD_NPROJ] bias (non-zero only in the q_pre block)
  const unsigned char* wn_img;   // the same weights as 5 UMMA images of [128 x 128] (3 bf16 pieces each) for the tensor-core path
  TdMlp k, v, q;          // q.tab unused
  const float* ew_w;      // ew_net_type 'r': [80], 'm' (x2h only): [128]; else NULL
  float ew_b;
  // x2h_out_fc: node_output MLP(256 -> 128 -> 128) on [aggregate | h] (reference models/uni_transformer.py:39-40,80-81)
  const unsigned char* out_wa_img;   // first Linear, columns that multiply the aggregate
  const unsigned char* out_wb_img;   // first Linear, columns that multiply h
  const float* out_b1;               // [128]
  TdMlp out;                         // LayerNorm affine + second Linear (ln_g, ln_b, b2, w2_img)
};

struct TdLayer {
  TdSubLayer x2h, h2x;
  const float* offsets;   // [20] gaussian centres of this layer (distance_expansion.offset)
  float coeff;            // -0.5/(offset[1]-offset[0])^2   (reference models/common.py:17)
};

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// LayerNorm(eps=1e-5, biased variance) + affine + ReLU over 128 features held 4 per lane (features lane+32c).
// Two-pass (mean, then centred second moment), as accurate as the reference's RowwiseMoments at fp32 tolerance.
__device__ __forceinline__ void ln_relu_128(float (&p)[4], const float* __restrict__ g, const float* __restrict__ b, int lane) {
  float s = warp_sum((p[0] + p[1]) + (p[2] + p[3]));
  float mean = s * (1.0f / 128.0f);
  float d0 = p[0] - mean, d1 = p[1] - mean, d2 = p[2] - mean, d3 = p[3] - mean;
  float var = warp_sum((d0 * d0 + d1 * d1) + (d2 * d2 + d3 * d3)) * (1.0f / 128.0f);
  float rstd = 1.0f / sqrtf(var + 1e-5f);
  p[0] = fmaxf(d0 * rstd * g[lane] + b[lane], 0.0f);
  p[1] = fmaxf(d1 * rstd * g[lane + 32] + b[lane + 32], 0.0f);
  p[2] = fmaxf(d2 * rstd * g[lane + 64] + b[lane + 64], 0.0f);
  p[3] = fmaxf(d3 * rstd * g[lane + 96] + b[lane + 96], 0.0f);
}

// ------------------------------------------------------------------------------------------------------
// 128 x NOUT x 128 fp32 tile GEMM out of shared memory (FFMA path).
//   As: [128][TD_LDA] row-major activations, Bs: [128][128] k-major weights.  512 threads:
//   ty = tid/16 (0..31) owns rows ty + 32*i (i<4), tx = tid%16 owns columns 4*tx..4*tx+3 and 64+4*tx..+3.
// ------------------------------------------------------------------------------------------------------
#define TD_LDA 132
#define TD_GEMM_THREADS 512

__device__ __forceinline__ void tile_gemm_128(const float* __restrict__ As, const float* __restrict__ Bs, float (&acc)[4][8],
                                              int ty, int tx) {
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.0f;
#pragma unroll 2
  for (int kk = 0; kk < 128; kk += 4) {
    float4 a[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) a[i] = *reinterpret_cast<const float4*>(As + (ty + 32 * i) * TD_LDA + kk);
#pragma unroll
    for (int k4 = 0; k4 < 4; ++k4) {
      float4 b0 = *reinterpret_cast<const float4*>(Bs + (kk + k4) * 128 + 4 * tx);
      float4 b1 = *reinterpret_cast<const float4*>(Bs + (kk + k4) * 128 + 64 + 4 * tx);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float av = (k4 == 0) ? a[i].x : (k4 == 1) ? a[i].y : (k4 == 2) ? a[i].z : a[i].w;
        acc[i][0] = fmaf(av, b0.x, acc[i][0]);
        acc[i][1] = fmaf(av, b0.y, acc[i][1]);
        acc[i][2] = fmaf(av, b0.z, acc[i][2]);
        acc[i][3] = fmaf(av, b0.w, acc[i][3]);
        acc[i][4] = fmaf(av, b1.x, acc[i][4]);
        acc[i][5] = fmaf(av, b1.y, acc[i][5]);
        acc[i][6] = fmaf(av, b1.z, acc[i][6]);
        acc[i][7] = fmaf(av, b1.w, acc[i][7]);
      }
    }
  }
}

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-DEVICE attribute (one process may own an engine on every GPU): each launcher
// keeps, per kernel, the size it has already opted into on each device.
#define TD_MAX_DEVICES 64
template <class Kernel>
inline void td_opt_in_smem(Kernel kernel, size_t bytes, size_t (&done)[TD_MAX_DEVICES]) {
  int dev = 0;
  const bool known = cudaGetDevice(&dev) == cudaSuccess && dev >= 0 && dev < TD_MAX_DEVICES;
  if (known && bytes <= done[dev]) return;
  cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (known) done[dev] = bytes;
}

// tdiff_last_error() text for entry points outside engine.cu; returns `code`
int td_set_err(int code, const char* fmt, ...);

// Launchers (defined in the .cu files, called by engine.cu).  All asynchronous on `st`.
// `stride` = slots per row (>= k); `hybrid` != 0: ligand rows = other ligand atoms + k nearest protein atoms (prot_ptr required)
void td_launch_knn(const float4* xm, const int* node_ptr, const int* prot_ptr, int n_graphs, int max_nodes_per_graph, int k, int stride, int hybrid,
                   int* src, cudaStream_t st);
void td_launch_knn_cache(const float4* xm, const int* node_ptr, const int* prot_ptr, int n_graphs, int max_ng, int k, unsigned long long* cache,
                         cudaStream_t st);
void td_launch_knn_update(const float4* xm, const int* node_ptr, const int* prot_ptr, int n_graphs, int max_ng, int k, int stride, int hybrid,
                          const unsigned long long* cache, int* src, cudaStream_t st);
void td_launch_edge_const(const float4* xm, const int* src, int* src_prev, int have_prev, int n_nodes, int k, const float* offsets, float coeff,
                          const float* w1t, const float* b1, const float* ln_g, const float* ln_b, const float* w2, float b2,
                          unsigned char* etype, float* e_w, unsigned char* rel_flag, unsigned char* touch_flag, int* work_list, int* n_work,
                          int gate_mode, cudaStream_t st);
void td_launch_dirty_propagate(const unsigned char* in, const int* src, int n_nodes, int k, unsigned char* out, cudaStream_t st);
void td_launch_restore_clean(const unsigned char* dirty, const float4* xm, const float* h_free, int n_nodes, float* h, cudaStream_t st);
void td_launch_rel_rows(const unsigned char* rel_flag, const float4* xm, int n_nodes, const int* lig_rows, int n_lig_rows, int pad, int* rel_rows,
                        int* rel_counts, cudaStream_t st);
void td_launch_protein_embed(const float* feat, int n_protein, int fdim, const float* w, const float* b, const int* prot_node,
                             float* h0, cudaStream_t st);
void td_launch_init_h(const float* h0, const float4* xm, const int* lig_v, const int* node_lig, const float* wl_t, const float* bl,
                      const float* w_time, const float* time_norm, const int* lig_graph, int n_nodes, float* h, cudaStream_t st);
void td_launch_node_proj(const float* h, int n_nodes, const float* wn_t, const float* bn, float* P, cudaStream_t st);
void td_launch_node_q(const float* P, int n_nodes, TdMlp q, float* qout, cudaStream_t st);
void td_launch_edge_mlp(const float* P, const float4* xm, const int* src, const unsigned char* etype, const int* row_nodes,
                        long long n_rows, int k, TdMlp m, const float* offsets, float coeff, float* out, int sm_count, cudaStream_t st);
void td_launch_edge_geom(const float4* xm, const int* src, const unsigned char* etype, int n_nodes, int k, float* dist, const TdEwR& ew, cudaStream_t st);
void td_launch_add_rows(const float* a, const float* b, float* out, long long n_floats, cudaStream_t st);
void td_launch_set_time(const int* step, int t_start, int n_timesteps, int n_graphs, float* time_norm, cudaStream_t st);
void td_launch_edge_mlp_tc(const float* P, const float4* xm, const int* src, const unsigned char* etype, const float* dist,
                           const int* row_nodes, long long n_rows, int k, TdMlp m, const unsigned char* w2_image, int pieces, const float* offsets, float coeff,
                           float* out, int sm_count, cudaStream_t st);
void td_launch_edge_mlp_v4(const float* P, int zero_row, const int* src, const unsigned char* etype, const float* dist, const int* row_nodes, long long n_dst,
                           long long split_dst, const int* d_counts, int k, const TdMlp& m, const float* h_offsets, float coeff,
                           const float* h_ln_g, const float* h_ln_b, const float* h_b2, const float* qnode, float* out, int out_by_slot,
                           const float* agg_logits, const float* agg_e_w, float* agg_h, int key_softmax, int sm_count, cudaStream_t st);
void td_launch_rows_tc(int mode, const float* in, int ldi, int in_off, long long n_rows, TdMlp m, const unsigned char* w_image, int pieces, float* out,
                       int ldo, int nblocks, const int* row_list, const int* d_n_rows, int sm_count, cudaStream_t st);
void td_launch_rel_compact(const unsigned char* flag, int n_nodes, int* rel_list, int* n_rel, cudaStream_t st);
void td_launch_aggregate_h(const float* kbuf, const float* vbuf, const float* e_w, const int* src, const float* q, const float* h_in,
                           float* h_out, int n_nodes, int k, cudaStream_t st);
void td_launch_aggregate_x(const float* kbuf, const float* v16, const float* e_w, const int* src, const float* q, const float4* xm_in,
                           const int* row_nodes, float4* xm_out, int n_rows, int k, cudaStream_t st);
void td_launch_aggregate_h_logits(const float* logits, const float* vbuf, const float* e_w, const int* src, const float* h_in, float* h_out,
                                  int n_nodes, int k, const float* ewm_w, float ewm_b, cudaStream_t st);
void td_launch_aggregate_x_logits(const float* logits, const float* v16, const float* e_w, const int* src, const float4* xm_in,
                                  const int* row_nodes, float4* xm_out, int n_rows, int k, cudaStream_t st);
void td_launch_head(const float* h, const int* lig_node, int n_lig, const float* w1t, const float* b1, const float* w2, const float* b2,
                    int n_classes, float* logits, cudaStream_t st);
void td_launch_check_stability(const float* pos, const int* atomic_num, const int* mol_ptr, int n_mol, int hs, int* nr_bonds, int* stable_atoms,
                               unsigned char* mol_stable, int* err, cudaStream_t st);
