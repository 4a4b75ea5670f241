// engine.cu -- host side of libtdiff.so: the C-ABI of include/tdiff.h, weight re-packing, HBM layout, per-step
// orchestration and CUDA-graph replay.  No torch, no CPU fallback: every entry point needs a CUDA device.
//
// HBM layout of a bound batch (N nodes in compose_context order, K = knn, Nl ligand atoms):
//   xm[2]   float4 [N]      (x, y, z, is_ligand) ping-pong: protein rows identical in both, a layer writes the ligand
//                           rows of the other buffer (models/uni_transformer.py:205-206 updates ligand atoms only)
//   h, h0   fp32 [N,128]    node features / cached protein embedding (step-invariant, models/molopt_score_model.py:333)
//   P       fp32 [N,640]    node projections of the split first layers [A_k | A_v | B_k | B_v | q_pre]
//   q       fp32 [N,128]    query MLP output
//   src     int32 [N*K]     dst-sorted neighbour slots (-1 = absent);  etype uint8 [N*K];  e_w fp32 [N*K]
//   kbuf, vbuf fp32 [N*K,128]; v16 fp32 [Nl*K,16]   per-edge keys / values (h2x uses the first Nl*K rows of kbuf)
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <map>
#include <string>
#include <vector>

#include "../../include/tdiff.h"
#include "sampler.cuh"
#include "tdiff_common.cuh"

static thread_local char g_err[1024] = "";
static int set_err(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
// the same error slot for the entry points defined in other translation units (prop.cu)
int td_set_err(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
#define CK(call)                                                                                       \
  do {                                                                                                 \
    cudaError_t _e = (call);                                                                           \
    if (_e != cudaSuccess) return set_err(TDIFF_ECUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  int ensure(size_t bytes) {
    if (bytes <= cap) return 0;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    size_t want = bytes + bytes / 8 + 256;
    if (cudaMalloc(&p, want) != cudaSuccess) { (void)cudaGetLastError(); if (cudaMalloc(&p, bytes) != cudaSuccess) { (void)cudaGetLastError(); return -1; } want = bytes; }
    cap = want;
    // test switch: fill fresh allocations with 0xFF (NaN floats, negative ints) so that a read of never-written memory shows up in
    // the parity tests instead of depending on what the allocator returns (the GPU test-suite runs with it, tests/conftest.py)
    static const bool poison = getenv("TDIFF_POISON") != nullptr;
    if (poison) cudaMemset(p, 0xFF, want);
    return 0;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
  template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

enum { EV_AGG_H = 0, EV_AGG_X = 1, EV_EDGE_MLP = 2, EV_TOTAL = 3, EV_KINDS = 4 };
struct EvPair { cudaEvent_t a, b; int kind; };

struct tdiff_engine {
  tdiff_config cfg;
  int device = 0, sm_count = 148;
  // ---- weights (one device arena)
  float* arena = nullptr;
  std::vector<float> host_arena;        // host copy of the packed fp32 weights (kernel-argument constants are read from it)
  unsigned char* img_arena = nullptr;   // bf16-split second-layer weights in the tensor-core shared-memory image
  int mlp_mode = 2;                     // 0: FP32 FFMA (edge_mlp.cu), 2: tcgen05 2-piece bf16 split / 3 products (default), 3: 3-piece / 6 products
  bool mlp_v4 = true;                   // mode 2 edge MLPs: edge_mlp_v4.cu (both Linear layers + every edge type's gaussian block on tcgen05) instead of edge_mlp_tc.cu
  std::vector<TdLayer> layers;
  const float *w_prot = nullptr, *b_prot = nullptr, *wl_t = nullptr, *bl = nullptr;
  const float *ew_w1t = nullptr, *ew_b1 = nullptr, *ew_g = nullptr, *ew_b = nullptr, *ew_w2 = nullptr, *ew_off = nullptr;
  float ew_b2 = 0.f, ew_coeff = -0.5f;
  // config-surface options (tdiff_config): blocks, edge-gate flavour, node_output MLP, time embedding
  int num_blocks = 1, ew_mode = 0 /* 0 global, 1 'r', 2 'm', 3 none */, out_fc = 0, time_emb = 0;
  const float* w_time = nullptr;        // time_emb 'simple': the ligand embedding's extra input column
  const float* zeros128 = nullptr;
  DevBuf ew_x2h, ew_h2x, hagg, time_norm;   // 'r' gates per slot (per layer, both sub-layers); x2h aggregate for node_output; t / T per graph
  const float *hd_w1t = nullptr, *hd_b1 = nullptr, *hd_w2 = nullptr, *hd_b2 = nullptr;
  const float *t_c0 = nullptr, *t_ct = nullptr, *t_logvar = nullptr, *t_la = nullptr, *t_l1ma = nullptr, *t_lca = nullptr, *t_l1mca = nullptr,
              *t_sra = nullptr, *t_srm1 = nullptr;
  // ---- batch
  bool bound = false, has_ligand = false, have_graph = false;
  bool restrict_last = false;           // sampling loop only: the last layer's x2h is evaluated for the relevant nodes only
  bool knn_incremental = false;         // protein-protein neighbour keys cached at bind time (TDIFF_KNN_FULL=1 disables)
  bool have_prev = false;               // src_prev / etype / e_w hold the previous forward's graph of this batch (edge_const reuse)
  // developer switches, read from the environment ONCE in tdiff_create (never on the per-layer path)
  bool env_no_fused_agg = false, env_no_restrict = false, env_no_graph = false, env_knn_full = false, env_no_slot_keep = false;
  int B = 0, N = 0, Np = 0, Nl = 0, K = 0, max_ng = 0, final_buf = 0;
  // cutoff_mode 'hybrid': KQ = the configured k (neighbours searched), K = slots per row = KQ + max ligand atoms per graph - 1 (set at
  // bind time); 'knn': K == KQ
  int KQ = 0, hybrid = 0;
  DevBuf node_ptr, prot_ptr, prot_node, prot_graph, lig_node, lig_graph, node_lig;
  DevBuf rel_flag, rel_list, n_rel, work_list, n_work, knn_cache;
  // class-sorted destination lists of the v4 edge kernel: protein destinations (padded with -1 to `row_pad`), then ligand destinations
  DevBuf x2h_rows, lig_rows, rel_rows, rel_counts;
  long long x2h_n_dst = 0, x2h_split = 0, lig_n_dst = 0;
  int row_pad = 4;                      // destinations per class are padded so that class boundaries fall on 128-row tile boundaries
  // Ligand-free cache (exact): protein atoms never move and their embedding is step-invariant, so a protein node that is neither
  // touched by a ligand atom nor (transitively, layer by layer) fed by a touched node has the same features after x2h layer l in
  // every denoising step.  Those values are computed once per bound batch (h_free[l]); per step the first `free_depth` x2h layers
  // only visit the dirty destinations (free_rows[l]) and the clean rows are restored from the cache.
  int free_depth = 0;                   // cached x2h layers of this batch (0 = off)
  int env_free_depth = 2;               // TDIFF_FREE_DEPTH (default 2; 0 disables)
  bool free_ready = false;
  DevBuf h_free, dirty, free_rows, free_counts, lig_save;
  long long free_stride = 0;            // ints per layer in free_rows
  DevBuf xm0, xm1, offset, h0, h, P, q, src, src_prev, etype, e_w, dist, kbuf, vbuf, v16, lig_pos, lig_v, logits;
  DevBuf step, err_flag, node_off, total_edges;
  DevBuf stage[8];   // staging for tdiff_sample_host
  // ---- instrumentation
  cudaStream_t own_stream = nullptr;   // capture stream (the caller's stream may be the legacy default stream, which cannot capture)
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  long long launches = 0;
  bool profiling = false;
  std::vector<EvPair> events;
  double ms_acc[EV_KINDS] = {0, 0, 0, 0};
  long long n_acc[EV_KINDS] = {0, 0, 0, 0};
};

// ---------------------------------------------------------------------------------------------- weights
namespace {
struct Packer {
  std::map<std::string, const tdiff_tensor*> byname;
  std::vector<float> host;
  std::vector<unsigned char> img;
  std::string missing;
  const float* get(const std::string& name, int64_t numel) {
    auto it = byname.find(name);
    if (it == byname.end() || it->second->numel != numel || it->second->data == nullptr) {
      if (missing.empty()) missing = name + (it == byname.end() ? " (absent)" : " (wrong size)");
      return nullptr;
    }
    return it->second->data;
  }
  size_t alloc(size_t n) {   // 256-byte aligned blocks
    size_t off = (host.size() + 63) / 64 * 64;
    host.resize(off + n, 0.0f);
    return off;
  }
};

struct MlpOff { size_t tab, ln_g, ln_b, w2t, b2; int nout; long long img, tabcls; };

// round-to-nearest-even fp32 -> bf16 bit pattern
inline uint16_t bf16_rn(float x) {
  uint32_t u; memcpy(&u, &x, 4);
  if ((u & 0x7fffffffu) > 0x7f800000u) return (uint16_t)((u >> 16) | 0x40);
  u += 0x7fffu + ((u >> 16) & 1u);
  return (uint16_t)(u >> 16);
}
inline float bf16_f(uint16_t b) { uint32_t u = (uint32_t)b << 16; float f; memcpy(&f, &u, 4); return f; }

// W2 [128 out (N), 128 in (K)] -> three bf16 pieces (w = w1 + w2 + w3), each stored as the shared-memory image the UMMA
// descriptor of edge_mlp_tc.cu expects: K-major, SWIZZLE_128B, two K-halves of [128 rows x 128 B], 16-byte chunks XOR row%8.
void pack_umma_image(const float* w2, std::vector<unsigned char>& img, size_t off, int nrows = 128) {
  for (int n = 0; n < nrows; ++n)
    for (int kk = 0; kk < 128; ++kk) {
      float r = w2[(size_t)n * 128 + kk];
      const size_t o = (size_t)(kk / 64) * ((size_t)nrows * 128) + (size_t)n * 128 + (size_t)((((kk % 64) / 8) ^ (n & 7)) * 16) + (size_t)(kk % 8) * 2;
      for (int p = 0; p < 3; ++p) {
        const uint16_t b = bf16_rn(r);
        r = r - bf16_f(b);
        memcpy(&img[off + (size_t)p * ((size_t)nrows * 256) + o], &b, 2);
      }
    }
}

// Gaussian/type blocks as the B operand of the small "pre" MMA of edge_mlp_v4.cu: per destination class one table of
// [128 out (N) x 64 K-slots] in two bf16 pieces, K-major SWIZZLE_128B (128-byte rows, 16-byte chunk index XOR row % 8).
// Class 0 (protein destination): slots 0-31 = type 3 (P->P), 32-63 = type 1 (L->P); class 1 (ligand destination): type 2 (P->L) / type 0 (L->L).
// Inside a 32-slot half: 8*c + i = gaussian 5*c + i (c < 4, i < 5), slot 29 = constant row (type column + bias), all other slots 0.
void pack_tabcls_image(const float* tab /*[4][21][128]*/, std::vector<unsigned char>& img, size_t off) {
  static const int type_of[2][2] = {{3, 1}, {2, 0}};
  for (int cls = 0; cls < 2; ++cls)
    for (int n = 0; n < 128; ++n)
      for (int slot = 0; slot < 64; ++slot) {
        const int half = slot >> 5, sl = slot & 31;
        int j = -1;
        if ((sl & 7) < 5) j = 5 * (sl >> 3) + (sl & 7);
        else if (sl == 29) j = 20;
        float r = j >= 0 ? tab[((size_t)type_of[cls][half] * TD_TAB + j) * TD_H + n] : 0.0f;
        const size_t o = (size_t)n * 128 + (size_t)(((slot >> 3) ^ (n & 7)) * 16) + (size_t)(slot & 7) * 2;
        for (int p = 0; p < 2; ++p) {
          const uint16_t b = bf16_rn(r);
          r = r - bf16_f(b);
          memcpy(&img[off + (size_t)cls * 32768 + (size_t)p * 16384 + o], &b, 2);
        }
      }
}

// edge MLP: first Linear [128, 4 + 80 + 128 + 128] split, LayerNorm affine, second Linear transposed
bool pack_edge_mlp(Packer& pk, const std::string& p, int nout, MlpOff& o, const float** w1_out) {
  const int KV = 4 + 4 * TD_NG + 2 * TD_H;
  const float* w1 = pk.get(p + ".net.0.weight", (int64_t)TD_H * KV);
  const float* b1 = pk.get(p + ".net.0.bias", TD_H);
  const float* g = pk.get(p + ".net.1.weight", TD_H);
  const float* b = pk.get(p + ".net.1.bias", TD_H);
  const float* w2 = pk.get(p + ".net.3.weight", (int64_t)nout * TD_H);
  const float* b2 = pk.get(p + ".net.3.bias", nout);
  if (!w1 || !b1 || !g || !b || !w2 || !b2) return false;
  o.nout = nout;
  o.tab = pk.alloc(4 * TD_TAB * TD_H);
  for (int t = 0; t < 4; ++t) {
    for (int j = 0; j < TD_NG; ++j)
      for (int f = 0; f < TD_H; ++f) pk.host[o.tab + (t * TD_TAB + j) * TD_H + f] = w1[(size_t)f * KV + 4 + t * TD_NG + j];
    for (int f = 0; f < TD_H; ++f) pk.host[o.tab + (t * TD_TAB + TD_NG) * TD_H + f] = w1[(size_t)f * KV + t] + b1[f];
  }
  o.ln_g = pk.alloc(TD_H); memcpy(&pk.host[o.ln_g], g, TD_H * sizeof(float));
  o.ln_b = pk.alloc(TD_H); memcpy(&pk.host[o.ln_b], b, TD_H * sizeof(float));
  o.w2t = pk.alloc((size_t)TD_H * nout);
  for (int kk = 0; kk < TD_H; ++kk)
    for (int n = 0; n < nout; ++n) pk.host[o.w2t + (size_t)kk * nout + n] = w2[(size_t)n * TD_H + kk];
  o.b2 = pk.alloc(nout); memcpy(&pk.host[o.b2], b2, nout * sizeof(float));
  o.img = -1; o.tabcls = -1;
  if (nout == TD_H || nout == 16) {
    o.img = (long long)pk.img.size();
    pk.img.resize(pk.img.size() + 3 * (size_t)nout * 256, 0);
    pack_umma_image(w2, pk.img, (size_t)o.img, nout);
    o.tabcls = (long long)pk.img.size();
    pk.img.resize(pk.img.size() + 2 * 32768, 0);
    pack_tabcls_image(&pk.host[o.tab], pk.img, (size_t)o.tabcls);
  }
  *w1_out = w1;
  return true;
}

struct SubOff {
  size_t wn_t, bn; long long wn_img; MlpOff k, v, q;
  long long ew_w = -1; float ew_b = 0.f;                       // ew_net_type 'r' / 'm'
  long long out_wa = -1, out_wb = -1, out_w2 = -1, out_b1 = -1, out_g = -1, out_b = -1, out_b2 = -1;   // x2h_out_fc node_output MLP
};

// optional per-sub-layer parameters: the 'r' / 'm' gate Linear and the node_output MLP (reference models/uni_transformer.py:34-40)
bool pack_sublayer_options(Packer& pk, const std::string& p, int ew_dim, bool out_fc, SubOff& so) {
  if (ew_dim > 0) {
    const float* w = pk.get(p + ".ew_net.0.weight", ew_dim);
    const float* b = pk.get(p + ".ew_net.0.bias", 1);
    if (!w || !b) return false;
    so.ew_w = (long long)pk.alloc(ew_dim);
    memcpy(&pk.host[so.ew_w], w, ew_dim * sizeof(float));
    so.ew_b = b[0];
  }
  if (out_fc) {
    const std::string np = p + ".node_output";
    const float* w1 = pk.get(np + ".net.0.weight", (int64_t)TD_H * 2 * TD_H);
    const float* b1 = pk.get(np + ".net.0.bias", TD_H);
    const float* g = pk.get(np + ".net.1.weight", TD_H);
    const float* b = pk.get(np + ".net.1.bias", TD_H);
    const float* w2 = pk.get(np + ".net.3.weight", (int64_t)TD_H * TD_H);
    const float* b2 = pk.get(np + ".net.3.bias", TD_H);
    if (!w1 || !b1 || !g || !b || !w2 || !b2) return false;
    std::vector<float> blk((size_t)TD_H * TD_H);
    for (int half = 0; half < 2; ++half) {                     // input columns [aggregate | h]
      for (int n = 0; n < TD_H; ++n)
        for (int kk = 0; kk < TD_H; ++kk) blk[(size_t)n * TD_H + kk] = w1[(size_t)n * 2 * TD_H + half * TD_H + kk];
      long long& dst = half == 0 ? so.out_wa : so.out_wb;
      dst = (long long)pk.img.size();
      pk.img.resize(pk.img.size() + 3 * 32768, 0);
      pack_umma_image(blk.data(), pk.img, (size_t)dst);
    }
    so.out_w2 = (long long)pk.img.size();
    pk.img.resize(pk.img.size() + 3 * 32768, 0);
    pack_umma_image(w2, pk.img, (size_t)so.out_w2);
    so.out_b1 = (long long)pk.alloc(TD_H); memcpy(&pk.host[so.out_b1], b1, TD_H * 4);
    so.out_g = (long long)pk.alloc(TD_H); memcpy(&pk.host[so.out_g], g, TD_H * 4);
    so.out_b = (long long)pk.alloc(TD_H); memcpy(&pk.host[so.out_b], b, TD_H * 4);
    so.out_b2 = (long long)pk.alloc(TD_H); memcpy(&pk.host[so.out_b2], b2, TD_H * 4);
  }
  return true;
}

bool pack_sublayer(Packer& pk, const std::string& p, const char* kn, const char* vn, const char* qn, int nout_v, SubOff& so) {
  const int KV = 4 + 4 * TD_NG + 2 * TD_H;
  const float *w1k = nullptr, *w1v = nullptr;
  if (!pack_edge_mlp(pk, p + "." + kn, TD_H, so.k, &w1k)) return false;
  if (!pack_edge_mlp(pk, p + "." + vn, nout_v, so.v, &w1v)) return false;
  const std::string qp = p + "." + qn;
  const float* w1q = pk.get(qp + ".net.0.weight", (int64_t)TD_H * TD_H);
  const float* b1q = pk.get(qp + ".net.0.bias", TD_H);
  const float* gq = pk.get(qp + ".net.1.weight", TD_H);
  const float* bq = pk.get(qp + ".net.1.bias", TD_H);
  const float* w2q = pk.get(qp + ".net.3.weight", (int64_t)TD_H * TD_H);
  const float* b2q = pk.get(qp + ".net.3.bias", TD_H);
  if (!w1q || !b1q || !gq || !bq || !w2q || !b2q) return false;
  so.q.nout = TD_H; so.q.tab = 0; so.q.tabcls = -1;
  so.q.img = (long long)pk.img.size();
  pk.img.resize(pk.img.size() + 3 * 32768, 0);
  pack_umma_image(w2q, pk.img, (size_t)so.q.img);
  so.q.ln_g = pk.alloc(TD_H); memcpy(&pk.host[so.q.ln_g], gq, TD_H * sizeof(float));
  so.q.ln_b = pk.alloc(TD_H); memcpy(&pk.host[so.q.ln_b], bq, TD_H * sizeof(float));
  so.q.w2t = pk.alloc((size_t)TD_H * TD_H);
  for (int kk = 0; kk < TD_H; ++kk)
    for (int n = 0; n < TD_H; ++n) pk.host[so.q.w2t + (size_t)kk * TD_H + n] = w2q[(size_t)n * TD_H + kk];
  so.q.b2 = pk.alloc(TD_H); memcpy(&pk.host[so.q.b2], b2q, TD_H * sizeof(float));
  so.wn_t = pk.alloc((size_t)TD_H * TD_NPROJ);
  so.bn = pk.alloc(TD_NPROJ);
  for (int kk = 0; kk < TD_H; ++kk) {
    float* row = &pk.host[so.wn_t + (size_t)kk * TD_NPROJ];
    for (int c = 0; c < TD_H; ++c) {
      row[c] = w1k[(size_t)c * KV + 4 + 4 * TD_NG + kk];                 // A_k: h[dst] block of hk/xk
      row[128 + c] = w1v[(size_t)c * KV + 4 + 4 * TD_NG + kk];           // A_v
      row[256 + c] = w1k[(size_t)c * KV + 4 + 4 * TD_NG + TD_H + kk];    // B_k: h[src] block
      row[384 + c] = w1v[(size_t)c * KV + 4 + 4 * TD_NG + TD_H + kk];    // B_v
      row[512 + c] = w1q[(size_t)c * TD_H + kk];                         // q first Linear
    }
  }
  for (int c = 0; c < TD_H; ++c) pk.host[so.bn + 512 + c] = b1q[c];
  // tensor-core images of the five 128-column blocks of the node projection
  so.wn_img = (long long)pk.img.size();
  pk.img.resize(pk.img.size() + 5 * 3 * 32768, 0);
  std::vector<float> blk((size_t)TD_H * TD_H);
  for (int y = 0; y < 5; ++y) {
    for (int n = 0; n < TD_H; ++n)
      for (int kk = 0; kk < TD_H; ++kk) blk[(size_t)n * TD_H + kk] = pk.host[so.wn_t + (size_t)kk * TD_NPROJ + y * TD_H + n];
    pack_umma_image(blk.data(), pk.img, (size_t)so.wn_img + (size_t)y * 3 * 32768);
  }
  return true;
}

TdMlp mk_mlp(const float* base, const unsigned char* img_base, const MlpOff& o, int offA, int offB) {
  TdMlp m;
  m.w2_img = (o.img >= 0 && img_base) ? img_base + o.img : nullptr;
  m.tabcls_img = (o.tabcls >= 0 && img_base) ? img_base + o.tabcls : nullptr;
  m.tab = base + o.tab; m.ln_g = base + o.ln_g; m.ln_b = base + o.ln_b; m.w2t = base + o.w2t; m.b2 = base + o.b2;
  m.nout = o.nout; m.offA = offA; m.offB = offB;
  return m;
}
}  // namespace

extern "C" const char* tdiff_last_error(void) { return g_err; }
extern "C" const char* tdiff_version(void) { return "tdiff-b200 0.1 (sm_100a)"; }

extern "C" int tdiff_create(const tdiff_config* cfg, const tdiff_tensor* sd, int n_entries, int device, tdiff_engine** out) {
  if (!cfg || !sd || !out) return set_err(TDIFF_EINVAL, "null argument");
  *out = nullptr;
  if (cfg->hidden_dim != TD_H || cfg->n_heads != TD_HEADS || cfg->num_r_gaussian != TD_NG)
    return set_err(TDIFF_EINVAL, "unsupported model shape: hidden_dim=%d n_heads=%d num_r_gaussian=%d (kernels are built for 128/16/20)",
                   cfg->hidden_dim, cfg->n_heads, cfg->num_r_gaussian);
  if (cfg->knn < 1 || cfg->knn > TD_KMAX) return set_err(TDIFF_EINVAL, "knn=%d outside 1..%d", cfg->knn, TD_KMAX);
  if (cfg->model_mean_type != 0 && cfg->model_mean_type != 1)
    return set_err(TDIFF_EINVAL, "model_mean_type=%d (0 = C0, 1 = noise)", cfg->model_mean_type);
  for (int r : cfg->reserved)
    if (r != 0) return set_err(TDIFF_EINVAL, "tdiff_config.reserved must be 0");
  if (cfg->cutoff_mode != 0 && cfg->cutoff_mode != 1) return set_err(TDIFF_EINVAL, "cutoff_mode=%d (0 = 'knn', 1 = 'hybrid')", cfg->cutoff_mode);
  if (cfg->num_blocks < 0 || cfg->num_blocks > 16 || cfg->ew_net_type < 0 || cfg->ew_net_type > 3 || (cfg->x2h_out_fc != 0 && cfg->x2h_out_fc != 1) ||
      (cfg->time_emb != 0 && cfg->time_emb != 1))
    return set_err(TDIFF_EINVAL, "bad option (num_blocks=%d ew_net_type=%d x2h_out_fc=%d time_emb=%d)", cfg->num_blocks, cfg->ew_net_type,
                   cfg->x2h_out_fc, cfg->time_emb);
  if (cfg->num_layers < 1 || cfg->num_classes < 1 || cfg->num_classes > TD_CMAX || cfg->protein_feat_dim < 1 || cfg->num_timesteps < 1)
    return set_err(TDIFF_EINVAL, "bad config (num_layers=%d num_classes=%d protein_feat_dim=%d num_timesteps=%d)", cfg->num_layers,
                   cfg->num_classes, cfg->protein_feat_dim, cfg->num_timesteps);
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    (void)cudaGetLastError();
    return set_err(TDIFF_ECUDA, "no CUDA device: libtdiff has no CPU fallback");
  }
  if (device < 0 || device >= ndev) return set_err(TDIFF_EINVAL, "device %d out of range (%d devices)", device, ndev);
  CK(cudaSetDevice(device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) return set_err(TDIFF_ECUDA, "device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);

  tdiff_engine* e = new tdiff_engine();
  e->cfg = *cfg; e->device = device; e->sm_count = prop.multiProcessorCount; e->K = e->KQ = cfg->knn; e->hybrid = cfg->cutoff_mode;
  e->num_blocks = cfg->num_blocks > 1 ? cfg->num_blocks : 1; e->ew_mode = cfg->ew_net_type; e->out_fc = cfg->x2h_out_fc; e->time_emb = cfg->time_emb;

  Packer pk;
  for (int i = 0; i < n_entries; ++i)
    if (sd[i].name) pk.byname[sd[i].name] = &sd[i];
  const int T = cfg->num_timesteps, KC = cfg->num_classes, F = cfg->protein_feat_dim, L = cfg->num_layers;
  struct { const char* name; size_t off; } tabs[9] = {{"posterior_mean_c0_coef", 0}, {"posterior_mean_ct_coef", 0}, {"posterior_logvar", 0},
      {"log_alphas_v", 0}, {"log_one_minus_alphas_v", 0}, {"log_alphas_cumprod_v", 0}, {"log_one_minus_alphas_cumprod_v", 0},
      {"sqrt_recip_alphas_cumprod", 0}, {"sqrt_recipm1_alphas_cumprod", 0}};
  for (auto& t : tabs) {
    const float* p = pk.get(t.name, T);
    t.off = pk.alloc(T);
    if (p) memcpy(&pk.host[t.off], p, T * sizeof(float));
  }
  // embeddings
  const float* wp = pk.get("protein_atom_emb.weight", (int64_t)(TD_H - 1) * F);
  const float* bp = pk.get("protein_atom_emb.bias", TD_H - 1);
  const int KIN = KC + (cfg->time_emb ? 1 : 0);           // ligand embedding input width: classes (+ the time column)
  const float* wl = pk.get("ligand_atom_emb.weight", (int64_t)(TD_H - 1) * KIN);
  const float* blp = pk.get("ligand_atom_emb.bias", TD_H - 1);
  size_t o_wp = pk.alloc((size_t)TD_H * F), o_bp = pk.alloc(TD_H), o_wl = pk.alloc((size_t)KC * TD_H), o_bl = pk.alloc(TD_H),
         o_wtime = pk.alloc(TD_H), o_zeros = pk.alloc(TD_H);
  if (wp && bp && wl && blp) {
    memcpy(&pk.host[o_wp], wp, (size_t)(TD_H - 1) * F * sizeof(float));
    memcpy(&pk.host[o_bp], bp, (TD_H - 1) * sizeof(float));
    for (int v = 0; v < KC; ++v)
      for (int f = 0; f < TD_H - 1; ++f) pk.host[o_wl + (size_t)v * TD_H + f] = wl[(size_t)f * KIN + v];
    if (cfg->time_emb)
      for (int f = 0; f < TD_H - 1; ++f) pk.host[o_wtime + f] = wl[(size_t)f * KIN + KC];
    memcpy(&pk.host[o_bl], blp, (TD_H - 1) * sizeof(float));
  }
  // global edge gate (models/uni_transformer.py:242-243,312-316)
  const bool has_gate = cfg->ew_net_type == 0;            // the edge_pred_layer only exists for ew_net_type 'global' (uni_transformer.py:242-243)
  const float* gw1 = has_gate ? pk.get("refine_net.edge_pred_layer.net.0.weight", (int64_t)TD_H * TD_NG) : nullptr;
  const float* gb1 = has_gate ? pk.get("refine_net.edge_pred_layer.net.0.bias", TD_H) : nullptr;
  const float* gg = has_gate ? pk.get("refine_net.edge_pred_layer.net.1.weight", TD_H) : nullptr;
  const float* gb = has_gate ? pk.get("refine_net.edge_pred_layer.net.1.bias", TD_H) : nullptr;
  const float* gw2 = has_gate ? pk.get("refine_net.edge_pred_layer.net.3.weight", TD_H) : nullptr;
  const float* gb2 = has_gate ? pk.get("refine_net.edge_pred_layer.net.3.bias", 1) : nullptr;
  const float* goff = pk.get("refine_net.distance_expansion.offset", TD_NG);
  size_t o_gw1 = pk.alloc((size_t)TD_NG * TD_H), o_gb1 = pk.alloc(TD_H), o_gg = pk.alloc(TD_H), o_gb = pk.alloc(TD_H), o_gw2 = pk.alloc(TD_H),
         o_goff = pk.alloc(TD_NG);
  if (goff) memcpy(&pk.host[o_goff], goff, TD_NG * 4);
  if (gw1 && gb1 && gg && gb && gw2 && gb2 && goff) {
    for (int j = 0; j < TD_NG; ++j)
      for (int f = 0; f < TD_H; ++f) pk.host[o_gw1 + (size_t)j * TD_H + f] = gw1[(size_t)f * TD_NG + j];
    memcpy(&pk.host[o_gb1], gb1, TD_H * 4); memcpy(&pk.host[o_gg], gg, TD_H * 4); memcpy(&pk.host[o_gb], gb, TD_H * 4);
    memcpy(&pk.host[o_gw2], gw2, TD_H * 4); memcpy(&pk.host[o_goff], goff, TD_NG * 4);
    e->ew_b2 = gb2[0];
    const float d = goff[1] - goff[0];
    e->ew_coeff = -0.5f / (d * d);
  }
  // head
  const float* hw1 = pk.get("v_inference.0.weight", (int64_t)TD_H * TD_H);
  const float* hb1 = pk.get("v_inference.0.bias", TD_H);
  const float* hw2 = pk.get("v_inference.2.weight", (int64_t)KC * TD_H);
  const float* hb2 = pk.get("v_inference.2.bias", KC);
  size_t o_hw1 = pk.alloc((size_t)TD_H * TD_H), o_hb1 = pk.alloc(TD_H), o_hw2 = pk.alloc((size_t)KC * TD_H), o_hb2 = pk.alloc(KC);
  if (hw1 && hb1 && hw2 && hb2) {
    for (int kk = 0; kk < TD_H; ++kk)
      for (int n = 0; n < TD_H; ++n) pk.host[o_hw1 + (size_t)kk * TD_H + n] = hw1[(size_t)n * TD_H + kk];
    memcpy(&pk.host[o_hb1], hb1, TD_H * 4); memcpy(&pk.host[o_hw2], hw2, (size_t)KC * TD_H * 4); memcpy(&pk.host[o_hb2], hb2, KC * 4);
  }
  // attention layers
  std::vector<SubOff> sx(L), sh(L);
  std::vector<size_t> o_off(L);
  std::vector<float> coeffs(L, -0.5f);
  for (int l = 0; l < L; ++l) {
    const std::string p = "refine_net.base_block." + std::to_string(l);
    if (!pack_sublayer(pk, p + ".x2h_layers.0", "hk_func", "hv_func", "hq_func", TD_H, sx[l])) break;
    if (!pack_sublayer(pk, p + ".h2x_layers.0", "xk_func", "xv_func", "xq_func", TD_HEADS, sh[l])) break;
    if (!pack_sublayer_options(pk, p + ".x2h_layers.0", cfg->ew_net_type == 1 ? 4 * TD_NG : cfg->ew_net_type == 2 ? TD_H : 0, cfg->x2h_out_fc != 0, sx[l])) break;
    if (!pack_sublayer_options(pk, p + ".h2x_layers.0", cfg->ew_net_type == 1 ? 4 * TD_NG : 0, false, sh[l])) break;
    const float* off = pk.get(p + ".distance_expansion.offset", TD_NG);
    o_off[l] = pk.alloc(TD_NG);
    if (off) {
      memcpy(&pk.host[o_off[l]], off, TD_NG * 4);
      const float d = off[1] - off[0];
      coeffs[l] = -0.5f / (d * d);
    }
  }
  if (!pk.missing.empty()) {
    delete e;
    return set_err(TDIFF_EWEIGHT, "state_dict entry %s", pk.missing.c_str());
  }
  const size_t bytes = pk.host.size() * sizeof(float);
  if (cudaMalloc(&e->arena, bytes) != cudaSuccess) { delete e; return set_err(TDIFF_ECUDA, "cudaMalloc(%zu) for weights failed", bytes); }
  if (cudaMemcpy(e->arena, pk.host.data(), bytes, cudaMemcpyHostToDevice) != cudaSuccess) {
    cudaFree(e->arena); delete e; return set_err(TDIFF_ECUDA, "weight upload failed");
  }
  if (!pk.img.empty()) {
    if (cudaMalloc(&e->img_arena, pk.img.size()) != cudaSuccess ||
        cudaMemcpy(e->img_arena, pk.img.data(), pk.img.size(), cudaMemcpyHostToDevice) != cudaSuccess) {
      cudaFree(e->arena); delete e; return set_err(TDIFF_ECUDA, "weight image upload failed");
    }
  }
  if (const char* mode = getenv("TDIFF_EDGE_MLP")) {
    if (!strcmp(mode, "simt")) e->mlp_mode = 0;
    else if (!strcmp(mode, "tc3")) e->mlp_mode = 2;
    else if (!strcmp(mode, "tc3v2")) { e->mlp_mode = 2; e->mlp_v4 = false; }
    else if (!strcmp(mode, "tc6")) e->mlp_mode = 3;
    else { cudaFree(e->arena); cudaFree(e->img_arena); delete e; return set_err(TDIFF_EINVAL, "TDIFF_EDGE_MLP=%s (simt|tc3|tc3v2|tc6)", mode); }
  }
  if ((cfg->ew_net_type != 0 || cfg->x2h_out_fc || cfg->cutoff_mode != 0) && !(e->mlp_mode == 2 && e->mlp_v4)) {
    cudaFree(e->arena); cudaFree(e->img_arena); delete e;
    return set_err(TDIFF_EINVAL, "ew_net_type != 'global', x2h_out_fc and cutoff_mode 'hybrid' are implemented (and tested) in the default engine mode only (unset TDIFF_EDGE_MLP)");
  }
  e->env_no_fused_agg = getenv("TDIFF_NO_FUSED_AGG") != nullptr;
  e->env_no_restrict = getenv("TDIFF_NO_RESTRICT") != nullptr;
  e->env_no_graph = getenv("TDIFF_NO_GRAPH") != nullptr;
  e->env_knn_full = getenv("TDIFF_KNN_FULL") != nullptr;
  e->env_no_slot_keep = getenv("TDIFF_NO_SLOT_KEEP") != nullptr;
  if (const char* fd = getenv("TDIFF_FREE_DEPTH")) e->env_free_depth = atoi(fd) < 0 ? 0 : (atoi(fd) > 8 ? 8 : atoi(fd));
  e->host_arena = pk.host;
  const float* A = e->arena;
  const unsigned char* IM = e->img_arena;
  e->t_c0 = A + tabs[0].off; e->t_ct = A + tabs[1].off; e->t_logvar = A + tabs[2].off; e->t_la = A + tabs[3].off;
  e->t_l1ma = A + tabs[4].off; e->t_lca = A + tabs[5].off; e->t_l1mca = A + tabs[6].off;
  e->t_sra = A + tabs[7].off; e->t_srm1 = A + tabs[8].off;
  e->w_prot = A + o_wp; e->b_prot = A + o_bp; e->wl_t = A + o_wl; e->bl = A + o_bl;
  e->w_time = cfg->time_emb ? A + o_wtime : nullptr; e->zeros128 = A + o_zeros;
  e->ew_w1t = A + o_gw1; e->ew_b1 = A + o_gb1; e->ew_g = A + o_gg; e->ew_b = A + o_gb; e->ew_w2 = A + o_gw2; e->ew_off = A + o_goff;
  e->hd_w1t = A + o_hw1; e->hd_b1 = A + o_hb1; e->hd_w2 = A + o_hw2; e->hd_b2 = A + o_hb2;
  e->layers.resize(L);
  for (int l = 0; l < L; ++l) {
    TdLayer& ly = e->layers[l];
    ly.offsets = A + o_off[l]; ly.coeff = coeffs[l];
    ly.x2h.wn_t = A + sx[l].wn_t; ly.x2h.bn = A + sx[l].bn; ly.x2h.wn_img = IM ? IM + sx[l].wn_img : nullptr;
    ly.x2h.k = mk_mlp(A, IM, sx[l].k, 0, 256); ly.x2h.v = mk_mlp(A, IM, sx[l].v, 128, 384); ly.x2h.q = mk_mlp(A, IM, sx[l].q, 512, 512);
    ly.h2x.wn_t = A + sh[l].wn_t; ly.h2x.bn = A + sh[l].bn; ly.h2x.wn_img = IM ? IM + sh[l].wn_img : nullptr;
    ly.h2x.k = mk_mlp(A, IM, sh[l].k, 0, 256); ly.h2x.v = mk_mlp(A, IM, sh[l].v, 128, 384); ly.h2x.q = mk_mlp(A, IM, sh[l].q, 512, 512);
    for (int sub = 0; sub < 2; ++sub) {
      TdSubLayer& sl = sub ? ly.h2x : ly.x2h;
      const SubOff& so = sub ? sh[l] : sx[l];
      sl.ew_w = so.ew_w >= 0 ? A + so.ew_w : nullptr; sl.ew_b = so.ew_b;
      sl.out_wa_img = so.out_wa >= 0 ? IM + so.out_wa : nullptr; sl.out_wb_img = so.out_wb >= 0 ? IM + so.out_wb : nullptr;
      sl.out_b1 = so.out_b1 >= 0 ? A + so.out_b1 : nullptr;
      memset(&sl.out, 0, sizeof(sl.out));
      if (so.out_w2 >= 0) {
        sl.out.w2_img = IM + so.out_w2; sl.out.ln_g = A + so.out_g; sl.out.ln_b = A + so.out_b; sl.out.b2 = A + so.out_b2; sl.out.nout = TD_H;
      }
    }
  }
  if (e->step.ensure(sizeof(int)) || e->err_flag.ensure(sizeof(int)) || e->total_edges.ensure(sizeof(long long))) {
    tdiff_destroy(e); return set_err(TDIFF_ECUDA, "cudaMalloc failed");
  }
  cudaMemset(e->err_flag.p, 0, sizeof(int));
  if (cudaStreamCreateWithFlags(&e->own_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&e->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&e->ev_join, cudaEventDisableTiming) != cudaSuccess) {
    tdiff_destroy(e); return set_err(TDIFF_ECUDA, "stream/event creation failed");
  }
  *out = e;
  return TDIFF_OK;
}

extern "C" void tdiff_destroy(tdiff_engine* e) {
  if (!e) return;
  cudaSetDevice(e->device);
  for (auto& ev : e->events) { cudaEventDestroy(ev.a); cudaEventDestroy(ev.b); }
  if (e->own_stream) cudaStreamDestroy(e->own_stream);
  if (e->ev_fork) cudaEventDestroy(e->ev_fork);
  if (e->ev_join) cudaEventDestroy(e->ev_join);
  DevBuf* bufs[] = {&e->node_ptr, &e->prot_ptr, &e->prot_node, &e->prot_graph, &e->lig_node, &e->lig_graph, &e->node_lig, &e->xm0, &e->xm1,
                    &e->rel_flag, &e->rel_list, &e->n_rel, &e->work_list, &e->n_work, &e->knn_cache, &e->x2h_rows, &e->lig_rows, &e->rel_rows, &e->rel_counts, &e->ew_x2h, &e->ew_h2x, &e->hagg, &e->time_norm, &e->h_free, &e->dirty, &e->free_rows, &e->free_counts, &e->lig_save, &e->offset, &e->h0, &e->h, &e->P, &e->q, &e->src, &e->src_prev, &e->etype, &e->e_w, &e->dist, &e->kbuf, &e->vbuf, &e->v16, &e->lig_pos,
                    &e->lig_v, &e->logits, &e->step, &e->err_flag, &e->node_off, &e->total_edges};
  for (auto* b : bufs) b->release();
  for (auto& b : e->stage) b.release();
  if (e->arena) cudaFree(e->arena);
  if (e->img_arena) cudaFree(e->img_arena);
  delete e;
}

// ---------------------------------------------------------------------------------------------- batch binding
extern "C" int tdiff_bind_batch(tdiff_engine* e, int B, const int32_t* pc, const int32_t* lc, const float* d_ppos, const float* d_pfeat,
                                int center_mode, void* stream) {
  if (!e || !pc || !lc || B < 1) return set_err(TDIFF_EINVAL, "bind_batch: bad arguments");
  if (center_mode != 0 && center_mode != 1) return set_err(TDIFF_EINVAL, "center_mode %d (0 'none' | 1 'protein')", center_mode);
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaSetDevice(e->device));
  long long N = 0, Np = 0, Nl = 0;
  int max_ng = 0;
  for (int g = 0; g < B; ++g) {
    if (pc[g] < 0 || lc[g] < 0) return set_err(TDIFF_EINVAL, "negative atom count in graph %d", g);
    Np += pc[g]; Nl += lc[g];
    if (pc[g] + lc[g] > max_ng) max_ng = pc[g] + lc[g];
  }
  N = Np + Nl;
  if (N <= 0) return set_err(TDIFF_EINVAL, "empty batch");
  if (e->hybrid) {
    // reference models/common.py:165-212: a ligand destination has (n_ligand - 1) ligand neighbours + k protein neighbours (torch.topk
    // raises when a graph has fewer than k protein atoms); the slot rows are sized for the largest ligand of the batch
    int max_lc = 0;
    for (int g = 0; g < B; ++g) {
      if (lc[g] > max_lc) max_lc = lc[g];
      if (lc[g] > 0 && pc[g] < e->KQ)
        return set_err(TDIFF_EINVAL, "cutoff_mode 'hybrid': graph %d has %d protein atoms < k = %d (torch.topk fails in the reference too)", g, pc[g], e->KQ);
    }
    const int need = e->KQ + (max_lc > 0 ? max_lc - 1 : 0);
    if (need > TD_KMAX)
      return set_err(TDIFF_EINVAL, "cutoff_mode 'hybrid': k + n_ligand - 1 = %d + %d - 1 exceeds the %d neighbour slots per node", e->KQ, max_lc, TD_KMAX);
    e->K = need;
  }
  if (N * (long long)e->K >= (1LL << 31) / 1) return set_err(TDIFF_EINVAL, "batch too large: N*k = %lld edge slots", N * e->K);
  if (max_ng > 2800) return set_err(TDIFF_EINVAL, "graph with %d nodes exceeds the k-NN kernel's shared-memory tile (2800)", max_ng);
  if (Np > 0 && (!d_ppos || !d_pfeat)) return set_err(TDIFF_EINVAL, "null protein arrays");
  const int K = e->K;
  std::vector<int> node_ptr(B + 1), prot_ptr(B + 1), prot_node(Np), prot_graph(Np), lig_node(Nl), lig_graph(Nl), node_lig(N, -1);
  int n = 0, p = 0, a = 0;
  for (int g = 0; g < B; ++g) {
    node_ptr[g] = n; prot_ptr[g] = p;
    for (int i = 0; i < pc[g]; ++i) { prot_node[p] = n; prot_graph[p] = g; ++p; ++n; }
    for (int i = 0; i < lc[g]; ++i) { lig_node[a] = n; lig_graph[a] = g; node_lig[n] = a; ++a; ++n; }
  }
  node_ptr[B] = n; prot_ptr[B] = p;
  e->bound = false; e->has_ligand = false; e->have_graph = false; e->have_prev = false;
  e->B = B; e->N = (int)N; e->Np = (int)Np; e->Nl = (int)Nl; e->max_ng = max_ng;
  const size_t slots = (size_t)N * K;
  int bad = 0;
  bad |= e->node_ptr.ensure((B + 1) * 4) | e->prot_ptr.ensure((B + 1) * 4) | e->prot_node.ensure(Np * 4 + 4) | e->prot_graph.ensure(Np * 4 + 4);
  bad |= e->lig_node.ensure(Nl * 4 + 4) | e->lig_graph.ensure(Nl * 4 + 4) | e->node_lig.ensure(N * 4);
  bad |= e->xm0.ensure(N * 16) | e->xm1.ensure(N * 16) | e->offset.ensure((size_t)B * 16);
  bad |= e->h0.ensure(N * TD_H * 4) | e->h.ensure(N * TD_H * 4) | e->P.ensure((size_t)(N + 1) * TD_NPROJ * 4) | e->q.ensure(N * TD_H * 4);
  bad |= e->src.ensure(slots * 4) | e->src_prev.ensure(slots * 4) | e->etype.ensure(slots) | e->e_w.ensure(slots * 4) | e->dist.ensure(slots * 4);
  // class-sorted destination lists (v4 edge kernel): each class padded so that its rows end on a 128-row tile boundary
  const bool v4 = e->mlp_mode == 2 && e->mlp_v4;
  int gcd128 = 128;
  while (K % gcd128) gcd128 >>= 1;
  e->row_pad = 128 / gcd128;
  const long long pad = e->row_pad, nPpad = (Np + pad - 1) / pad * pad, nLpad = (Nl + pad - 1) / pad * pad;
  e->x2h_n_dst = nPpad + nLpad; e->x2h_split = nPpad; e->lig_n_dst = nLpad;
  std::vector<int> x2h_rows((size_t)(nPpad + nLpad), -1), lig_rows((size_t)nLpad, -1);
  for (long long i = 0; i < Np; ++i) x2h_rows[i] = prot_node[i];
  for (long long i = 0; i < Nl; ++i) { x2h_rows[nPpad + i] = lig_node[i]; lig_rows[i] = lig_node[i]; }
  if (v4) bad |= e->x2h_rows.ensure(x2h_rows.size() * 4 + 4) | e->lig_rows.ensure(lig_rows.size() * 4 + 4) | e->rel_rows.ensure(x2h_rows.size() * 4 + 4) |
                 e->rel_counts.ensure(16);
  // per-edge buffers: v4 keeps 16 attention logits / weights per row and, with the aggregation fused into the value launch (k == 32),
  // no [E,128] tensor at all; the earlier execution modes materialise keys and values
  const bool fuse = v4 && K == 32 && !e->env_no_fused_agg && e->ew_mode != 2;      // 'm' gates need the value rows (unfused aggregation)
  if (e->ew_mode == 1) bad |= e->ew_x2h.ensure(slots * 4) | e->ew_h2x.ensure(slots * 4);
  if (e->out_fc) bad |= e->hagg.ensure((size_t)N * TD_H * 4);
  if (e->time_emb) bad |= e->time_norm.ensure((size_t)B * 4 + 16);
  bad |= e->kbuf.ensure(v4 ? (size_t)(nPpad + nLpad) * K * TD_HEADS * 4 + 64 : slots * TD_H * 4);
  if (!fuse) bad |= e->vbuf.ensure(slots * TD_H * 4);
  bad |= e->v16.ensure((size_t)nLpad * K * TD_HEADS * 4 + 16);
  // ligand-free cache: needs the fused path and, in every graph, more than k protein atoms (so that parked ligand atoms can never be
  // among a protein atom's neighbours) and at least one ligand atom
  int min_pc = 1 << 30;
  for (int g = 0; g < B; ++g) if (pc[g] < min_pc) min_pc = pc[g];
  e->free_ready = false;
  e->free_depth = (fuse && !e->hybrid && Nl > 0 && min_pc > K) ? e->env_free_depth : 0;      // (only block 0 of a multi-block network uses it)
  if (e->free_depth > (int)e->layers.size() - 1) e->free_depth = (int)e->layers.size() - 1;
  if (e->free_depth > 0)
    bad |= e->h_free.ensure((size_t)e->free_depth * N * TD_H * 4) | e->dirty.ensure((size_t)e->free_depth * N + 16) |
           e->free_rows.ensure((size_t)e->free_depth * x2h_rows.size() * 4 + 4) | e->free_counts.ensure((size_t)e->free_depth * 16) |
           e->lig_save.ensure((size_t)Nl * 20 + 32);
  e->free_stride = (long long)x2h_rows.size();
  bad |= e->lig_pos.ensure(Nl * 16 + 16) | e->lig_v.ensure(Nl * 4 + 4) | e->logits.ensure((size_t)Nl * e->cfg.num_classes * 4 + 4);
  bad |= e->node_off.ensure(N * 8) | e->rel_flag.ensure(N + 16) | e->rel_list.ensure(N * 4 + 64) | e->n_rel.ensure(16) | e->work_list.ensure(N * 4 + 64) | e->n_work.ensure(16);
  e->knn_incremental = !e->env_knn_full && Np > 0;
  if (e->knn_incremental) bad |= e->knn_cache.ensure((size_t)N * (e->KQ + 1) * 8);
  if (bad) return set_err(TDIFF_ECUDA, "out of device memory binding a batch of %lld nodes (%zu edge slots)", N, slots);
  CK(cudaMemcpyAsync(e->node_ptr.p, node_ptr.data(), (B + 1) * 4, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(e->prot_ptr.p, prot_ptr.data(), (B + 1) * 4, cudaMemcpyHostToDevice, st));
  if (Np) {
    CK(cudaMemcpyAsync(e->prot_node.p, prot_node.data(), Np * 4, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(e->prot_graph.p, prot_graph.data(), Np * 4, cudaMemcpyHostToDevice, st));
  }
  if (Nl) {
    CK(cudaMemcpyAsync(e->lig_node.p, lig_node.data(), Nl * 4, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(e->lig_graph.p, lig_graph.data(), Nl * 4, cudaMemcpyHostToDevice, st));
  }
  CK(cudaMemcpyAsync(e->node_lig.p, node_lig.data(), N * 4, cudaMemcpyHostToDevice, st));
  if (v4) {
    if (!x2h_rows.empty()) CK(cudaMemcpyAsync(e->x2h_rows.p, x2h_rows.data(), x2h_rows.size() * 4, cudaMemcpyHostToDevice, st));
    if (!lig_rows.empty()) CK(cudaMemcpyAsync(e->lig_rows.p, lig_rows.data(), lig_rows.size() * 4, cudaMemcpyHostToDevice, st));
  }
  CK(cudaStreamSynchronize(st));   // host vectors go out of scope
  CK(cudaMemsetAsync(e->offset.p, 0, (size_t)B * 16, st));
  if (e->time_emb) CK(cudaMemsetAsync(e->time_norm.p, 0, (size_t)B * 4, st));
  CK(cudaMemsetAsync(e->h0.p, 0, (size_t)N * TD_H * 4, st));
  CK(cudaMemsetAsync(e->xm0.p, 0, (size_t)N * 16, st));
  CK(cudaMemsetAsync(e->xm1.p, 0, (size_t)N * 16, st));
  CK(cudaMemsetAsync(e->etype.p, 0, slots, st));            // bit 7 of an edge type is the "keep" mark of the incremental edge gate
  // row N of the projection table stays all-zero: the edge kernel's gather warps read it for absent neighbour slots (no per-row branch)
  CK(cudaMemsetAsync(e->P.as<float>() + (size_t)N * TD_NPROJ, 0, (size_t)TD_NPROJ * 4, st));
  if (center_mode == 1) td_launch_segment_mean3(d_ppos, e->prot_ptr.as<int>(), B, e->offset.as<float4>(), st);
  td_launch_place_protein(d_ppos, e->prot_node.as<int>(), e->prot_graph.as<int>(), e->offset.as<float4>(), (int)Np, e->xm0.as<float4>(),
                          e->xm1.as<float4>(), st);
  td_launch_protein_embed(d_pfeat, (int)Np, e->cfg.protein_feat_dim, e->w_prot, e->b_prot, e->prot_node.as<int>(), e->h0.as<float>(), st);
  e->launches += 3;
  if (e->knn_incremental) {      // protein atoms never move: their protein-only neighbour keys are computed once per bound batch
    td_launch_knn_cache(e->xm0.as<float4>(), e->node_ptr.as<int>(), e->prot_ptr.as<int>(), B, max_ng, e->KQ, e->knn_cache.as<unsigned long long>(), st);
    e->launches += 1;
  }
  CK(cudaGetLastError());
  e->bound = true;
  return TDIFF_OK;
}

extern "C" int tdiff_set_ligand(tdiff_engine* e, const float* d_pos, const int64_t* d_v, int apply_center, void* stream) {
  if (!e || !e->bound) return set_err(TDIFF_ESTATE, "set_ligand before bind_batch");
  if (e->Nl > 0 && !d_pos) return set_err(TDIFF_EINVAL, "null ligand positions");
  if (!e->has_ligand && e->Nl > 0 && !d_v) return set_err(TDIFF_EINVAL, "ligand types required on first set_ligand");
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaSetDevice(e->device));
  td_launch_set_ligand(d_pos, (const long long*)d_v, e->lig_graph.as<int>(), e->offset.as<float4>(), apply_center, e->Nl,
                       e->cfg.num_classes, e->lig_pos.as<float4>(), e->lig_v.as<int>(), e->err_flag.as<int>(), st);
  e->launches += 1;
  if (d_v) {
    int flag = 0;
    CK(cudaMemcpyAsync(&flag, e->err_flag.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (flag) {
      cudaMemsetAsync(e->err_flag.p, 0, sizeof(int), st);
      e->has_ligand = false;          // rejected indices were replaced by 0 (set_ligand_kernel); the state must be set again
      return set_err(TDIFF_EINVAL, "ligand atom type index >= num_classes (%d)", e->cfg.num_classes);
    }
  }
  CK(cudaGetLastError());
  e->has_ligand = true;
  return TDIFF_OK;
}

extern "C" int tdiff_get_ligand(tdiff_engine* e, float* d_pos, int64_t* d_v, int add_offset, void* stream) {
  if (!e || !e->has_ligand) return set_err(TDIFF_ESTATE, "get_ligand before set_ligand");
  CK(cudaSetDevice(e->device));
  td_launch_get_ligand(e->lig_pos.as<float4>(), e->lig_v.as<int>(), e->lig_graph.as<int>(), e->offset.as<float4>(), add_offset, e->Nl, d_pos,
                       (long long*)d_v, (cudaStream_t)stream);
  e->launches += 1;
  CK(cudaGetLastError());
  return TDIFF_OK;
}

extern "C" int tdiff_get_offset(tdiff_engine* e, float* d_offset, void* stream) {
  if (!e || !e->bound || !d_offset) return set_err(TDIFF_ESTATE, "get_offset before bind_batch");
  CK(cudaSetDevice(e->device));
  td_launch_gather_xyz(e->offset.as<float4>(), nullptr, e->B, d_offset, (cudaStream_t)stream);
  e->launches += 1;
  CK(cudaGetLastError());
  return TDIFF_OK;
}

// ---------------------------------------------------------------------------------------------- forward
namespace {
struct Prof {
  tdiff_engine* e; cudaStream_t st; int kind; bool on; EvPair ev;
  Prof(tdiff_engine* e_, cudaStream_t st_, int kind_) : e(e_), st(st_), kind(kind_), on(e_->profiling) {
    if (on) { cudaEventCreate(&ev.a); cudaEventCreate(&ev.b); ev.kind = kind; cudaEventRecord(ev.a, st); }
  }
  ~Prof() { if (on) { cudaEventRecord(ev.b, st); e->events.push_back(ev); } }
};

// per-edge MLP dispatch.  `list`: which destination set the launch covers.
//   v4 (default): class-sorted destination lists; `qnode` != NULL marks a key MLP whose output is 16 attention logits (or, with
//   `key_softmax`, softmax weights * e_w) per row; `agg_logits` / `agg_h` make the value launch perform the attention aggregation.
//   earlier modes: tcgen05 second Linear with keys / values in HBM (edge_mlp_tc.cu) or the FP32 FFMA build (edge_mlp.cu).
enum RowList { ROWS_ALL = 0, ROWS_LIGAND = 1, ROWS_RELEVANT = 2 };
bool fused_logits(const tdiff_engine* e) { return e->mlp_mode == 2 && e->mlp_v4; }
void edge_mlp(tdiff_engine* e, const float* P, const float4* xm, const int* src, const unsigned char* etype, RowList list, int K, const TdMlp& m,
              const float* offsets, float coeff, float* out, cudaStream_t st, const float* e_w, const float* qnode = nullptr,
              const float* agg_logits = nullptr, float* agg_h = nullptr, int key_softmax = 0, int free_layer = -1) {
  if (fused_logits(e) && m.w2_img && m.tabcls_img) {
    const int* rows = list == ROWS_ALL ? e->x2h_rows.as<int>() : list == ROWS_LIGAND ? e->lig_rows.as<int>() : e->rel_rows.as<int>();
    const int* counts = list == ROWS_RELEVANT ? e->rel_counts.as<int>() : nullptr;
    if (free_layer >= 0) {           // ligand-free cache: only the dirty destinations of this layer (device-compacted, class-sorted)
      rows = e->free_rows.as<int>() + (size_t)free_layer * e->free_stride;
      counts = e->free_counts.as<int>() + 4 * free_layer;
    }
    const long long n_dst = list == ROWS_LIGAND ? e->lig_n_dst : e->x2h_n_dst;          // ROWS_RELEVANT: upper bound, real counts on the device
    const long long split = list == ROWS_LIGAND ? 0 : e->x2h_split;
    // plain (unfused) x2h outputs are consumed by slot index (aggregate_h_logits_kernel); everything else by row index
    const int by_slot = (list != ROWS_LIGAND && !key_softmax && agg_logits == nullptr) ? 1 : 0;
    td_launch_edge_mlp_v4(P, e->N, src, etype, e->dist.as<float>(), rows, n_dst, split, counts, K, m,
                          e->host_arena.data() + (offsets - e->arena), coeff, e->host_arena.data() + (m.ln_g - e->arena), e->host_arena.data() + (m.ln_b - e->arena),
                          e->host_arena.data() + (m.b2 - e->arena), qnode, out, by_slot, agg_logits, e_w, agg_h, key_softmax,
                          e->sm_count, st);
    return;
  }
  const int* row_nodes = list == ROWS_LIGAND ? e->lig_node.as<int>() : nullptr;
  const long long n_rows = (long long)(list == ROWS_LIGAND ? e->Nl : e->N) * K;
  if (e->mlp_mode != 0 && m.nout == TD_H && m.w2_img)
    td_launch_edge_mlp_tc(P, xm, src, etype, e->dist.as<float>(), row_nodes, n_rows, K, m, m.w2_img, e->mlp_mode, offsets, coeff, out, e->sm_count, st);
  else
    td_launch_edge_mlp(P, xm, src, etype, row_nodes, n_rows, K, m, offsets, coeff, out, e->sm_count, st);
}

// node-side GEMMs: P = h . Wn^T + bn ; q = relu(LN(P[:,512:640])) . W2q^T + b2q   (tensor cores unless TDIFF_EDGE_MLP=simt)
// `rows` / `d_n` (optional): restrict to a node subset given as a device list (+ device count); other rows of P / q are left stale
void node_side(tdiff_engine* e, const float* h, int N, const TdSubLayer& sl, float* P, float* q, cudaStream_t st, const int* rows = nullptr,
               const int* d_n = nullptr) {
  if (e->mlp_mode != 0 && sl.wn_img && sl.q.w2_img) {
    TdMlp pm = sl.q;
    pm.b2 = sl.bn;                 // mode 1 reads the per-column-block bias through m.b2
    td_launch_rows_tc(1, h, TD_H, 0, N, pm, sl.wn_img, e->mlp_mode, P, TD_NPROJ, TD_NPROJ / TD_H, rows, d_n, e->sm_count, st);
    td_launch_rows_tc(2, P, TD_NPROJ, 512, N, sl.q, sl.q.w2_img, e->mlp_mode, q, TD_H, 1, rows, d_n, e->sm_count, st);
  } else {
    td_launch_node_proj(h, N, sl.wn_t, sl.bn, P, st);
    td_launch_node_q(P, N, sl.q, q, st);
  }
}

// One evaluation of the network on the bound batch (reference ScorePosNet3D.forward -> UniTransformerO2TwoUpdateGeneral.forward)
// `free_build` > 0: ligand-free cache construction -- only the first `free_build` x2h layers, features saved after each (ligand parked far away)
void run_forward(tdiff_engine* e, cudaStream_t st, int fix_x, int free_build = 0) {
  const int N = e->N, Nl = e->Nl, K = e->K;
  float4* xm[2] = {e->xm0.as<float4>(), e->xm1.as<float4>()};
  const int* src = e->src.as<int>();
  const unsigned char* etype = e->etype.as<unsigned char>();
  float* h = e->h.as<float>();
  float* P = e->P.as<float>();
  float* q = e->q.as<float>();
  td_launch_scatter_ligand_pos(e->lig_pos.as<float4>(), e->lig_node.as<int>(), Nl, xm[0], st);
  td_launch_init_h(e->h0.as<float>(), xm[0], e->lig_v.as<int>(), e->node_lig.as<int>(), e->wl_t, e->bl, e->w_time, e->time_norm.as<float>(),
                   e->lig_graph.as<int>(), N, h, st);
  e->launches += 2;
  int cur = 0;
  const int n_blocks = free_build ? 1 : e->num_blocks;
  for (int blk = 0; blk < n_blocks; ++blk) {
    // ---- graph of this block from the current coordinates (reference models/uni_transformer.py:306-318)
    const int use_free = (!free_build && e->free_ready && blk == 0) ? e->free_depth : 0;
    const bool last_blk = blk + 1 == n_blocks;
    if (e->knn_incremental)
      td_launch_knn_update(xm[cur], e->node_ptr.as<int>(), e->prot_ptr.as<int>(), e->B, e->max_ng, e->KQ, K, e->hybrid, e->knn_cache.as<unsigned long long>(),
                           e->src.as<int>(), st);
    else
      td_launch_knn(xm[cur], e->node_ptr.as<int>(), e->prot_ptr.as<int>(), e->B, e->max_ng, e->KQ, K, e->hybrid, e->src.as<int>(), st);
    td_launch_edge_const(xm[cur], src, e->src_prev.as<int>(), e->have_prev ? 1 : 0, N, K, e->ew_off, e->ew_coeff, e->ew_w1t, e->ew_b1, e->ew_g, e->ew_b, e->ew_w2,
                         e->ew_b2, e->etype.as<unsigned char>(), e->e_w.as<float>(), e->rel_flag.as<unsigned char>(),
                         use_free ? e->dirty.as<unsigned char>() : nullptr, e->work_list.as<int>(), e->n_work.as<int>(), (e->ew_mode != 0 ? 1 : 0) | (e->env_no_slot_keep ? 2 : 0), st);
    e->have_prev = true;
    for (int l = 0; l < use_free; ++l) {             // dirty sets layer by layer and their class-sorted destination lists
      unsigned char* dl = e->dirty.as<unsigned char>() + (size_t)l * N;
      if (l > 0) td_launch_dirty_propagate(dl - N, src, N, K, dl, st);
      td_launch_rel_rows(dl, xm[cur], N, e->lig_rows.as<int>(), (int)e->lig_n_dst, e->row_pad, e->free_rows.as<int>() + (size_t)l * e->free_stride,
                         e->free_counts.as<int>() + 4 * l, st);
      e->launches += l > 0 ? 3 : 2;
    }
    td_launch_rel_compact(e->rel_flag.as<unsigned char>(), N, e->rel_list.as<int>(), e->n_rel.as<int>(), st);
    e->launches += 4;
    if (fused_logits(e) && e->restrict_last && last_blk) {       // class-sorted list of the relevant destinations for the last x2h
      td_launch_rel_rows(e->rel_flag.as<unsigned char>(), xm[cur], N, e->lig_rows.as<int>(), (int)e->lig_n_dst, e->row_pad, e->rel_rows.as<int>(),
                         e->rel_counts.as<int>(), st);
      e->launches += 2;
    }
    const float4* xm_blk = xm[cur];                  // coordinates the block's graph was built from (protein flags for the cache kernels)
    const size_t n_layers = free_build ? (size_t)free_build : e->layers.size();
    for (size_t l = 0; l < n_layers; ++l) {
      const TdLayer& ly = e->layers[l];
      const int fl = (int)l < use_free ? (int)l : -1;
      // per-sub-layer edge gates: the global gate, or the layer's own 'r' gates (evaluated with the edge lengths), or 1
      const float* ew_x = e->ew_mode == 1 ? e->ew_x2h.as<float>() : e->e_w.as<float>();
      const float* ew_h = e->ew_mode == 1 ? e->ew_h2x.as<float>() : e->e_w.as<float>();
      // ---- x2h: h <- h + sum_e alpha * v * e_w   (+ node_output MLP with x2h_out_fc)
      node_side(e, h, N, ly.x2h, P, q, st);
      if (e->mlp_mode != 0) {
        TdEwR ew = {nullptr, nullptr, 0.f, 0.f, ly.offsets, ly.coeff, nullptr, nullptr};
        if (e->ew_mode == 1) { ew.w_x2h = ly.x2h.ew_w; ew.w_h2x = ly.h2x.ew_w; ew.b_x2h = ly.x2h.ew_b; ew.b_h2x = ly.h2x.ew_b; ew.out_x2h = e->ew_x2h.as<float>(); ew.out_h2x = e->ew_h2x.as<float>(); }
        td_launch_edge_geom(xm[cur], src, etype, N, K, e->dist.as<float>(), ew, st);
        e->launches += 1;
      }
      // k == 32: a 128-row tile is 4 complete destinations -> the value launch also performs the softmax aggregation (h += ...)
      const bool fuse_agg = fused_logits(e) && K == 32 && !e->env_no_fused_agg && e->ew_mode != 2;
      // sampling loop, last layer: only the ligand atoms' features feed the type head and only ligand atoms + their neighbours feed
      // the last h2x, so x2h is evaluated for those destinations only (device-compacted list; final_h of other nodes is not produced)
      const bool sub = fuse_agg && e->restrict_last && last_blk && l + 1 == e->layers.size() && !e->env_no_restrict && !e->out_fc;
      const RowList rl = sub ? ROWS_RELEVANT : ROWS_ALL;
      float* agg_target = h;
      if (e->out_fc) {               // node_output needs the bare aggregate: accumulate into a zeroed buffer instead of h
        agg_target = e->hagg.as<float>();
        cudaMemsetAsync(agg_target, 0, (size_t)N * TD_H * 4, st);
      }
      {
        Prof pr(e, st, EV_EDGE_MLP);
        edge_mlp(e, P, xm[cur], src, etype, rl, K, ly.x2h.k, ly.offsets, ly.coeff, e->kbuf.as<float>(), st, ew_x, fused_logits(e) ? q : nullptr, nullptr,
                 nullptr, fuse_agg ? 1 : 0, fl);
        edge_mlp(e, P, xm[cur], src, etype, rl, K, ly.x2h.v, ly.offsets, ly.coeff, e->vbuf.as<float>(), st, ew_x, nullptr,
                 fuse_agg ? e->kbuf.as<float>() : nullptr, fuse_agg ? agg_target : nullptr, 0, fl);
      }
      if (!fuse_agg) {
        Prof pr(e, st, EV_AGG_H);
        if (fused_logits(e))
          td_launch_aggregate_h_logits(e->kbuf.as<float>(), e->vbuf.as<float>(), ew_x, src, e->out_fc ? agg_target : h, agg_target, N, K,
                                       e->ew_mode == 2 ? ly.x2h.ew_w : nullptr, ly.x2h.ew_b, st);
        else td_launch_aggregate_h(e->kbuf.as<float>(), e->vbuf.as<float>(), e->e_w.as<float>(), src, q, h, h, N, K, st);
      }
      e->launches += fuse_agg ? 4 : 5;
      if (e->out_fc) {               // h <- h + node_output([aggregate | h])   (reference models/uni_transformer.py:80-83); P is free here
        float* t1 = P;
        float* t2 = P + (size_t)N * TD_H;
        TdMlp m1 = ly.x2h.out;
        m1.b2 = e->zeros128;
        td_launch_rows_tc(1, agg_target, TD_H, 0, N, m1, ly.x2h.out_wa_img, e->mlp_mode, t1, TD_H, 1, nullptr, nullptr, e->sm_count, st);
        m1.b2 = ly.x2h.out_b1;
        td_launch_rows_tc(1, h, TD_H, 0, N, m1, ly.x2h.out_wb_img, e->mlp_mode, t2, TD_H, 1, nullptr, nullptr, e->sm_count, st);
        td_launch_add_rows(t1, t2, t1, (long long)N * TD_H, st);
        td_launch_rows_tc(2, t1, TD_H, 0, N, ly.x2h.out, ly.x2h.out.w2_img, e->mlp_mode, t2, TD_H, 1, nullptr, nullptr, e->sm_count, st);
        td_launch_add_rows(h, t2, h, (long long)N * TD_H, st);
        e->launches += 6;
      }
      if (fl >= 0) {                 // clean protein rows: cached ligand-free features of this layer
        td_launch_restore_clean(e->dirty.as<unsigned char>() + (size_t)fl * N, xm_blk, e->h_free.as<float>() + (size_t)fl * N * TD_H, N, h, st);
        e->launches += 1;
      }
      if (free_build) {
        cudaMemcpyAsync(e->h_free.as<float>() + l * (size_t)N * TD_H, h, (size_t)N * TD_H * 4, cudaMemcpyDeviceToDevice, st);
        continue;
      }
      if (fix_x || Nl == 0) continue;     // h2x only moves ligand atoms; with fix_x its result is discarded (:204-206)
      // ---- h2x: x_lig <- x_lig + mean_heads sum_e alpha * v * e_w * (x_dst - x_src), destinations = ligand atoms only
      {
        const bool rel = fused_logits(e) && !e->env_no_restrict;      // h2x only reads P / q of ligand atoms and their neighbours
        node_side(e, h, N, ly.h2x, P, q, st, rel ? e->rel_list.as<int>() : nullptr, rel ? e->n_rel.as<int>() : nullptr);
      }
      {
        Prof pr(e, st, EV_EDGE_MLP);
        edge_mlp(e, P, xm[cur], src, etype, ROWS_LIGAND, K, ly.h2x.k, ly.offsets, ly.coeff, e->kbuf.as<float>(), st, ew_h, fused_logits(e) ? q : nullptr);
        edge_mlp(e, P, xm[cur], src, etype, ROWS_LIGAND, K, ly.h2x.v, ly.offsets, ly.coeff, e->v16.as<float>(), st, ew_h);
      }
      {
        Prof pr(e, st, EV_AGG_X);
        if (fused_logits(e))
          td_launch_aggregate_x_logits(e->kbuf.as<float>(), e->v16.as<float>(), ew_h, src, xm[cur], e->lig_node.as<int>(), xm[cur ^ 1], Nl, K, st);
        else
          td_launch_aggregate_x(e->kbuf.as<float>(), e->v16.as<float>(), e->e_w.as<float>(), src, q, xm[cur], e->lig_node.as<int>(), xm[cur ^ 1], Nl, K, st);
      }
      e->launches += 5;
      cur ^= 1;
    }
  }
  if (free_build) return;
  td_launch_head(h, e->lig_node.as<int>(), Nl, e->hd_w1t, e->hd_b1, e->hd_w2, e->hd_b2, e->cfg.num_classes, e->logits.as<float>(), st);
  e->launches += 1;
  e->final_buf = cur;
  e->have_graph = true;
  e->have_prev = true;
}
}  // namespace

extern "C" int tdiff_set_time(tdiff_engine* e, const float* d_time_norm, void* stream) {
  if (!e || !e->bound) return set_err(TDIFF_ESTATE, "set_time before bind_batch");
  if (!e->time_emb) return TDIFF_OK;           // no time embedding in this model: nothing to set
  if (!d_time_norm) return set_err(TDIFF_EINVAL, "null time array");
  CK(cudaSetDevice(e->device));
  CK(cudaMemcpyAsync(e->time_norm.p, d_time_norm, (size_t)e->B * 4, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return TDIFF_OK;
}

extern "C" int tdiff_forward(tdiff_engine* e, float* d_pred_pos, float* d_pred_logits, float* d_final_h, int fix_x, void* stream) {
  if (!e || !e->bound || !e->has_ligand) return set_err(TDIFF_ESTATE, "forward needs bind_batch + set_ligand first");
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaSetDevice(e->device));
  Prof* total = new Prof(e, st, EV_TOTAL);
  run_forward(e, st, fix_x);
  delete total;
  const float4* xf = e->final_buf ? e->xm1.as<float4>() : e->xm0.as<float4>();
  if (d_pred_pos) { td_launch_gather_xyz(xf, e->lig_node.as<int>(), e->Nl, d_pred_pos, st); e->launches += 1; }
  if (d_pred_logits && e->Nl) CK(cudaMemcpyAsync(d_pred_logits, e->logits.p, (size_t)e->Nl * e->cfg.num_classes * 4, cudaMemcpyDeviceToDevice, st));
  if (d_final_h) CK(cudaMemcpyAsync(d_final_h, e->h.p, (size_t)e->N * TD_H * 4, cudaMemcpyDeviceToDevice, st));
  CK(cudaGetLastError());
  return TDIFF_OK;
}

extern "C" int64_t tdiff_num_edges(tdiff_engine* e, void* stream) {
  if (!e || !e->have_graph) return set_err(TDIFF_ESTATE, "no graph built yet (run forward first)");
  cudaStream_t st = (cudaStream_t)stream;
  if (cudaSetDevice(e->device) != cudaSuccess) return set_err(TDIFF_ECUDA, "cudaSetDevice failed");
  td_launch_edge_count_scan(e->src.as<int>(), e->N, e->K, e->node_off.as<long long>(), e->total_edges.as<long long>(), st);
  e->launches += 1;
  long long tot = 0;
  if (cudaMemcpyAsync(&tot, e->total_edges.p, 8, cudaMemcpyDeviceToHost, st) != cudaSuccess || cudaStreamSynchronize(st) != cudaSuccess)
    return set_err(TDIFF_ECUDA, "num_edges: %s", cudaGetErrorString(cudaGetLastError()));
  return tot;
}

extern "C" int tdiff_get_edge_index(tdiff_engine* e, int64_t* d_edge_index, void* stream) {
  if (!e || !e->have_graph || !d_edge_index) return set_err(TDIFF_ESTATE, "no graph built yet (run forward first)");
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaSetDevice(e->device));
  td_launch_edge_count_scan(e->src.as<int>(), e->N, e->K, e->node_off.as<long long>(), e->total_edges.as<long long>(), st);
  td_launch_edge_compact(e->src.as<int>(), nullptr, e->N, e->K, e->node_off.as<long long>(), e->total_edges.as<long long>(),
                         (long long*)d_edge_index, nullptr, st);
  e->launches += 2;
  CK(cudaGetLastError());
  return TDIFF_OK;
}

extern "C" int tdiff_get_edge_weight(tdiff_engine* e, float* d_e_w, void* stream) {
  if (!e || !e->have_graph || !d_e_w) return set_err(TDIFF_ESTATE, "no graph built yet (run forward first)");
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaSetDevice(e->device));
  td_launch_edge_count_scan(e->src.as<int>(), e->N, e->K, e->node_off.as<long long>(), e->total_edges.as<long long>(), st);
  td_launch_edge_compact(e->src.as<int>(), e->e_w.as<float>(), e->N, e->K, e->node_off.as<long long>(), e->total_edges.as<long long>(), nullptr,
                         d_e_w, st);
  e->launches += 2;
  CK(cudaGetLastError());
  return TDIFF_OK;
}

extern "C" int tdiff_get_node_pos(tdiff_engine* e, float* d_x, void* stream) {
  if (!e || !e->have_graph || !d_x) return set_err(TDIFF_ESTATE, "no forward run yet");
  CK(cudaSetDevice(e->device));
  td_launch_gather_xyz(e->final_buf ? e->xm1.as<float4>() : e->xm0.as<float4>(), nullptr, e->N, d_x, (cudaStream_t)stream);
  e->launches += 1;
  CK(cudaGetLastError());
  return TDIFF_OK;
}

// ---------------------------------------------------------------------------------------------- sampling loop
namespace {
// Ligand-free features of the first `free_depth` x2h layers (once per bound batch): the ligand atoms are parked far away so that no
// protein atom has one among its neighbours, the ordinary kernels run, and the protein rows are exactly what a clean node gets later.
void build_free_cache(tdiff_engine* e, cudaStream_t st) {
  const size_t Nl = (size_t)e->Nl;
  char* sv = e->lig_save.as<char>();
  cudaMemcpyAsync(sv, e->lig_pos.p, Nl * 16, cudaMemcpyDeviceToDevice, st);
  cudaMemcpyAsync(sv + Nl * 16, e->lig_v.p, Nl * 4, cudaMemcpyDeviceToDevice, st);
  td_launch_park_ligand(e->lig_pos.as<float4>(), e->lig_v.as<int>(), e->Nl, st);
  const bool had_prev = e->have_prev;
  e->have_prev = false;
  run_forward(e, st, 1, e->free_depth);
  e->have_prev = false;               // src_prev now holds the parked graph: the next forward re-evaluates every edge constant
  (void)had_prev;
  cudaMemcpyAsync(e->lig_pos.p, sv, Nl * 16, cudaMemcpyDeviceToDevice, st);
  cudaMemcpyAsync(e->lig_v.p, sv + Nl * 16, Nl * 4, cudaMemcpyDeviceToDevice, st);
  e->launches += 1;
  e->free_ready = true;
}

void run_step(tdiff_engine* e, cudaStream_t st, const TdStepArgs& base) {
  if (e->time_emb) {               // every graph is at time step t_start - step (reference models/molopt_score_model.py:651)
    td_launch_set_time(base.step, base.t_start, e->cfg.num_timesteps, e->B, e->time_norm.as<float>(), st);
    e->launches += 1;
  }
  e->restrict_last = true;
  run_forward(e, st, 0);
  e->restrict_last = false;
  TdStepArgs A = base;
  A.xm_final = e->final_buf ? e->xm1.as<float4>() : e->xm0.as<float4>();
  td_launch_step_epilogue(A, st);
  e->launches += 2;
}
}  // namespace

extern "C" int tdiff_sample(tdiff_engine* e, int num_steps, const float* d_pos_noise, const float* d_v_uniform, uint64_t seed,
                            float* d_pos_traj, int64_t* d_v_traj, float* d_v0_traj, float* d_vt_traj, int pos_only, void* stream) {
  if (!e || !e->bound || !e->has_ligand) return set_err(TDIFF_ESTATE, "sample needs bind_batch + set_ligand first");
  const int T = e->cfg.num_timesteps;
  if (num_steps < 0 || num_steps > T) return set_err(TDIFF_EINVAL, "num_steps=%d outside 0..%d", num_steps, T);
  if ((d_pos_noise == nullptr) != (d_v_uniform == nullptr) && !pos_only)
    return set_err(TDIFF_EINVAL, "noise tape needs both pos_noise and v_uniform (or neither for Philox)");
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaSetDevice(e->device));
  if (num_steps == 0) return TDIFF_OK;
  TdStepArgs A;
  memset(&A, 0, sizeof(A));
  A.n_lig = e->Nl; A.n_classes = e->cfg.num_classes; A.t_start = T - 1; A.pos_only = pos_only;
  A.step = e->step.as<int>(); A.lig_node = e->lig_node.as<int>(); A.lig_graph = e->lig_graph.as<int>();
  A.logits = e->logits.as<float>(); A.offset = e->offset.as<float4>();
  A.c0 = e->t_c0; A.ct = e->t_ct; A.logvar = e->t_logvar; A.la_v = e->t_la; A.l1ma_v = e->t_l1ma; A.lca_v = e->t_lca; A.l1mca_v = e->t_l1mca;
  A.sra = e->t_sra; A.srm1 = e->t_srm1; A.mean_noise = e->cfg.model_mean_type == 1;
  A.log_k = (float)log((double)e->cfg.num_classes);
  A.pos_noise = d_pos_noise; A.v_uniform = d_v_uniform; A.seed = seed;
  A.lig_pos = e->lig_pos.as<float4>(); A.lig_v = e->lig_v.as<int>();
  A.pos_traj = d_pos_traj; A.v_traj = (long long*)d_v_traj; A.v0_traj = d_v0_traj; A.vt_traj = d_vt_traj;
  CK(cudaMemsetAsync(e->step.p, 0, sizeof(int), st));
  if (e->free_depth > 0 && !e->free_ready) build_free_cache(e, st);
  const bool eager = e->profiling || e->env_no_graph;
  Prof* total = new Prof(e, st, EV_TOTAL);
  // first step eagerly (module loading, shared-memory attributes), the rest replayed from one captured graph
  run_step(e, st, A);
  int done = 1;
  if (!eager && num_steps > 2) {
    // fork onto the engine's own stream: capture there (the caller's stream may be the legacy default stream), replay, join back
    cudaStream_t cs = e->own_stream;
    CK(cudaEventRecord(e->ev_fork, st));
    CK(cudaStreamWaitEvent(cs, e->ev_fork, 0));
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    const long long before = e->launches;
    cudaError_t ce = cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal);
    if (ce == cudaSuccess) {
      run_step(e, cs, A);
      ce = cudaStreamEndCapture(cs, &graph);
    }
    const long long per_step = e->launches - before;
    e->launches = before;
    if (ce == cudaSuccess) ce = cudaGraphInstantiate(&exec, graph, 0);
    if (ce != cudaSuccess) {
      if (graph) cudaGraphDestroy(graph);
      (void)cudaGetLastError();
      delete total;
      return set_err(TDIFF_ECUDA, "CUDA graph capture of the sampling step failed: %s", cudaGetErrorString(ce));
    }
    for (; done < num_steps; ++done) {
      ce = cudaGraphLaunch(exec, cs);
      if (ce != cudaSuccess) break;
      e->launches += per_step;
    }
    if (ce == cudaSuccess) ce = cudaEventRecord(e->ev_join, cs);
    if (ce == cudaSuccess) ce = cudaStreamWaitEvent(st, e->ev_join, 0);
    cudaGraphExecDestroy(exec);      // deferred by the runtime until the launched replays have finished
    cudaGraphDestroy(graph);
    if (ce != cudaSuccess) { delete total; return set_err(TDIFF_ECUDA, "cudaGraphLaunch failed: %s", cudaGetErrorString(ce)); }
  }
  for (; done < num_steps; ++done) run_step(e, st, A);
  delete total;
  CK(cudaGetLastError());
  return TDIFF_OK;
}

extern "C" int tdiff_sample_host(tdiff_engine* e, int B, const int32_t* pc, const int32_t* lc, const float* h_ppos, const float* h_pfeat,
                                 const float* h_lpos, const int64_t* h_lv, int center_mode, int num_steps, const float* h_pos_noise,
                                 const float* h_v_uniform, uint64_t seed, float* h_out_pos, int64_t* h_out_v, float* h_pos_traj,
                                 int64_t* h_v_traj, float* h_v0_traj, float* h_vt_traj, int pos_only, void* stream) {
  if (!e || !pc || !lc || B < 1) return set_err(TDIFF_EINVAL, "sample_host: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaSetDevice(e->device));
  size_t Np = 0, Nl = 0;
  for (int g = 0; g < B; ++g) { Np += pc[g] > 0 ? pc[g] : 0; Nl += lc[g] > 0 ? lc[g] : 0; }
  const int F = e->cfg.protein_feat_dim, KC = e->cfg.num_classes;
  const size_t S = num_steps > 0 ? num_steps : 0;
  DevBuf* sb = e->stage;
  int bad = sb[0].ensure(Np * 12 + 16) | sb[1].ensure(Np * F * 4 + 16) | sb[2].ensure(Nl * 12 + 16) | sb[3].ensure(Nl * 8 + 16);
  if (h_pos_noise) bad |= sb[4].ensure(S * Nl * 12 + 16);
  if (h_v_uniform) bad |= sb[5].ensure(S * Nl * KC * 4 + 16);
  // trajectories share one staging block: pos [S,Nl,3] f32 | v [S,Nl] i64 | v0 [S,Nl,K] | vt [S,Nl,K]
  const size_t o_pos = 0, o_v = (o_pos + (h_pos_traj ? S * Nl * 12 : 0) + 15) / 16 * 16,      // int64 rows need 8-byte alignment (S*Nl may be odd)
               o_v0 = (o_v + (h_v_traj ? S * Nl * 8 : 0) + 15) / 16 * 16,
               o_vt = o_v0 + (h_v0_traj ? S * Nl * KC * 4 : 0), o_end = o_vt + (h_vt_traj ? S * Nl * KC * 4 : 0);
  bad |= sb[6].ensure(o_end + 16) | sb[7].ensure(Nl * 12 + Nl * 8 + 32);
  if (bad) return set_err(TDIFF_ECUDA, "out of device memory staging host buffers");
  if (Np) {
    CK(cudaMemcpyAsync(sb[0].p, h_ppos, Np * 12, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(sb[1].p, h_pfeat, Np * F * 4, cudaMemcpyHostToDevice, st));
  }
  if (Nl) {
    CK(cudaMemcpyAsync(sb[2].p, h_lpos, Nl * 12, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(sb[3].p, h_lv, Nl * 8, cudaMemcpyHostToDevice, st));
  }
  if (h_pos_noise && S * Nl) CK(cudaMemcpyAsync(sb[4].p, h_pos_noise, S * Nl * 12, cudaMemcpyHostToDevice, st));
  if (h_v_uniform && S * Nl) CK(cudaMemcpyAsync(sb[5].p, h_v_uniform, S * Nl * KC * 4, cudaMemcpyHostToDevice, st));
  int rc = tdiff_bind_batch(e, B, pc, lc, sb[0].as<float>(), sb[1].as<float>(), center_mode, st);
  if (rc) return rc;
  rc = tdiff_set_ligand(e, sb[2].as<float>(), sb[3].as<int64_t>(), center_mode == 1, st);
  if (rc) return rc;
  char* tb = sb[6].as<char>();
  rc = tdiff_sample(e, num_steps, h_pos_noise ? sb[4].as<float>() : nullptr, h_v_uniform ? sb[5].as<float>() : nullptr, seed,
                    h_pos_traj ? (float*)(tb + o_pos) : nullptr, h_v_traj ? (int64_t*)(tb + o_v) : nullptr,
                    h_v0_traj ? (float*)(tb + o_v0) : nullptr, h_vt_traj ? (float*)(tb + o_vt) : nullptr, pos_only, st);
  if (rc) return rc;
  float* d_opos = sb[7].as<float>();
  int64_t* d_ov = (int64_t*)(sb[7].as<char>() + (Nl * 12 + 15) / 16 * 16);
  rc = tdiff_get_ligand(e, d_opos, d_ov, 1, st);
  if (rc) return rc;
  if (Nl) {
    if (h_out_pos) CK(cudaMemcpyAsync(h_out_pos, d_opos, Nl * 12, cudaMemcpyDeviceToHost, st));
    if (h_out_v) CK(cudaMemcpyAsync(h_out_v, d_ov, Nl * 8, cudaMemcpyDeviceToHost, st));
    if (S) {
      if (h_pos_traj) CK(cudaMemcpyAsync(h_pos_traj, tb + o_pos, S * Nl * 12, cudaMemcpyDeviceToHost, st));
      if (h_v_traj) CK(cudaMemcpyAsync(h_v_traj, tb + o_v, S * Nl * 8, cudaMemcpyDeviceToHost, st));
      if (h_v0_traj) CK(cudaMemcpyAsync(h_v0_traj, tb + o_v0, S * Nl * KC * 4, cudaMemcpyDeviceToHost, st));
      if (h_vt_traj) CK(cudaMemcpyAsync(h_vt_traj, tb + o_vt, S * Nl * KC * 4, cudaMemcpyDeviceToHost, st));
    }
  }
  CK(cudaStreamSynchronize(st));
  return TDIFF_OK;
}

// ---------------------------------------------------------------------------------------------- stand-alone operators
extern "C" int tdiff_knn_graph(const float* d_x, int n_nodes, const int32_t* h_counts, int n_graphs, int k, int32_t* d_src_slots,
                               int64_t* d_edge_index, int64_t* h_n_edges, void* stream) {
  if (!d_x || !h_counts || !d_src_slots || n_nodes < 0 || n_graphs < 1 || k < 1 || k > TD_KMAX) return set_err(TDIFF_EINVAL, "knn_graph: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  std::vector<int> ptr(n_graphs + 1, 0);
  int max_ng = 0;
  for (int g = 0; g < n_graphs; ++g) {
    if (h_counts[g] < 0) return set_err(TDIFF_EINVAL, "negative count");
    ptr[g + 1] = ptr[g] + h_counts[g];
    if (h_counts[g] > max_ng) max_ng = h_counts[g];
  }
  if (ptr[n_graphs] != n_nodes) return set_err(TDIFF_EINVAL, "graph counts sum to %d, expected %d nodes", ptr[n_graphs], n_nodes);
  if (max_ng > 2800) return set_err(TDIFF_EINVAL, "graph with %d nodes exceeds the k-NN kernel's shared-memory tile (2800)", max_ng);
  if (n_nodes == 0) { if (h_n_edges) *h_n_edges = 0; return TDIFF_OK; }
  DevBuf xm, dptr, off, tot;
  int rc = TDIFF_OK;
  if (xm.ensure((size_t)n_nodes * 16) || dptr.ensure((n_graphs + 1) * 4) || off.ensure((size_t)n_nodes * 8) || tot.ensure(8)) {
    rc = set_err(TDIFF_ECUDA, "out of device memory");
  } else {
    cudaMemcpyAsync(dptr.p, ptr.data(), (n_graphs + 1) * 4, cudaMemcpyHostToDevice, st);
    td_launch_pack_xyzm(d_x, nullptr, n_nodes, xm.as<float4>(), st);
    td_launch_knn(xm.as<float4>(), dptr.as<int>(), nullptr, n_graphs, max_ng, k, k, 0, d_src_slots, st);
    td_launch_edge_count_scan(d_src_slots, n_nodes, k, off.as<long long>(), tot.as<long long>(), st);
    if (d_edge_index) td_launch_edge_compact(d_src_slots, nullptr, n_nodes, k, off.as<long long>(), tot.as<long long>(), (long long*)d_edge_index, nullptr, st);
    long long t = 0;
    cudaMemcpyAsync(&t, tot.p, 8, cudaMemcpyDeviceToHost, st);
    cudaError_t ce = cudaStreamSynchronize(st);
    if (ce == cudaSuccess) ce = cudaGetLastError();
    if (ce != cudaSuccess) rc = set_err(TDIFF_ECUDA, "knn_graph: %s", cudaGetErrorString(ce));
    else if (h_n_edges) *h_n_edges = t;
  }
  xm.release(); dptr.release(); off.release(); tot.release();
  return rc;
}

extern "C" int tdiff_attn_aggregate_h(const float* d_k, const float* d_v, const float* d_e_w, const int32_t* d_src, const float* d_q,
                                      const float* d_h_in, float* d_h_out, int n_nodes, int kk, void* stream) {
  if (!d_k || !d_v || !d_e_w || !d_src || !d_q || !d_h_in || !d_h_out || n_nodes < 0 || kk < 1 || kk > TD_KMAX)
    return set_err(TDIFF_EINVAL, "attn_aggregate_h: bad arguments");
  td_launch_aggregate_h(d_k, d_v, d_e_w, d_src, d_q, d_h_in, d_h_out, n_nodes, kk, (cudaStream_t)stream);
  CK(cudaGetLastError());
  return TDIFF_OK;
}

extern "C" int tdiff_attn_aggregate_x(const float* d_k, const float* d_v16, const float* d_e_w, const int32_t* d_src, const float* d_q,
                                      const float* d_x, const uint8_t* d_mask, float* d_x_out, int n_nodes, int kk, void* stream) {
  if (!d_k || !d_v16 || !d_e_w || !d_src || !d_q || !d_x || !d_mask || !d_x_out || n_nodes < 0 || kk < 1 || kk > TD_KMAX)
    return set_err(TDIFF_EINVAL, "attn_aggregate_x: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  if (n_nodes == 0) return TDIFF_OK;
  DevBuf a, b;
  if (a.ensure((size_t)n_nodes * 16) || b.ensure((size_t)n_nodes * 16)) { a.release(); b.release(); return set_err(TDIFF_ECUDA, "out of device memory"); }
  td_launch_pack_xyzm(d_x, d_mask, n_nodes, a.as<float4>(), st);
  td_launch_aggregate_x(d_k, d_v16, d_e_w, d_src, d_q, a.as<float4>(), nullptr, b.as<float4>(), n_nodes, kk, st);
  td_launch_gather_xyz(b.as<float4>(), nullptr, n_nodes, d_x_out, st);
  cudaError_t ce = cudaStreamSynchronize(st);
  if (ce == cudaSuccess) ce = cudaGetLastError();
  a.release(); b.release();
  if (ce != cudaSuccess) return set_err(TDIFF_ECUDA, "attn_aggregate_x: %s", cudaGetErrorString(ce));
  return TDIFF_OK;
}

extern "C" int tdiff_scatter_mean3(const float* d_src, const int32_t* h_counts, int n_segments, float* d_out, void* stream) {
  if (!d_src || !h_counts || !d_out || n_segments < 1) return set_err(TDIFF_EINVAL, "scatter_mean3: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  std::vector<int> ptr(n_segments + 1, 0);
  for (int g = 0; g < n_segments; ++g) ptr[g + 1] = ptr[g] + (h_counts[g] > 0 ? h_counts[g] : 0);
  DevBuf dptr, o4;
  if (dptr.ensure((n_segments + 1) * 4) || o4.ensure((size_t)n_segments * 16)) { dptr.release(); o4.release(); return set_err(TDIFF_ECUDA, "out of device memory"); }
  cudaMemcpyAsync(dptr.p, ptr.data(), (n_segments + 1) * 4, cudaMemcpyHostToDevice, st);
  td_launch_segment_mean3(d_src, dptr.as<int>(), n_segments, o4.as<float4>(), st);
  td_launch_gather_xyz(o4.as<float4>(), nullptr, n_segments, d_out, st);
  cudaError_t ce = cudaStreamSynchronize(st);
  if (ce == cudaSuccess) ce = cudaGetLastError();
  dptr.release(); o4.release();
  if (ce != cudaSuccess) return set_err(TDIFF_ECUDA, "scatter_mean3: %s", cudaGetErrorString(ce));
  return TDIFF_OK;
}

extern "C" int tdiff_check_stability(const float* d_pos, const int32_t* d_atomic_num, const int32_t* h_counts, int n_mol, int hs, int32_t* d_nr_bonds,
                                     int32_t* d_stable_atoms, uint8_t* d_mol_stable, void* stream) {
  if (!d_pos || !d_atomic_num || !h_counts || !d_stable_atoms || !d_mol_stable || n_mol < 0) return set_err(TDIFF_EINVAL, "check_stability: bad arguments");
  if (n_mol == 0) return TDIFF_OK;
  cudaStream_t st = (cudaStream_t)stream;
  std::vector<int> ptr(n_mol + 1, 0);
  for (int m = 0; m < n_mol; ++m) {
    if (h_counts[m] < 0) return set_err(TDIFF_EINVAL, "negative atom count");
    ptr[m + 1] = ptr[m] + h_counts[m];
  }
  DevBuf dptr, derr;
  if (dptr.ensure((n_mol + 1) * 4) || derr.ensure(4)) { dptr.release(); derr.release(); return set_err(TDIFF_ECUDA, "out of device memory"); }
  cudaMemcpyAsync(dptr.p, ptr.data(), (n_mol + 1) * 4, cudaMemcpyHostToDevice, st);
  cudaMemsetAsync(derr.p, 0, 4, st);
  td_launch_check_stability(d_pos, d_atomic_num, dptr.as<int>(), n_mol, hs, d_nr_bonds, d_stable_atoms, d_mol_stable, derr.as<int>(), st);
  int flag = 0;
  cudaMemcpyAsync(&flag, derr.p, 4, cudaMemcpyDeviceToHost, st);
  cudaError_t ce = cudaStreamSynchronize(st);
  if (ce == cudaSuccess) ce = cudaGetLastError();
  dptr.release(); derr.release();
  if (ce != cudaSuccess) return set_err(TDIFF_ECUDA, "check_stability: %s", cudaGetErrorString(ce));
  if (flag) return set_err(TDIFF_EINVAL, "check_stability: atomic number outside the reference's table (H C N O F P S Cl)");
  return TDIFF_OK;
}

// ---------------------------------------------------------------------------------------------- instrumentation
extern "C" int64_t tdiff_launch_count(tdiff_engine* e) { return e ? e->launches : 0; }
extern "C" int tdiff_edge_mlp_mode(tdiff_engine* e) { return !e ? TDIFF_EINVAL : (e->mlp_mode == 2 && e->mlp_v4) ? 5 : e->mlp_mode; }

extern "C" int tdiff_profile(tdiff_engine* e, int enable) {
  if (!e) return set_err(TDIFF_EINVAL, "null engine");
  e->profiling = enable != 0;
  if (enable) {
    for (int i = 0; i < EV_KINDS; ++i) { e->ms_acc[i] = 0; e->n_acc[i] = 0; }
  }
  return TDIFF_OK;
}

extern "C" int tdiff_profile_read(tdiff_engine* e, double* ms_h, int64_t* n_h, double* ms_x, int64_t* n_x, double* ms_mlp, int64_t* n_mlp,
                                  double* ms_total) {
  if (!e) return set_err(TDIFF_EINVAL, "null engine");
  CK(cudaSetDevice(e->device));
  CK(cudaDeviceSynchronize());
  for (auto& ev : e->events) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ev.a, ev.b) == cudaSuccess) { e->ms_acc[ev.kind] += ms; e->n_acc[ev.kind] += 1; }
    cudaEventDestroy(ev.a); cudaEventDestroy(ev.b);
  }
  e->events.clear();
  if (ms_h) *ms_h = e->ms_acc[EV_AGG_H];
  if (n_h) *n_h = e->n_acc[EV_AGG_H];
  if (ms_x) *ms_x = e->ms_acc[EV_AGG_X];
  if (n_x) *n_x = e->n_acc[EV_AGG_X];
  if (ms_mlp) *ms_mlp = e->ms_acc[EV_EDGE_MLP];
  if (n_mlp) *n_mlp = e->n_acc[EV_EDGE_MLP];
  if (ms_total) *ms_total = e->ms_acc[EV_TOTAL];
  return TDIFF_OK;
}
