// prop.cu -- binding-affinity regressor (PropPredNet / PropPredNetEnc with the EnEquiEncoder) on the 5th-gen tensor cores.
//
// Reference: models/property_pred/prop_model.py:27-165, models/property_pred/prop_egnn.py:8-83 (update_x=False, norm=False, ReLU).
// Per layer, with W1 [256 x (G+512)] split exactly by column blocks [gaussians | h_dst | h_src]:
//   P = h . [W1_dst ; W1_src]^T                                   node GEMM, [N,256] x [256,512]
//   m = relu(W2 . relu(G(d) . W1_g^T + P_dst[dst] + P_src[src] + b1) + b2)        edge kernel, per (dst, slot)
//   e = sigmoid(w . m + b),  mi[dst] = sum_slots e * m                             fused in the edge kernel's epilogue
//   h = h + node_mlp([mi | h])                                    node GEMMs, [N,512] x [512,256] and [N,256] x [256,256]
//
// Every matrix product runs on tcgen05.mma kind::f16 in the project's fp32-faithful split: each fp32 operand is x = x1 + x2 with
// x1 = bf16(x), x2 = bf16(x - x1) (16 mantissa bits), and a.b = a1b1 + a1b2 + a2b1 is accumulated in fp32 in TMEM.  Weight pieces
// are pre-swizzled on the host into the K-major SWIZZLE_128B shared-memory image (one 64-wide K chunk = [rows x 128 B] per piece).
//
// Edge tile (DESIGN.md section 9): 128 rows = 2 destinations x 64 neighbour slots.  Slots j >= k and absent neighbours (-1, graphs
// with <= k atoms) are zero rows.  Padding each destination to 64 rows costs 64/48 = 1.33x the MMA work at k = 48, and buys:
//   * an aggregation that is a fixed-order column sum over the 64 rows of one destination, read back from shared memory: no atomics,
//     no [E,256] message tensor in HBM, and a destination's result never depends on which other destinations share its tile
//     (a complex scored alone is bit-identical to the same complex inside a batch);
//   * TMEM: D1 (first Linear, 256 columns) + D2 (second Linear, 256 columns) = all 512 columns, so one CTA per SM.
// W2's two bf16 pieces are 2 x 128 KB and do not fit next to the activation tile, so W2 is streamed in four K-chunks of 64 KB
// (both pieces) through one 64 KB buffer that first holds the gaussian block W1_g.  Shared memory: 128 KB activations + 64 KB weights.
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/tdiff.h"
#include "tdiff_common.cuh"

namespace {

constexpr int kH = 256;                     // hidden width the kernels are built for
constexpr int kChunkA = 128 * 128;          // one A piece chunk: 128 rows x 64 bf16 (128 B) = 16 KB
constexpr int kChunkB = kH * 128;           // one B piece chunk: 256 rows x 128 B = 32 KB

// ------------------------------------------------------------------------------------------------ PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tPROP_WAIT:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra PROP_DONE;\n\tbra PROP_WAIT;\n\tPROP_DONE:\n\t}" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
template <int NCOLS>
__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "n"(NCOLS) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int NCOLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(NCOLS) : "memory");
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&f)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
        "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) f[i] = __uint_as_float(r[i]);
}
// K-major SWIZZLE_128B descriptor, 8-row groups 1024 B apart (same fields as edge_mlp_tc.cu)
__device__ __forceinline__ uint64_t desc_sw128(uint32_t a) {
  return (uint64_t)((a >> 4) & 0x3FFF) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
// F32 accumulate, BF16 A/B, both K-major, N = 256, M = 128
constexpr uint32_t kIdesc256 = (1u << 4) | (1u << 7) | (1u << 10) | ((256u >> 3) << 17) | ((128u >> 4) << 24);

__device__ __forceinline__ uint32_t cvt_bf16x2(float hi, float lo) {
  uint32_t d;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
  return d;
}
__device__ __forceinline__ void sts128(uint32_t addr, uint4 v) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
// 8 consecutive K values of `row` (16-byte chunk `c16` of a 64-wide K chunk) -> two bf16 pieces at a_chunk and a_chunk + kChunkA
__device__ __forceinline__ void store_split8(uint32_t a_chunk, int row, int c16, const float (&v)[8]) {
  const uint32_t off = row * 128 + ((c16 ^ (row & 7)) << 4);
  uint32_t hi[4], lo[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    hi[i] = cvt_bf16x2(v[2 * i + 1], v[2 * i]);
    const float r0 = v[2 * i] - __uint_as_float(hi[i] << 16), r1 = v[2 * i + 1] - __uint_as_float(hi[i] & 0xffff0000u);   // exact
    lo[i] = cvt_bf16x2(r1, r0);
  }
  sts128(a_chunk + off, make_uint4(hi[0], hi[1], hi[2], hi[3]));
  sts128(a_chunk + kChunkA + off, make_uint4(lo[0], lo[1], lo[2], lo[3]));
}
// one 64-wide K chunk of both weight pieces (2 x 32 KB, already in the smem image layout) -> shared memory, all threads
__device__ __forceinline__ void load_b_chunk(unsigned char* sB, const unsigned char* img_piece0, size_t piece_stride) {
  uint4* d = reinterpret_cast<uint4*>(sB);
  const uint4* s0 = reinterpret_cast<const uint4*>(img_piece0);
  const uint4* s1 = reinterpret_cast<const uint4*>(img_piece0 + piece_stride);
  for (int i = threadIdx.x; i < kChunkB / 16; i += blockDim.x) {
    d[i] = __ldg(s0 + i);
    d[kChunkB / 16 + i] = __ldg(s1 + i);
  }
}
// D (+)= A.B^T over one 64-wide K chunk: a1b1, a1b2, a2b1 (smallest terms last), 4 instructions of K = 16 each
__device__ __forceinline__ void mma_chunk(uint32_t d_tmem, uint32_t a_chunk, uint32_t b_chunk, bool accumulate) {
  uint32_t acc = accumulate ? 1u : 0u;
#pragma unroll
  for (int t = 0; t < 3; ++t) {
    const int pa = t == 2 ? 1 : 0, pb = t == 1 ? 1 : 0;
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      umma_bf16(d_tmem, desc_sw128(a_chunk + pa * kChunkA + kk * 32), desc_sw128(b_chunk + pb * kChunkB + kk * 32), kIdesc256, acc);
      acc = 1;
    }
  }
}

// ------------------------------------------------------------------------------------------------ node GEMM
// out[row, 256*y + c] = act(sum_k A[row,k] W[256*y + c, k] + bias[256*y + c]) (+ residual[row, ...]),  A = [a0[:, :k0] | a1[:, :k1] | 0 pad].
// One CTA (4 warps) per 128 rows x 256 columns; thread t owns tile row t (TMEM lane t).  out_rows (optional) scatters row i to out_rows[i].
struct GemmArgs {
  const float* a0; int lda0, k0;
  const float* a1; int lda1, k1;
  int m, kp;                  // rows, K padded to a multiple of 64
  const unsigned char* w_img; int n_img;   // image of W [n_img x kp]
  const float* bias; int relu;
  const float* residual;      // [m, ldo] or nullptr (added after the bias: h + (W x + b))
  float* out; int ldo;
  const int* out_rows;
};

__device__ __forceinline__ void load_a8(const GemmArgs& g, long long row, int kc, float (&v)[8]) {
  if (row >= g.m) {
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = 0.f;
    return;
  }
  if (kc + 8 <= g.k0 && ((g.lda0 | kc) & 3) == 0 && (reinterpret_cast<uintptr_t>(g.a0) & 15) == 0) {
    const float4* p = reinterpret_cast<const float4*>(g.a0 + (size_t)row * g.lda0 + kc);
    const float4 x = __ldg(p), y = __ldg(p + 1);
    v[0] = x.x; v[1] = x.y; v[2] = x.z; v[3] = x.w; v[4] = y.x; v[5] = y.y; v[6] = y.z; v[7] = y.w;
    return;
  }
  if (kc >= g.k0 && kc + 8 <= g.k0 + g.k1 && ((g.lda1 | (kc - g.k0)) & 3) == 0 && (reinterpret_cast<uintptr_t>(g.a1) & 15) == 0) {
    const float4* p = reinterpret_cast<const float4*>(g.a1 + (size_t)row * g.lda1 + (kc - g.k0));
    const float4 x = __ldg(p), y = __ldg(p + 1);
    v[0] = x.x; v[1] = x.y; v[2] = x.z; v[3] = x.w; v[4] = y.x; v[5] = y.y; v[6] = y.z; v[7] = y.w;
    return;
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int k = kc + i;
    v[i] = k < g.k0 ? g.a0[(size_t)row * g.lda0 + k] : (k < g.k0 + g.k1 ? g.a1[(size_t)row * g.lda1 + (k - g.k0)] : 0.f);
  }
}

__global__ void __launch_bounds__(128) prop_gemm_kernel(GemmArgs g) {
  extern __shared__ unsigned char smem_raw[];
  unsigned char* base = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  unsigned char* sA = base;                          // 2 pieces x 16 KB
  unsigned char* sB = sA + 2 * kChunkA;              // 2 pieces x 32 KB
  uint64_t* bar = reinterpret_cast<uint64_t*>(sB + 2 * kChunkB);
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(bar + 1);
  const int tid = threadIdx.x, warp = tid >> 5;
  if (tid == 0) { mbar_init(smem_u32(bar), 1); fence_barrier_init(); }
  if (warp == 0) tmem_alloc<256>(smem_u32(s_tmem));
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *s_tmem;
  const long long row = (long long)blockIdx.x * 128 + tid;
  const int y = blockIdx.y;
  const int nk = g.kp / 64;
  for (int c = 0; c < nk; ++c) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float v[8];
      load_a8(g, row, c * 64 + j * 8, v);
      store_split8(smem_u32(sA), tid, j, v);
    }
    load_b_chunk(sB, g.w_img + (size_t)c * 2 * g.n_img * 128 + (size_t)y * kChunkB, (size_t)g.n_img * 128);
    fence_proxy_async();
    __syncthreads();
    if (tid == 0) {
      tc_fence_after();
      mma_chunk(tmem, smem_u32(sA), smem_u32(sB), c > 0);
      umma_commit(smem_u32(bar));
    }
    mbar_wait(smem_u32(bar), (uint32_t)(c & 1));      // the MMAs have read sA / sB: they may be overwritten
    tc_fence_after();
  }
  // tcgen05.ld is warp-collective: every lane loads, only rows < m store
  const bool live = row < g.m;
  const long long orow = live ? (g.out_rows ? g.out_rows[row] : row) : 0;
  float* o = g.out + (size_t)orow * g.ldo + y * kH;
  const float* res = g.residual ? g.residual + (size_t)orow * g.ldo + y * kH : nullptr;
  const float* b = g.bias + y * kH;
#pragma unroll 1
  for (int c0 = 0; c0 < kH; c0 += 32) {
    float f[32];
    tmem_ld32(tmem + ((uint32_t)(warp * 32) << 16) + (uint32_t)c0, f);
    if (!live) continue;
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      float t = f[i] + b[c0 + i];
      if (g.relu) t = fmaxf(t, 0.f);
      if (res) t = res[c0 + i] + t;
      f[i] = t;
    }
#pragma unroll
    for (int i = 0; i < 32; i += 4) *reinterpret_cast<float4*>(o + c0 + i) = make_float4(f[i], f[i + 1], f[i + 2], f[i + 3]);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) { tc_fence_after(); tmem_dealloc<256>(tmem); }
}

// ------------------------------------------------------------------------------------------------ edge kernel
struct EdgeArgs {
  const float4* pos;          // [n] composed positions
  const int* src;             // [n*k] neighbour slots, -1 = absent
  const float* P;             // [n, 512]: h . W1_dst^T | h . W1_src^T
  const unsigned char* wg_img;   // W1 gaussian block [256 x 64] image
  const unsigned char* w2_img;   // W2 [256 x 256] image
  const float* b1; const float* b2; const float* wgate; float bgate;
  const float* offsets; int n_gauss; float coeff;
  int n, k;
  float* mi;                  // [n, 256]
};

__global__ void __launch_bounds__(128, 1) prop_edge_kernel(EdgeArgs a) {
  extern __shared__ unsigned char smem_raw[];
  unsigned char* base = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  unsigned char* sA = base;                          // 4 K-chunks x 2 pieces x 16 KB (chunk 0 first holds the gaussian tile)
  unsigned char* sB = sA + 8 * kChunkA;              // 2 pieces x 32 KB; reused as the [128][33] reduction buffer at the end
  uint64_t* bar = reinterpret_cast<uint64_t*>(sB + 2 * kChunkB);
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(bar + 1);
  const int tid = threadIdx.x, warp = tid >> 5;
  if (tid == 0) { mbar_init(smem_u32(bar), 1); fence_barrier_init(); }
  if (warp == 0) tmem_alloc<512>(smem_u32(s_tmem));
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *s_tmem;
  const uint32_t d1 = tmem, d2 = tmem + 256;
  const uint32_t lane_off = (uint32_t)(warp * 32) << 16;

  // row -> (destination, slot)
  const int dst = blockIdx.x * 2 + (tid >> 6), slot = tid & 63;
  int s = -1;
  if (dst < a.n && slot < a.k) s = a.src[(size_t)dst * a.k + slot];
  const bool valid = s >= 0;
  // ---- gaussian tile (K = 64) + W1_g
  {
    float dist = 0.f;
    if (valid) {
      const float4 p = a.pos[dst], q = a.pos[s];
      const float dx = p.x - q.x, dy = p.y - q.y, dz = p.z - q.z;
      dist = sqrtf(__fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz)));
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float v[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int gi = j * 8 + i;
        float t = 0.f;
        if (valid && gi < a.n_gauss) {
          const float d = dist - a.offsets[gi];
          t = expf(a.coeff * (d * d));
        }
        v[i] = t;
      }
      store_split8(smem_u32(sA), tid, j, v);
    }
  }
  load_b_chunk(sB, a.wg_img, (size_t)kChunkB);
  fence_proxy_async();
  __syncthreads();
  uint32_t phase = 0;
  if (tid == 0) {
    tc_fence_after();
    mma_chunk(d1, smem_u32(sA), smem_u32(sB), false);
    umma_commit(smem_u32(bar));
  }
  mbar_wait(smem_u32(bar), phase);
  phase ^= 1;
  tc_fence_after();
  // ---- + P_dst[dst] + P_src[src] + b1, ReLU -> second-Linear activation tile (zero rows for absent edges)
  {
    const float* pd = a.P + (size_t)(valid ? dst : 0) * 512;
    const float* ps = a.P + (size_t)(valid ? s : 0) * 512 + 256;
#pragma unroll 1
    for (int c0 = 0; c0 < kH; c0 += 32) {
      float f[32];
      tmem_ld32(d1 + lane_off + (uint32_t)c0, f);
#pragma unroll
      for (int i = 0; i < 32; i += 4) {
        const float4 x = __ldg(reinterpret_cast<const float4*>(pd + c0 + i)), z = __ldg(reinterpret_cast<const float4*>(ps + c0 + i));
        const float4 b = __ldg(reinterpret_cast<const float4*>(a.b1 + c0 + i));
        f[i] = valid ? fmaxf(((f[i] + b.x) + x.x) + z.x, 0.f) : 0.f;
        f[i + 1] = valid ? fmaxf(((f[i + 1] + b.y) + x.y) + z.y, 0.f) : 0.f;
        f[i + 2] = valid ? fmaxf(((f[i + 2] + b.z) + x.z) + z.z, 0.f) : 0.f;
        f[i + 3] = valid ? fmaxf(((f[i + 3] + b.w) + x.w) + z.w, 0.f) : 0.f;
      }
      const uint32_t chunk = smem_u32(sA) + (uint32_t)(c0 >> 6) * 2 * kChunkA;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = f[j * 8 + i];
        store_split8(chunk, tid, ((c0 & 63) >> 3) + j, v);
      }
    }
  }
  // ---- second Linear, W2 streamed in four K-chunks
#pragma unroll 1
  for (int c = 0; c < 4; ++c) {
    load_b_chunk(sB, a.w2_img + (size_t)c * 2 * kChunkB, (size_t)kChunkB);
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    if (tid == 0) {
      tc_fence_after();
      mma_chunk(d2, smem_u32(sA) + c * 2 * kChunkA, smem_u32(sB), c > 0);
      umma_commit(smem_u32(bar));
    }
    mbar_wait(smem_u32(bar), phase);
    phase ^= 1;
    tc_fence_after();
  }
  // ---- epilogue: m = relu(D2 + b2); e = sigmoid(w . m + b); mi[dst] = sum over the destination's 64 rows of e*m (fixed order)
  float dot = 0.f;
#pragma unroll 1
  for (int c0 = 0; c0 < kH; c0 += 32) {
    float f[32];
    tmem_ld32(d2 + lane_off + (uint32_t)c0, f);
#pragma unroll
    for (int i = 0; i < 32; ++i) dot = fmaf(fmaxf(f[i] + __ldg(a.b2 + c0 + i), 0.f), __ldg(a.wgate + c0 + i), dot);
  }
  const float e = valid ? 1.0f / (1.0f + expf(-(dot + a.bgate))) : 0.f;
  float* red = reinterpret_cast<float*>(sB);         // [128][33]
  const int out_dst = blockIdx.x * 2 + (tid >> 5 & 1), col = tid & 31;
#pragma unroll 1
  for (int c0 = 0; c0 < kH; c0 += 32) {
    float f[32];
    tmem_ld32(d2 + lane_off + (uint32_t)c0, f);
#pragma unroll
    for (int i = 0; i < 32; ++i) red[tid * 33 + i] = e * fmaxf(f[i] + __ldg(a.b2 + c0 + i), 0.f);
    __syncthreads();
    if (tid < 64) {                                  // thread (d, col): rows d*64 .. d*64+63 in slot order
      const float* r = red + (tid >> 5) * 64 * 33 + col;
      float sum = 0.f;
#pragma unroll 8
      for (int j = 0; j < 64; ++j) sum += r[j * 33];
      if (out_dst < a.n) a.mi[(size_t)out_dst * kH + c0 + col] = sum;
    }
    __syncthreads();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) { tc_fence_after(); tmem_dealloc<512>(tmem); }
}

// ------------------------------------------------------------------------------------------------ small kernels
__global__ void compose_pos_kernel(const float* __restrict__ ppos, const float* __restrict__ lpos, const int* __restrict__ prow,
                                   const int* __restrict__ lrow, int np, int nl, float4* __restrict__ pos) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < np) pos[prow[i]] = make_float4(ppos[3 * i], ppos[3 * i + 1], ppos[3 * i + 2], 0.f);
  else if (i < np + nl) {
    const int j = i - np;
    pos[lrow[j]] = make_float4(lpos[3 * j], lpos[3 * j + 1], lpos[3 * j + 2], 0.f);
  }
}

// pre[g] = [sum over the graph's nodes of h | enc_graph[g]]   (sequential node order per column: deterministic)
__global__ void pool_kernel(const float* __restrict__ h, const int* __restrict__ node_ptr, const float* __restrict__ enc_graph, int gdim,
                            float* __restrict__ pre) {
  const int g = blockIdx.x, w = kH + gdim;
  for (int c = threadIdx.x; c < w; c += blockDim.x) {
    float s = 0.f;
    if (c < kH) {
      for (int n = node_ptr[g]; n < node_ptr[g + 1]; ++n) s += h[(size_t)n * kH + c];
    } else {
      s = enc_graph[(size_t)g * gdim + (c - kH)];
    }
    pre[(size_t)g * w + c] = s;
  }
}

// out_block: Linear(256+gdim, 256) -> ShiftedSoftplus -> Linear(256, out_dim), then the output_kind column select
__global__ void readout_kernel(const float* __restrict__ pre, int kin, const float* __restrict__ w0, const float* __restrict__ b0,
                               const float* __restrict__ w2, const float* __restrict__ b2, int out_dim, const long long* __restrict__ kind,
                               float* __restrict__ out, int* __restrict__ err) {
  __shared__ float y[kH];
  const int g = blockIdx.x, c = threadIdx.x;
  const float* x = pre + (size_t)g * kin;
  float s = 0.f;
  for (int k = 0; k < kin; ++k) s = fmaf(w0[(size_t)c * kin + k], x[k], s);
  s += b0[c];
  const float sp = s > 20.f ? s : log1pf(expf(s));                 // F.softplus (beta 1, threshold 20)
  y[c] = sp - 0.6931471824645996f;                                  // - fp32(log 2)  (models/common.py:156-162)
  __syncthreads();
  if (c < out_dim) {
    float o = 0.f;
    for (int k = 0; k < kH; ++k) o = fmaf(w2[(size_t)c * kH + k], y[k], o);
    o += b2[c];
    if (!kind) {
      out[(size_t)g * out_dim + c] = o;
    } else {
      const long long kd = kind[g];
      if (kd < 1 || kd > out_dim) { if (c == 0) atomicExch(err, 1); }
      else if (kd - 1 == c) out[g] = o;
    }
  }
}

uint16_t bf16_rn_host(float x) {
  uint32_t u;
  memcpy(&u, &x, 4);
  if ((u & 0x7fffffffu) > 0x7f800000u) return (uint16_t)((u >> 16) | 0x40);
  u += 0x7fffu + ((u >> 16) & 1u);
  return (uint16_t)(u >> 16);
}
float bf16_f_host(uint16_t b) {
  const uint32_t u = (uint32_t)b << 16;
  float f;
  memcpy(&f, &u, 4);
  return f;
}

// W[n][k] = get(n, k) for n < nrows, k < K (zero for K <= k < kp) -> two bf16 pieces, per 64-wide K chunk: piece 0 then piece 1,
// each [nrows x 128 B] in the K-major SWIZZLE_128B layout (16-byte chunk index XOR row % 8)
template <class Get>
std::vector<unsigned char> pack_image(int nrows, int K, int kp, Get get) {
  std::vector<unsigned char> img((size_t)kp * nrows * 4, 0);
  for (int n = 0; n < nrows; ++n)
    for (int k = 0; k < K; ++k) {
      const float w = get(n, k);
      const uint16_t hi = bf16_rn_host(w), lo = bf16_rn_host(w - bf16_f_host(hi));
      const size_t o = (size_t)(k / 64) * 2 * nrows * 128 + (size_t)n * 128 + (size_t)((((k % 64) / 8) ^ (n & 7)) * 16) + (size_t)(k % 8) * 2;
      memcpy(&img[o], &hi, 2);
      memcpy(&img[o + (size_t)nrows * 128], &lo, 2);
    }
  return img;
}

struct PBuf {
  void* p = nullptr;
  size_t cap = 0;
  int ensure(size_t bytes) {
    if (bytes <= cap) return 0;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    if (cudaMalloc(&p, bytes) != cudaSuccess) { (void)cudaGetLastError(); return -1; }
    cap = bytes;
    static const bool poison = getenv("TDIFF_POISON") != nullptr;     // test switch: see DevBuf in engine.cu
    if (poison) cudaMemset(p, 0xFF, bytes);
    return 0;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
  template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

struct PropLayer {
  const unsigned char *wds, *wg, *w2, *wn0, *wn2;
  const float *b1, *b2, *wgate, *bn0, *bn2;
  float bgate;
};

}  // namespace

struct tdiff_prop {
  tdiff_prop_config cfg;
  int device = 0;
  float coeff = 0.f;
  std::vector<void*> allocs;
  const float *offsets = nullptr, *zero512 = nullptr;
  const unsigned char *emb_p = nullptr, *emb_l = nullptr, *enc0 = nullptr, *enc2 = nullptr;
  const float *emb_pb = nullptr, *emb_lb = nullptr, *enc0b = nullptr, *enc2b = nullptr, *out_w0 = nullptr, *out_b0 = nullptr, *out_w2 = nullptr,
              *out_b2 = nullptr;
  std::vector<PropLayer> layers;
  PBuf pos, maps, src, h, P, mi, tmp, pre, err;
  bool profiling = false;
  double ms_edge = 0.0;
  long long n_edge = 0, n_edge_rows = 0;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
};

namespace {

template <class T>
const T* upload(tdiff_prop* p, const void* data, size_t bytes) {
  void* d = nullptr;
  if (cudaMalloc(&d, bytes) != cudaSuccess) return nullptr;
  p->allocs.push_back(d);
  if (cudaMemcpy(d, data, bytes, cudaMemcpyHostToDevice) != cudaSuccess) return nullptr;
  return reinterpret_cast<const T*>(d);
}

int kpad(int k) { return (k + 63) / 64 * 64; }

void launch_gemm(const GemmArgs& g, cudaStream_t st) {
  if (g.m <= 0) return;
  const size_t smem = 1024 + 2 * kChunkA + 2 * kChunkB + 64;
  static size_t opted[TD_MAX_DEVICES] = {0};
  td_opt_in_smem(prop_gemm_kernel, smem, opted);
  dim3 grid((unsigned)((g.m + 127) / 128), (unsigned)(g.n_img / kH));
  prop_gemm_kernel<<<grid, 128, smem, st>>>(g);
}

void launch_edge(const EdgeArgs& a, cudaStream_t st) {
  if (a.n <= 0) return;
  const size_t smem = 1024 + 8 * kChunkA + 2 * kChunkB + 64;
  static size_t opted[TD_MAX_DEVICES] = {0};
  td_opt_in_smem(prop_edge_kernel, smem, opted);
  prop_edge_kernel<<<(unsigned)((a.n + 1) / 2), 128, smem, st>>>(a);
}

GemmArgs gemm(const float* a0, int lda0, int k0, const float* a1, int lda1, int k1, int m, const unsigned char* img, int n_img, const float* bias,
              int relu, const float* residual, float* out, int ldo, const int* out_rows) {
  GemmArgs g;
  g.a0 = a0; g.lda0 = lda0; g.k0 = k0; g.a1 = a1; g.lda1 = lda1; g.k1 = k1;
  g.m = m; g.kp = kpad(k0 + k1); g.w_img = img; g.n_img = n_img; g.bias = bias; g.relu = relu; g.residual = residual;
  g.out = out; g.ldo = ldo; g.out_rows = out_rows;
  return g;
}

}  // namespace

extern "C" void tdiff_prop_destroy(tdiff_prop* p) {
  if (!p) return;
  cudaSetDevice(p->device);
  for (void* a : p->allocs) cudaFree(a);
  p->pos.release(); p->maps.release(); p->src.release(); p->h.release(); p->P.release(); p->mi.release(); p->tmp.release();
  p->pre.release(); p->err.release();
  if (p->ev0) cudaEventDestroy(p->ev0);
  if (p->ev1) cudaEventDestroy(p->ev1);
  delete p;
}

extern "C" int tdiff_prop_create(const tdiff_prop_config* cfg, const tdiff_tensor* sd, int n_entries, int device, tdiff_prop** out) {
  if (!cfg || !sd || !out || n_entries < 0) return td_set_err(TDIFF_EINVAL, "null argument");
  *out = nullptr;
  const tdiff_prop_config& c = *cfg;
  if (c.hidden_dim != kH) return td_set_err(TDIFF_EINVAL, "hidden_dim=%d: the kernels are built for 256", c.hidden_dim);
  if (c.knn < 1 || c.knn > TD_KMAX) return td_set_err(TDIFF_EINVAL, "knn=%d outside 1..%d", c.knn, TD_KMAX);
  if (c.num_r_gaussian < 2 || c.num_r_gaussian > 64) return td_set_err(TDIFF_EINVAL, "num_r_gaussian=%d outside 2..64", c.num_r_gaussian);
  if (c.edge_dim != 0 || c.norm != 0) return td_set_err(TDIFF_EINVAL, "edge_dim=%d norm=%d: only edge_dim 0 and norm False are implemented", c.edge_dim, c.norm);
  if (c.num_layers < 1 || c.protein_feat_dim < 1 || c.ligand_feat_dim < 1 || c.enc_ligand_dim < 0 || c.enc_node_dim < 0 || c.enc_graph_dim < 0 ||
      c.output_dim < 1 || c.output_dim > 32)
    return td_set_err(TDIFF_EINVAL, "bad config (num_layers=%d protein_feat_dim=%d ligand_feat_dim=%d enc dims %d/%d/%d output_dim=%d)", c.num_layers,
                      c.protein_feat_dim, c.ligand_feat_dim, c.enc_ligand_dim, c.enc_node_dim, c.enc_graph_dim, c.output_dim);
  if (c.protein_feat_dim + 0 > 4096 || c.ligand_feat_dim + c.enc_ligand_dim > 4096 || c.enc_node_dim > 4096 || c.enc_graph_dim > 4096)
    return td_set_err(TDIFF_EINVAL, "feature width above 4096");
  for (int r : c.reserved)
    if (r != 0) return td_set_err(TDIFF_EINVAL, "tdiff_prop_config.reserved must be 0");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    (void)cudaGetLastError();
    return td_set_err(TDIFF_ECUDA, "no CUDA device: libtdiff has no CPU fallback");
  }
  if (device < 0 || device >= ndev) return td_set_err(TDIFF_EINVAL, "device %d out of range (%d devices)", device, ndev);
  if (cudaSetDevice(device) != cudaSuccess) return td_set_err(TDIFF_ECUDA, "cudaSetDevice(%d) failed", device);
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess || prop.major < 10)
    return td_set_err(TDIFF_ECUDA, "device %d is not sm_100a; this library is built for sm_100a only", device);

  // ---- state_dict lookup: every entry must be known and every expected entry present with its shape
  const int H = kH, G = c.num_r_gaussian, L = c.num_layers;
  std::vector<std::pair<std::string, long long>> want;
  auto lin = [&](const std::string& k, long long o, long long i) { want.push_back({k + ".weight", o * i}); want.push_back({k + ".bias", o}); };
  lin("protein_atom_emb", H, c.protein_feat_dim);
  lin("ligand_atom_emb", H, c.ligand_feat_dim + c.enc_ligand_dim);
  want.push_back({"encoder.distance_expansion.offset", G});
  for (int l = 0; l < L; ++l) {
    const std::string p = "encoder.net." + std::to_string(l);
    want.push_back({p + ".r_expansion.offset", G});
    lin(p + ".edge_mlp.net.0", H, 2 * H + G);
    lin(p + ".edge_mlp.net.2", H, H);
    lin(p + ".edge_inf.0", 1, H);
    lin(p + ".node_mlp.net.0", H, 2 * H);
    lin(p + ".node_mlp.net.2", H, H);
  }
  if (c.enc_node_dim > 0) { lin("enc_node_layer.0", H, H + c.enc_node_dim); lin("enc_node_layer.2", H, H); }
  lin("out_block.0", H, H + c.enc_graph_dim);
  lin("out_block.2", c.output_dim, H);
  std::vector<const float*> got(want.size(), nullptr);
  for (int i = 0; i < n_entries; ++i) {
    if (!sd[i].name || !sd[i].data) return td_set_err(TDIFF_EWEIGHT, "state_dict entry %d has no name or data", i);
    size_t j = 0;
    while (j < want.size() && want[j].first != sd[i].name) ++j;
    if (j == want.size()) return td_set_err(TDIFF_EWEIGHT, "unexpected state_dict entry %s", sd[i].name);
    if (sd[i].numel != want[j].second)
      return td_set_err(TDIFF_EWEIGHT, "state_dict entry %s has %lld elements, expected %lld", sd[i].name, (long long)sd[i].numel, want[j].second);
    got[j] = sd[i].data;
  }
  for (size_t j = 0; j < want.size(); ++j)
    if (!got[j]) return td_set_err(TDIFF_EWEIGHT, "missing state_dict entry %s", want[j].first.c_str());
  auto W = [&](const std::string& k) {
    for (size_t j = 0; j < want.size(); ++j)
      if (want[j].first == k) return got[j];
    return (const float*)nullptr;
  };

  tdiff_prop* p = new tdiff_prop();
  p->cfg = c;
  p->device = device;
  bool ok = true;
  auto up = [&](const float* d, size_t n) { const float* r = upload<float>(p, d, n * 4); ok = ok && r; return r; };
  auto upimg = [&](const std::vector<unsigned char>& img) { const unsigned char* r = upload<unsigned char>(p, img.data(), img.size()); ok = ok && r; return r; };
  auto img_of = [&](const float* w, int nrows, int ld, int col0, int K) {
    return upimg(pack_image(nrows, K, kpad(K), [&](int n, int k) { return w[(size_t)n * ld + col0 + k]; }));
  };
  const float* off = W("encoder.distance_expansion.offset");
  p->offsets = up(off, G);
  p->coeff = (float)(-0.5 / std::pow((double)(off[1] - off[0]), 2.0));        // models/common.py:17 (.item() of the fp32 difference)
  std::vector<float> zeros(512, 0.f);
  p->zero512 = up(zeros.data(), 512);
  const int Kl = c.ligand_feat_dim + c.enc_ligand_dim;
  p->emb_p = img_of(W("protein_atom_emb.weight"), H, c.protein_feat_dim, 0, c.protein_feat_dim);
  p->emb_pb = up(W("protein_atom_emb.bias"), H);
  p->emb_l = img_of(W("ligand_atom_emb.weight"), H, Kl, 0, Kl);
  p->emb_lb = up(W("ligand_atom_emb.bias"), H);
  for (int l = 0; l < L && ok; ++l) {
    const std::string pre = "encoder.net." + std::to_string(l);
    const float* w1 = W(pre + ".edge_mlp.net.0.weight");
    const int ld1 = 2 * H + G;
    PropLayer ly;
    // [W1_dst ; W1_src] as one [512 x 256] weight: output columns 0-255 project destinations, 256-511 sources
    ly.wds = upimg(pack_image(2 * H, H, H, [&](int n, int k) { return w1[(size_t)(n % H) * ld1 + G + (n / H) * H + k]; }));
    ly.wg = img_of(w1, H, ld1, 0, G);
    ly.w2 = img_of(W(pre + ".edge_mlp.net.2.weight"), H, H, 0, H);
    ly.wn0 = img_of(W(pre + ".node_mlp.net.0.weight"), H, 2 * H, 0, 2 * H);
    ly.wn2 = img_of(W(pre + ".node_mlp.net.2.weight"), H, H, 0, H);
    ly.b1 = up(W(pre + ".edge_mlp.net.0.bias"), H);
    ly.b2 = up(W(pre + ".edge_mlp.net.2.bias"), H);
    ly.wgate = up(W(pre + ".edge_inf.0.weight"), H);
    ly.bgate = W(pre + ".edge_inf.0.bias")[0];
    ly.bn0 = up(W(pre + ".node_mlp.net.0.bias"), H);
    ly.bn2 = up(W(pre + ".node_mlp.net.2.bias"), H);
    p->layers.push_back(ly);
  }
  if (c.enc_node_dim > 0) {
    p->enc0 = img_of(W("enc_node_layer.0.weight"), H, H + c.enc_node_dim, 0, H + c.enc_node_dim);
    p->enc0b = up(W("enc_node_layer.0.bias"), H);
    p->enc2 = img_of(W("enc_node_layer.2.weight"), H, H, 0, H);
    p->enc2b = up(W("enc_node_layer.2.bias"), H);
  }
  p->out_w0 = up(W("out_block.0.weight"), (size_t)H * (H + c.enc_graph_dim));
  p->out_b0 = up(W("out_block.0.bias"), H);
  p->out_w2 = up(W("out_block.2.weight"), (size_t)c.output_dim * H);
  p->out_b2 = up(W("out_block.2.bias"), c.output_dim);
  if (ok) ok = cudaEventCreate(&p->ev0) == cudaSuccess && cudaEventCreate(&p->ev1) == cudaSuccess;
  if (!ok) {
    (void)cudaGetLastError();
    tdiff_prop_destroy(p);
    return td_set_err(TDIFF_ECUDA, "weight upload failed (out of device memory?)");
  }
  *out = p;
  return TDIFF_OK;
}

extern "C" int tdiff_prop_forward(tdiff_prop* p, int B, const int32_t* pc, const int32_t* lc, const float* d_ppos, const float* d_pfeat,
                                  const float* d_lpos, const float* d_lfeat, const float* d_enc_ligand, const float* d_enc_node,
                                  const float* d_enc_graph, const int64_t* d_kind, float* d_out, float* d_h_out, void* stream) {
  if (!p || !pc || !lc || B < 1 || !d_out) return td_set_err(TDIFF_EINVAL, "prop_forward: bad arguments");
  const tdiff_prop_config& c = p->cfg;
  if ((c.enc_ligand_dim > 0) != (d_enc_ligand != nullptr))
    return td_set_err(TDIFF_EINVAL, "enc_ligand_feature %s but the model has enc_ligand_dim=%d", d_enc_ligand ? "given" : "missing", c.enc_ligand_dim);
  if ((c.enc_graph_dim > 0) != (d_enc_graph != nullptr))
    return td_set_err(TDIFF_EINVAL, "enc_graph_feature %s but the model has enc_graph_dim=%d", d_enc_graph ? "given" : "missing", c.enc_graph_dim);
  if (d_enc_node && c.enc_node_dim == 0) return td_set_err(TDIFF_EINVAL, "enc_node_feature given but the model has no enc_node_layer");
  std::vector<int> node_ptr(B + 1, 0), prow, lrow;
  long long N = 0, Np = 0, Nl = 0;
  int max_ng = 0;
  for (int g = 0; g < B; ++g) {
    if (pc[g] < 0 || lc[g] < 0) return td_set_err(TDIFF_EINVAL, "negative atom count in graph %d", g);
    N += (long long)pc[g] + lc[g];
    if (N > (1LL << 31) / TD_KMAX) return td_set_err(TDIFF_EINVAL, "batch too large");
    node_ptr[g + 1] = (int)N;
    max_ng = pc[g] + lc[g] > max_ng ? pc[g] + lc[g] : max_ng;
  }
  if (max_ng > 2800) return td_set_err(TDIFF_EINVAL, "graph with %d atoms exceeds the k-NN kernel's shared-memory tile (2800)", max_ng);
  for (int g = 0; g < B; ++g) {
    for (int i = 0; i < pc[g]; ++i) prow.push_back(node_ptr[g] + i);
    for (int i = 0; i < lc[g]; ++i) lrow.push_back(node_ptr[g] + pc[g] + i);
  }
  Np = (long long)prow.size(); Nl = (long long)lrow.size();
  if (N == 0) return td_set_err(TDIFF_EINVAL, "empty batch");
  if ((Np > 0 && (!d_ppos || !d_pfeat)) || (Nl > 0 && (!d_lpos || !d_lfeat))) return td_set_err(TDIFF_EINVAL, "null atom arrays");
  if (cudaSetDevice(p->device) != cudaSuccess) return td_set_err(TDIFF_ECUDA, "cudaSetDevice failed");
  cudaStream_t st = (cudaStream_t)stream;
  const int k = c.knn, H = kH;
  if (p->pos.ensure((size_t)N * 16) || p->maps.ensure((size_t)(N + B + 1) * 4) || p->src.ensure((size_t)N * k * 4) ||
      p->h.ensure((size_t)N * H * 4) || p->P.ensure((size_t)N * 2 * H * 4) || p->mi.ensure((size_t)N * H * 4) || p->tmp.ensure((size_t)N * H * 4) ||
      p->pre.ensure((size_t)B * (H + c.enc_graph_dim) * 4) || p->err.ensure(4))
    return td_set_err(TDIFF_ECUDA, "out of device memory for a batch of %lld atoms", N);
  int* d_prow = p->maps.as<int>();
  int* d_lrow = d_prow + Np;
  int* d_ptr = d_lrow + Nl;
  // pageable host memory: the copies are staged before cudaMemcpyAsync returns
  if (Np) cudaMemcpyAsync(d_prow, prow.data(), Np * 4, cudaMemcpyHostToDevice, st);
  if (Nl) cudaMemcpyAsync(d_lrow, lrow.data(), Nl * 4, cudaMemcpyHostToDevice, st);
  cudaMemcpyAsync(d_ptr, node_ptr.data(), (B + 1) * 4, cudaMemcpyHostToDevice, st);
  cudaMemsetAsync(p->err.p, 0, 4, st);
  float4* pos = p->pos.as<float4>();
  float *h = p->h.as<float>(), *P = p->P.as<float>(), *mi = p->mi.as<float>(), *tmp = p->tmp.as<float>();
  compose_pos_kernel<<<(unsigned)((N + 255) / 256), 256, 0, st>>>(d_ppos, d_lpos, d_prow, d_lrow, (int)Np, (int)Nl, pos);
  // embeddings, written straight into the composed node order
  launch_gemm(gemm(d_pfeat, c.protein_feat_dim, c.protein_feat_dim, nullptr, 0, 0, (int)Np, p->emb_p, H, p->emb_pb, 0, nullptr, h, H, d_prow), st);
  launch_gemm(gemm(d_lfeat, c.ligand_feat_dim, c.ligand_feat_dim, d_enc_ligand, c.enc_ligand_dim, c.enc_ligand_dim, (int)Nl, p->emb_l, H, p->emb_lb, 0,
                   nullptr, h, H, d_lrow), st);
  td_launch_knn(pos, d_ptr, nullptr, B, max_ng, k, k, 0, p->src.as<int>(), st);
  for (const PropLayer& ly : p->layers) {
    launch_gemm(gemm(h, H, H, nullptr, 0, 0, (int)N, ly.wds, 2 * H, p->zero512, 0, nullptr, P, 2 * H, nullptr), st);
    EdgeArgs a;
    a.pos = pos; a.src = p->src.as<int>(); a.P = P; a.wg_img = ly.wg; a.w2_img = ly.w2; a.b1 = ly.b1; a.b2 = ly.b2; a.wgate = ly.wgate;
    a.bgate = ly.bgate; a.offsets = p->offsets; a.n_gauss = c.num_r_gaussian; a.coeff = p->coeff; a.n = (int)N; a.k = k; a.mi = mi;
    if (p->profiling) cudaEventRecord(p->ev0, st);
    launch_edge(a, st);
    if (p->profiling) {
      cudaEventRecord(p->ev1, st);
      cudaEventSynchronize(p->ev1);
      float ms = 0.f;
      cudaEventElapsedTime(&ms, p->ev0, p->ev1);
      p->ms_edge += ms;
      p->n_edge += 1;
      p->n_edge_rows += (N + 1) / 2 * 128;
    }
    launch_gemm(gemm(mi, H, H, h, H, H, (int)N, ly.wn0, H, ly.bn0, 1, nullptr, tmp, H, nullptr), st);
    launch_gemm(gemm(tmp, H, H, nullptr, 0, 0, (int)N, ly.wn2, H, ly.bn2, 0, h, h, H, nullptr), st);
  }
  if (d_h_out) cudaMemcpyAsync(d_h_out, h, (size_t)N * H * 4, cudaMemcpyDeviceToDevice, st);
  const float* hf = h;
  if (d_enc_node) {
    launch_gemm(gemm(h, H, H, d_enc_node, c.enc_node_dim, c.enc_node_dim, (int)N, p->enc0, H, p->enc0b, 1, nullptr, tmp, H, nullptr), st);
    launch_gemm(gemm(tmp, H, H, nullptr, 0, 0, (int)N, p->enc2, H, p->enc2b, 0, nullptr, mi, H, nullptr), st);
    hf = mi;
  }
  pool_kernel<<<B, 256, 0, st>>>(hf, d_ptr, d_enc_graph, c.enc_graph_dim, p->pre.as<float>());
  readout_kernel<<<B, kH, 0, st>>>(p->pre.as<float>(), H + c.enc_graph_dim, p->out_w0, p->out_b0, p->out_w2, p->out_b2, c.output_dim,
                                  (const long long*)d_kind, d_out, p->err.as<int>());
  int bad = 0;
  cudaMemcpyAsync(&bad, p->err.p, 4, cudaMemcpyDeviceToHost, st);
  cudaError_t ce = cudaStreamSynchronize(st);
  if (ce == cudaSuccess) ce = cudaGetLastError();
  if (ce != cudaSuccess) return td_set_err(TDIFF_ECUDA, "prop_forward: %s", cudaGetErrorString(ce));
  if (bad) return td_set_err(TDIFF_EINVAL, "output_kind outside 1..%d", c.output_dim);
  return TDIFF_OK;
}

extern "C" int tdiff_prop_profile(tdiff_prop* p, int enable) {
  if (!p) return td_set_err(TDIFF_EINVAL, "null model");
  p->profiling = enable != 0;
  if (enable) { p->ms_edge = 0.0; p->n_edge = 0; p->n_edge_rows = 0; }
  return TDIFF_OK;
}

extern "C" int tdiff_prop_profile_read(tdiff_prop* p, double* ms_edge, int64_t* n_edge, int64_t* n_rows) {
  if (!p) return td_set_err(TDIFF_EINVAL, "null model");
  if (ms_edge) *ms_edge = p->ms_edge;
  if (n_edge) *n_edge = p->n_edge;
  if (n_rows) *n_rows = p->n_edge_rows;
  return TDIFF_OK;
}
