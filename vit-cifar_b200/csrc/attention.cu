// attention.cu — fused short-sequence attention (layers.py:92-101), forward and backward.
//
// T is 17 or 65 (<= 128), head_dim 32 (64 for the scaled config; 96 and 128 as panels of those, see below): the whole (T x T) score tile of one
// (image, head) lives on chip.  bf16 path: one CTA per (image, head), one warp per 16 query rows,
// QKᵀ and PV on mma.sync.m16n8k16 bf16 tensor-core tiles fed by ldmatrix from padded shared memory
// (tcgen05's 128-row tiles do not fit a 65x65x32 problem), softmax in registers with quad shuffles;
// only the per-row log-sum-exp is kept for backward, which recomputes P.  fp32 path (check mode):
// plain FFMA with the score tile in shared memory.
#include <cuda.h>

#include "common.cuh"
#include "gemm_internal.h"

namespace vitb {

// ---------------------------------------------------------------------------------------------
// mma / ldmatrix wrappers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], const void* p) {
  const uint32_t a = (uint32_t)__cvta_generic_to_shared(p);
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(a));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t (&r)[4], const void* p) {
  const uint32_t a = (uint32_t)__cvta_generic_to_shared(p);
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(a));
}
__device__ __forceinline__ void stsm_x4(void* p, uint32_t r0, uint32_t r1, uint32_t r2, uint32_t r3) {
  const uint32_t a = (uint32_t)__cvta_generic_to_shared(p);
  asm volatile("stmatrix.sync.aligned.m8n8.x4.shared.b16 [%0], {%1,%2,%3,%4};" ::"r"(a), "r"(r0), "r"(r1), "r"(r2), "r"(r3) : "memory");
}
__device__ __forceinline__ void mma_bf16(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ float quad_sum(float v) {
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  v += __shfl_xor_sync(0xffffffffu, v, 2);
  return v;
}
__device__ __forceinline__ float quad_max(float v) {
  v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 1));
  v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 2));
  return v;
}

constexpr float kLog2e = 1.4426950408889634f;

__device__ __forceinline__ float ex2_fast(float x) {  // one MUFU.EX2; ex2(-inf) = 0
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// key-column masking without per-element selects: the T valid keys fill `nfull` 8-key tiles completely and `rem` columns of
// the next one; tiles beyond are never computed (their scores are -inf), the partial tile gets an additive 0 / -inf per thread.
struct KeyMask {
  int nfull, rem;
  float pm0, pm1;  // additive mask of this thread's two columns (2t, 2t+1) in the partial tile
};
__device__ __forceinline__ KeyMask make_key_mask(int T, int lane) {
  KeyMask m;
  m.nfull = T >> 3;
  m.rem = T & 7;
  const int t = lane & 3;
  m.pm0 = (2 * t < m.rem) ? 0.f : -INFINITY;
  m.pm1 = (2 * t + 1 < m.rem) ? 0.f : -INFINITY;
  return m;
}

// ---------------------------------------------------------------------------------------------
// TMA plumbing.  A head tile is a (D x T) box of a 3-D tensor map {columns, tokens, images}: one instruction loads it,
// token rows >= T are out of bounds and arrive as zeros (the padding the MMA tiles need), rows land densely (2*D bytes)
// under the hardware swizzle (64B for D = 32, 128B for D = 64) so ldmatrix is conflict-free without padding.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count)); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  long long t0 = 0;
  for (uint32_t it = 0;; ++it) {
    asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n" : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    if (done) return;
    if (it == 64) t0 = clock64();
    if (it > 64 && (it & 1023) == 0 && clock64() - t0 > 4000000000LL) {  // a protocol bug traps instead of hanging the GPU
      printf("vitb attention: mbarrier wait timed out (block %d thread %d)\n", blockIdx.x, threadIdx.x);
      __trap();
    }
  }
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(dst),
               "l"((uint64_t)map), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void tma_prefetch_3d(const CUtensorMap* map, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.prefetch.tensor.3d.L2.global [%0, {%1, %2, %3}];" ::"l"((uint64_t)map), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* map, uint32_t src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"((uint64_t)map), "r"(src), "r"(c0), "r"(c1),
               "r"(c2)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// byte offset of 16-byte chunk `chunk` of row `row` inside a swizzled (rows x D) bf16 tile
template <int D>
__device__ __forceinline__ uint32_t swz(int row) { return D == 32 ? (uint32_t)((row >> 1) & 3) : (uint32_t)(row & 7); }
template <int D>
__device__ __forceinline__ uint32_t tile_off(int row, uint32_t chunk) { return (uint32_t)row * (2 * D) + ((chunk ^ swz<D>(row)) << 4); }

// per-lane pieces of the three ldmatrix address patterns (all row offsets added later are multiples of 8: the swizzle term of a
// lane never changes, so an address is  base + (row0 + lane_row) * 2D + ((chunk0 ^ lane_x) << 4)  with chunk0 a constant)
template <int D>
struct LaneAddr {
  uint32_t a_row, a_x;  // A fragments (16 rows x 16 k):   row = lane & 15,                       chunk = 2 kk + (lane >> 4)
  uint32_t b_row, b_x;  // B fragments (8 keys x 32 k):    row = lane & 7,                        chunk = 4 k2 + (lane >> 3)
  uint32_t t_row, t_x;  // transposed B (16 k-rows x 16):  row = (lane & 7) + 8 ((lane >> 3) & 1), chunk = 2 jp + (lane >> 4)
  __device__ __forceinline__ LaneAddr(int lane) {
    a_row = lane & 15; a_x = (uint32_t)(lane >> 4) ^ swz<D>(a_row);
    b_row = lane & 7;  b_x = (uint32_t)(lane >> 3) ^ swz<D>(b_row);
    t_row = (lane & 7) + ((lane >> 3) & 1) * 8; t_x = (uint32_t)(lane >> 4) ^ swz<D>(t_row);
  }
  __device__ __forceinline__ uint32_t a(int row0, int kk) const { return (row0 + a_row) * (2 * D) + (((uint32_t)(2 * kk) ^ a_x) << 4); }
  __device__ __forceinline__ uint32_t b(int row0, int k2) const { return (row0 + b_row) * (2 * D) + (((uint32_t)(4 * k2) ^ b_x) << 4); }
  __device__ __forceinline__ uint32_t t(int row0, int jp) const { return (row0 + t_row) * (2 * D) + (((uint32_t)(2 * jp) ^ t_x) << 4); }
};
__device__ __forceinline__ void ldsm_x4_s(uint32_t (&r)[4], uint32_t a) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(a));
}
__device__ __forceinline__ void ldsm_x4_t_s(uint32_t (&r)[4], uint32_t a) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(a));
}

// S[16 x TP] = Q_rows(16w..) · Kᵀ   (raw, unscaled; masked key columns = -inf) -> s[j][4], j = key tile of 8
template <int D, int NT16>
__device__ __forceinline__ void qk_tile(float (&s)[2 * NT16][4], uint32_t sA, uint32_t sB, int warp, const LaneAddr<D>& la, const KeyMask& km) {
  uint32_t a[D / 16][4];
#pragma unroll
  for (int kk = 0; kk < D / 16; ++kk) ldsm_x4_s(a[kk], sA + la.a(16 * warp, kk));
#pragma unroll
  for (int j = 0; j < 2 * NT16; ++j) {
    if (j < km.nfull || (j == km.nfull && km.rem != 0)) {  // warp-uniform
      s[j][0] = s[j][1] = s[j][2] = s[j][3] = 0.f;
#pragma unroll
      for (int k2 = 0; k2 < D / 32; ++k2) {
        uint32_t b[4];
        ldsm_x4_s(b, sB + la.b(8 * j, k2));
        mma_bf16(s[j], a[2 * k2], b[0], b[1]);
        mma_bf16(s[j], a[2 * k2 + 1], b[2], b[3]);
      }
      if (j == km.nfull) {
        s[j][0] += km.pm0; s[j][2] += km.pm0;
        s[j][1] += km.pm1; s[j][3] += km.pm1;
      }
    } else {
      s[j][0] = s[j][1] = s[j][2] = s[j][3] = -INFINITY;
    }
  }
}

// acc[16 x D] += P(regs, 16 x TP) · B(TP x D) with B rows = reduction index (ldmatrix.trans)
template <int D, int NT16>
__device__ __forceinline__ void pv_tile(float (&acc)[D / 8][4], const float (&p)[2 * NT16][4], uint32_t sB, const LaneAddr<D>& la) {
#pragma unroll
  for (int kk = 0; kk < NT16; ++kk) {
    uint32_t a[4];
    a[0] = pack_bf16x2(p[2 * kk][0], p[2 * kk][1]);
    a[1] = pack_bf16x2(p[2 * kk][2], p[2 * kk][3]);
    a[2] = pack_bf16x2(p[2 * kk + 1][0], p[2 * kk + 1][1]);
    a[3] = pack_bf16x2(p[2 * kk + 1][2], p[2 * kk + 1][3]);
#pragma unroll
    for (int jp = 0; jp < D / 16; ++jp) {
      uint32_t b[4];
      ldsm_x4_t_s(b, sB + la.t(16 * kk, jp));
      mma_bf16(acc[2 * jp], a, b[0], b[1]);
      mma_bf16(acc[2 * jp + 1], a, b[2], b[3]);
    }
  }
}

// write a warp's 16 x D fp32 fragment tile as bf16 into rows row0.. (a multiple of 16) of a swizzled tile; a later TMA store
// moves the tile out.  Rows g and g + 8 share their swizzle term, so an address is base + ((chunk ^ x) << 4).
template <int D>
__device__ __forceinline__ void stage_rows16(const float (&acc)[D / 8][4], uint32_t sTile, int row0, int lane) {
  const int g = lane >> 2, t = lane & 3;
  const uint32_t x = swz<D>(g);
  const uint32_t base = sTile + (uint32_t)(row0 + g) * (2 * D) + 4 * t;
#pragma unroll
  for (int jn = 0; jn < D / 8; ++jn) {
    const uint32_t a = base + (((uint32_t)jn ^ x) << 4);
    asm volatile("st.shared.b32 [%0], %1;" ::"r"(a), "r"(pack_bf16x2(acc[jn][0], acc[jn][1])) : "memory");
    asm volatile("st.shared.b32 [%0], %1;" ::"r"(a + 8 * 2 * D), "r"(pack_bf16x2(acc[jn][2], acc[jn][3])) : "memory");
  }
}

// ---------------------------------------------------------------------------------------------
// bf16 forward: persistent CTAs walk (image, head) items; one thread streams the next item's Q/K/V tiles in with TMA
// (double buffer, mbarrier) while the CTA computes the current one; the output tile leaves through a TMA store
// ---------------------------------------------------------------------------------------------
// CTAs per SM of the forward kernel at 3-5 row tiles (T = 33..80).  5 fit in shared memory (5 x 42 KB) if the kernel stays within
// 80 registers, and ptxas gets there from 93 with 20 bytes of spills — measured SLOWER (74.8 vs 67.8 us at B = 1024, T = 65,
// profiles/r2_attn_experiments.md): the kernel is bound by its dependent ldmatrix / mma.sync / shuffle chains, which the tighter
// register allocation lengthens by more than the fifth CTA hides.
#ifndef VITB_ATTN_FWD_CTAS
#define VITB_ATTN_FWD_CTAS 4
#endif
template <int D, int NT16>
__global__ void __launch_bounds__(32 * NT16, (NT16 <= 2 ? 8 : (NT16 <= 5 ? (D == 32 ? VITB_ATTN_FWD_CTAS : 2) : 1)))
    attn_fwd_bf16_kernel(const __grid_constant__ CUtensorMap m_qkv, const __grid_constant__ CUtensorMap m_o, float* __restrict__ lse,
                         float* __restrict__ attn_map, int n_items, int T, int heads, float scale) {
  constexpr int TP = 16 * NT16;
  constexpr uint32_t TILE_B = TP * D * 2;
  extern __shared__ uint8_t smem_attn_raw[];
  const uint32_t sbase = (smem_u32(smem_attn_raw) + 1023u) & ~1023u;  // [2][3] input tiles, [2] output tiles, 2 barriers
  const uint32_t sO0 = sbase + 6 * TILE_B;
  const uint32_t bars = sO0 + 2 * TILE_B;
  const int Hd = heads * D;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  pdl_trigger();
  if (tid == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)&m_qkv) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)&m_o) : "memory");
    mbar_init(bars, 1);
    mbar_init(bars + 8, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  pdl_wait();  // inputs come from the preceding kernel
  auto issue = [&](int item, int buf) {  // one thread
    const int b = item / heads, h = item % heads;
    const uint32_t dst = sbase + (uint32_t)buf * 3 * TILE_B, bar = bars + 8 * buf;
    mbar_arrive_expect_tx(bar, 3 * TILE_B);
    tma_load_3d(dst, &m_qkv, bar, h * D, 0, b);
    tma_load_3d(dst + TILE_B, &m_qkv, bar, Hd + h * D, 0, b);
    tma_load_3d(dst + 2 * TILE_B, &m_qkv, bar, 2 * Hd + h * D, 0, b);
  };
  int item = blockIdx.x;
  if (tid == 0 && item < n_items) issue(item, 0);
  const int g = lane >> 2, t = lane & 3;
  const float sl2 = scale * kLog2e;
  const KeyMask km = make_key_mask(T, lane);
  const LaneAddr<D> la(lane);
  for (int it = 0; item < n_items; item += gridDim.x, ++it) {
    const int cur = it & 1;
    const uint32_t sO = sO0 + (uint32_t)cur * TILE_B;
    // every warp has finished with the other input buffer (the barrier of the previous iteration comes after its compute)
    if (tid == 0) {
      const int nxt = item + gridDim.x;
      if (nxt < n_items) issue(nxt, cur ^ 1);
    }
    mbar_wait(bars + 8 * cur, (uint32_t)(it >> 1) & 1u);
    const uint32_t sQ = sbase + (uint32_t)cur * 3 * TILE_B, sK = sQ + TILE_B, sV = sK + TILE_B;
    const int b = item / heads, h = item % heads;

    float s[2 * NT16][4];
    qk_tile<D, NT16>(s, sQ, sK, warp, la, km);
    float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll
    for (int j = 0; j < 2 * NT16; ++j) {
      m0 = fmaxf(m0, fmaxf(s[j][0], s[j][1]));
      m1 = fmaxf(m1, fmaxf(s[j][2], s[j][3]));
    }
    m0 = quad_max(m0);
    m1 = quad_max(m1);
    // p = 2^(s * scale*log2e - max * scale*log2e): one FFMA + one MUFU per element; P stays unnormalised through the PV
    // product (its largest entry is exactly 1) and the 16 x D output is scaled by 1 / rowsum instead
    const float ms0 = m0 * sl2, ms1 = m1 * sl2;
    float sum0 = 0.f, sum1 = 0.f;
#pragma unroll
    for (int j = 0; j < 2 * NT16; ++j) {
      s[j][0] = ex2_fast(fmaf(s[j][0], sl2, -ms0));
      s[j][1] = ex2_fast(fmaf(s[j][1], sl2, -ms0));
      s[j][2] = ex2_fast(fmaf(s[j][2], sl2, -ms1));
      s[j][3] = ex2_fast(fmaf(s[j][3], sl2, -ms1));
      sum0 += s[j][0] + s[j][1];
      sum1 += s[j][2] + s[j][3];
    }
    sum0 = quad_sum(sum0);
    sum1 = quad_sum(sum1);
    const float inv0 = 1.0f / sum0, inv1 = 1.0f / sum1;
    const int r0 = 16 * warp + g, r1 = r0 + 8;
    if (t == 0) {
      float* l = lse + ((int64_t)b * heads + h) * T;
      if (r0 < T) l[r0] = m0 * scale + logf(sum0);
      if (r1 < T) l[r1] = m1 * scale + logf(sum1);
    }
    if (attn_map != nullptr) {  // save_attn_map protocol (layers.py:99-100)
      float* am = attn_map + ((int64_t)b * heads + h) * T * T;
#pragma unroll
      for (int j = 0; j < 2 * NT16; ++j) {
        const int c = 8 * j + 2 * t;
        if (r0 < T) { if (c < T) am[(int64_t)r0 * T + c] = s[j][0] * inv0; if (c + 1 < T) am[(int64_t)r0 * T + c + 1] = s[j][1] * inv0; }
        if (r1 < T) { if (c < T) am[(int64_t)r1 * T + c] = s[j][2] * inv1; if (c + 1 < T) am[(int64_t)r1 * T + c + 1] = s[j][3] * inv1; }
      }
    }
    float acc[D / 8][4];
#pragma unroll
    for (int jn = 0; jn < D / 8; ++jn) acc[jn][0] = acc[jn][1] = acc[jn][2] = acc[jn][3] = 0.f;
    pv_tile<D, NT16>(acc, s, sV, la);
#pragma unroll
    for (int jn = 0; jn < D / 8; ++jn) {
      acc[jn][0] *= inv0; acc[jn][1] *= inv0; acc[jn][2] *= inv1; acc[jn][3] *= inv1;
    }
    stage_rows16<D>(acc, sO, 16 * warp, lane);
    fence_async_smem();  // generic-proxy writes of the output tile -> visible to the TMA store
    // The store of the previous item (other output tile, issued a whole iteration ago) must have read its tile before the barrier
    // releases the warps into the iteration that rewrites it.
    if (tid == 0) tma_store_wait_read();
    __syncthreads();
    if (tid == 0) {
      tma_store_3d(&m_o, sO, h * D, 0, b);  // token rows >= T are clipped by the tensor map
      tma_store_commit();
    }
  }
  if (tid == 0) tma_store_wait_read();  // shared memory must stay alive until the last store has read it
}

// ---------------------------------------------------------------------------------------------
// bf16 backward
// ---------------------------------------------------------------------------------------------
// acc[16 keys x D] += Aᵀ-tile from sPS (stored [query][key], padded rows) · sB (swizzled [query][D] tile); reduction over queries
template <int D, int NT16>
__device__ __forceinline__ void tn_tile(float (&acc)[D / 8][4], const bf16* sPS, uint32_t sB, int warp, int lane, const LaneAddr<D>& la) {
  constexpr int LP = 16 * NT16 + 8;
#pragma unroll
  for (int kq = 0; kq < NT16; ++kq) {
    uint32_t a[4];
    ldsm_x4_t(a, sPS + (16 * kq + (lane & 7) + ((lane >> 4) & 1) * 8) * LP + 16 * warp + ((lane >> 3) & 1) * 8);
#pragma unroll
    for (int jp = 0; jp < D / 16; ++jp) {
      uint32_t b[4];
      ldsm_x4_t_s(b, sB + la.t(16 * kq, jp));
      mma_bf16(acc[2 * jp], a, b[0], b[1]);
      mma_bf16(acc[2 * jp + 1], a, b[2], b[3]);
    }
  }
}

// One CTA per (image, head); low register count (scores are processed in 16-key chunks) so that 4 CTAs share an SM.
//   D_i = sum_d dO_id * O_id  (= rowsum(P ∘ dP), flash-attention identity) from the saved forward output, so a chunk's
//   dS can be formed without holding the whole score row.
// Q, K, V, dO and O tiles arrive through five TMA loads (zero rows beyond T included), dQ/dK/dV leave through three TMA stores.
template <int D, int NT16>
__global__ void __launch_bounds__(32 * NT16, (D == 32 ? (NT16 <= 2 ? 8 : (NT16 <= 5 ? 4 : 1)) : (NT16 <= 2 ? 4 : (NT16 <= 5 ? 2 : 1))))
    attn_bwd_bf16_kernel(const __grid_constant__ CUtensorMap m_qkv, const __grid_constant__ CUtensorMap m_o, const __grid_constant__ CUtensorMap m_do,
                         const __grid_constant__ CUtensorMap m_dqkv, const float* __restrict__ lse, int T, int heads, float scale, int pf_dist) {
  constexpr int TP = 16 * NT16, LP = TP + 8, CH = D / 8;
  constexpr uint32_t TILE_B = TP * D * 2;
  extern __shared__ uint8_t smem_attn_raw[];
  const uint32_t sbase = (smem_u32(smem_attn_raw) + 1023u) & ~1023u;
  uint8_t* gen = smem_attn_raw + (sbase - smem_u32(smem_attn_raw));
  const uint32_t sQ = sbase, sK = sQ + TILE_B, sV = sK + TILE_B, sdO = sV + TILE_B, sO = sdO + TILE_B;
  bf16* sP = reinterpret_cast<bf16*>(gen + 5 * TILE_B);  // [TP][LP]
  bf16* sdS = sP + TP * LP;                               // [TP][LP]
  float* sD = reinterpret_cast<float*>(sdS + TP * LP);    // [TP]
  const uint32_t bar = smem_u32(sD + 2 * TP);
  const int b = blockIdx.x / heads, h = blockIdx.x % heads;
  const int Hd = heads * D;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  pdl_trigger();
  pdl_wait();  // inputs come from the preceding kernels
  if (tid == 0) {
    mbar_init(bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    mbar_arrive_expect_tx(bar, 5 * TILE_B);
    tma_load_3d(sQ, &m_qkv, bar, h * D, 0, b);
    tma_load_3d(sK, &m_qkv, bar, Hd + h * D, 0, b);
    tma_load_3d(sV, &m_qkv, bar, 2 * Hd + h * D, 0, b);
    tma_load_3d(sdO, &m_do, bar, h * D, 0, b);
    tma_load_3d(sO, &m_o, bar, h * D, 0, b);
    // CTAs are not persistent here: ask L2 for the tiles of the item that takes this CTA's place about one wave later, so its
    // loads do not pay the full HBM latency with nothing else to do
    const int nxt = (int)blockIdx.x + pf_dist;
    if (nxt < (int)gridDim.x) {
      const int nb = nxt / heads, nh = nxt % heads;
      tma_prefetch_3d(&m_qkv, nh * D, 0, nb);
      tma_prefetch_3d(&m_qkv, Hd + nh * D, 0, nb);
      tma_prefetch_3d(&m_qkv, 2 * Hd + nh * D, 0, nb);
      tma_prefetch_3d(&m_do, nh * D, 0, nb);
      tma_prefetch_3d(&m_o, nh * D, 0, nb);
    }
  }
  const int g = lane >> 2;
  const int r0 = 16 * warp + g, r1 = r0 + 8;
  // lse * log2(e) of this thread's two query rows (0 beyond T)
  const float* lrow = lse + ((int64_t)b * heads + h) * T;
  const float l0 = r0 < T ? lrow[r0] * kLog2e : 0.f, l1 = r1 < T ? lrow[r1] * kLog2e : 0.f;
  __syncthreads();  // barrier initialised before anyone waits
  mbar_wait(bar, 0);
  // D_i = sum_d dO_id * O_id from the two tiles, each warp for its own 16 query rows: CH lanes per row, 8 elements each
  // (zero rows give D = 0)
  for (int idx = lane; idx < 16 * CH; idx += 32) {
    const int r = 16 * warp + idx / CH, c = idx % CH;
    uint32_t a0, a1, a2, a3, q0, q1, q2, q3;
    const uint32_t off = tile_off<D>(r, c);
    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(a0), "=r"(a1), "=r"(a2), "=r"(a3) : "r"(sdO + off));
    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(q0), "=r"(q1), "=r"(q2), "=r"(q3) : "r"(sO + off));
    const float2 x0 = unpack_bf16x2(a0), x1 = unpack_bf16x2(a1), x2 = unpack_bf16x2(a2), x3 = unpack_bf16x2(a3);
    const float2 y0 = unpack_bf16x2(q0), y1 = unpack_bf16x2(q1), y2 = unpack_bf16x2(q2), y3 = unpack_bf16x2(q3);
    float v = (x0.x * y0.x + x0.y * y0.y) + (x1.x * y1.x + x1.y * y1.y) + (x2.x * y2.x + x2.y * y2.y) + (x3.x * y3.x + x3.y * y3.y);
#pragma unroll
    for (int off2 = CH / 2; off2 > 0; off2 >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off2);  // CH (4 or 8) adjacent lanes share a row
    if (c == 0) sD[r] = v;
  }
  __syncwarp();

  const float sl2 = scale * kLog2e;
  const float d0 = sD[r0], d1 = sD[r1];
  const KeyMask km = make_key_mask(T, lane);
  const LaneAddr<D> la(lane);
  uint32_t aq[D / 16][4], ado[D / 16][4];
#pragma unroll
  for (int kk = 0; kk < D / 16; ++kk) {
    ldsm_x4_s(aq[kk], sQ + la.a(16 * warp, kk));
    ldsm_x4_s(ado[kk], sdO + la.a(16 * warp, kk));
  }
  float dq[D / 8][4];
#pragma unroll
  for (int jn = 0; jn < D / 8; ++jn) dq[jn][0] = dq[jn][1] = dq[jn][2] = dq[jn][3] = 0.f;
#pragma unroll
  for (int jc = 0; jc < NT16; ++jc) {  // 16 keys per chunk
    float s[2][4], dp[2][4];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int j = 2 * jc + u;
      s[u][0] = s[u][1] = s[u][2] = s[u][3] = 0.f;
      dp[u][0] = dp[u][1] = dp[u][2] = dp[u][3] = 0.f;
      if (j < km.nfull || (j == km.nfull && km.rem != 0)) {  // warp-uniform: key tiles beyond T contribute P = dS = 0
#pragma unroll
        for (int k2 = 0; k2 < D / 32; ++k2) {
          uint32_t bk[4], bv[4];
          ldsm_x4_s(bk, sK + la.b(8 * j, k2));
          ldsm_x4_s(bv, sV + la.b(8 * j, k2));
          mma_bf16(s[u], aq[2 * k2], bk[0], bk[1]);
          mma_bf16(s[u], aq[2 * k2 + 1], bk[2], bk[3]);
          mma_bf16(dp[u], ado[2 * k2], bv[0], bv[1]);
          mma_bf16(dp[u], ado[2 * k2 + 1], bv[2], bv[3]);
        }
        if (j == km.nfull) {  // partial tile: masked key columns get score -inf -> P = 0
          s[u][0] += km.pm0; s[u][2] += km.pm0;
          s[u][1] += km.pm1; s[u][3] += km.pm1;
        }
        // Query rows >= T need no mask: their Q and dO rows are zero padding and D = lse = 0 there, so P = 1, dP = 0, dS = 0 and
        // P only multiplies zero dO rows in dV.
        s[u][0] = ex2_fast(fmaf(s[u][0], sl2, -l0));
        s[u][1] = ex2_fast(fmaf(s[u][1], sl2, -l0));
        s[u][2] = ex2_fast(fmaf(s[u][2], sl2, -l1));
        s[u][3] = ex2_fast(fmaf(s[u][3], sl2, -l1));
        // dS = P ∘ (dP − D) / sqrt(features)
        dp[u][0] = s[u][0] * (dp[u][0] - d0) * scale;
        dp[u][1] = s[u][1] * (dp[u][1] - d0) * scale;
        dp[u][2] = s[u][2] * (dp[u][2] - d1) * scale;
        dp[u][3] = s[u][3] * (dp[u][3] - d1) * scale;
      }
    }
    uint32_t pa[4], da[4];  // A-operand fragments of this 16 x 16 chunk (also exactly what stmatrix stores)
    pa[0] = pack_bf16x2(s[0][0], s[0][1]); pa[1] = pack_bf16x2(s[0][2], s[0][3]);
    pa[2] = pack_bf16x2(s[1][0], s[1][1]); pa[3] = pack_bf16x2(s[1][2], s[1][3]);
    da[0] = pack_bf16x2(dp[0][0], dp[0][1]); da[1] = pack_bf16x2(dp[0][2], dp[0][3]);
    da[2] = pack_bf16x2(dp[1][0], dp[1][1]); da[3] = pack_bf16x2(dp[1][2], dp[1][3]);
    // matrices: (rows 0-7, keys 0-7), (rows 8-15, keys 0-7), (rows 0-7, keys 8-15), (rows 8-15, keys 8-15) of the chunk
    const int srow = 16 * warp + ((lane >> 3) & 1) * 8 + (lane & 7), scol = 16 * jc + (lane >> 4) * 8;
    stsm_x4(sP + srow * LP + scol, pa[0], pa[1], pa[2], pa[3]);
    stsm_x4(sdS + srow * LP + scol, da[0], da[1], da[2], da[3]);
    // dQ += dS_chunk · K_chunk  (K rows = reduction index -> ldmatrix.trans)
#pragma unroll
    for (int jp = 0; jp < D / 16; ++jp) {
      uint32_t bb[4];
      ldsm_x4_t_s(bb, sK + la.t(16 * jc, jp));
      mma_bf16(dq[2 * jp], da, bb[0], bb[1]);
      mma_bf16(dq[2 * jp + 1], da, bb[2], bb[3]);
    }
  }
  __syncthreads();  // sP / sdS complete

  // this warp now owns key rows 16w..16w+15:  dV = Pᵀ · dO,  dK = dSᵀ · Q
  float dv[D / 8][4], dk[D / 8][4];
#pragma unroll
  for (int jn = 0; jn < D / 8; ++jn) {
    dv[jn][0] = dv[jn][1] = dv[jn][2] = dv[jn][3] = 0.f;
    dk[jn][0] = dk[jn][1] = dk[jn][2] = dk[jn][3] = 0.f;
  }
  tn_tile<D, NT16>(dv, sP, sdO, warp, lane, la);
  tn_tile<D, NT16>(dk, sdS, sQ, warp, lane, la);
  __syncthreads();  // everyone is done reading sQ/sK/sV/sdO: the Q/K/V tiles become the staging tiles of dQ/dK/dV

  stage_rows16<D>(dq, sQ, 16 * warp, lane);
  stage_rows16<D>(dk, sK, 16 * warp, lane);
  stage_rows16<D>(dv, sV, 16 * warp, lane);
  fence_async_smem();
  __syncthreads();
  if (tid == 0) {
    tma_store_3d(&m_dqkv, sQ, h * D, 0, b);  // token rows >= T are clipped by the tensor map
    tma_store_3d(&m_dqkv, sK, Hd + h * D, 0, b);
    tma_store_3d(&m_dqkv, sV, 2 * Hd + h * D, 0, b);
    tma_store_commit();
    tma_store_wait_read();  // shared memory must stay alive until the stores have read it
  }
}

// ---------------------------------------------------------------------------------------------
// bf16 attention at head dimensions 96 and 128.  A 192- or 256-byte row has no TMA swizzle mode, so a head is split into P panels
// of W = 32 or 64 columns (D = W·P: 3 x 32 or 2 x 64), each one TMA box of the W-column head tile above, under that tile's swizzle.
// Panel p of a (TP x D) tile lives at p·TP·W·2 and is addressed with LaneAddr<W>.  QKᵀ reduces over P x W/16 k-steps; the
// outputs are accumulated, staged and stored panel by panel, so the per-thread accumulators stay those of a W-column head.
// ---------------------------------------------------------------------------------------------
constexpr size_t kMaxSmemPerBlock = 227 * 1024;
constexpr size_t kSmemPerSM = 228 * 1024;  // of which each resident CTA reserves 1 KB

template <int W, int P, int NT16>
struct PanelTile {
  static constexpr int TP = 16 * NT16, LP = TP + 8, D = W * P;
  static constexpr uint32_t PANEL_B = TP * W * 2, TILE_B = P * PANEL_B;
  static constexpr uint32_t PS_B = TP * LP * 2;  // one padded [TP][LP] bf16 score tile (P or dS)
  // forward: [2][3] input tiles, one output tile (a second one does not fit at D = 128, T > 80), 2 barriers
  static constexpr size_t fwd_smem = (size_t)7 * TILE_B + 16 + 1024;
  // backward: Q, K, V, dO tiles; O shares its region with dS (O is read only to form D_i, before dS is first written); P; D_i
  static constexpr uint32_t ODS_B = TILE_B > PS_B ? TILE_B : PS_B;
  static constexpr size_t bwd_smem = (size_t)4 * TILE_B + ODS_B + PS_B + 2 * TP * sizeof(float) + 16 + 1024;
  static_assert(fwd_smem <= kMaxSmemPerBlock && bwd_smem <= kMaxSmemPerBlock, "panelled attention tile set exceeds 227 KB");
  // CTAs that fit an SM by shared memory: the register bound asks no more of ptxas than that
  static constexpr int ctas(size_t smem) { return (int)(kSmemPerSM / (smem + 1024)) < 8 ? (int)(kSmemPerSM / (smem + 1024)) : 8; }
};

// S[16 x TP] = Q_rows(16w..) · Kᵀ over P panels (raw, unscaled; masked key columns = -inf) -> s[j][4], j = key tile of 8
template <int W, int P, int NT16>
__device__ __forceinline__ void qk_tile_panels(float (&s)[2 * NT16][4], uint32_t sA, uint32_t sB, int warp, const LaneAddr<W>& la,
                                               const KeyMask& km) {
  constexpr uint32_t PB = PanelTile<W, P, NT16>::PANEL_B;
  uint32_t a[P][W / 16][4];
#pragma unroll
  for (int p = 0; p < P; ++p)
#pragma unroll
    for (int kk = 0; kk < W / 16; ++kk) ldsm_x4_s(a[p][kk], sA + p * PB + la.a(16 * warp, kk));
#pragma unroll
  for (int j = 0; j < 2 * NT16; ++j) {
    if (j < km.nfull || (j == km.nfull && km.rem != 0)) {  // warp-uniform
      s[j][0] = s[j][1] = s[j][2] = s[j][3] = 0.f;
#pragma unroll
      for (int p = 0; p < P; ++p)
#pragma unroll
        for (int k2 = 0; k2 < W / 32; ++k2) {
          uint32_t b[4];
          ldsm_x4_s(b, sB + p * PB + la.b(8 * j, k2));
          mma_bf16(s[j], a[p][2 * k2], b[0], b[1]);
          mma_bf16(s[j], a[p][2 * k2 + 1], b[2], b[3]);
        }
      if (j == km.nfull) {
        s[j][0] += km.pm0; s[j][2] += km.pm0;
        s[j][1] += km.pm1; s[j][3] += km.pm1;
      }
    } else {
      s[j][0] = s[j][1] = s[j][2] = s[j][3] = -INFINITY;
    }
  }
}

// Forward: as attn_fwd_bf16_kernel<D, NT16> (persistent CTAs, double-buffered TMA input), with one output tile: the previous item's
// store must have read it before the PV product of the next item is staged.
template <int W, int P, int NT16>
__global__ void __launch_bounds__(32 * NT16, PanelTile<W, P, NT16>::ctas(PanelTile<W, P, NT16>::fwd_smem))
    attn_fwd_bf16_kernel(const __grid_constant__ CUtensorMap m_qkv, const __grid_constant__ CUtensorMap m_o, float* __restrict__ lse,
                         float* __restrict__ attn_map, int n_items, int T, int heads, float scale) {
  using PT = PanelTile<W, P, NT16>;
  constexpr int D = PT::D;
  constexpr uint32_t PB = PT::PANEL_B, TILE_B = PT::TILE_B;
  extern __shared__ uint8_t smem_attn_raw[];
  const uint32_t sbase = (smem_u32(smem_attn_raw) + 1023u) & ~1023u;  // [2][3] input tiles, 1 output tile, 2 barriers
  const uint32_t sO = sbase + 6 * TILE_B;
  const uint32_t bars = sO + TILE_B;
  const int Hd = heads * D;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  pdl_trigger();
  if (tid == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)&m_qkv) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)&m_o) : "memory");
    mbar_init(bars, 1);
    mbar_init(bars + 8, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  pdl_wait();  // inputs come from the preceding kernel
  auto issue = [&](int item, int buf) {  // one thread: 3 tensors x P panels on one barrier
    const int b = item / heads, h = item % heads;
    const uint32_t dst = sbase + (uint32_t)buf * 3 * TILE_B, bar = bars + 8 * buf;
    mbar_arrive_expect_tx(bar, 3 * TILE_B);
#pragma unroll
    for (int p = 0; p < P; ++p) {
      tma_load_3d(dst + p * PB, &m_qkv, bar, h * D + p * W, 0, b);
      tma_load_3d(dst + TILE_B + p * PB, &m_qkv, bar, Hd + h * D + p * W, 0, b);
      tma_load_3d(dst + 2 * TILE_B + p * PB, &m_qkv, bar, 2 * Hd + h * D + p * W, 0, b);
    }
  };
  int item = blockIdx.x;
  if (tid == 0 && item < n_items) issue(item, 0);
  const int g = lane >> 2, t = lane & 3;
  const float sl2 = scale * kLog2e;
  const KeyMask km = make_key_mask(T, lane);
  const LaneAddr<W> la(lane);
  for (int it = 0; item < n_items; item += gridDim.x, ++it) {
    const int cur = it & 1;
    // every warp has finished with the other input buffer (the barrier of the previous iteration comes after its compute)
    if (tid == 0) {
      const int nxt = item + gridDim.x;
      if (nxt < n_items) issue(nxt, cur ^ 1);
    }
    mbar_wait(bars + 8 * cur, (uint32_t)(it >> 1) & 1u);
    const uint32_t sQ = sbase + (uint32_t)cur * 3 * TILE_B, sK = sQ + TILE_B, sV = sK + TILE_B;
    const int b = item / heads, h = item % heads;

    float s[2 * NT16][4];
    qk_tile_panels<W, P, NT16>(s, sQ, sK, warp, la, km);
    float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll
    for (int j = 0; j < 2 * NT16; ++j) {
      m0 = fmaxf(m0, fmaxf(s[j][0], s[j][1]));
      m1 = fmaxf(m1, fmaxf(s[j][2], s[j][3]));
    }
    m0 = quad_max(m0);
    m1 = quad_max(m1);
    const float ms0 = m0 * sl2, ms1 = m1 * sl2;
    float sum0 = 0.f, sum1 = 0.f;
#pragma unroll
    for (int j = 0; j < 2 * NT16; ++j) {
      s[j][0] = ex2_fast(fmaf(s[j][0], sl2, -ms0));
      s[j][1] = ex2_fast(fmaf(s[j][1], sl2, -ms0));
      s[j][2] = ex2_fast(fmaf(s[j][2], sl2, -ms1));
      s[j][3] = ex2_fast(fmaf(s[j][3], sl2, -ms1));
      sum0 += s[j][0] + s[j][1];
      sum1 += s[j][2] + s[j][3];
    }
    sum0 = quad_sum(sum0);
    sum1 = quad_sum(sum1);
    const float inv0 = 1.0f / sum0, inv1 = 1.0f / sum1;
    const int r0 = 16 * warp + g, r1 = r0 + 8;
    if (t == 0) {
      float* l = lse + ((int64_t)b * heads + h) * T;
      if (r0 < T) l[r0] = m0 * scale + logf(sum0);
      if (r1 < T) l[r1] = m1 * scale + logf(sum1);
    }
    if (attn_map != nullptr) {  // save_attn_map protocol (layers.py:99-100)
      float* am = attn_map + ((int64_t)b * heads + h) * T * T;
#pragma unroll
      for (int j = 0; j < 2 * NT16; ++j) {
        const int c = 8 * j + 2 * t;
        if (r0 < T) { if (c < T) am[(int64_t)r0 * T + c] = s[j][0] * inv0; if (c + 1 < T) am[(int64_t)r0 * T + c + 1] = s[j][1] * inv0; }
        if (r1 < T) { if (c < T) am[(int64_t)r1 * T + c] = s[j][2] * inv1; if (c + 1 < T) am[(int64_t)r1 * T + c + 1] = s[j][3] * inv1; }
      }
    }
    // the previous item's store (issued a whole item ago) has read the output tile before any warp rewrites it
    if (tid == 0) tma_store_wait_read();
    __syncthreads();
#pragma unroll
    for (int p = 0; p < P; ++p) {
      float acc[W / 8][4];
#pragma unroll
      for (int jn = 0; jn < W / 8; ++jn) acc[jn][0] = acc[jn][1] = acc[jn][2] = acc[jn][3] = 0.f;
      pv_tile<W, NT16>(acc, s, sV + p * PB, la);
#pragma unroll
      for (int jn = 0; jn < W / 8; ++jn) {
        acc[jn][0] *= inv0; acc[jn][1] *= inv0; acc[jn][2] *= inv1; acc[jn][3] *= inv1;
      }
      stage_rows16<W>(acc, sO + p * PB, 16 * warp, lane);
    }
    fence_async_smem();  // generic-proxy writes of the output tile -> visible to the TMA store
    __syncthreads();     // also: every warp is done with this item's input buffer
    if (tid == 0) {
#pragma unroll
      for (int p = 0; p < P; ++p) tma_store_3d(&m_o, sO + p * PB, h * D + p * W, 0, b);  // token rows >= T are clipped
      tma_store_commit();
    }
  }
  if (tid == 0) tma_store_wait_read();  // shared memory must stay alive until the last store has read it
}

// acc[16 queries x W] += sPS rows 16w.. (stored [query][key], padded rows) · sB (swizzled [key][W] panel); reduction over keys
template <int W, int NT16>
__device__ __forceinline__ void nn_tile(float (&acc)[W / 8][4], const bf16* sPS, uint32_t sB, int warp, int lane, const LaneAddr<W>& la) {
  constexpr int LP = 16 * NT16 + 8;
#pragma unroll
  for (int kc = 0; kc < NT16; ++kc) {
    uint32_t a[4];
    ldsm_x4(a, sPS + (16 * warp + (lane & 15)) * LP + 16 * kc + (lane >> 4) * 8);
#pragma unroll
    for (int jp = 0; jp < W / 16; ++jp) {
      uint32_t b[4];
      ldsm_x4_t_s(b, sB + la.t(16 * kc, jp));
      mma_bf16(acc[2 * jp], a, b[0], b[1]);
      mma_bf16(acc[2 * jp + 1], a, b[2], b[3]);
    }
  }
}

// Backward: one CTA per (image, head), as attn_bwd_bf16_kernel<D, NT16>, except that phase 1 only forms P and dS; dQ = dS·K,
// dK = dSᵀ·Q and dV = Pᵀ·dO are all computed in phase 2, one W-column panel at a time from shared memory.  Staging: dV goes to
// the V tile (free after phase 1), dK to the dO tile (free after dV), dQ to the Q tile (free after dK).
template <int W, int P, int NT16>
__global__ void __launch_bounds__(32 * NT16, PanelTile<W, P, NT16>::ctas(PanelTile<W, P, NT16>::bwd_smem))
    attn_bwd_bf16_kernel(const __grid_constant__ CUtensorMap m_qkv, const __grid_constant__ CUtensorMap m_o, const __grid_constant__ CUtensorMap m_do,
                         const __grid_constant__ CUtensorMap m_dqkv, const float* __restrict__ lse, int T, int heads, float scale, int pf_dist) {
  using PT = PanelTile<W, P, NT16>;
  constexpr int D = PT::D, TP = PT::TP, LP = PT::LP, CH = W / 8;
  constexpr uint32_t PB = PT::PANEL_B, TILE_B = PT::TILE_B;
  extern __shared__ uint8_t smem_attn_raw[];
  const uint32_t sbase = (smem_u32(smem_attn_raw) + 1023u) & ~1023u;
  uint8_t* gen = smem_attn_raw + (sbase - smem_u32(smem_attn_raw));
  const uint32_t sQ = sbase, sK = sQ + TILE_B, sV = sK + TILE_B, sdO = sV + TILE_B, sO = sdO + TILE_B;
  bf16* sdS = reinterpret_cast<bf16*>(gen + 4 * TILE_B);           // [TP][LP], over the O tile
  bf16* sP = reinterpret_cast<bf16*>(gen + 4 * TILE_B + PT::ODS_B);  // [TP][LP]
  float* sD = reinterpret_cast<float*>(sP + TP * LP);                // [TP]
  const uint32_t bar = smem_u32(sD + 2 * TP);
  const int b = blockIdx.x / heads, h = blockIdx.x % heads;
  const int Hd = heads * D;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  pdl_trigger();
  pdl_wait();  // inputs come from the preceding kernels
  if (tid == 0) {
    mbar_init(bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    mbar_arrive_expect_tx(bar, 5 * TILE_B);
#pragma unroll
    for (int p = 0; p < P; ++p) {
      tma_load_3d(sQ + p * PB, &m_qkv, bar, h * D + p * W, 0, b);
      tma_load_3d(sK + p * PB, &m_qkv, bar, Hd + h * D + p * W, 0, b);
      tma_load_3d(sV + p * PB, &m_qkv, bar, 2 * Hd + h * D + p * W, 0, b);
      tma_load_3d(sdO + p * PB, &m_do, bar, h * D + p * W, 0, b);
      tma_load_3d(sO + p * PB, &m_o, bar, h * D + p * W, 0, b);
    }
    const int nxt = (int)blockIdx.x + pf_dist;  // L2 prefetch of the item about one wave later (see attn_bwd_bf16_kernel<D, NT16>)
    if (nxt < (int)gridDim.x) {
      const int nb = nxt / heads, nh = nxt % heads;
#pragma unroll
      for (int p = 0; p < P; ++p) {
        tma_prefetch_3d(&m_qkv, nh * D + p * W, 0, nb);
        tma_prefetch_3d(&m_qkv, Hd + nh * D + p * W, 0, nb);
        tma_prefetch_3d(&m_qkv, 2 * Hd + nh * D + p * W, 0, nb);
        tma_prefetch_3d(&m_do, nh * D + p * W, 0, nb);
        tma_prefetch_3d(&m_o, nh * D + p * W, 0, nb);
      }
    }
  }
  const int g = lane >> 2;
  const int r0 = 16 * warp + g, r1 = r0 + 8;
  const float* lrow = lse + ((int64_t)b * heads + h) * T;
  const float l0 = r0 < T ? lrow[r0] * kLog2e : 0.f, l1 = r1 < T ? lrow[r1] * kLog2e : 0.f;
  __syncthreads();  // barrier initialised before anyone waits
  mbar_wait(bar, 0);
  // D_i = sum_d dO_id * O_id for this warp's 16 query rows: CH adjacent lanes per row, each summing its 16-byte chunk over panels
  for (int idx = lane; idx < 16 * CH; idx += 32) {
    const int r = 16 * warp + idx / CH, c = idx % CH;
    float v = 0.f;
#pragma unroll
    for (int p = 0; p < P; ++p) {
      uint32_t a0, a1, a2, a3, q0, q1, q2, q3;
      const uint32_t off = p * PB + tile_off<W>(r, c);
      asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(a0), "=r"(a1), "=r"(a2), "=r"(a3) : "r"(sdO + off));
      asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(q0), "=r"(q1), "=r"(q2), "=r"(q3) : "r"(sO + off));
      const float2 x0 = unpack_bf16x2(a0), x1 = unpack_bf16x2(a1), x2 = unpack_bf16x2(a2), x3 = unpack_bf16x2(a3);
      const float2 y0 = unpack_bf16x2(q0), y1 = unpack_bf16x2(q1), y2 = unpack_bf16x2(q2), y3 = unpack_bf16x2(q3);
      v += (x0.x * y0.x + x0.y * y0.y) + (x1.x * y1.x + x1.y * y1.y) + (x2.x * y2.x + x2.y * y2.y) + (x3.x * y3.x + x3.y * y3.y);
    }
#pragma unroll
    for (int off2 = CH / 2; off2 > 0; off2 >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off2);
    if (c == 0) sD[r] = v;
  }
  __syncthreads();  // every warp has read the O tile: its region becomes sdS

  const float sl2 = scale * kLog2e;
  const float d0 = sD[r0], d1 = sD[r1];
  const KeyMask km = make_key_mask(T, lane);
  const LaneAddr<W> la(lane);
  uint32_t aq[P][W / 16][4], ado[P][W / 16][4];
#pragma unroll
  for (int p = 0; p < P; ++p)
#pragma unroll
    for (int kk = 0; kk < W / 16; ++kk) {
      ldsm_x4_s(aq[p][kk], sQ + p * PB + la.a(16 * warp, kk));
      ldsm_x4_s(ado[p][kk], sdO + p * PB + la.a(16 * warp, kk));
    }
#pragma unroll
  for (int jc = 0; jc < NT16; ++jc) {  // 16 keys per chunk
    float s[2][4], dp[2][4];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int j = 2 * jc + u;
      s[u][0] = s[u][1] = s[u][2] = s[u][3] = 0.f;
      dp[u][0] = dp[u][1] = dp[u][2] = dp[u][3] = 0.f;
      if (j < km.nfull || (j == km.nfull && km.rem != 0)) {  // warp-uniform: key tiles beyond T contribute P = dS = 0
#pragma unroll
        for (int p = 0; p < P; ++p)
#pragma unroll
          for (int k2 = 0; k2 < W / 32; ++k2) {
            uint32_t bk[4], bv[4];
            ldsm_x4_s(bk, sK + p * PB + la.b(8 * j, k2));
            ldsm_x4_s(bv, sV + p * PB + la.b(8 * j, k2));
            mma_bf16(s[u], aq[p][2 * k2], bk[0], bk[1]);
            mma_bf16(s[u], aq[p][2 * k2 + 1], bk[2], bk[3]);
            mma_bf16(dp[u], ado[p][2 * k2], bv[0], bv[1]);
            mma_bf16(dp[u], ado[p][2 * k2 + 1], bv[2], bv[3]);
          }
        if (j == km.nfull) {
          s[u][0] += km.pm0; s[u][2] += km.pm0;
          s[u][1] += km.pm1; s[u][3] += km.pm1;
        }
        // query rows >= T: zero Q / dO rows and D = lse = 0 give P = 1, dS = 0, and P only meets zero dO rows in dV
        s[u][0] = ex2_fast(fmaf(s[u][0], sl2, -l0));
        s[u][1] = ex2_fast(fmaf(s[u][1], sl2, -l0));
        s[u][2] = ex2_fast(fmaf(s[u][2], sl2, -l1));
        s[u][3] = ex2_fast(fmaf(s[u][3], sl2, -l1));
        dp[u][0] = s[u][0] * (dp[u][0] - d0) * scale;
        dp[u][1] = s[u][1] * (dp[u][1] - d0) * scale;
        dp[u][2] = s[u][2] * (dp[u][2] - d1) * scale;
        dp[u][3] = s[u][3] * (dp[u][3] - d1) * scale;
      }
    }
    const int srow = 16 * warp + ((lane >> 3) & 1) * 8 + (lane & 7), scol = 16 * jc + (lane >> 4) * 8;
    stsm_x4(sP + srow * LP + scol, pack_bf16x2(s[0][0], s[0][1]), pack_bf16x2(s[0][2], s[0][3]), pack_bf16x2(s[1][0], s[1][1]),
            pack_bf16x2(s[1][2], s[1][3]));
    stsm_x4(sdS + srow * LP + scol, pack_bf16x2(dp[0][0], dp[0][1]), pack_bf16x2(dp[0][2], dp[0][3]), pack_bf16x2(dp[1][0], dp[1][1]),
            pack_bf16x2(dp[1][2], dp[1][3]));
  }
  __syncthreads();  // sP / sdS complete; V is free

  // phase 2, per W-column panel: this warp owns key rows 16w.. of dV and dK and query rows 16w.. of dQ
  float acc[W / 8][4];
  auto zero = [&]() {
#pragma unroll
    for (int jn = 0; jn < W / 8; ++jn) acc[jn][0] = acc[jn][1] = acc[jn][2] = acc[jn][3] = 0.f;
  };
#pragma unroll
  for (int p = 0; p < P; ++p) {  // dV = Pᵀ · dO -> V tile
    zero();
    tn_tile<W, NT16>(acc, sP, sdO + p * PB, warp, lane, la);
    stage_rows16<W>(acc, sV + p * PB, 16 * warp, lane);
  }
  fence_async_smem();
  __syncthreads();  // dV staged; every warp is done reading dO
  if (tid == 0)
#pragma unroll
    for (int p = 0; p < P; ++p) tma_store_3d(&m_dqkv, sV + p * PB, 2 * Hd + h * D + p * W, 0, b);  // rows >= T are clipped
#pragma unroll
  for (int p = 0; p < P; ++p) {  // dK = dSᵀ · Q -> dO tile
    zero();
    tn_tile<W, NT16>(acc, sdS, sQ + p * PB, warp, lane, la);
    stage_rows16<W>(acc, sdO + p * PB, 16 * warp, lane);
  }
  fence_async_smem();
  __syncthreads();  // dK staged; every warp is done reading Q
  if (tid == 0)
#pragma unroll
    for (int p = 0; p < P; ++p) tma_store_3d(&m_dqkv, sdO + p * PB, Hd + h * D + p * W, 0, b);
#pragma unroll
  for (int p = 0; p < P; ++p) {  // dQ = dS · K -> Q tile
    zero();
    nn_tile<W, NT16>(acc, sdS, sK + p * PB, warp, lane, la);
    stage_rows16<W>(acc, sQ + p * PB, 16 * warp, lane);
  }
  fence_async_smem();
  __syncthreads();
  if (tid == 0) {
#pragma unroll
    for (int p = 0; p < P; ++p) tma_store_3d(&m_dqkv, sQ + p * PB, h * D + p * W, 0, b);
    tma_store_commit();
    tma_store_wait_read();  // shared memory must stay alive until the stores have read it
  }
}

// ---------------------------------------------------------------------------------------------
// fp32 check-mode kernels (FFMA, score tile in shared memory)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
    attn_fwd_f32_kernel(const float* __restrict__ qkv, float* __restrict__ o, float* __restrict__ lse, float* __restrict__ attn_map,
                        int T, int heads, int D, float scale) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ __align__(16) uint8_t smem_attn[];
  float* sQ = reinterpret_cast<float*>(smem_attn);
  float* sK = sQ + T * D;
  float* sV = sK + T * D;
  float* sS = sV + T * D;  // T x T
  const int b = blockIdx.x / heads, h = blockIdx.x % heads, Hd = heads * D;
  const int tid = threadIdx.x, nthr = blockDim.x;
  const float* base = qkv + (int64_t)b * T * 3 * Hd + h * D;
  for (int i = tid; i < T * D; i += nthr) {
    const int r = i / D, c = i % D;
    sQ[i] = base[(int64_t)r * 3 * Hd + c];
    sK[i] = base[(int64_t)r * 3 * Hd + Hd + c];
    sV[i] = base[(int64_t)r * 3 * Hd + 2 * Hd + c];
  }
  __syncthreads();
  for (int i = tid; i < T * T; i += nthr) {
    const int r = i / T, c = i % T;
    float acc = 0.f;
    for (int d = 0; d < D; ++d) acc = fmaf(sQ[r * D + d], sK[c * D + d], acc);
    sS[i] = acc * scale;
  }
  __syncthreads();
  for (int r = tid; r < T; r += nthr) {
    float m = -INFINITY;
    for (int c = 0; c < T; ++c) m = fmaxf(m, sS[r * T + c]);
    float sum = 0.f;
    for (int c = 0; c < T; ++c) {
      const float e = expf(sS[r * T + c] - m);
      sS[r * T + c] = e;
      sum += e;
    }
    const float inv = 1.0f / sum;
    for (int c = 0; c < T; ++c) sS[r * T + c] *= inv;
    lse[((int64_t)b * heads + h) * T + r] = m + logf(sum);
  }
  __syncthreads();
  if (attn_map != nullptr)
    for (int i = tid; i < T * T; i += nthr) attn_map[((int64_t)b * heads + h) * T * T + i] = sS[i];
  for (int i = tid; i < T * D; i += nthr) {
    const int r = i / D, d = i % D;
    float acc = 0.f;
    for (int c = 0; c < T; ++c) acc = fmaf(sS[r * T + c], sV[c * D + d], acc);
    o[((int64_t)b * T + r) * Hd + h * D + d] = acc;
  }
}

__global__ void __launch_bounds__(128)
    attn_bwd_f32_kernel(const float* __restrict__ qkv, const float* __restrict__ d_o, const float* __restrict__ lse,
                        float* __restrict__ dqkv, int T, int heads, int D, float scale) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ __align__(16) uint8_t smem_attn[];
  float* sQ = reinterpret_cast<float*>(smem_attn);
  float* sK = sQ + T * D;
  float* sV = sK + T * D;
  float* sdO = sV + T * D;
  float* sP = sdO + T * D;  // T x T
  float* sdS = sP + T * T;  // T x T
  const int b = blockIdx.x / heads, h = blockIdx.x % heads, Hd = heads * D;
  const int tid = threadIdx.x, nthr = blockDim.x;
  const float* base = qkv + (int64_t)b * T * 3 * Hd + h * D;
  for (int i = tid; i < T * D; i += nthr) {
    const int r = i / D, c = i % D;
    sQ[i] = base[(int64_t)r * 3 * Hd + c];
    sK[i] = base[(int64_t)r * 3 * Hd + Hd + c];
    sV[i] = base[(int64_t)r * 3 * Hd + 2 * Hd + c];
    sdO[i] = d_o[((int64_t)b * T + r) * Hd + h * D + c];
  }
  __syncthreads();
  const float* l = lse + ((int64_t)b * heads + h) * T;
  for (int i = tid; i < T * T; i += nthr) {
    const int r = i / T, c = i % T;
    float acc = 0.f, dp = 0.f;
    for (int d = 0; d < D; ++d) {
      acc = fmaf(sQ[r * D + d], sK[c * D + d], acc);
      dp = fmaf(sdO[r * D + d], sV[c * D + d], dp);
    }
    sP[i] = expf(acc * scale - l[r]);
    sdS[i] = dp;
  }
  __syncthreads();
  for (int r = tid; r < T; r += nthr) {
    float dsum = 0.f;
    for (int c = 0; c < T; ++c) dsum = fmaf(sP[r * T + c], sdS[r * T + c], dsum);
    for (int c = 0; c < T; ++c) sdS[r * T + c] = sP[r * T + c] * (sdS[r * T + c] - dsum) * scale;
  }
  __syncthreads();
  float* gd = dqkv + (int64_t)b * T * 3 * Hd + h * D;
  for (int i = tid; i < T * D; i += nthr) {
    const int r = i / D, d = i % D;
    float q = 0.f, k = 0.f, v = 0.f;
    for (int c = 0; c < T; ++c) {
      q = fmaf(sdS[r * T + c], sK[c * D + d], q);    // dQ[r] = sum_c dS[r][c] K[c]
      k = fmaf(sdS[c * T + r], sQ[c * D + d], k);    // dK[r] = sum_c dS[c][r] Q[c]
      v = fmaf(sP[c * T + r], sdO[c * D + d], v);    // dV[r] = sum_c P[c][r] dO[c]
    }
    gd[(int64_t)r * 3 * Hd + d] = q;
    gd[(int64_t)r * 3 * Hd + Hd + d] = k;
    gd[(int64_t)r * 3 * Hd + 2 * Hd + d] = v;
  }
}

// ---------------------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------------------
// tensor maps of one head tile: box = (D columns, 16*NT16 token rows, 1 image) of a (columns, T, B) view
template <int D, int NT16>
static int head_tile_map(CUtensorMap* map, const void* ptr, int cols, int T, int B) {
  return make_tma_map_3d_bf16(map, ptr, (uint64_t)cols, (uint64_t)T, (uint64_t)B, (uint64_t)cols * 2, (uint64_t)T * cols * 2, D, 16 * NT16, 1, D == 32 ? 64 : 128);
}

template <int D, int NT16>
static int launch_fwd_bf16(const void* qkv, void* o, float* lse, float* am, int B, int T, int heads, float scale, cudaStream_t st) {
  constexpr int TP = 16 * NT16;
  constexpr size_t smem = (size_t)8 * TP * D * 2 + 16 + 1024;
  auto kern = attn_fwd_bf16_kernel<D, NT16>;
  static int per_sm = 0;  // resident CTAs per SM of this instantiation (the kernel is persistent: the grid is exactly one wave)
  if (per_sm == 0) {
    VITB_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    VITB_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 32 * NT16, smem));
    if (per_sm < 1) per_sm = 1;
  }
  const int Hd = heads * D;
  CUtensorMap m_qkv, m_o;
  if (head_tile_map<D, NT16>(&m_qkv, qkv, 3 * Hd, T, B)) return -1;
  if (head_tile_map<D, NT16>(&m_o, o, Hd, T, B)) return -1;
  const int items = B * heads;
  const int grid = items < kNumSMs * per_sm ? items : kNumSMs * per_sm;
  VITB_LAUNCH((kern), grid, 32 * NT16, smem, st, m_qkv, m_o, lse, am, items, T, heads, scale);
  VITB_LAUNCH_OK();
  return 0;
}
template <int D, int NT16>
static int launch_bwd_bf16(const void* qkv, const void* o, const void* d_o, const float* lse, void* dqkv, int B, int T, int heads, float scale,
                           cudaStream_t st) {
  constexpr int TP = 16 * NT16, LP = TP + 8;
  constexpr size_t smem = (size_t)5 * TP * D * 2 + (size_t)2 * TP * LP * 2 + (size_t)2 * TP * sizeof(float) + 16 + 1024;
  auto kern = attn_bwd_bf16_kernel<D, NT16>;
  static bool configured = false;
  if (!configured) {
    VITB_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = true;
  }
  const int Hd = heads * D;
  CUtensorMap m_qkv, m_o, m_do, m_dqkv;
  if (head_tile_map<D, NT16>(&m_qkv, qkv, 3 * Hd, T, B)) return -1;
  if (head_tile_map<D, NT16>(&m_o, o, Hd, T, B)) return -1;
  if (head_tile_map<D, NT16>(&m_do, d_o, Hd, T, B)) return -1;
  if (head_tile_map<D, NT16>(&m_dqkv, dqkv, 3 * Hd, T, B)) return -1;
  int per_sm = 1;
  VITB_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 32 * NT16, smem));
  VITB_LAUNCH((kern), B * heads, 32 * NT16, smem, st, m_qkv, m_o, m_do, m_dqkv, lse, T, heads, scale, kNumSMs * (per_sm > 0 ? per_sm : 1));
  VITB_LAUNCH_OK();
  return 0;
}

// D = 96 / 128: P panels of W columns, each tensor map a W-column box
template <int D>
struct Panels {
  static_assert(D == 96 || D == 128, "panelled attention covers head dimensions 96 and 128");
  static constexpr int W = D == 96 ? 32 : 64, P = D / W;
};

template <int D, int NT16>
static int launch_fwd_bf16_panels(const void* qkv, void* o, float* lse, float* am, int B, int T, int heads, float scale, cudaStream_t st) {
  constexpr int W = Panels<D>::W, P = Panels<D>::P;
  constexpr size_t smem = PanelTile<W, P, NT16>::fwd_smem;
  auto kern = attn_fwd_bf16_kernel<W, P, NT16>;
  static int per_sm = 0;  // resident CTAs per SM of this instantiation (the kernel is persistent: the grid is exactly one wave)
  if (per_sm == 0) {
    VITB_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    VITB_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 32 * NT16, smem));
    if (per_sm < 1) per_sm = 1;
  }
  const int Hd = heads * D;
  CUtensorMap m_qkv, m_o;
  if (head_tile_map<W, NT16>(&m_qkv, qkv, 3 * Hd, T, B)) return -1;
  if (head_tile_map<W, NT16>(&m_o, o, Hd, T, B)) return -1;
  const int items = B * heads;
  const int grid = items < kNumSMs * per_sm ? items : kNumSMs * per_sm;
  VITB_LAUNCH((kern), grid, 32 * NT16, smem, st, m_qkv, m_o, lse, am, items, T, heads, scale);
  VITB_LAUNCH_OK();
  return 0;
}
template <int D, int NT16>
static int launch_bwd_bf16_panels(const void* qkv, const void* o, const void* d_o, const float* lse, void* dqkv, int B, int T, int heads,
                                  float scale, cudaStream_t st) {
  constexpr int W = Panels<D>::W, P = Panels<D>::P;
  constexpr size_t smem = PanelTile<W, P, NT16>::bwd_smem;
  auto kern = attn_bwd_bf16_kernel<W, P, NT16>;
  static int per_sm = 0;
  if (per_sm == 0) {
    VITB_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    VITB_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 32 * NT16, smem));
    if (per_sm < 1) per_sm = 1;
  }
  const int Hd = heads * D;
  CUtensorMap m_qkv, m_o, m_do, m_dqkv;
  if (head_tile_map<W, NT16>(&m_qkv, qkv, 3 * Hd, T, B)) return -1;
  if (head_tile_map<W, NT16>(&m_o, o, Hd, T, B)) return -1;
  if (head_tile_map<W, NT16>(&m_do, d_o, Hd, T, B)) return -1;
  if (head_tile_map<W, NT16>(&m_dqkv, dqkv, 3 * Hd, T, B)) return -1;
  VITB_LAUNCH((kern), B * heads, 32 * NT16, smem, st, m_qkv, m_o, m_do, m_dqkv, lse, T, heads, scale, kNumSMs * per_sm);
  VITB_LAUNCH_OK();
  return 0;
}

#define VITB_ATTN_NT16(FN, D, ...)                    \
  do {                                                \
    if (nt <= 1) return FN<D, 1>(__VA_ARGS__);        \
    if (nt <= 2) return FN<D, 2>(__VA_ARGS__);        \
    if (nt <= 4) return FN<D, 4>(__VA_ARGS__);        \
    if (nt <= 5) return FN<D, 5>(__VA_ARGS__);        \
    return FN<D, 8>(__VA_ARGS__);                     \
  } while (0)
#define VITB_ATTN_DISPATCH(FN, ...)                                 \
  do {                                                              \
    const int nt = (T + 15) / 16;                                   \
    if (d == 32) VITB_ATTN_NT16(FN, 32, __VA_ARGS__);               \
    if (d == 64) VITB_ATTN_NT16(FN, 64, __VA_ARGS__);               \
    if (d == 96) VITB_ATTN_NT16(FN##_panels, 96, __VA_ARGS__);      \
    VITB_ATTN_NT16(FN##_panels, 128, __VA_ARGS__);                  \
  } while (0)

static int set_dyn_smem(const void* fn, size_t smem) {
  if (smem > 48 * 1024) VITB_CUDA_OK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  return 0;
}

}  // namespace vitb

using namespace vitb;

extern "C" {

int vitb_attn_fwd(const void* qkv, void* o, float* lse, float* attn_map, int B, int T, int heads, int d, float scale, int dt, void* stream) {
  VITB_REQUIRE(qkv && o && lse, "attn_fwd: null pointer");
  VITB_REQUIRE(B > 0 && T > 0 && T <= 128 && heads > 0 && (d == 32 || d == 64 || d == 96 || d == 128),
               "attn_fwd: unsupported shape B=%d T=%d heads=%d d=%d (T<=128, d in {32,64,96,128})", B, T, heads, d);
  cudaStream_t st = (cudaStream_t)stream;
  if (dt == VITB_BF16) {
    VITB_ATTN_DISPATCH(launch_fwd_bf16, qkv, o, lse, attn_map, B, T, heads, scale, st);
  }
  const size_t smem = ((size_t)3 * T * d + (size_t)T * T) * sizeof(float);
  VITB_REQUIRE(d <= 64 || smem <= kMaxSmemPerBlock, "attn_fwd: fp32 tiles at T=%d d=%d need %zu bytes of shared memory (> 227 KB)", T, d, smem);
  if (set_dyn_smem((const void*)attn_fwd_f32_kernel, smem)) return -1;
  VITB_LAUNCH((attn_fwd_f32_kernel), B * heads, 128, smem, st, (const float*)qkv, (float*)o, lse, attn_map, T, heads, d, scale);
  VITB_LAUNCH_OK();
  return 0;
}

int vitb_attn_bwd(const void* qkv, const void* o, const void* d_o, const float* lse, void* dqkv, int B, int T, int heads, int d, float scale,
                  int dt, void* stream) {
  VITB_REQUIRE(qkv && o && d_o && lse && dqkv, "attn_bwd: null pointer");
  VITB_REQUIRE(B > 0 && T > 0 && T <= 128 && heads > 0 && (d == 32 || d == 64 || d == 96 || d == 128),
               "attn_bwd: unsupported shape B=%d T=%d heads=%d d=%d (T<=128, d in {32,64,96,128})", B, T, heads, d);
  cudaStream_t st = (cudaStream_t)stream;
  if (dt == VITB_BF16) {
    VITB_ATTN_DISPATCH(launch_bwd_bf16, qkv, o, d_o, lse, dqkv, B, T, heads, scale, st);
  }
  const size_t smem = ((size_t)4 * T * d + (size_t)2 * T * T) * sizeof(float);
  VITB_REQUIRE(d <= 64 || smem <= kMaxSmemPerBlock, "attn_bwd: fp32 tiles at T=%d d=%d need %zu bytes of shared memory (> 227 KB)", T, d, smem);
  if (set_dyn_smem((const void*)attn_bwd_f32_kernel, smem)) return -1;
  VITB_LAUNCH((attn_bwd_f32_kernel), B * heads, 128, smem, st, (const float*)qkv, (const float*)d_o, lse, (float*)dqkv, T, heads, d, scale);
  VITB_LAUNCH_OK();
  return 0;
}

}  // extern "C"
