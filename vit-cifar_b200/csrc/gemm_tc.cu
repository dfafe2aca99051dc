// gemm_tc.cu — bf16 tensor-core GEMM for sm_100a: TMA (128B swizzle) -> shared-memory ring ->
// tcgen05.mma (kind::f16, bf16 x bf16 -> fp32 in TMEM) -> tcgen05.ld epilogue with fused
// bias / GELU / residual / pre-activation save / GELU-backward, or fp32 split-K partials.
//
// One persistent kernel, three roles: TMA producer warp(s), MMA issuer warp(s), 8 epilogue warps; TMEM
// accumulator stages so the epilogue of tile i overlaps the MMAs of tile i+1.
// NS = 2 ("dual stream"): a 128x128x16 MMA occupies the tensor pipe for 64 cycles, but ONE issuing thread
// needs ~50 cycles per MMA plus ~300 per barrier wait / tcgen05.commit round trip (measured, tools/mma_bench.cu
// and tools/gemm_timeline.py), so a single producer/issuer pair leaves the pipe half idle at this tile width.
// Two independent producer/issuer pairs ("streams") walk alternate tiles of the CTA's tile list with their own
// smem rings, barriers and TMEM accumulators (and share the resident weight block); the pipe interleaves them.  The epilogue never touches global memory with per-thread row accesses: every epilogue
// warp owns a 32-row x 64-column slab, stages bf16 results in 128B-swizzled shared memory and moves
// whole slabs with TMA (store for C / pre-activation, load for the residual / GELU-backward operand).
// wgrad additionally computes the bias gradient with one extra N=16 MMA per k-step against an
// all-ones operand (column sums of dY for free on the tensor pipe).  Operand layouts are chosen per GEMM so no tensor is ever transposed in memory:
//   fwd   C[M,N]  = A[M,K]   · W[N,K]ᵀ : A K-major,  B K-major
//   dgrad dX[M,K] = dY[M,N]  · W[N,K]  : A K-major,  B MN-major (reduction runs over W's rows)
//   wgrad dW[N,K] = dY[M,N]ᵀ · X[M,K]  : A MN-major, B MN-major (reduction runs over the rows of both)
#include <cuda.h>
#include <stdlib.h>

#include "common.cuh"
#include "gemm_internal.h"

namespace vitb {

constexpr int BM = 128;          // UMMA M (cta_group::1)
constexpr int BK = 64;           // one 128-byte swizzle atom of bf16 along the contiguous dimension
constexpr int UK = 16;           // K per tcgen05.mma for 16-bit inputs
constexpr int kEpiWarps = 8;
// epilogue warps of an instantiation: 4 TMEM lane quarters x (BN / 64) column groups of 64 in the slab epilogue of the 192-wide
// forward / dgrad tiles (12 warps), 8 everywhere else
constexpr int epi_warps_for(int bn, int nslab) { return (bn == 192 && nslab > 0) ? 12 : kEpiWarps; }
constexpr int tc_threads(int ns, int ew = kEpiWarps) { return (2 * ns + ew) * 32; }  // NS TMA warps + NS MMA warps + the epilogue warps
constexpr uint32_t kTmemCols = 512;  // NS x ACC accumulators of 128 columns (+ 16-column bias-gradient accumulators in wgrad)
constexpr int kSlabBytes = 32 * 128;  // 32 rows x 64 bf16, 128B swizzle

struct TcArgs {
  int M;             // valid output rows (C rows; for wgrad: N_out)
  int N;             // output columns (multiple of BN)
  int num_m_blocks, num_n_blocks, splits;
  int kblocks_total, kblocks_per_split;
  int has_in;        // tma_in valid: residual (EPI_FWD) or z for gelu' (EPI_DGRAD)
  int has_pre;       // tma_pre valid: store the pre-activation
  float* dbias_part; // wgrad: [splits][M] fp32 partial column sums of dY (or null)
  int valid_n;       // RAW epilogue: columns >= valid_n are not stored (patch-embedding wgrad: K = 48 inside a 128 tile)
  int a3_pp;         // > 0: the MN-major A operand is a (B, T, H) tensor read through a 3-D map, a3_pp token rows per image
  int a3_off;        //      first token row used (1 when a cls row is skipped)
  long long* dbg;    // optional per-CTA cycle counters (tools/gemm_timeline.py); null in production
  int pair;          // resident fwd/dgrad launched as cta_group::2 pairs (num_m_blocks then counts 256-row blocks, tma_b boxes are half tiles)
  int pf_tiles;      // fwd/dgrad: prefetch the A tile this many tiles (per stream) ahead into L2; 0 = off
  int pf_kblocks;    // wgrad: prefetch operands this many k-blocks ahead into L2; 0 = off
  int pf_in;         // resident fwd/dgrad: also prefetch the epilogue's input operand (residual / z) of the tile pf_tiles ahead
  int dbg_flags;     // tools only: 1 = epilogue skips its work (accumulator handed straight back), 2 = producer loads nothing
  DropParams drop;   // thr != 0: nn.Dropout on the output, after GELU / gelu' and before the residual (mask over the flattened [M, N] output)
  int out3;          // EPI_FWD: tma_out is a 3-D (columns, tokens, images) map of a (B, T, H) tensor — the patch embedding writes GEMM
                     // row m to token e.rm_offset + m % e.rm_group of image m / e.rm_group and adds e.pos[token] (vit.py:68-70)
  EpiParams e;
};

// ---------------------------------------------------------------------------------------------
// PTX wrappers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// Wait with a wall-clock bound: a protocol bug traps (launch error) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  long long t0 = 0;
  for (uint32_t it = 0;; ++it) {
    asm volatile(
        "{\n.reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n}\n"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    if (done) return;
    if (it == 64) t0 = clock64();
    if (it > 64 && (it & 1023) == 0 && clock64() - t0 > 4000000000LL) {
      printf("vitb gemm_tc: mbarrier wait timed out (block %d thread %d bar %u parity %u)\n", blockIdx.x, threadIdx.x, bar, parity);
      __trap();
    }
  }
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"((uint64_t)map), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"((uint64_t)map), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// L2 prefetch of a box: costs no shared memory, so operands can be requested from HBM much further ahead than the ring holds
__device__ __forceinline__ void tma_prefetch_2d(const CUtensorMap* map, int c0, int c1) {
  asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global [%0, {%1, %2}];" ::"l"((uint64_t)map), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, uint32_t src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"((uint64_t)map), "r"(src), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* map, uint32_t src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
               ::"l"((uint64_t)map), "r"(src), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
#ifndef VITB_TC_TAIL_WAIT_READ
#define VITB_TC_TAIL_WAIT_READ 1
#endif
constexpr bool kTailWaitRead = VITB_TC_TAIL_WAIT_READ != 0;
#ifndef VITB_TC_BIAS_PREFETCH
#define VITB_TC_BIAS_PREFETCH 1
#endif
constexpr bool kBiasPrefetch = VITB_TC_BIAS_PREFETCH != 0;
__device__ __forceinline__ void prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// ---- cta_group::2 (a pair of CTAs on adjacent SMs computes one 256-row tile; only the leader issues MMAs) ----
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t mapa_rank(uint32_t addr, uint32_t rank) {  // the same shared-memory offset in CTA `rank` of the cluster
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_remote(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// TMA load into THIS CTA's shared memory that signals an mbarrier of the pair's leader CTA
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* map, uint32_t leader_bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"((uint64_t)map), "r"(leader_bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tc_commit_pair(uint32_t bar) {  // arrives on the barrier at this offset in BOTH CTAs
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar), "h"((uint16_t)3)
               : "memory");
}
__device__ __forceinline__ void tc_mma_bf16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n.reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n}\n"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tc_mma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n.reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}\n"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tc_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tc_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ int ceil_div_dev(int a, int b) { return (a + b - 1) / b; }

// shared-memory matrix descriptor (SWIZZLE_128B, descriptor version 1)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;  // version
  d |= (uint64_t)2 << 61;  // SWIZZLE_128B
  return d;
}

// The high word of every descriptor used here is one constant (SBO = 1024 B, version 1, SWIZZLE_128B); the low word is
// (address >> 4) | (LBO >> 4) << 16, so walking k or the ring is a single add on a precomputed low word.
constexpr uint32_t kDescHi = ((1024u >> 4) & 0x3FFFu) | (1u << 14) | (2u << 29);
__device__ __forceinline__ uint32_t desc_lo(uint32_t saddr, uint32_t lbo_bytes) { return ((saddr & 0x3FFFFu) >> 4) | (((lbo_bytes >> 4) & 0x3FFFu) << 16); }
__device__ __forceinline__ uint64_t desc_from_lo(uint32_t lo) { return ((uint64_t)kDescHi << 32) | (uint64_t)lo; }
// one lane of a converged warp; code under `if (elect_one())` is compiled as warp-uniform (no per-lane waterfall loops
// around the uniform-datapath tcgen05 / TMA instructions, which cost more than the MMAs they issue)
__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile("{\n.reg .pred P1;\nelect.sync _|P1, 0xffffffff;\nselp.u32 %0, 1, 0, P1;\n}\n" : "=r"(pred));
  return pred != 0;
}

constexpr int kMaxResKB = 6;  // resident-B mode keeps up to 6 k-blocks (K <= 384) of the weight tile in shared memory

// shared-memory plan: [resident B slab (W_RES)] [ring: STAGES x KPS x (A | B) tiles] [epilogue slabs / ones operand] [barriers] [tmem slot]
// A ring stage holds KPS consecutive k-blocks behind ONE full/empty barrier pair: the MMA-issuing thread pays its
// wait + commit round trip (which the tensor pipe cannot hide: tools/mma_bench.cu) once per 4*KPS MMAs.
template <int BN, int NS, int STAGES, int KPS, int NSLAB, bool W_RES, int CG = 1>
struct TcSmem {
  static constexpr int kAcc = (NS == 2 && NSLAB == 0) ? 1 : 2;  // TMEM accumulator stages per stream (wgrad items are long: 1 is enough)
  static constexpr int kEW = epi_warps_for(BN, NSLAB);
  static constexpr uint32_t kABytes = BM * BK * 2;
  static constexpr uint32_t kBBytes = (BN / CG) * BK * 2;  // a CTA of a pair holds half of the B tile
  static constexpr uint32_t kSubBytes = W_RES ? kABytes : kABytes + kBBytes;  // one k-block
  static constexpr uint32_t kStageBytes = KPS * kSubBytes;
  static constexpr uint32_t kResBytes = W_RES ? kMaxResKB * kBBytes : 0;
  static constexpr uint32_t kRingOff = kResBytes;
  static constexpr uint32_t kRingBytes = STAGES * kStageBytes;  // per stream
  static constexpr uint32_t kEpiOff = kRingOff + NS * kRingBytes;
  static constexpr uint32_t kEpiBytes = NSLAB > 0 ? kEW * NSLAB * kSlabBytes : 2048;  // NSLAB slabs per epilogue warp, or the all-ones wgrad operand
  static constexpr uint32_t kBarOff = kEpiOff + kEpiBytes;
  static constexpr uint32_t kBarsPerStream = 2 * STAGES + 4;  // full[STAGES] empty[STAGES] tfull[2] tempty[2]
  static constexpr uint32_t kNumBars = NS * kBarsPerStream + kEW + 1;
  static constexpr uint32_t kTotal = kBarOff + kNumBars * 8 + 16;
  static constexpr uint32_t kDynBytes = kTotal + 1024;  // slack for manual 1024-byte alignment
};

// ---------------------------------------------------------------------------------------------
// epilogue helpers: one thread = one row of a 32 x 64 slab (128 B per row, 128B swizzle: 16-byte chunk j of
// row r lives at chunk position j ^ (r & 7), the layout TMA reads/writes with CU_TENSOR_MAP_SWIZZLE_128B;
// a quarter-warp's 16-byte accesses then fall in 8 distinct bank groups -> conflict-free)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void slab_store_row64(uint32_t slab, int r, const float (&f)[64]) {
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const uint32_t addr = slab + (uint32_t)r * 128u + (uint32_t)((j ^ (r & 7)) << 4);
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(pack_bf16x2(f[8 * j + 0], f[8 * j + 1])),
                 "r"(pack_bf16x2(f[8 * j + 2], f[8 * j + 3])), "r"(pack_bf16x2(f[8 * j + 4], f[8 * j + 5])),
                 "r"(pack_bf16x2(f[8 * j + 6], f[8 * j + 7]))
                 : "memory");
  }
}
__device__ __forceinline__ void slab_load_chunk8(uint32_t slab, int r, int j, float (&f)[8]) {
  const uint32_t addr = slab + (uint32_t)r * 128u + (uint32_t)((j ^ (r & 7)) << 4);
  uint32_t a, b, c, d;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(a), "=r"(b), "=r"(c), "=r"(d) : "r"(addr) : "memory");
  float2 x = unpack_bf16x2(a), y = unpack_bf16x2(b), z = unpack_bf16x2(c), w = unpack_bf16x2(d);
  f[0] = x.x; f[1] = x.y; f[2] = y.x; f[3] = y.y; f[4] = z.x; f[5] = z.y; f[6] = w.x; f[7] = w.y;
}

// ---------------------------------------------------------------------------------------------
// the kernel
// ---------------------------------------------------------------------------------------------
// W_RES ("resident weights", fwd / dgrad with K <= 384): the CTA owns ONE 128-column block of the output, loads that
// block's B operand (all k-blocks) into shared memory once, and streams only A tiles for its share of the m-blocks —
// half the L2->SM traffic per tile of the streaming mode, which is what bounds these 384-wide GEMMs.
// CG = 2 ("pair", resident fwd / dgrad only): two CTAs on adjacent SMs form a cluster and compute one 256-row tile with
// tcgen05.mma.cta_group::2 — each loads its own 128 rows of A and keeps HALF of the weight block (48 KB instead of 96 KB), which
// buys every stream a fourth ring stage (ring depth is what bounds these kernels, DESIGN.md 3a).  The leader CTA issues the MMAs
// for both; full / accumulator-empty barriers live in the leader (the peer's TMA loads and epilogue warps signal them remotely),
// empty / accumulator-full barriers exist in both CTAs and are signalled by multicast tcgen05.commit.
#define VITB_TC_KERNEL gemm_tc_kernel
#define VITB_TC_TAIL false
#include "gemm_tc_kernel.cuh"
#undef VITB_TC_KERNEL
#undef VITB_TC_TAIL
#define VITB_TC_KERNEL gemm_tc_tail_kernel
#define VITB_TC_TAIL true
#include "gemm_tc_kernel.cuh"
#undef VITB_TC_KERNEL
#undef VITB_TC_TAIL

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess || qres != cudaDriverEntryPointSuccess) return nullptr;
  fn = (EncodeTiledFn)p;
  return fn;
}

// 2-D bf16 tensor [outer][inner] (inner contiguous), box = 64 x box_outer, 128-byte swizzle
static int make_map(CUtensorMap* map, const void* ptr, uint64_t inner, uint64_t outer, uint64_t pitch_elems, uint32_t box_outer) {
  EncodeTiledFn fn = get_encode_fn();
  VITB_REQUIRE(fn != nullptr, "cuTensorMapEncodeTiled not available from the driver");
  VITB_REQUIRE(((uintptr_t)ptr % 16 == 0) && (pitch_elems * 2) % 16 == 0, "gemm_tc: operand must be 16-byte aligned with a 16-byte multiple pitch");
  cuuint64_t gdim[2] = {inner, outer};
  cuuint64_t gstr[1] = {pitch_elems * 2};
  cuuint32_t box[2] = {64, box_outer};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  VITB_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed with CUresult %d (inner=%llu outer=%llu pitch=%llu box=%u)", (int)r,
               (unsigned long long)inner, (unsigned long long)outer, (unsigned long long)pitch_elems, box_outer);
  return 0;
}

// 3-D bf16 tensor (B, T, H) read as 64 H-columns x `rows` token rows x `imgs` images (128B swizzle): the MN-major A operand
// of the patch-embedding wgrad, which must skip the cls row of every image
static int make_map3(CUtensorMap* map, const void* ptr, uint64_t H, uint64_t Tn, uint64_t B, uint32_t rows, uint32_t imgs) {
  EncodeTiledFn fn = get_encode_fn();
  VITB_REQUIRE(fn != nullptr, "cuTensorMapEncodeTiled not available from the driver");
  cuuint64_t gdim[3] = {H, Tn, B};
  cuuint64_t gstr[2] = {H * 2, Tn * H * 2};
  cuuint32_t box[3] = {64, rows, imgs};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(ptr), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  VITB_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(3d) failed with CUresult %d", (int)r);
  return 0;
}

int make_tma_map_3d_bf16(CUtensorMap* map, const void* ptr, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t stride1_bytes, uint64_t stride2_bytes,
                         uint32_t box0, uint32_t box1, uint32_t box2, int swizzle_bytes) {
  EncodeTiledFn fn = get_encode_fn();
  VITB_REQUIRE(fn != nullptr, "cuTensorMapEncodeTiled not available from the driver");
  VITB_REQUIRE(((uintptr_t)ptr % 16 == 0) && stride1_bytes % 16 == 0 && stride2_bytes % 16 == 0, "tensor map: operand must be 16-byte aligned with 16-byte multiple strides");
  cuuint64_t gdim[3] = {d0, d1, d2};
  cuuint64_t gstr[2] = {stride1_bytes, stride2_bytes};
  cuuint32_t box[3] = {box0, box1, box2};
  cuuint32_t estr[3] = {1, 1, 1};
  const CUtensorMapSwizzle sw = swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                                : swizzle_bytes == 32 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_NONE;
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(ptr), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  VITB_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(3d) failed with CUresult %d (dims %llu %llu %llu box %u %u %u)", (int)r, (unsigned long long)d0,
               (unsigned long long)d1, (unsigned long long)d2, box0, box1, box2);
  return 0;
}

struct TcMaps {
  CUtensorMap a, b, out, pre, in;
};

template <int BN, bool A_MN, bool B_MN, int NS, int STAGES, int KPS, int NSLAB, bool W_RES, int CG = 1, bool DROP = false, bool TAIL = false>
static int launch_tc_impl(const TcMaps& m, const TcArgs& args, cudaStream_t st) {
  using S = TcSmem<BN, NS, STAGES, KPS, NSLAB, W_RES, CG>;
  static_assert(S::kDynBytes <= 232448, "shared memory plan exceeds 227 KB");
  auto kern = gemm_tc_kernel<BN, A_MN, B_MN, NS, STAGES, KPS, NSLAB, W_RES, CG, DROP>;
  if constexpr (TAIL) kern = gemm_tc_tail_kernel<BN, A_MN, B_MN, NS, STAGES, KPS, NSLAB, W_RES, CG, DROP>;
  static bool configured = false;  // per instantiation
  if (!configured) {
    VITB_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S::kDynBytes));
    configured = true;
  }
  int grid;
  if (W_RES) {
    int units = kNumSMs / CG;
    if (CG == 2) {
      // every pair must be resident at once (persistent kernel): ask the driver how many 2-CTA clusters of this kernel fit
      static int max_clusters = -1;
      if (max_clusters < 0) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(kNumSMs / 2 * 2);
        cfg.blockDim = dim3(tc_threads(NS, S::kEW));
        cfg.dynamicSmemBytes = S::kDynBytes;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        int n = 0;
        VITB_CUDA_OK(cudaOccupancyMaxActiveClusters(&n, kern, &cfg));
        max_clusters = n;
        if (getenv("VITB_DEBUG")) fprintf(stderr, "vitb gemm_tc: max active 2-CTA clusters = %d\n", n);
      }
      if (units > max_clusters) units = max_clusters;
      VITB_REQUIRE(units >= args.num_n_blocks, "gemm_tc pair mode: only %d clusters fit", units);
    }
    grid = CG * (units / args.num_n_blocks) * args.num_n_blocks;  // (members per column block) x (column blocks) [x 2 CTAs per pair]
  } else {
    const int tiles = args.num_m_blocks * args.num_n_blocks * args.splits;
    grid = tiles < kNumSMs ? tiles : kNumSMs;
  }
  if (CG == 2) {
    VITB_CUDA_OK(::vitb::launch_kernel_cluster(kern, grid, tc_threads(NS, S::kEW), S::kDynBytes, st, 2, m.a, m.b, m.out, m.pre, m.in, args));
  } else {
    VITB_LAUNCH((kern), grid, tc_threads(NS, S::kEW), S::kDynBytes, st, m.a, m.b, m.out, m.pre, m.in, args);
  }
  VITB_LAUNCH_OK();
  return 0;
}

constexpr int kBN = 128;
static int env_int(const char* name, int dflt) { const char* v = getenv(name); return v ? atoi(v) : dflt; }

static long long* g_tc_dbg = nullptr;  // set through vitb_debug_gemm_timeline (tools only)
static int g_tc_force_mode = 0;        // 0 auto, 1 never resident, 2 always resident (when legal)
static int g_tc_dbg_flags = 0;
// L2 prefetch distances (tools / VITB_GEMM_PF_* can change them)
static int g_tc_pf_tiles = env_int("VITB_GEMM_PF_TILES", 2), g_tc_pf_kblocks = env_int("VITB_GEMM_PF_KBLOCKS", 8);
static int g_tc_pf_in = env_int("VITB_GEMM_PF_IN", 0);

static bool use_resident_weights(const TcArgs& a) {
  if (a.e.mode == EPI_RAW_F32 || a.splits != 1 || a.kblocks_total > kMaxResKB || a.num_n_blocks > kNumSMs) return false;
  if (g_tc_force_mode == 1) return false;
  if (g_tc_force_mode == 2) return true;
  const int members = kNumSMs / a.num_n_blocks;
  return a.num_m_blocks >= 2 * members;  // enough row blocks per CTA to amortise loading the weight block
}

// cta_group::2 pairs (CG = 2) for the resident-weight kernels were an experiment of round 1: parity-correct on 256-row-aligned M and
// exactly as fast as the single-CTA kernel (fwd 66560x384x384: 26.1 vs 26.3 us, profiles/r1_gemm_timeline_cta_pair_experiment.log),
// with an unresolved deadlock when the last pair's peer tile lies entirely beyond M.  The kernel template keeps its CG parameter
// (the barrier / multicast-commit plumbing is the starting point for full-width tiles), but the library instantiates CG = 1 only:
// no code ships that the GPU test suite does not run.
// The smem rings get whatever the resident weights and the epilogue slabs leave free (227 KB per CTA):
//   slabs per epilogue warp = 1 (output; shared with the input operand and, sequentially, with a pre-activation output);
//   0 = fp32 direct-store epilogue (wgrad)
//   <NS, STAGES, KPS> dual stream: wgrad 2 x 3 x 32 KB;  resident 2 x 3 x 16 KB;  streaming 2 x 3 x 32 KB.
//   g_tc_streams = 1 (tools) selects the single-stream plans.
static int g_tc_streams = 2;
static int g_tc_wgrad_bn = 192;  // wgrad tile width; tools can force 128

// TAIL: forward / dgrad with a partial last column block (output width 64 mod 128), 128-wide tiles: the same plans as below
// except the single-stream ones that only tools select
template <int BN, bool A_MN, bool B_MN, bool TAIL = false>
static int launch_tc(const TcMaps& m, const TcArgs& args_in, cudaStream_t st) {
  TcArgs args = args_in;
  args.dbg = g_tc_dbg;
  args.dbg_flags = g_tc_dbg_flags;
  args.pf_tiles = g_tc_pf_tiles;
  args.pf_kblocks = g_tc_pf_kblocks;
  args.pf_in = g_tc_pf_in;
  if constexpr (TAIL) {
    static_assert(BN == 128 && !A_MN, "partial column tiles: 128-wide forward / dgrad");
    const bool res = use_resident_weights(args);
    if (args.drop.thr != 0) {
      if (res) return launch_tc_impl<BN, A_MN, B_MN, 2, 3, 1, 1, true, 1, true, true>(m, args, st);
      return launch_tc_impl<BN, A_MN, B_MN, 2, 3, 1, 1, false, 1, true, true>(m, args, st);
    }
    if (res) return launch_tc_impl<BN, A_MN, B_MN, 2, 3, 1, 1, true, 1, false, true>(m, args, st);
    if (args.kblocks_total <= 6 && args.num_m_blocks * args.num_n_blocks <= 2 * kNumSMs)
      return launch_tc_impl<BN, A_MN, B_MN, 1, 3, 2, 1, false, 1, false, true>(m, args, st);
    return launch_tc_impl<BN, A_MN, B_MN, 2, 3, 1, 1, false, 1, false, true>(m, args, st);
  } else if constexpr (BN != 128) {
    // wide tiles (BN = 192): a 128x192x16 MMA holds the pipe for 96 cycles, which one issuing thread can sustain, and the
    // operand bytes per FLOP drop by a sixth; single stream.  wgrad: 5 stages x 40 KB, fp32 direct-store epilogue;
    // forward / dgrad (A K-major): 4 stages x 40 KB and a 12-warp slab epilogue
    if constexpr (A_MN) return launch_tc_impl<BN, A_MN, B_MN, 1, 5, 1, 0, false>(m, args, st);
    else return launch_tc_impl<BN, A_MN, B_MN, 1, 4, 1, 1, false>(m, args, st);
  } else {
  const bool res = !A_MN && use_resident_weights(args);
  if constexpr (!A_MN) {
    if (args.drop.thr != 0) {  // dropout in the epilogue: the two dual-stream plans carry it
      if (res) return launch_tc_impl<BN, A_MN, B_MN, 2, 3, 1, 1, true, 1, true>(m, args, st);
      return launch_tc_impl<BN, A_MN, B_MN, 2, 3, 1, 1, false, 1, true>(m, args, st);
    }
  }
  if (g_tc_streams == 1) {
    if (args.e.mode == EPI_RAW_F32) return launch_tc_impl<BN, A_MN, B_MN, 1, 3, 2, 0, false>(m, args, st);
    if (res) return launch_tc_impl<BN, A_MN, B_MN, 1, 3, 2, 1, true>(m, args, st);
    return launch_tc_impl<BN, A_MN, B_MN, 1, 3, 2, 1, false>(m, args, st);
  }
  if (args.e.mode == EPI_RAW_F32) return launch_tc_impl<BN, A_MN, B_MN, 2, 3, 1, 0, false>(m, args, st);
  // (a pre-activation output shares the output slab, see the epilogue: every variant keeps 3 ring stages per stream)
  if (res) return launch_tc_impl<BN, A_MN, B_MN, 2, 3, 1, 1, true>(m, args, st);
  // Small problems (at most two tiles per SM, K <= 384: batch 128, T = 17): the kernel is one load latency + one tile of MMAs +
  // one epilogue long.  One stream with the WHOLE reduction of a tile in flight (3 stages x 2 k-blocks = 192 KB) needs a single
  // round trip to memory where two 3 x 1 rings need two (VITB_GEMM_SMALL_DEEP=0 switches it off).
  static const bool small_deep = getenv("VITB_GEMM_SMALL_DEEP") ? atoi(getenv("VITB_GEMM_SMALL_DEEP")) != 0 : true;
  if (small_deep && args.kblocks_total <= 6 && args.num_m_blocks * args.num_n_blocks * args.splits <= 2 * kNumSMs)
    return launch_tc_impl<BN, A_MN, B_MN, 1, 3, 2, 1, false>(m, args, st);
  return launch_tc_impl<BN, A_MN, B_MN, 2, 3, 1, 1, false>(m, args, st);
  }
}

// K needs only a 16-byte row pitch: a partial last k-block is zero-filled by TMA.  N % 128 == 64: a partial last column block
// (the TAIL kernels)
static bool tc_shape_ok(int M, int N, int K) { return M >= 32 && N % 64 == 0 && K % 8 == 0; }

// 128 x 192 output tiles for forward / dgrad (12-warp slab epilogue).  Used (a) when they turn a problem of more than one
// wave of 128 x 128 tiles into a single wave (8,320 rows x 384 columns: 130 tiles instead of 195 on 148 SMs — the kernel is then one
// tile long instead of two), and (b) VITB_GEMM_BN192_STREAM=1 (experiment): for outputs whose weight slice cannot be resident
// (reduction > 384, e.g. the QKV dgrad), where two column blocks instead of three read A twice instead of three times.
static bool use_bn192(int M, int Nout, int Kred) {
  static const int mode = getenv("VITB_GEMM_BN192") ? atoi(getenv("VITB_GEMM_BN192")) : 1;
  static const bool stream = getenv("VITB_GEMM_BN192_STREAM") && atoi(getenv("VITB_GEMM_BN192_STREAM")) != 0;
  if (mode == 0 || Nout % 192 != 0) return false;
  const int mb = ceil_div(M, BM);
  if (mb * (Nout / 192) <= kNumSMs && mb * ceil_div(Nout, 128) > kNumSMs) return true;
  if (stream && Kred > kMaxResKB * BK && mb * (Nout / 192) >= 4 * kNumSMs) return true;
  return false;
}

static int check_dt(int dt) {
  VITB_REQUIRE(dt == VITB_F32 || dt == VITB_BF16, "dt must be VITB_F32 or VITB_BF16 (got %d)", dt);
  return 0;
}

// ---------------------------------------------------------------------------------------------
// patch embedding on the tensor cores (called from gemm_simt.cu's front end)
// ---------------------------------------------------------------------------------------------
bool tc_patch_ok(int PP, int H, int K) {
  // (the 32-row epilogue slabs must be whole tokens of one image or whole images: PP a multiple or a divisor of 32)
  return H % 64 == 0 && K % 8 == 0 && K <= 256 && ((PP >= 64 && PP % 64 == 0) || (PP < 64 && 64 % PP == 0)) && (PP % 32 == 0 || 32 % PP == 0);
}

// out (B, Tn, H) bf16: token rows off .. off + PP - 1 of every image = words · wᵀ + bias + pos[token]  (vit.py:66-70; the cls row is
// written by the caller).  The epilogue stores straight into the (B, T, H) tensor through a 3-D map: no intermediate buffer.
int tc_patch_fwd(const void* words, const void* w_bf16, const float* bias, const float* pos, const void* pos_bf16, void* out, int B, int PP, int Tn,
                 int off, int H, int K, cudaStream_t st) {
  const int M = B * PP;
  TcMaps m;
  if (make_map(&m.a, words, K, M, K, BM)) return -1;
  if (make_map(&m.b, w_bf16, K, H, K, kBN)) return -1;
  const uint32_t toks = PP >= 32 ? 32 : (uint32_t)PP, imgs = PP >= 32 ? 1 : (uint32_t)(32 / PP);
  if (make_tma_map_3d_bf16(&m.out, out, (uint64_t)H, (uint64_t)Tn, (uint64_t)B, (uint64_t)H * 2, (uint64_t)Tn * H * 2, 64, toks, imgs, 128)) return -1;
  m.pre = m.out; m.in = m.out;
  TcArgs t = {};
  t.M = M; t.N = H; t.num_m_blocks = ceil_div(M, BM); t.num_n_blocks = ceil_div(H, kBN); t.splits = 1;
  t.kblocks_total = ceil_div(K, BK); t.kblocks_per_split = t.kblocks_total; t.valid_n = H;
  t.e.mode = EPI_FWD; t.e.bias = bias; t.e.out = out; t.e.ldc = H;
  t.out3 = 1; t.e.rm_group = PP; t.e.rm_stride = Tn; t.e.rm_offset = off;
  if (pos_bf16 != nullptr && PP % 32 == 0) {
    // pos_emb rides in like a residual: each epilogue warp TMA-loads the 32 token rows of its slab from the bf16 copy (the
    // kernel has next to no L1 beside its shared memory: per-thread fp32 loads of pos cost more than the GEMM, 45 vs 20 us)
    if (make_map(&m.in, pos_bf16, H, Tn, H, 32)) return -1;
    t.has_in = 1;
    t.e.residual = pos_bf16;
  } else {
    t.e.pos = pos;  // 32 rows of a slab span several images (PP < 32): per-thread fp32 loads
  }
  if (H % kBN != 0) return launch_tc<kBN, false, false, true>(m, t, st);
  return launch_tc<kBN, false, false>(m, t, st);
}

static void patch_wgrad_plan(int B, int PP, int H, int* splits, int* kb_total, int* kb_per) {
  const int tiles = ceil_div(H, BM);  // one 128-wide n block holds all K <= 128 columns (two for K = 192)
  const int total = ceil_div(B * PP, BK);
  int s = (kNumSMs * g_tc_streams) / (tiles > 0 ? tiles : 1);  // one work item per stream of every CTA
  if (s < 1) s = 1;
  if (s > total) s = total;
  const int per = ceil_div(total, s);
  *splits = ceil_div(total, per);
  *kb_total = total;
  *kb_per = per;
}

size_t tc_patch_wgrad_ws_bytes(int B, int PP, int H, int K) {
  int splits, a, b;
  patch_wgrad_plan(B, PP, H, &splits, &a, &b);
  return align_up((size_t)splits * H * K * sizeof(float), 256) + align_up((size_t)splits * H * sizeof(float), 256);
}

int tc_patch_wgrad(const void* dout, const void* words, float* dw, float* dbias, void* ws, size_t ws_bytes, int B, int Tn, int PP,
                   int has_cls, int H, int K, cudaStream_t st) {
  VITB_REQUIRE(ws && ws_bytes >= tc_patch_wgrad_ws_bytes(B, PP, H, K), "patch wgrad: workspace too small");
  int splits, kb_total, kb_per;
  patch_wgrad_plan(B, PP, H, &splits, &kb_total, &kb_per);
  float* part = (float*)ws;
  float* bpart = (float*)((char*)ws + align_up((size_t)splits * H * K * sizeof(float), 256));
  TcMaps m;
  const uint32_t rows = PP >= 64 ? 64 : PP, imgs = PP >= 64 ? 1 : 64 / PP;
  if (make_map3(&m.a, dout, H, Tn, B, rows, imgs)) return -1;
  if (make_map(&m.b, words, K, (uint64_t)B * PP, K, 64)) return -1;
  m.out = m.b; m.pre = m.b; m.in = m.b;
  TcArgs t = {};
  t.M = H; t.N = ceil_div(K, kBN) * kBN; t.num_m_blocks = ceil_div(H, BM); t.num_n_blocks = ceil_div(K, kBN); t.splits = splits;
  t.kblocks_total = kb_total; t.kblocks_per_split = kb_per;
  t.e.mode = EPI_RAW_F32; t.e.ldc = K; t.e.out = part; t.valid_n = K;
  t.dbias_part = bpart;
  t.a3_pp = PP; t.a3_off = has_cls ? 1 : 0;
  int rc = launch_tc<kBN, true, true>(m, t, st);
  if (rc) return rc;
  const int64_t n = (int64_t)H * K;
  VITB_CUDA_OK(::vitb::launch_finalize2(part, n, dw, bpart, H, dbias, splits, st));
  return 0;
}

}  // namespace vitb

#include "gemm_bwd_fused.cuh"

using namespace vitb;

// ---------------------------------------------------------------------------------------------
// fused backward of a Linear (gemm_bwd_fused.cuh): host side
// ---------------------------------------------------------------------------------------------
static bool bw_fused_shape_ok(int M, int N, int K) { return M >= 1 && N % 128 == 0 && N >= 128 && N <= 384 && K % 128 == 0 && K / 128 <= kNumSMs; }
// CTAs per 128-column block of K: every SM gets one CTA, but no CTA without a row block
static int bw_members(int M, int K) {
  const int nb = K / 128, mblocks = ceil_div(M, BM);
  int mem = kNumSMs / nb;
  if (mem > mblocks) mem = mblocks;
  return mem < 1 ? 1 : mem;
}

template <int NB>
static int launch_bw_fused(const CUtensorMap& m_dy, const CUtensorMap& m_x, const CUtensorMap& m_w, const CUtensorMap& m_out, const CUtensorMap& m_in,
                           const BwArgs& a, cudaStream_t st) {
  using S = BwSmem<NB>;
  static_assert(S::kDynBytes <= 232448, "shared memory plan exceeds 227 KB");
  auto kern = gemm_bwd_fused_kernel<NB>;
  static bool configured = false;
  if (!configured) {
    VITB_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S::kDynBytes));
    configured = true;
  }
  VITB_LAUNCH((kern), (a.K / 128) * a.members, 384, S::kDynBytes, st, m_dy, m_x, m_w, m_out, m_in, a);
  VITB_LAUNCH_OK();
  return 0;
}

extern "C" {

size_t vitb_gemm_bwd_fused_ws_bytes(int M, int N, int K, int dt) {
  if (dt != VITB_BF16 || !bw_fused_shape_ok(M, N, K)) return 0;
  const size_t mem = (size_t)bw_members(M, K);
  return align_up(mem * N * K * sizeof(float), 256) + align_up(mem * 4 * K * sizeof(float), 256) + 256;
}

int vitb_gemm_bwd_fused(const void* dy, const void* x, const void* w, const void* z, void* dx, float* dw, float* dx_colsum, void* ws, size_t ws_bytes,
                        int M, int N, int K, int dt, void* stream) {
  VITB_REQUIRE(dy && x && w && dx && dw && ws, "gemm_bwd_fused: null pointer");
  const size_t need = vitb_gemm_bwd_fused_ws_bytes(M, N, K, dt);
  VITB_REQUIRE(need != 0, "gemm_bwd_fused: no fused kernel for M=%d N=%d K=%d dt=%d (bf16, N in {128, 256, 384}, K a multiple of 128): use dgrad + wgrad", M,
               N, K, dt);
  VITB_REQUIRE(ws_bytes >= need, "gemm_bwd_fused: workspace too small (%zu < %zu)", ws_bytes, need);
  if (void* d = defer_alloc(need)) ws = d;  // deferred second pass: the partials live in the arena until vitb_defer_flush
  cudaStream_t st = (cudaStream_t)stream;
  CUtensorMap m_dy, m_x, m_w, m_out, m_in;
  if (make_map(&m_dy, dy, N, M, N, BM)) return -1;   // boxes of 64 columns x 128 rows
  if (make_map(&m_x, x, K, M, K, 64)) return -1;     // 64 x 64
  if (make_map(&m_w, w, K, N, K, 64)) return -1;     // 64 output columns x 64 reduction rows
  if (make_map(&m_out, dx, K, M, K, 32)) return -1;  // epilogue slabs: 64 x 32
  m_in = m_out;
  if (z && make_map(&m_in, z, K, M, K, 32)) return -1;
  BwArgs a = {};
  a.M = M; a.N = N; a.K = K;
  a.num_m_blocks = ceil_div(M, BM);
  a.members = bw_members(M, K);
  a.has_in = z != nullptr;
  a.dw_part = (float*)ws;
  a.csum_part = dx_colsum ? (float*)((char*)ws + align_up((size_t)a.members * N * K * sizeof(float), 256)) : nullptr;
  a.pf_tiles = g_tc_pf_tiles;
  int rc;
  switch (N / 128) {
    case 1: rc = launch_bw_fused<1>(m_dy, m_x, m_w, m_out, m_in, a, st); break;
    case 2: rc = launch_bw_fused<2>(m_dy, m_x, m_w, m_out, m_in, a, st); break;
    default: rc = launch_bw_fused<3>(m_dy, m_x, m_w, m_out, m_in, a, st); break;
  }
  if (rc) return rc;
  if (a.members > 1) {
    VITB_CUDA_OK(::vitb::launch_finalize(a.dw_part, a.members, (int64_t)N * K, dw, nullptr, nullptr, 1, st));
  } else {
    VITB_CUDA_OK(cudaMemcpyAsync(dw, a.dw_part, (size_t)N * K * sizeof(float), cudaMemcpyDeviceToDevice, st));
  }
  if (dx_colsum) VITB_CUDA_OK(::vitb::launch_finalize(a.csum_part, a.members * 4, K, dx_colsum, nullptr, nullptr, 1, st));
  return 0;
}

/* tools only (not in vitb200.h): dbg = device buffer of 148*8 int64 cycle counters, or NULL; mode 0 auto / 1 streaming / 2 resident */
int vitb_debug_gemm_prefetch(int tiles, int kblocks) {
  g_tc_pf_tiles = tiles;
  g_tc_pf_kblocks = kblocks;
  return 0;
}

int vitb_debug_gemm_timeline(long long* dbg, int mode) {
  g_tc_dbg = dbg;
  g_tc_force_mode = mode & 0xf;
  g_tc_streams = (mode & 0x10) ? 1 : 2;
  g_tc_wgrad_bn = (mode & 0x20) ? 128 : 192;
  g_tc_dbg_flags = mode >> 8;
  return 0;
}

int vitb_gemm_bias_act_fwd(const void* a, const void* w, const float* bias, const void* residual, void* c, void* preact,
                           int M, int N, int K, int flags, int dt, void* stream) {
  return vitb_gemm_bias_act_fwd_drop(a, w, bias, residual, c, preact, M, N, K, flags, dt, nullptr, stream);
}

int vitb_gemm_bias_act_fwd_drop(const void* a, const void* w, const float* bias, const void* residual, void* c, void* preact,
                                int M, int N, int K, int flags, int dt, const vitb_dropout_t* drop, void* stream) {
  VITB_REQUIRE(a && w && c, "gemm_fwd: null pointer");
  VITB_REQUIRE(M > 0 && N > 0 && K > 0, "gemm_fwd: bad shape M=%d N=%d K=%d", M, N, K);
  if (check_dt(dt)) return -1;
  DropParams dp;
  VITB_REQUIRE(make_drop_params(drop, &dp), "gemm_fwd: dropout p = %f outside [0, 1)", (double)drop->p);
  VITB_REQUIRE(dp.thr == 0 || (!(flags & VITB_GEMM_OUT_F32) && N % 8 == 0), "gemm_fwd: dropout needs an activation-type output with N %% 8 == 0");
  cudaStream_t st = (cudaStream_t)stream;
  if (dp.thr != 0 && !(dt == VITB_BF16 && tc_shape_ok(M, N, K))) {
    // no tensor-core epilogue for this shape / type: the plain kernel without the residual, then the stand-alone pass adds mask and residual
    int rc = vitb_gemm_bias_act_fwd(a, w, bias, nullptr, c, preact, M, N, K, flags, dt, stream);
    if (rc) return rc;
    return vitb_dropout(c, residual, c, (int64_t)M * N, drop->p, drop->seed, drop->site, drop->step, drop->step_dev, dt, stream);
  }
  EpiParams e = {};
  e.mode = EPI_FWD; e.gelu = (flags & VITB_GEMM_GELU) ? 1 : 0; e.out_f32 = (flags & VITB_GEMM_OUT_F32) ? 1 : 0;
  e.bias = bias; e.residual = residual; e.out = c; e.preact = preact; e.ldc = N;
  if (dt == VITB_BF16 && tc_shape_ok(M, N, K) && !e.out_f32) {
    TcMaps m;
    if (make_map(&m.a, a, K, M, K, BM)) return -1;
    if (make_map(&m.b, w, K, N, K, kBN)) return -1;
    if (make_map(&m.out, c, N, M, N, 32)) return -1;
    m.pre = m.out; m.in = m.out;
    if (preact && make_map(&m.pre, preact, N, M, N, 32)) return -1;
    if (residual && make_map(&m.in, residual, N, M, N, 32)) return -1;
    TcArgs t = {};
    t.M = M; t.N = N; t.num_m_blocks = ceil_div(M, BM); t.num_n_blocks = ceil_div(N, kBN); t.splits = 1;
    t.kblocks_total = ceil_div(K, BK); t.kblocks_per_split = t.kblocks_total; t.e = e; t.valid_n = N;
    t.has_in = residual != nullptr; t.has_pre = preact != nullptr;
    t.drop = dp;
    if (dp.thr == 0 && use_bn192(M, N, K)) {
      if (make_map(&m.b, w, K, N, K, 192)) return -1;
      t.num_n_blocks = N / 192;
      return launch_tc<192, false, false>(m, t, st);
    }
    if (N % kBN != 0) return launch_tc<kBN, false, false, true>(m, t, st);
    return launch_tc<kBN, false, false>(m, t, st);
  }
  if (e.out_f32 && !e.gelu && !residual && !preact && head_shape_ok(M, N, K)) return head_fwd_launch(a, w, bias, (float*)c, M, N, K, dt, st);
  SimtGemmArgs g = {};
  g.a = a; g.b = w; g.M = M; g.N = N; g.K = K;
  g.a_sm = K; g.a_sk = 1; g.b_sk = 1; g.b_sn = K; g.e = e;
  return simt_gemm_launch(g, dt, dt, dt, 1, st);
}

int vitb_gemm_dgrad(const void* dy, const void* w, const void* z, void* dx, int M, int N, int K, int flags, int dt, void* stream) {
  return vitb_gemm_dgrad_drop(dy, w, z, dx, M, N, K, flags, dt, nullptr, stream);
}

int vitb_gemm_dgrad_drop(const void* dy, const void* w, const void* z, void* dx, int M, int N, int K, int flags, int dt,
                         const vitb_dropout_t* drop, void* stream) {
  VITB_REQUIRE(dy && w && dx, "gemm_dgrad: null pointer");
  VITB_REQUIRE(M > 0 && N > 0 && K > 0, "gemm_dgrad: bad shape M=%d N=%d K=%d", M, N, K);
  if (check_dt(dt)) return -1;
  DropParams dp;
  VITB_REQUIRE(make_drop_params(drop, &dp), "gemm_dgrad: dropout p = %f outside [0, 1)", (double)drop->p);
  VITB_REQUIRE(dp.thr == 0 || K % 8 == 0, "gemm_dgrad: dropout needs K %% 8 == 0");
  cudaStream_t st = (cudaStream_t)stream;
  const int dy_f32 = (flags & VITB_GEMM_DY_F32) ? 1 : 0;
  if (dp.thr != 0 && !(dt == VITB_BF16 && !dy_f32 && tc_shape_ok(M, K, N))) {
    int rc = vitb_gemm_dgrad(dy, w, z, dx, M, N, K, flags, dt, stream);
    if (rc) return rc;
    return vitb_dropout(dx, nullptr, dx, (int64_t)M * K, drop->p, drop->seed, drop->site, drop->step, drop->step_dev, dt, stream);
  }
  EpiParams e = {};
  e.mode = EPI_DGRAD; e.out = dx; e.aux = z; e.ldc = K;
  // GEMM view: C[M, K] = dY[M, N] (K-major, reduction N) x W[N, K] (MN-major: reduction over rows)
  if (dt == VITB_BF16 && !dy_f32 && tc_shape_ok(M, K, N)) {
    TcMaps m;
    if (make_map(&m.a, dy, N, M, N, BM)) return -1;
    if (make_map(&m.b, w, K, N, K, 64)) return -1;  // box: 64 output columns x 64 reduction rows
    if (make_map(&m.out, dx, K, M, K, 32)) return -1;
    m.pre = m.out; m.in = m.out;
    if (z && make_map(&m.in, z, K, M, K, 32)) return -1;
    TcArgs t = {};
    t.M = M; t.N = K; t.num_m_blocks = ceil_div(M, BM); t.num_n_blocks = ceil_div(K, kBN); t.splits = 1;
    t.kblocks_total = ceil_div(N, BK); t.kblocks_per_split = t.kblocks_total; t.e = e; t.valid_n = K;
    t.has_in = z != nullptr;
    t.drop = dp;
    if (dp.thr == 0 && use_bn192(M, K, N)) {  // (the MN-major weight boxes are 64 columns wide: the same map serves both tile widths)
      t.num_n_blocks = K / 192;
      return launch_tc<192, false, true>(m, t, st);
    }
    if (K % kBN != 0) return launch_tc<kBN, false, true, true>(m, t, st);
    return launch_tc<kBN, false, true>(m, t, st);
  }
  if (dy_f32 && !z && head_shape_ok(M, N, K)) return head_dgrad_launch((const float*)dy, w, dx, M, N, K, dt, st);
  SimtGemmArgs g = {};
  g.a = dy; g.b = w; g.M = M; g.N = K; g.K = N;
  g.a_sm = N; g.a_sk = 1; g.b_sk = K; g.b_sn = 1; g.e = e;
  return simt_gemm_launch(g, dy_f32 ? VITB_F32 : dt, dt, dt, 1, st);
}

// split plan for wgrad on the tensor-core path
// 192-wide tiles (single stream) win on narrow outputs, where they save a third of the fp32 partials' column blocks and a sixth of
// the operand traffic; wide outputs (QKV: 9 row blocks) do better with 128-wide tiles on both streams (measured 68 vs 74 us)
static int wgrad_bn(int N, int K) {
  static const int max_rows = getenv("VITB_WGRAD_WIDE_MAX_ROWBLOCKS") ? atoi(getenv("VITB_WGRAD_WIDE_MAX_ROWBLOCKS")) : 4;  // tuning hook
  return (g_tc_wgrad_bn == 192 && K % 192 == 0 && ceil_div(N, BM) <= max_rows) ? 192 : kBN;
}

static void wgrad_tc_plan(int M, int N, int K, int* splits, int* kb_total, int* kb_per) {
  const int bn = wgrad_bn(N, K);
  const int tiles = ceil_div(N, BM) * ceil_div(K, bn);
  const int total = ceil_div(M, BK);
  // 192-wide tiles run single-stream: one work item per CTA.  128-wide tiles: one item per stream of every CTA when the output is
  // wide (QKV: 27 tiles); narrow outputs (9 tiles) keep one item per CTA, where twice the fp32 partials cost more than the second
  // stream gains
  int s = (kNumSMs * ((bn == 128 && tiles >= 18) ? g_tc_streams : 1)) / (tiles > 0 ? tiles : 1);
  // tuning hook: at least this many 64-row k-blocks per work item (fewer, longer items and fewer fp32 partials for small batches)
  static const int min_kb = env_int("VITB_WGRAD_MIN_KBLOCKS", 1);
  if (min_kb > 1 && s > total / min_kb) s = total / min_kb;
  // Short reductions (small batch / few tokens): fewer, longer work items.  A weight gradient runs on the side stream next to the
  // critical path; with 130-272 k-blocks to reduce, 22-24 splits per tile put 6 x 24 CTAs of a few k-blocks each on the machine and
  // write 24 fp32 partial tiles, 8-11 splits finish as soon in wall-clock terms, leave two thirds of the SMs to the critical path and
  // cut the partials (and the flush that re-reads them) to a third.  Measured (profiles/r2_wgrad_splits_ab.md): B=128 1.376 -> 1.272 ms
  // at 8 splits (6: 1.347), T=17 at B=1024 1.997 -> 1.888 ms at 11 (8: 1.913, 16: 1.947), T=17 at B=128 0.910 -> 0.844 ms at 8;
  // B=1024 (1040 k-blocks) is flat from 8 to 24 (12: 6.047 vs 6.071 ms).  VITB_WGRAD_MAX_SPLITS = n caps at n, -1 removes the cap.
  static const int max_splits = env_int("VITB_WGRAD_MAX_SPLITS", 0);
  // 8 splits up to 130 k-blocks, 10-11 at 260-272, 12 from 310 (B = 256: 1.944 -> 1.819 ms at 10, 1.837 at 8; B = 512: 3.184 -> 3.101 ms at 12)
  // From 1000 k-blocks (B = 1024 at T = 65) the old plan stays: the step is the same within the run-to-run band (6.047 vs 6.071 ms,
  // 6.044 vs 6.210 ms) but a 12-split kernel takes twice as long by itself (0.30 instead of 0.39 of the tensor peak in isolation).
  int rule = 8 + (total - 130) / 45;
  rule = rule < 8 ? 8 : (rule > 12 ? 12 : rule);
  if (total >= 1000) rule = s;
  const int cap = max_splits > 0 ? max_splits : (max_splits < 0 ? s : rule);
  if (s > cap) s = cap;
  if (s < 1) s = 1;
  if (s > total) s = total;
  const int per = ceil_div(total, s);
  *splits = ceil_div(total, per);
  *kb_total = total;
  *kb_per = per;
}

// N or K % 128 == 64: partial last row / column blocks; TMA zero-fills the operands past the edge and the fp32 epilogue stores
// only rows < N (dW and bias-gradient rows) and columns < K
static bool wgrad_tc_ok(int N, int K, int flags, int dt) {
  return dt == VITB_BF16 && !(flags & VITB_GEMM_DY_F32) && N % 64 == 0 && K % 64 == 0;
}

static int wgrad_simt_splits(int M, int N, int K) { return simt_pick_splits(ceil_div(N, 64) * ceil_div(K, 64), M); }

// workspace: [dW partials: splits*N*K][dbias partials: splits*N][colsum scratch (SIMT path)]
/* tools / tests only (not in vitb200.h): splits of the reduction a bf16 tensor-core weight gradient of this shape would use */
int vitb_debug_wgrad_splits(int M, int N, int K) {
  if (!wgrad_tc_ok(N, K, 0, VITB_BF16) || M <= 0) return 0;
  int splits, a, b;
  wgrad_tc_plan(M, N, K, &splits, &a, &b);
  return splits;
}

size_t vitb_gemm_wgrad_ws_bytes(int M, int N, int K, int dt) {
  if (M <= 0 || N <= 0 || K <= 0) return 0;
  int splits;
  if (wgrad_tc_ok(N, K, 0, dt)) {
    int a, b;
    wgrad_tc_plan(M, N, K, &splits, &a, &b);
  } else {
    splits = wgrad_simt_splits(M, N, K);
  }
  const size_t part = align_up((size_t)(splits > 1 ? splits : 0) * N * K * sizeof(float), 256);
  const size_t bpart = align_up((size_t)splits * N * sizeof(float), 256);
  return part + bpart + align_up(vitb_colsum_ws_bytes(M, N), 256) + 256;
}

int vitb_gemm_wgrad_dbias(const void* dy, const void* x, float* dw, float* dbias, void* ws, size_t ws_bytes, int M, int N, int K,
                          int flags, int dt, void* stream) {
  VITB_REQUIRE(dy && x && dw, "gemm_wgrad: null pointer");
  VITB_REQUIRE(M > 0 && N > 0 && K > 0, "gemm_wgrad: bad shape M=%d N=%d K=%d", M, N, K);
  if (check_dt(dt)) return -1;
  VITB_REQUIRE(ws_bytes >= vitb_gemm_wgrad_ws_bytes(M, N, K, dt) && (ws != nullptr), "gemm_wgrad: workspace too small (%zu < %zu)", ws_bytes,
               vitb_gemm_wgrad_ws_bytes(M, N, K, dt));
  cudaStream_t st = (cudaStream_t)stream;
  const int dy_dt = (flags & VITB_GEMM_DY_F32) ? VITB_F32 : dt;
  int splits;
  if (wgrad_tc_ok(N, K, flags, dt))  // deferred second pass (vitb_defer_begin): the partials live in the arena until the flush
    if (void* d = defer_alloc(vitb_gemm_wgrad_ws_bytes(M, N, K, dt))) ws = d;
  float* part = (float*)ws;
  if (wgrad_tc_ok(N, K, flags, dt)) {
    int kb_total, kb_per;
    wgrad_tc_plan(M, N, K, &splits, &kb_total, &kb_per);
    const size_t part_bytes = align_up((size_t)(splits > 1 ? splits : 0) * N * K * sizeof(float), 256);
    float* bpart = (float*)((char*)ws + part_bytes);
    // GEMM view: C[N, K] = dYᵀ (A MN-major: [M rows][N contiguous]) x X (B MN-major: [M rows][K contiguous]), reduction M
    TcMaps m;
    if (make_map(&m.a, dy, N, M, N, 64)) return -1;
    if (make_map(&m.b, x, K, M, K, 64)) return -1;
    m.out = m.a; m.pre = m.a; m.in = m.a;  // unused in RAW mode
    TcArgs t = {};
    const int bn = wgrad_bn(N, K);
    t.M = N; t.N = K; t.num_m_blocks = ceil_div(N, BM); t.num_n_blocks = ceil_div(K, bn); t.splits = splits;
    t.kblocks_total = kb_total; t.kblocks_per_split = kb_per;
    t.e.mode = EPI_RAW_F32; t.e.ldc = K; t.e.out = splits > 1 ? part : dw; t.valid_n = K;
    t.dbias_part = dbias ? (splits > 1 ? bpart : dbias) : nullptr;  // bias gradient rides on the tensor pipe (ones-operand MMA)
    int rc = bn == 192 ? launch_tc<192, true, true>(m, t, st) : launch_tc<kBN, true, true>(m, t, st);
    if (rc) return rc;
    if (splits > 1) {
      const int64_t n = (int64_t)N * K;
      if (dbias) VITB_CUDA_OK(::vitb::launch_finalize2(part, n, dw, bpart, N, dbias, splits, st));  // dW and the bias gradient in one launch
      else VITB_CUDA_OK(::vitb::launch_finalize(part, splits, n, dw, nullptr, nullptr, 1, st));
    }
    return 0;
  }
  if ((flags & VITB_GEMM_DY_F32) && head_shape_ok(M, N, K)) return head_wgrad_launch((const float*)dy, x, dw, dbias, M, N, K, dt, st);
  splits = wgrad_simt_splits(M, N, K);
  const size_t part_bytes = align_up((size_t)(splits > 1 ? splits : 0) * N * K * sizeof(float), 256);
  {
    SimtGemmArgs g = {};
    g.a = dy; g.b = x; g.M = N; g.N = K; g.K = M;
    g.a_sm = 1; g.a_sk = N; g.b_sk = K; g.b_sn = 1;
    g.e.mode = EPI_RAW_F32; g.e.ldc = K; g.e.out = splits > 1 ? part : dw;
    int rc = simt_gemm_launch(g, dy_dt, dt, VITB_F32, splits, st);
    if (rc) return rc;
  }
  if (splits > 1) {
    const int64_t n = (int64_t)N * K;
    VITB_CUDA_OK(::vitb::launch_finalize(part, splits, n, dw, nullptr, nullptr, 1, st));
  }
  if (dbias != nullptr) {
    if (N % 128 == 0) {
      char* cws = (char*)ws + part_bytes + align_up((size_t)splits * N * sizeof(float), 256);
      return vitb_colsum(dy, dbias, cws, vitb_colsum_ws_bytes(M, N), M, N, dy_dt, stream);
    }
    return colsum_small_launch(dy, dbias, M, N, N, dy_dt, st);
  }
  return 0;
}

}  // extern "C"
