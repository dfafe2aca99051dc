// elementwise.cu — HBM-bound kernels: LayerNorm fwd/bwd (+residual grad, +column sums), GELU backward
// with fused bias-gradient column sums, column sums, token pooling, fp32->bf16 shadow cast.
// All are one-pass, 8/16-byte vectorised, warp-shuffle reductions, fp32 math on bf16/fp32 storage.
#include <stdarg.h>

#include <stdlib.h>

#include <vector>

#include "common.cuh"

namespace vitb {

static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

bool pdl_enabled() {
  static const bool on = getenv("VITB_PDL") ? atoi(getenv("VITB_PDL")) != 0 : true;  // default on since round 2 (VITB_PDL=0 switches it off)
  return on;
}
static PersistWindow g_persist = {nullptr, 0, 1.0f};
const PersistWindow& persist_window() { return g_persist; }
void set_persist_window(void* base, size_t bytes, float hit_ratio) { g_persist = {base, bytes, hit_ratio}; }
static unsigned long long g_launches = 0;  // host-side, single launching thread per process
void count_launch() { ++g_launches; }

// ---- deferred reductions (common.cuh) ----
struct DeferState {
  char* arena = nullptr;
  size_t cap = 0, used = 0, high = 0;
  bool active = false;
  std::vector<ReduceJob> plain, tall;
};
static thread_local DeferState g_defer;
bool defer_active() { return g_defer.active; }
bool defer_owns(const void* p) { return g_defer.active && (const char*)p >= g_defer.arena && (const char*)p < g_defer.arena + g_defer.cap; }
void* defer_alloc(size_t bytes) {
  if (!g_defer.active) return nullptr;
  const size_t need = align_up(bytes, 256);
  g_defer.high += need;  // what a large enough arena would have held (vitb_defer_used)
  if (g_defer.used + need > g_defer.cap) return nullptr;
  void* p = g_defer.arena + g_defer.used;
  g_defer.used += need;
  return p;
}
void defer_add(const float* src, int nparts, int64_t cols, float* dst) {
  ReduceJob j = {src, dst, nparts, (int)cols};
  (finalize_is_tall(nparts, cols) ? g_defer.tall : g_defer.plain).push_back(j);
}

// the job that owns block `bid`: binary search over the first-block table (a linear scan over up to 120 entries cost more than
// the reduction itself when a step has hundreds of thousands of small blocks — the scaled ViT lost 1 ms per step to it)
__device__ __forceinline__ int find_job(const ReduceBatch& b, int bid) {
  int lo = 0, hi = b.njobs - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (bid >= b.block_start[mid]) lo = mid; else hi = mid - 1;
  }
  return lo;
}
// columns chunks (of 128) per block of the plain pass: few partials -> many chunks, so that a block always has ~12k floats to add
__host__ __device__ __forceinline__ int plain_chunks_per_block(int nparts) {
  const int c = 96 / (nparts > 0 ? nparts : 1);
  return c < 1 ? 1 : (c > 64 ? 64 : c);
}
// block (32, 8): the plain fixed-order pass of common.cuh, chunk by chunk, for the job that owns this block
__global__ void __launch_bounds__(256) reduce_jobs_plain_kernel(const ReduceBatch b) {
  pdl_trigger();
  pdl_wait();
  const int j = find_job(b, (int)blockIdx.x);
  const ReduceJob& job = b.jobs[j];
  const int nchunks = (job.cols + 127) / 128, per = plain_chunks_per_block(job.nparts);
  const int c0 = ((int)blockIdx.x - b.block_start[j]) * per;
  for (int c = c0; c < c0 + per && c < nchunks; ++c) {
    finalize_block_cols(job.src, job.nparts, job.cols, job.dst, c, nchunks);
    __syncthreads();  // the shared reduction buffer is reused by the next chunk
  }
}
// block (8, 64): the tall pass
__global__ void __launch_bounds__(512) reduce_jobs_tall_kernel(const ReduceBatch b) {
  pdl_trigger();
  pdl_wait();
  const int j = find_job(b, (int)blockIdx.x);
  const ReduceJob& job = b.jobs[j];
  finalize_tall_block(job.src, job.nparts, job.cols, job.dst, (int)blockIdx.x - b.block_start[j]);
}

static int flush_jobs(const std::vector<ReduceJob>& jobs, bool tall, cudaStream_t st) {
  for (size_t i0 = 0; i0 < jobs.size(); i0 += kMaxReduceJobs) {
    ReduceBatch b = {};
    const size_t n = jobs.size() - i0 < (size_t)kMaxReduceJobs ? jobs.size() - i0 : (size_t)kMaxReduceJobs;
    b.njobs = (int)n;
    int blocks = 0;
    for (size_t i = 0; i < n; ++i) {
      b.jobs[i] = jobs[i0 + i];
      b.block_start[i] = blocks;
      const int chunks = (b.jobs[i].cols + 127) / 128, per = plain_chunks_per_block(b.jobs[i].nparts);
      blocks += tall ? (b.jobs[i].cols + 31) / 32 : (chunks + per - 1) / per;
    }
    b.block_start[n] = blocks;
    if (tall) VITB_LAUNCH((reduce_jobs_tall_kernel), blocks, dim3(8, 64), 0, st, b);
    else VITB_LAUNCH((reduce_jobs_plain_kernel), blocks, dim3(32, 8), 0, st, b);
    VITB_LAUNCH_OK();
  }
  return 0;
}

// ---------------------------------------------------------------------------------------------
// cast
// ---------------------------------------------------------------------------------------------
__global__ void cast_f32_bf16_kernel(const float* __restrict__ src, bf16* __restrict__ dst, int64_t n) {
  pdl_trigger();
  pdl_wait();
  const int64_t n4 = n >> 2;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride)
    st4(dst + i * 4, ld4(src + i * 4));
  if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
    const int64_t i = (n4 << 2) + threadIdx.x;
    dst[i] = __float2bfloat16_rn(src[i]);
  }
}

// ---------------------------------------------------------------------------------------------
// LayerNorm forward: one warp per row, VEC float4-groups per lane (H = 128*VEC)
// ---------------------------------------------------------------------------------------------
// raw (storage-type) 4-element groups, so that the next row can be prefetched without converting it yet
template <typename T> struct Raw4;
template <> struct Raw4<float> { float4 v; };
template <> struct Raw4<bf16> { uint2 v; };
__device__ __forceinline__ Raw4<float> ldraw(const float* p) { Raw4<float> r; r.v = *reinterpret_cast<const float4*>(p); return r; }
__device__ __forceinline__ Raw4<bf16> ldraw(const bf16* p) { Raw4<bf16> r; r.v = *reinterpret_cast<const uint2*>(p); return r; }
__device__ __forceinline__ float4 cvt4(const Raw4<float>& r) { return r.v; }
__device__ __forceinline__ float4 cvt4(const Raw4<bf16>& r) {
  const float2 a = unpack_bf16x2(r.v.x), b = unpack_bf16x2(r.v.y);
  return make_float4(a.x, a.y, b.x, b.y);
}

// A warp takes kLnFwdRows consecutive rows and issues the loads of all of them before the first reduction: a row is only
// 768 bytes at H = 384 (24 bytes per lane), so one row per warp leaves too few bytes in flight per SM between block launches.
constexpr int kLnFwdRows = 4;
template <typename T, int VEC>
__global__ void __launch_bounds__(256, 4) ln_fwd_kernel(const T* __restrict__ x, int64_t xs,
                                                     const float* __restrict__ gamma,
                                                     const float* __restrict__ beta, T* __restrict__ y,
                                                     float* __restrict__ mean, float* __restrict__ rstd,
                                                     int rows, float eps) {
  pdl_trigger();
  pdl_wait();
  constexpr int H = VEC * 128;
  constexpr int R = kLnFwdRows;
  const int lane = threadIdx.x & 31;
  const int row0 = (blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * R;
  if (row0 >= rows) return;
  Raw4<T> raw[R][VEC];  // storage type until used: 4 rows of bf16 are 24 registers
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int row = min(row0 + r, rows - 1);  // rows past the end re-read the last row (never stored)
    const T* xr = x + (int64_t)row * xs;
#pragma unroll
    for (int i = 0; i < VEC; ++i) raw[r][i] = ldraw(xr + (i * 32 + lane) * 4);
  }
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int row = row0 + r;
    float4 v[VEC];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      v[i] = cvt4(raw[r][i]);
      s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    }
    const float mu = warp_sum(s) * (1.0f / H);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      const float a = v[i].x - mu, b = v[i].y - mu, c = v[i].z - mu, d = v[i].w - mu;
      q += (a * a + b * b) + (c * c + d * d);
    }
    const float rs = rsqrtf(warp_sum(q) * (1.0f / H) + eps);
    if (row < rows) {
      T* yr = y + (int64_t)row * H;
#pragma unroll
      for (int i = 0; i < VEC; ++i) {
        const float4 g = ld4(gamma + (i * 32 + lane) * 4), bt = ld4(beta + (i * 32 + lane) * 4);  // L1 hits after the first row
        float4 o;
        o.x = (v[i].x - mu) * rs * g.x + bt.x;
        o.y = (v[i].y - mu) * rs * g.y + bt.y;
        o.z = (v[i].z - mu) * rs * g.z + bt.z;
        o.w = (v[i].w - mu) * rs * g.w + bt.w;
        st4(yr + (i * 32 + lane) * 4, o);
      }
      if (lane == 0) {
        mean[row] = mu;
        rstd[row] = rs;
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// LayerNorm backward (+ residual gradient add, + dgamma/dbeta/colsum(dx) partials)
// grid-stride over rows, one warp per row; per-block partials -> ws[3][gridDim.x][H]
// ---------------------------------------------------------------------------------------------
constexpr int kLnBwdWarps = 8;


// value as it reads back from a tensor of type T
__device__ __forceinline__ float round_as(float v, const float*) { return v; }
__device__ __forceinline__ float round_as(float v, const bf16*) { return __bfloat162float(__float2bfloat16_rn(v)); }

// OUT2: a second output dx2 = dropout(dx) [* gelu'(z2)] with the column sums over dx2 instead of dx — the first kernel of the
// next backward stage folded into this one (vitb_layernorm_bwd_fused); dx2 is computed from dx AS STORED, so it equals what the
// stand-alone kernels (vitb_dropout / vitb_gelu_bwd_colsum_drop) produce from this kernel's dx bit for bit.
template <typename T, int VEC, bool HAS_RES, bool COLSUM, bool OUT2 = false>
__global__ void __launch_bounds__(kLnBwdWarps * 32, 2)  // grid = 2 x SMs must be one wave: keep <= 128 registers
    ln_bwd_kernel(const T* __restrict__ dy, const T* __restrict__ x, int64_t xs,
                  const float* __restrict__ gamma, const float* __restrict__ mean,
                  const float* __restrict__ rstd, const T* __restrict__ dres, T* __restrict__ dx,
                  int64_t dxs, float* __restrict__ ws, int rows, const T* __restrict__ z2 = nullptr, T* __restrict__ dx2 = nullptr,
                  DropParams dp = DropParams{}) {
  pdl_trigger();
  pdl_wait();
  constexpr int H = VEC * 128;
  const bool dropping = OUT2 && dp.thr != 0;
  const uint32_t dstep = dropping ? drop_step(dp) : 0u;
  __shared__ float red[kLnBwdWarps][H];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  float4 gam[VEC], dg[VEC], db[VEC], dc[VEC];
#pragma unroll
  for (int i = 0; i < VEC; ++i) {
    gam[i] = ld4(gamma + (i * 32 + lane) * 4);
    dg[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    db[i] = dg[i];
    dc[i] = dg[i];
  }
  const int stride = gridDim.x * kLnBwdWarps;
  int row = blockIdx.x * kLnBwdWarps + warp;
  Raw4<T> rx[VEC], rdy[VEC], rdr[VEC];
  float mu = 0.f, rs = 0.f;
  const bool has_z = OUT2 && z2 != nullptr;
  auto fetch = [&](int r) {
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      const int c = (i * 32 + lane) * 4;
      rx[i] = ldraw(x + (int64_t)r * xs + c);
      rdy[i] = ldraw(dy + (int64_t)r * H + c);
      if (HAS_RES) rdr[i] = ldraw(dres + (int64_t)r * H + c);
    }
    mu = mean[r];
    rs = rstd[r];
  };
  if (row < rows) fetch(row);
  while (row < rows) {
    // convert the current row, then immediately start the loads of the next one (software pipeline)
    float4 xh[VEC], d[VEC], res[VEC];
    const float cmu = mu, crs = rs;
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      xh[i] = cvt4(rx[i]);
      d[i] = cvt4(rdy[i]);
      if (HAS_RES) res[i] = cvt4(rdr[i]);
    }
    const int cur = row;
    row += stride;
    if (row < rows) fetch(row);

    float c1 = 0.f, c2 = 0.f;
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      xh[i].x = (xh[i].x - cmu) * crs;
      xh[i].y = (xh[i].y - cmu) * crs;
      xh[i].z = (xh[i].z - cmu) * crs;
      xh[i].w = (xh[i].w - cmu) * crs;
      // parameter gradients use dy, the input gradient uses g = dy * gamma
      dg[i].x += d[i].x * xh[i].x; dg[i].y += d[i].y * xh[i].y;
      dg[i].z += d[i].z * xh[i].z; dg[i].w += d[i].w * xh[i].w;
      db[i].x += d[i].x; db[i].y += d[i].y; db[i].z += d[i].z; db[i].w += d[i].w;
      d[i].x *= gam[i].x; d[i].y *= gam[i].y; d[i].z *= gam[i].z; d[i].w *= gam[i].w;
      c1 += (d[i].x + d[i].y) + (d[i].z + d[i].w);
      c2 += (d[i].x * xh[i].x + d[i].y * xh[i].y) + (d[i].z * xh[i].z + d[i].w * xh[i].w);
    }
    // z2 of the current row: issued before the reductions, whose shuffles cover part of the latency.  (Prefetching it one row
    // ahead with the other operands was measured slower: 6.21 vs 6.19 ms per step, 14 B of spills at the 128-register cap.)
    Raw4<T> rz[VEC];
    if (has_z) {
#pragma unroll
      for (int i = 0; i < VEC; ++i) rz[i] = ldraw(z2 + (int64_t)cur * H + (i * 32 + lane) * 4);
    }
    c1 = warp_sum(c1) * (1.0f / H);
    c2 = warp_sum(c2) * (1.0f / H);
    T* dxr = dx + (int64_t)cur * dxs;
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      const int c = (i * 32 + lane) * 4;
      float4 o;
      o.x = crs * (d[i].x - c1 - xh[i].x * c2);
      o.y = crs * (d[i].y - c1 - xh[i].y * c2);
      o.z = crs * (d[i].z - c1 - xh[i].z * c2);
      o.w = crs * (d[i].w - c1 - xh[i].w * c2);
      if (HAS_RES) { o.x += res[i].x; o.y += res[i].y; o.z += res[i].z; o.w += res[i].w; }
      st4(dxr + c, o);
      if (OUT2) {
        const T* tag = nullptr;
        float4 q = make_float4(round_as(o.x, tag), round_as(o.y, tag), round_as(o.z, tag), round_as(o.w, tag));
        if (dropping) drop_apply4(q, dp, dstep, (uint64_t)cur * H + c);
        if (has_z) {
          const float4 zz = cvt4(rz[i]);
          q.x *= gelu_grad_f(zz.x); q.y *= gelu_grad_f(zz.y); q.z *= gelu_grad_f(zz.z); q.w *= gelu_grad_f(zz.w);
        }
        st4(dx2 + (int64_t)cur * H + c, q);
        if (COLSUM) { dc[i].x += q.x; dc[i].y += q.y; dc[i].z += q.z; dc[i].w += q.w; }
      } else if (COLSUM) {
        dc[i].x += o.x; dc[i].y += o.y; dc[i].z += o.z; dc[i].w += o.w;
      }
    }
  }
  // block reduction of the partial vectors, one at a time through the same smem
  const int nparts = gridDim.x;
#pragma unroll 1
  for (int k = 0; k < (COLSUM ? 3 : 2); ++k) {
    __syncthreads();
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      const float4 v = k == 0 ? dg[i] : (k == 1 ? db[i] : dc[i]);
      *reinterpret_cast<float4*>(&red[warp][(i * 32 + lane) * 4]) = v;
    }
    __syncthreads();
    for (int c = threadIdx.x; c < H; c += blockDim.x) {
      float s = 0.f;
#pragma unroll
      for (int w = 0; w < kLnBwdWarps; ++w) s += red[w][c];
      ws[((size_t)k * nparts + blockIdx.x) * H + c] = s;
    }
  }
}

static int ln_bwd_blocks(int rows) {
  int b = ceil_div(rows, kLnBwdWarps);
  return b < 2 * kNumSMs ? (b < 1 ? 1 : b) : 2 * kNumSMs;
}

// ---------------------------------------------------------------------------------------------
// row-streaming kernels with per-column partial sums: GELU backward, plain column sums
// block = (TX column groups of 4) x (TY rows); grid = (row parts, column chunks)
// ---------------------------------------------------------------------------------------------
template <typename T, bool GELU_BWD>
__global__ void __launch_bounds__(256)
    rows_colsum_kernel(const T* __restrict__ a, const T* __restrict__ z, T* __restrict__ out,
                       float* __restrict__ ws, int rows, int cols, DropParams dp) {
  pdl_trigger();
  pdl_wait();
  const bool dropping = GELU_BWD && dp.thr != 0;  // dropout backward on the incoming gradient (GELU -> Dropout, layers.py:37-38)
  const uint32_t dstep = dropping ? drop_step(dp) : 0u;
  __shared__ float4 red[256];
  const int tx = threadIdx.x, ty = threadIdx.y, TX = blockDim.x, TY = blockDim.y;
  const int c = (blockIdx.y * TX + tx) * 4;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  const int step = gridDim.x * TY;
  int r = blockIdx.x * TY + ty;
  for (; r + step < rows; r += 2 * step) {  // two independent rows in flight per thread
    const size_t off0 = (size_t)r * cols + c, off1 = (size_t)(r + step) * cols + c;
    float4 v0 = ld4(a + off0), v1 = ld4(a + off1);
    if (GELU_BWD) {
      if (dropping) {
        drop_apply4(v0, dp, dstep, off0);
        drop_apply4(v1, dp, dstep, off1);
      }
      const float4 z0 = ld4(z + off0), z1 = ld4(z + off1);
      v0.x *= gelu_grad_f(z0.x); v0.y *= gelu_grad_f(z0.y); v0.z *= gelu_grad_f(z0.z); v0.w *= gelu_grad_f(z0.w);
      v1.x *= gelu_grad_f(z1.x); v1.y *= gelu_grad_f(z1.y); v1.z *= gelu_grad_f(z1.z); v1.w *= gelu_grad_f(z1.w);
      st4(out + off0, v0);
      st4(out + off1, v1);
    }
    acc.x += v0.x + v1.x; acc.y += v0.y + v1.y; acc.z += v0.z + v1.z; acc.w += v0.w + v1.w;
  }
  for (; r < rows; r += step) {
    const size_t off = (size_t)r * cols + c;
    float4 v = ld4(a + off);
    if (GELU_BWD) {
      if (dropping) drop_apply4(v, dp, dstep, off);
      const float4 zz = ld4(z + off);
      v.x *= gelu_grad_f(zz.x); v.y *= gelu_grad_f(zz.y); v.z *= gelu_grad_f(zz.z); v.w *= gelu_grad_f(zz.w);
      st4(out + off, v);
    }
    acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
  }
  if (ws == nullptr) return;
  red[ty * TX + tx] = acc;
  __syncthreads();
  if (ty == 0) {
    for (int j = 1; j < TY; ++j) {
      const float4 o = red[j * TX + tx];
      acc.x += o.x; acc.y += o.y; acc.z += o.z; acc.w += o.w;
    }
    *reinterpret_cast<float4*>(ws + (size_t)blockIdx.x * cols + c) = acc;
  }
}

// bf16 GELU backward, 16-byte accesses: a thread owns 8 consecutive columns of a few rows.  block = (cols / 8, TY), rows strided
// over the grid.
__device__ __forceinline__ void unpack8(const uint4& u, float (&f)[8]) {
  const float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y), c = unpack_bf16x2(u.z), d = unpack_bf16x2(u.w);
  f[0] = a.x; f[1] = a.y; f[2] = b.x; f[3] = b.y; f[4] = c.x; f[5] = c.y; f[6] = d.x; f[7] = d.y;
}
__global__ void __launch_bounds__(512)
    gelu_bwd_bf16x8_kernel(const bf16* __restrict__ a, const bf16* __restrict__ z, bf16* __restrict__ out, float* __restrict__ ws, int rows, int cols,
                           DropParams dp) {
  pdl_trigger();
  pdl_wait();
  const bool dropping = dp.thr != 0;
  const uint32_t dstep = dropping ? drop_step(dp) : 0u;
  extern __shared__ float red8[];  // [TY][cols]
  const int tx = threadIdx.x, ty = threadIdx.y, TY = blockDim.y;
  const int c = tx * 8;
  float acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i] = 0.f;
  const int step = gridDim.x * TY;
  auto one = [&](const uint4& av, const uint4& zv, size_t off) -> uint4 {
    float x[8], g[8];
    unpack8(av, x);
    unpack8(zv, g);
    if (dropping) drop_apply8(x, drop_words(dp, dstep, (uint64_t)off >> 3), dp.thr, dp.scale);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      x[i] *= gelu_grad_f(g[i]);
      acc[i] += x[i];
    }
    return make_uint4(pack_bf16x2(x[0], x[1]), pack_bf16x2(x[2], x[3]), pack_bf16x2(x[4], x[5]), pack_bf16x2(x[6], x[7]));
  };
  int r = blockIdx.x * TY + ty;
  for (; r + 3 * step < rows; r += 4 * step) {
    // all eight loads first, all four stores last: no store sits between the loads, so they issue back to back
    uint4 av[4], zv[4], ov[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const size_t off = (size_t)(r + k * step) * cols + c;
      av[k] = __ldg(reinterpret_cast<const uint4*>(a + off));
      zv[k] = __ldg(reinterpret_cast<const uint4*>(z + off));
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) ov[k] = one(av[k], zv[k], (size_t)(r + k * step) * cols + c);
#pragma unroll
    for (int k = 0; k < 4; ++k) *reinterpret_cast<uint4*>(out + (size_t)(r + k * step) * cols + c) = ov[k];
  }
  for (; r < rows; r += step) {
    const size_t off = (size_t)r * cols + c;
    *reinterpret_cast<uint4*>(out + off) = one(__ldg(reinterpret_cast<const uint4*>(a + off)), __ldg(reinterpret_cast<const uint4*>(z + off)), off);
  }
  if (ws == nullptr) return;
#pragma unroll
  for (int i = 0; i < 8; ++i) red8[ty * cols + c + i] = acc[i];
  __syncthreads();
  for (int j = ty * blockDim.x + tx; j < cols; j += blockDim.x * TY) {
    float sum = 0.f;
    for (int y = 0; y < TY; ++y) sum += red8[y * cols + j];
    ws[(size_t)blockIdx.x * cols + j] = sum;
  }
}
static bool gelu8_geom(int rows, int cols, int* ty, int* gx) {
  if (cols % 8 != 0 || cols / 8 > 128 || cols / 8 < 16) return false;
  const int tx = cols / 8;
  int y = 512 / tx;
  if (y > 8) y = 8;
  if (y < 1) return false;
  // ptxas sinks every load to its use, so the bytes in flight come from resident threads, not from per-thread unrolling: fill
  // the SMs (5 blocks of <= 512 threads each at 32 registers)
  int g = ceil_div(rows, y * 4);
  if (g > 5 * kNumSMs) g = 5 * kNumSMs;
  if (g < 1) g = 1;
  *ty = y;
  *gx = g;
  return true;
}

struct RowsGeom {
  int tx, ty, gx, gy;
};
static bool rows_geom(int rows, int cols, RowsGeom* g) {
  if (cols % 128 != 0) return false;
  const int cg = cols / 4;
  int tx = 32;
  for (int cand : {128, 96, 64, 32})
    if (cg % cand == 0) { tx = cand; break; }
  g->tx = tx;
  g->ty = 256 / tx;
  g->gy = cg / tx;
  int gx = ceil_div(rows, g->ty * 4);
  const int cap = (4 * kNumSMs + g->gy - 1) / g->gy;
  if (gx > cap) gx = cap;
  if (gx < 1) gx = 1;
  g->gx = gx;
  return true;
}

template <typename T>
static int launch_rows_colsum(bool gelu, const void* a, const void* z, void* out, float* colsum,
                              void* ws, size_t ws_bytes, int rows, int cols, cudaStream_t st, const DropParams& dp = DropParams{}) {
  RowsGeom g;
  VITB_REQUIRE(rows_geom(rows, cols, &g), "colsum: cols=%d must be a multiple of 128", cols);
  int ty8 = 0, gx8 = 0;
  if (gelu && sizeof(T) == 2 && gelu8_geom(rows, cols, &ty8, &gx8) && ((uintptr_t)a | (uintptr_t)z | (uintptr_t)out) % 16 == 0 &&
      (colsum == nullptr || (ws != nullptr && ws_bytes >= (size_t)gx8 * cols * sizeof(float)))) {
    float* w8 = colsum != nullptr ? (float*)ws : nullptr;
    VITB_LAUNCH((gelu_bwd_bf16x8_kernel), gx8, dim3(cols / 8, ty8), (size_t)ty8 * cols * sizeof(float), st, (const bf16*)a, (const bf16*)z, (bf16*)out, w8, rows, cols, dp);
    VITB_LAUNCH_OK();
    if (colsum != nullptr) VITB_CUDA_OK(::vitb::launch_finalize(w8, gx8, cols, colsum, nullptr, nullptr, 1, st));
    return 0;
  }
  float* wsf = nullptr;
  if (colsum != nullptr) {
    VITB_REQUIRE(ws != nullptr && ws_bytes >= (size_t)g.gx * cols * sizeof(float),
                 "colsum: workspace too small (%zu < %zu)", ws_bytes, (size_t)g.gx * cols * sizeof(float));
    wsf = (float*)ws;
  }
  dim3 grid(g.gx, g.gy), block(g.tx, g.ty);
  if (gelu)
    VITB_LAUNCH((rows_colsum_kernel<T, true>), grid, block, 0, st, (const T*)a, (const T*)z, (T*)out, wsf, rows, cols, dp);
  else
    VITB_LAUNCH((rows_colsum_kernel<T, false>), grid, block, 0, st, (const T*)a, nullptr, nullptr, wsf, rows, cols, DropParams{});
  VITB_LAUNCH_OK();
  if (colsum != nullptr) VITB_CUDA_OK(::vitb::launch_finalize(wsf, g.gx, cols, colsum, nullptr, nullptr, 1, st));
  return 0;
}

// ---------------------------------------------------------------------------------------------
// pooling (vit.py:72-75)
// ---------------------------------------------------------------------------------------------
template <typename T>
__global__ void pool_fwd_kernel(const T* __restrict__ x, T* __restrict__ y, int B, int Tn, int H, int mode) {
  pdl_trigger();
  pdl_wait();
  const int b = blockIdx.x;
  for (int c = threadIdx.x * 4; c < H; c += blockDim.x * 4) {
    float4 acc = ld4(x + ((size_t)b * Tn) * H + c);
    if (mode == 1) {
      for (int t = 1; t < Tn; ++t) {
        const float4 v = ld4(x + ((size_t)b * Tn + t) * H + c);
        acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
      }
      const float inv = 1.0f / Tn;
      acc.x *= inv; acc.y *= inv; acc.z *= inv; acc.w *= inv;
    }
    st4(y + (size_t)b * H + c, acc);
  }
}

template <typename T>
__global__ void pool_bwd_kernel(const T* __restrict__ dy, T* __restrict__ dx, int B, int Tn, int H, int mode) {
  pdl_trigger();
  pdl_wait();
  const size_t total4 = (size_t)B * Tn * H / 4;
  const float inv = 1.0f / Tn;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total4; i += (size_t)gridDim.x * blockDim.x) {
    const size_t e = i * 4;
    const int c = (int)(e % H);
    const size_t bt = e / H;
    const int t = (int)(bt % Tn);
    const size_t b = bt / Tn;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (mode == 1) {
      v = ld4(dy + b * H + c);
      v.x *= inv; v.y *= inv; v.z *= inv; v.w *= inv;
    } else if (t == 0) {
      v = ld4(dy + b * H + c);
    }
    st4(dx + e, v);
  }
}

// mode 2: only the cls rows (token 0) of dx are written; the other rows must already be zero (a static, pre-zeroed buffer)
template <typename T>
__global__ void pool_bwd_cls_rows_kernel(const T* __restrict__ dy, T* __restrict__ dx, int B, int Tn, int H) {
  pdl_trigger();
  pdl_wait();
  const int64_t total4 = (int64_t)B * H / 4;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total4; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t e = i * 4;
    const int c = (int)(e % H);
    const int64_t b = e / H;
    st4(dx + (b * Tn) * H + c, ld4(dy + b * H + c));
  }
}

// ---------------------------------------------------------------------------------------------
// training-time input pipeline on the device (utils.py:337-355): RandomCrop(S, padding) + RandomHorizontalFlip + ToTensor +
// Normalize as one gather from the raw uint8 HWC batch; the random draws (per-image offsets, flip flags) are inputs.
//   out[b, c, y, x] = (src(r, y + dy[b] - pad, xs + dx[b] - pad, c) / 255 - mean[c]) / std[c],  xs = flip[b] ? S-1-x : x,
//   src = 0 outside the image (torchvision pads the PIL image with black before ToTensor / Normalize)
// r = b for a contiguous batch; with idx (the DataLoader's batch assembly, utils.py:452-470) r = idx[b], a row of an N-image
// resident dataset, and labels_dst[b] = labels_src[r].  A row outside [0, N) is never read: its image is NaN and its label -1.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
    augment_kernel(const uint8_t* __restrict__ src, const int32_t* __restrict__ idx, int N, const int64_t* __restrict__ labels_src,
                   int64_t* __restrict__ labels_dst, const int32_t* __restrict__ dx, const int32_t* __restrict__ dy, const uint8_t* __restrict__ flip,
                   float m0, float m1, float m2, float s0, float s1, float s2, float* __restrict__ out, int B, int S, int pad) {
  pdl_trigger();
  pdl_wait();
  const int64_t stride = (int64_t)gridDim.x * blockDim.x, first = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx)
    for (int64_t b = first; b < B; b += stride) {
      const int r = idx[b];
      labels_dst[b] = (r >= 0 && r < N) ? labels_src[r] : -1;
    }
  const int64_t total = (int64_t)B * S * S;
  for (int64_t i = first; i < total; i += stride) {
    const int x = (int)(i % S), y = (int)((i / S) % S), b = (int)(i / ((int64_t)S * S));
    float* o = out + (int64_t)b * 3 * S * S + (int64_t)y * S + x;
    const int r = idx ? idx[b] : b;
    if (idx && (r < 0 || r >= N)) {
      o[0] = o[(int64_t)S * S] = o[(int64_t)2 * S * S] = __int_as_float(0x7fffffff);
      continue;
    }
    const int ox = dx ? dx[b] : pad, oy = dy ? dy[b] : pad;
    const int xs = (flip && flip[b]) ? S - 1 - x : x;  // flip acts on the cropped image
    const int sx = xs + ox - pad, sy = y + oy - pad;
    float rr = 0.f, g = 0.f, bl = 0.f;
    if (sx >= 0 && sx < S && sy >= 0 && sy < S) {
      const uint8_t* p = src + (((int64_t)r * S + sy) * S + sx) * 3;
      rr = (float)p[0] * (1.0f / 255.0f); g = (float)p[1] * (1.0f / 255.0f); bl = (float)p[2] * (1.0f / 255.0f);
    }
    o[0] = (rr - m0) / s0;
    o[(int64_t)S * S] = (g - m1) / s1;
    o[(int64_t)2 * S * S] = (bl - m2) / s2;
  }
}

// ---------------------------------------------------------------------------------------------
// batch-level CutMix / MixUp (da.py:51-93, applied at network.py:149-158) on fp32 (B, C, S, S) batches:
//   mode 0 (CutMix)  out[b, c, i, j] = img[perm[b], c, i, j] if x1 <= i < x2 and y1 <= j < y2 else img[b, c, i, j]
//                    (the reference indexes rows with its "x" and columns with its "y": img[:, :, x1:x2, y1:y2], da.py:68)
//   mode 1 (MixUp)   out = lam * img[b] + (1 - lam) * img[perm[b]]                                     (da.py:90)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
    batch_mix_kernel(const float* __restrict__ img, const int32_t* __restrict__ perm, float* __restrict__ out, int64_t per_image, int B, int S, int mode,
                     float lam, float oml, int x1, int x2, int y1, int y2) {
  pdl_trigger();
  pdl_wait();
  const int64_t total4 = (int64_t)B * per_image / 4;
  for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < total4; q += (int64_t)gridDim.x * blockDim.x) {
    const int64_t e = q * 4;
    const int b = (int)(e / per_image);
    const int64_t r = e - (int64_t)b * per_image;
    const float4 a = ld4(img + e);
    const float4 o = ld4(img + (int64_t)perm[b] * per_image + r);
    float4 v;
    if (mode == 1) {
      // two rounded products and a rounded sum, as torch evaluates lam * x + (1 - lam) * x[index] (no contraction)
      v = make_float4(__fadd_rn(__fmul_rn(lam, a.x), __fmul_rn(oml, o.x)), __fadd_rn(__fmul_rn(lam, a.y), __fmul_rn(oml, o.y)),
                      __fadd_rn(__fmul_rn(lam, a.z), __fmul_rn(oml, o.z)), __fadd_rn(__fmul_rn(lam, a.w), __fmul_rn(oml, o.w)));
    } else {
      const int pix = (int)(r % ((int64_t)S * S));
      const int i = pix / S, j = pix % S;  // S % 4 == 0: the four elements share the row
      const bool row_in = i >= x1 && i < x2;
      v.x = (row_in && j >= y1 && j < y2) ? o.x : a.x;
      v.y = (row_in && j + 1 >= y1 && j + 1 < y2) ? o.y : a.y;
      v.z = (row_in && j + 2 >= y1 && j + 2 < y2) ? o.z : a.z;
      v.w = (row_in && j + 3 >= y1 && j + 3 < y2) ? o.w : a.w;
    }
    st4(out + e, v);
  }
}

// ---------------------------------------------------------------------------------------------
// dropout (nn.Dropout at layers.py:35, 38, 102): out = x * keep / (1 - p) (+ residual)
//
// The keep mask (common.cuh: DropParams, philox4x32_10) is a pure function of (seed, site, step, element index); the backward
// pass calls the same function on the gradient with the same (seed, site, step) and regenerates it.
// ---------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
    dropout_kernel(const T* x, const T* residual, T* out, int64_t groups,  // no __restrict__: in-place (out == x) is allowed
                   uint32_t thr, float scale,
                   uint2 key, uint32_t site, uint32_t step, const uint32_t* __restrict__ step_dev) {
  pdl_trigger();
  pdl_wait();
  if (step_dev != nullptr) step = *step_dev;
  for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < groups; g += (int64_t)gridDim.x * blockDim.x) {
    const uint4 r = philox4x32_10(make_uint4((uint32_t)g, (uint32_t)((uint64_t)g >> 32), site, step), key);
    const uint32_t w[4] = {r.x, r.y, r.z, r.w};
    const int64_t e = g * 8;
    float4 v[2] = {ld4(x + e), ld4(x + e + 4)};
    float f[8] = {v[0].x, v[0].y, v[0].z, v[0].w, v[1].x, v[1].y, v[1].z, v[1].w};
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const uint32_t u = (w[j >> 1] >> (16 * (j & 1))) & 0xffffu;
      f[j] = u >= thr ? f[j] * scale : 0.f;
    }
    if (residual != nullptr) {
      const float4 a = ld4(residual + e), b = ld4(residual + e + 4);
      f[0] += a.x; f[1] += a.y; f[2] += a.z; f[3] += a.w; f[4] += b.x; f[5] += b.y; f[6] += b.z; f[7] += b.w;
    }
    st4(out + e, make_float4(f[0], f[1], f[2], f[3]));
    st4(out + e + 4, make_float4(f[4], f[5], f[6], f[7]));
  }
}

}  // namespace vitb

using namespace vitb;

// ---------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------
extern "C" {

int vitb_version(void) { return VITB_ABI_VERSION; }
const char* vitb_last_error(void) { return g_err; }
unsigned long long vitb_launch_count(void) { return g_launches; }

int vitb_device_supported(void) {
  int dev = 0, major = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 0;
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) return 0;
  return major == 10 ? 1 : 0;
}

int vitb_set_l2_persisting_window(void* base, size_t bytes, size_t carve_out_bytes) {
  if (base == nullptr || bytes == 0) {
    set_persist_window(nullptr, 0, 1.0f);
    return 0;
  }
  int dev = 0, max_window = 0, max_persist = 0;
  VITB_CUDA_OK(cudaGetDevice(&dev));
  VITB_CUDA_OK(cudaDeviceGetAttribute(&max_window, cudaDevAttrMaxAccessPolicyWindowSize, dev));
  VITB_CUDA_OK(cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, dev));
  VITB_REQUIRE(max_window > 0 && max_persist > 0, "l2 persistence: not supported by this device");
  if (carve_out_bytes > (size_t)max_persist) carve_out_bytes = (size_t)max_persist;
  if (bytes > (size_t)max_window) bytes = (size_t)max_window;
  VITB_CUDA_OK(cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, carve_out_bytes));
  // a window larger than the carve-out keeps a random carve_out / bytes share of its lines resident instead of thrashing
  const float ratio = bytes <= carve_out_bytes ? 1.0f : (float)((double)carve_out_bytes / (double)bytes);
  set_persist_window(base, bytes, ratio);
  return 0;
}

int vitb_cast_f32_to_bf16(const float* src, void* dst, int64_t n, void* stream) {
  VITB_REQUIRE(src && dst && n >= 0, "cast: null pointer");
  if (n == 0) return 0;
  VITB_REQUIRE(((uintptr_t)src % 16 == 0) && ((uintptr_t)dst % 8 == 0), "cast: buffers must be 16/8-byte aligned");
  int blocks = (int)ceil_div64(n / 4 + 1, 256);
  if (blocks > 8 * kNumSMs) blocks = 8 * kNumSMs;
  VITB_LAUNCH((cast_f32_bf16_kernel), blocks, 256, 0, (cudaStream_t)stream, src, (bf16*)dst, n);
  VITB_LAUNCH_OK();
  return 0;
}

#define VITB_DISPATCH_VEC(H, ...)                                                     \
  switch ((H) / 128) {                                                                \
    case 1: { constexpr int VEC = 1; __VA_ARGS__; } break;                            \
    case 2: { constexpr int VEC = 2; __VA_ARGS__; } break;                            \
    case 3: { constexpr int VEC = 3; __VA_ARGS__; } break;                            \
    case 4: { constexpr int VEC = 4; __VA_ARGS__; } break;                            \
    case 6: { constexpr int VEC = 6; __VA_ARGS__; } break;                            \
    case 8: { constexpr int VEC = 8; __VA_ARGS__; } break;                            \
    default: ::vitb::set_error("layernorm: H=%d unsupported (128*{1,2,3,4,6,8})", H); return -1; \
  }

int vitb_layernorm_fwd(const void* x, int64_t xs, const float* gamma, const float* beta, void* y,
                       float* mean, float* rstd, int rows, int H, float eps, int dt, void* stream) {
  VITB_REQUIRE(x && gamma && beta && y && mean && rstd, "layernorm_fwd: null pointer");
  VITB_REQUIRE(rows >= 0 && H % 128 == 0 && xs % 4 == 0, "layernorm_fwd: bad shape rows=%d H=%d stride=%lld", rows, H, (long long)xs);
  if (rows == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  const int blocks = ceil_div(rows, 8 * kLnFwdRows);
  if (dt == VITB_BF16) {
    VITB_DISPATCH_VEC(H, (VITB_LAUNCH((ln_fwd_kernel<bf16, VEC>), blocks, 256, 0, st, (const bf16*)x, xs, gamma, beta, (bf16*)y, mean, rstd, rows, eps)));
  } else {
    VITB_DISPATCH_VEC(H, (VITB_LAUNCH((ln_fwd_kernel<float, VEC>), blocks, 256, 0, st, (const float*)x, xs, gamma, beta, (float*)y, mean, rstd, rows, eps)));
  }
  VITB_LAUNCH_OK();
  return 0;
}

size_t vitb_layernorm_bwd_ws_bytes(int rows, int H) {
  return (size_t)3 * ln_bwd_blocks(rows) * H * sizeof(float);
}

int vitb_layernorm_bwd_fused(const void* dy, const void* x, int64_t xs, const float* gamma, const float* mean, const float* rstd,
                             const void* dres, void* dx, int64_t dxs, float* dgamma, float* dbeta, const void* z, void* dx2,
                             float* dx2_colsum, const vitb_dropout_t* drop, void* ws, size_t ws_bytes, int rows, int H, int dt,
                             void* stream) {
  VITB_REQUIRE(dy && x && gamma && mean && rstd && dres && dx && dgamma && dbeta && dx2 && dx2_colsum && ws, "layernorm_bwd_fused: null pointer");
  VITB_REQUIRE(rows > 0 && H % 128 == 0 && xs % 4 == 0 && dxs % 4 == 0, "layernorm_bwd_fused: bad shape");
  VITB_REQUIRE(ws_bytes >= vitb_layernorm_bwd_ws_bytes(rows, H), "layernorm_bwd_fused: workspace too small");
  VITB_REQUIRE(dx2 != dx && dx2 != dy && dx2 != dres, "layernorm_bwd_fused: dx2 must not alias another operand");
  DropParams dp;
  VITB_REQUIRE(make_drop_params(drop, &dp), "layernorm_bwd_fused: dropout p = %f outside [0, 1)", (double)drop->p);
  if (void* d = defer_alloc(vitb_layernorm_bwd_ws_bytes(rows, H))) ws = d;  // deferred second pass: the partials must outlive this call
  cudaStream_t st = (cudaStream_t)stream;
  const int blocks = ln_bwd_blocks(rows);
  if (dt == VITB_BF16) {
    VITB_DISPATCH_VEC(H, (VITB_LAUNCH((ln_bwd_kernel<bf16, VEC, true, true, true>), blocks, kLnBwdWarps * 32, 0, st, (const bf16*)dy, (const bf16*)x, xs,
                                      gamma, mean, rstd, (const bf16*)dres, (bf16*)dx, dxs, (float*)ws, rows, (const bf16*)z, (bf16*)dx2, dp)));
  } else {
    VITB_DISPATCH_VEC(H, (VITB_LAUNCH((ln_bwd_kernel<float, VEC, true, true, true>), blocks, kLnBwdWarps * 32, 0, st, (const float*)dy, (const float*)x,
                                      xs, gamma, mean, rstd, (const float*)dres, (float*)dx, dxs, (float*)ws, rows, (const float*)z, (float*)dx2, dp)));
  }
  VITB_LAUNCH_OK();
  VITB_CUDA_OK(::vitb::launch_finalize((const float*)ws, blocks, H, dgamma, dbeta, dx2_colsum, 3, st));
  return 0;
}

int vitb_layernorm_bwd(const void* dy, const void* x, int64_t xs, const float* gamma, const float* mean,
                       const float* rstd, const void* dres, void* dx, int64_t dxs, float* dgamma,
                       float* dbeta, float* dx_colsum, void* ws, size_t ws_bytes, int rows, int H, int dt,
                       void* stream) {
  VITB_REQUIRE(dy && x && gamma && mean && rstd && dx && dgamma && dbeta && ws, "layernorm_bwd: null pointer");
  VITB_REQUIRE(rows > 0 && H % 128 == 0 && xs % 4 == 0 && dxs % 4 == 0, "layernorm_bwd: bad shape");
  VITB_REQUIRE(ws_bytes >= vitb_layernorm_bwd_ws_bytes(rows, H), "layernorm_bwd: workspace too small");
  if (void* d = defer_alloc(vitb_layernorm_bwd_ws_bytes(rows, H))) ws = d;  // deferred second pass: the partials must outlive this call
  cudaStream_t st = (cudaStream_t)stream;
  const int blocks = ln_bwd_blocks(rows);
  const bool res = dres != nullptr, cs = dx_colsum != nullptr;
#define VITB_LN_BWD(T, RES, CS)                                                                                              \
  VITB_DISPATCH_VEC(H, (VITB_LAUNCH((ln_bwd_kernel<T, VEC, RES, CS>), blocks, kLnBwdWarps * 32, 0, st, (const T*)dy, (const T*)x, xs, gamma, mean, rstd, \
                                                                                         (const T*)dres, (T*)dx, dxs, (float*)ws, rows, nullptr, nullptr, DropParams{})))
  if (dt == VITB_BF16) {
    if (res && cs) { VITB_LN_BWD(bf16, true, true); } else if (res) { VITB_LN_BWD(bf16, true, false); }
    else if (cs) { VITB_LN_BWD(bf16, false, true); } else { VITB_LN_BWD(bf16, false, false); }
  } else {
    if (res && cs) { VITB_LN_BWD(float, true, true); } else if (res) { VITB_LN_BWD(float, true, false); }
    else if (cs) { VITB_LN_BWD(float, false, true); } else { VITB_LN_BWD(float, false, false); }
  }
#undef VITB_LN_BWD
  VITB_LAUNCH_OK();
  VITB_CUDA_OK(::vitb::launch_finalize((const float*)ws, blocks, H, dgamma, dbeta, dx_colsum, 3, st));
  return 0;
}

size_t vitb_colsum_ws_bytes(int rows, int cols) {
  RowsGeom g;
  if (!rows_geom(rows, cols, &g)) return 0;
  int ty8 = 0, gx8 = 0;
  if (!gelu8_geom(rows, cols, &ty8, &gx8)) gx8 = 0;
  return (size_t)(g.gx > gx8 ? g.gx : gx8) * cols * sizeof(float);
}

int vitb_gelu_bwd_colsum(const void* dy, const void* z, void* dz, float* colsum, void* ws, size_t ws_bytes,
                         int rows, int cols, int dt, void* stream) {
  return vitb_gelu_bwd_colsum_drop(dy, z, dz, colsum, ws, ws_bytes, rows, cols, dt, nullptr, stream);
}

int vitb_gelu_bwd_colsum_drop(const void* dy, const void* z, void* dz, float* colsum, void* ws, size_t ws_bytes, int rows, int cols,
                              int dt, const vitb_dropout_t* drop, void* stream) {
  VITB_REQUIRE(dy && z && dz && rows > 0, "gelu_bwd: null pointer / empty");
  DropParams dp;
  VITB_REQUIRE(make_drop_params(drop, &dp), "gelu_bwd: dropout p = %f outside [0, 1)", (double)drop->p);
  VITB_REQUIRE(dp.thr == 0 || cols % 8 == 0, "gelu_bwd: dropout needs cols %% 8 == 0");
  if (colsum != nullptr)
    if (void* d = defer_alloc(vitb_colsum_ws_bytes(rows, cols))) { ws = d; ws_bytes = vitb_colsum_ws_bytes(rows, cols); }
  if (dt == VITB_BF16) return launch_rows_colsum<bf16>(true, dy, z, dz, colsum, ws, ws_bytes, rows, cols, (cudaStream_t)stream, dp);
  return launch_rows_colsum<float>(true, dy, z, dz, colsum, ws, ws_bytes, rows, cols, (cudaStream_t)stream, dp);
}

int vitb_colsum(const void* x, float* colsum, void* ws, size_t ws_bytes, int rows, int cols, int dt, void* stream) {
  VITB_REQUIRE(x && colsum && rows > 0, "colsum: null pointer / empty");
  if (dt == VITB_BF16) return launch_rows_colsum<bf16>(false, x, nullptr, nullptr, colsum, ws, ws_bytes, rows, cols, (cudaStream_t)stream);
  return launch_rows_colsum<float>(false, x, nullptr, nullptr, colsum, ws, ws_bytes, rows, cols, (cudaStream_t)stream);
}

int vitb_defer_begin(void* arena, size_t arena_bytes) {
  VITB_REQUIRE(arena != nullptr && arena_bytes >= 256 && (uintptr_t)arena % 256 == 0, "defer_begin: need a 256-byte aligned device arena");
  // (a begin without a flush — an exception between the two on the host — simply starts over: nothing was launched for the dropped jobs)
  g_defer.arena = (char*)arena; g_defer.cap = arena_bytes; g_defer.used = 0; g_defer.high = 0; g_defer.active = true;
  g_defer.plain.clear(); g_defer.tall.clear();
  return 0;
}

int vitb_defer_flush(void* stream) {
  VITB_REQUIRE(g_defer.active, "defer_flush: vitb_defer_begin has not been called");
  g_defer.active = false;
  int rc = flush_jobs(g_defer.plain, false, (cudaStream_t)stream);
  if (rc == 0) rc = flush_jobs(g_defer.tall, true, (cudaStream_t)stream);
  g_defer.plain.clear(); g_defer.tall.clear();
  return rc;
}

int vitb_defer_flush_partial(void* stream) {
  VITB_REQUIRE(g_defer.active, "defer_flush_partial: vitb_defer_begin has not been called");
  int rc = flush_jobs(g_defer.plain, false, (cudaStream_t)stream);
  if (rc == 0) rc = flush_jobs(g_defer.tall, true, (cudaStream_t)stream);
  g_defer.plain.clear(); g_defer.tall.clear();  // the window stays open; the arena keeps growing
  return rc;
}

size_t vitb_defer_used(void) { return g_defer.high; }

int vitb_augment_crop_flip_normalize(const uint8_t* img_u8, const int32_t* dx, const int32_t* dy, const uint8_t* flip, const float* mean3,
                                     const float* std3, float* out, int B, int S, int pad, void* stream) {
  VITB_REQUIRE(img_u8 && out && mean3 && std3, "augment: null pointer");
  VITB_REQUIRE(B > 0 && S > 0 && pad >= 0, "augment: bad shape B=%d S=%d pad=%d", B, S, pad);
  VITB_REQUIRE(std3[0] != 0.f && std3[1] != 0.f && std3[2] != 0.f, "augment: zero std");
  const int64_t total = (int64_t)B * S * S;
  int blocks = (int)ceil_div64(total, 256);
  if (blocks > 16 * kNumSMs) blocks = 16 * kNumSMs;
  VITB_LAUNCH((augment_kernel), blocks, 256, 0, (cudaStream_t)stream, img_u8, (const int32_t*)nullptr, 0, (const int64_t*)nullptr, (int64_t*)nullptr,
              dx, dy, flip, mean3[0], mean3[1], mean3[2], std3[0], std3[1], std3[2], out, B, S, pad);
  VITB_LAUNCH_OK();
  return 0;
}

int vitb_augment_crop_flip_normalize_gather(const uint8_t* data_u8, const int64_t* labels_src, int N, const int32_t* idx, const int32_t* dx,
                                            const int32_t* dy, const uint8_t* flip, const float* mean3, const float* std3, float* out,
                                            int64_t* labels_dst, int B, int S, int pad, void* stream) {
  VITB_REQUIRE(data_u8 && labels_src && idx && out && labels_dst && mean3 && std3, "augment_gather: null pointer");
  VITB_REQUIRE(N > 0 && B > 0 && S > 0 && pad >= 0, "augment_gather: bad shape N=%d B=%d S=%d pad=%d", N, B, S, pad);
  VITB_REQUIRE(std3[0] != 0.f && std3[1] != 0.f && std3[2] != 0.f, "augment_gather: zero std");
  const int64_t total = (int64_t)B * S * S;
  int blocks = (int)ceil_div64(total, 256);
  if (blocks > 16 * kNumSMs) blocks = 16 * kNumSMs;
  VITB_LAUNCH((augment_kernel), blocks, 256, 0, (cudaStream_t)stream, data_u8, idx, N, labels_src, labels_dst, dx, dy, flip, mean3[0], mean3[1],
              mean3[2], std3[0], std3[1], std3[2], out, B, S, pad);
  VITB_LAUNCH_OK();
  return 0;
}

int vitb_batch_mix(const float* img, const int32_t* perm, float* out, int B, int C, int S, int mode, double lam, int x1, int x2, int y1, int y2,
                   void* stream) {
  VITB_REQUIRE(img && perm && out && img != out, "batch_mix: null pointer, or out aliases img (every image is read by two outputs)");
  VITB_REQUIRE(B > 0 && C > 0 && S > 0 && S % 4 == 0, "batch_mix: bad shape B=%d C=%d S=%d (S must be a multiple of 4)", B, C, S);
  VITB_REQUIRE(mode == 0 || mode == 1, "batch_mix: mode %d (0 = CutMix, 1 = MixUp)", mode);
  VITB_REQUIRE(mode == 1 || (0 <= x1 && x1 <= x2 && x2 <= S && 0 <= y1 && y1 <= y2 && y2 <= S), "batch_mix: box [%d,%d) x [%d,%d) outside the image", x1, x2,
               y1, y2);
  const int64_t per_image = (int64_t)C * S * S;
  int blocks = (int)ceil_div64((int64_t)B * per_image / 4, 256);
  if (blocks > 16 * kNumSMs) blocks = 16 * kNumSMs;
  VITB_LAUNCH((batch_mix_kernel), blocks, 256, 0, (cudaStream_t)stream, img, perm, out, per_image, B, S, mode, (float)lam, (float)(1.0 - lam), x1, x2,
              y1, y2);
  VITB_LAUNCH_OK();
  return 0;
}

uint32_t vitb_dropout_threshold(float p) {
  const double t = (double)p * 65536.0 + 0.5;
  return t <= 0.0 ? 0u : (t >= 65535.0 ? 65535u : (uint32_t)t);
}

int vitb_dropout(const void* x, const void* residual, void* out, int64_t n, float p, uint64_t seed, uint32_t site, uint32_t step,
                 const uint32_t* step_dev, int dt, void* stream) {
  VITB_REQUIRE(x && out && n > 0, "dropout: null pointer / empty");
  VITB_REQUIRE(n % 8 == 0, "dropout: the element count (%lld) must be a multiple of 8", (long long)n);
  VITB_REQUIRE(p >= 0.f && p < 1.f, "dropout: p = %f outside [0, 1)", (double)p);
  const int64_t groups = n / 8;
  const int blocks = (int)(ceil_div64(groups, 256) < 16 * (int64_t)kNumSMs ? ceil_div64(groups, 256) : 16 * (int64_t)kNumSMs);
  const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
  const float scale = 1.0f / (1.0f - p);
  const uint32_t thr = vitb_dropout_threshold(p);
  if (dt == VITB_BF16)
    VITB_LAUNCH((dropout_kernel<bf16>), blocks, 256, 0, (cudaStream_t)stream, (const bf16*)x, (const bf16*)residual, (bf16*)out, groups, thr, scale, key, site,
                step, step_dev);
  else
    VITB_LAUNCH((dropout_kernel<float>), blocks, 256, 0, (cudaStream_t)stream, (const float*)x, (const float*)residual, (float*)out, groups, thr, scale, key,
                site, step, step_dev);
  VITB_LAUNCH_OK();
  return 0;
}

int vitb_pool_fwd(const void* x, void* y, int B, int T, int H, int mode, int dt, void* stream) {
  VITB_REQUIRE(x && y && B > 0 && T > 0 && H % 4 == 0 && (mode == 0 || mode == 1), "pool_fwd: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  if (dt == VITB_BF16) VITB_LAUNCH((pool_fwd_kernel<bf16>), B, 128, 0, st, (const bf16*)x, (bf16*)y, B, T, H, mode);
  else VITB_LAUNCH((pool_fwd_kernel<float>), B, 128, 0, st, (const float*)x, (float*)y, B, T, H, mode);
  VITB_LAUNCH_OK();
  return 0;
}

int vitb_pool_bwd(const void* dy, void* dx, int B, int T, int H, int mode, int dt, void* stream) {
  VITB_REQUIRE(dy && dx && B > 0 && T > 0 && H % 4 == 0 && (mode == 0 || mode == 1 || mode == 2), "pool_bwd: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  if (mode == 2) {  // cls rows only, the rest of dx is already zero
    const int nb = (int)ceil_div64((int64_t)B * H / 4, 256);
    if (dt == VITB_BF16) VITB_LAUNCH((pool_bwd_cls_rows_kernel<bf16>), nb, 256, 0, st, (const bf16*)dy, (bf16*)dx, B, T, H);
    else VITB_LAUNCH((pool_bwd_cls_rows_kernel<float>), nb, 256, 0, st, (const float*)dy, (float*)dx, B, T, H);
    VITB_LAUNCH_OK();
    return 0;
  }
  int blocks = (int)ceil_div64((int64_t)B * T * H / 4, 256);
  if (blocks > 8 * kNumSMs) blocks = 8 * kNumSMs;
  if (dt == VITB_BF16) VITB_LAUNCH((pool_bwd_kernel<bf16>), blocks, 256, 0, st, (const bf16*)dy, (bf16*)dx, B, T, H, mode);
  else VITB_LAUNCH((pool_bwd_kernel<float>), blocks, 256, 0, st, (const float*)dy, (float*)dx, B, T, H, mode);
  VITB_LAUNCH_OK();
  return 0;
}

}  // extern "C"
