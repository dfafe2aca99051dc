// loss_adam.cu — fused label-smoothing cross-entropy (fwd+bwd in one pass) and flat-buffer Adam.
#include "common.cuh"

namespace vitb {

// ---------------------------------------------------------------------------------------------
// LS-CE: criterions.py:13-19.  One CTA, one thread per image (C is 10 or 100: a row is a few cache lines), rows r, r + 1024, ...;
// the batch mean is reduced in a fixed order (lane shuffles, then the 32 warp sums serially) -> bit-reproducible.
// ---------------------------------------------------------------------------------------------
// Two-target form (CutMix / MixUp, network.py:149-167): loss = lam * L(z, a) + (1 - lam) * L(z, b), i.e. the smoothed target
// distribution is q = lam * q_a + (1 - lam) * q_b.  labels_b == nullptr is the plain loss.  lam comes from device memory when
// lam_dev != nullptr (so a captured CUDA graph sees a new value every step).
// One block of 1024 threads (the loss is ONE number: a single block sums it in a fixed order without scratch memory).  A row is
// owned by a group of G lanes (G = 16 for C <= 16, else 32) that keeps its C <= 256 logits in registers: coalesced loads, one pass
// over memory, xor-tree reductions inside the group.  (Round 1's one-thread-per-row loop took 141 us at B = 1024, C = 100: three
// uncoalesced passes over the row per thread.)  C > 8 G falls back to the serial row loop.
constexpr int kLsMaxV = 8;  // logits per lane, at most

template <int G>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
template <int G>
__device__ __forceinline__ float group_max(float v) {
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// The per-row arithmetic every loss kernel shares (the training losses and vitb_eval_metrics): from a row's max mx, logit sum sz
// and sum_j exp(z_j - mx) se, lse = log sum_j exp(z_j) and the smoothed loss sum_j -q_j (z_j - lse) of target logit zy, with
// q_y = conf = 1 - s and q_j = off = s / (C - 1) elsewhere (criterions.py:13-19)
__device__ __forceinline__ float ls_ce_lse(float mx, float se) { return mx + logf(se); }
__device__ __forceinline__ float ls_ce_row_loss(float zy, float sz, float lse, int C, float conf, float off) {
  return -(conf * (zy - lse) + off * ((sz - zy) - (float)(C - 1) * lse));
}

// (eval_metrics_kernel walks each row's columns in the same per-lane order, j = lane + G i with i ascending, so that its per-image
// loss equals the one averaged here for C <= 256: a change of that order here must be made there too)
// kLsR rows per group and iteration, all their loads (logits, labels) issued before the first reduction: a row is a chain of
// load -> reduce -> exp -> reduce -> log -> gather z[y] of about two thousand cycles, and a group walks B / (1024 / G) rows
// (V = logits per lane, R = rows per iteration: 1024 threads leave 64 registers per thread)
template <int G, int kLsV, int kLsR>
__device__ __forceinline__ float ls_ce_rows(const float* __restrict__ logits, const int64_t* __restrict__ labels, const int64_t* __restrict__ labels_b,
                                            float lam, float* __restrict__ dlogits, int B, int C, int nv, float conf, float off, float gs) {
  // groups of the whole grid (one block in ls_ce_kernel, many in ls_ce_blocks_kernel)
  const int gl = threadIdx.x % G, gid = (int)blockIdx.x * (blockDim.x / G) + threadIdx.x / G, ngroups = (int)gridDim.x * (blockDim.x / G);
  float acc = 0.f;
  for (int base = 0; base < B; base += ngroups * kLsR) {  // (uniform trip count: the shuffles below need every lane of the warp)
    float v[kLsR][kLsV], mx[kLsR], sz[kLsR], se[kLsR];
    int y[kLsR], yb[kLsR];
    bool live[kLsR];
#pragma unroll
    for (int q = 0; q < kLsR; ++q) {
      const int r = base + q * ngroups + gid;
      live[q] = r < nv;
      mx[q] = -INFINITY;
      sz[q] = 0.f;
#pragma unroll
      for (int i = 0; i < kLsV; ++i) {
        const int j = gl + i * G;
        v[q][i] = (live[q] && j < C) ? logits[(size_t)r * C + j] : -INFINITY;
      }
      y[q] = live[q] ? (int)labels[r] : 0;
      yb[q] = (live[q] && labels_b != nullptr) ? (int)labels_b[r] : y[q];
    }
#pragma unroll
    for (int q = 0; q < kLsR; ++q) {
#pragma unroll
      for (int i = 0; i < kLsV; ++i)
        if (live[q] && gl + i * G < C) {
          mx[q] = fmaxf(mx[q], v[q][i]);
          sz[q] += v[q][i];
        }
    }
#pragma unroll
    for (int q = 0; q < kLsR; ++q) {
      mx[q] = group_max<G>(mx[q]);
      sz[q] = group_sum<G>(sz[q]);
    }
#pragma unroll
    for (int q = 0; q < kLsR; ++q) {
      se[q] = 0.f;
#pragma unroll
      for (int i = 0; i < kLsV; ++i)
        if (live[q] && gl + i * G < C) se[q] += expf(v[q][i] - mx[q]);
    }
#pragma unroll
    for (int q = 0; q < kLsR; ++q) se[q] = group_sum<G>(se[q]);
#pragma unroll
    for (int q = 0; q < kLsR; ++q) {
      const int r = base + q * ngroups + gid;
      if (r < B && !live[q] && dlogits != nullptr) {
        for (int j = gl; j < C; j += G) dlogits[(size_t)r * C + j] = 0.f;
      }
      if (!live[q]) continue;
      const float lse = ls_ce_lse(mx[q], se[q]);
      const float zy = logits[(size_t)r * C + y[q]], zb = logits[(size_t)r * C + yb[q]];
      // the loss for each target, then the lam mix (criterions.py:13-19 applied twice, network.py:163-165)
      const float la = ls_ce_row_loss(zy, sz[q], lse, C, conf, off);
      const float lb = ls_ce_row_loss(zb, sz[q], lse, C, conf, off);
      if (gl == 0) acc += lam * la + (1.0f - lam) * lb;
      if (dlogits != nullptr) {
#pragma unroll
        for (int i = 0; i < kLsV; ++i) {
          const int j = gl + i * G;
          if (j < C) {
            const float p = expf(v[q][i] - lse);
            const float t = lam * (j == y[q] ? conf : off) + (1.0f - lam) * (j == yb[q] ? conf : off);
            dlogits[(size_t)r * C + j] = (p - t) * gs;
          }
        }
      }
    }
  }
  return acc;
}

__global__ void __launch_bounds__(1024)
    ls_ce_kernel(const float* __restrict__ logits, const int64_t* __restrict__ labels, const int64_t* __restrict__ labels_b, float lam_host,
                 const float* __restrict__ lam_dev, const int* __restrict__ n_valid_dev, float* __restrict__ loss, float* __restrict__ dlogits, int B,
                 int C, float smoothing, float grad_scale) {
  pdl_trigger();
  pdl_wait();
  __shared__ float part[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const float off = smoothing / (float)(C - 1);
  const float conf = 1.0f - smoothing;
  // a partial last batch of an epoch in a fixed-size (graph-captured) step: only the first n_valid rows are images; the mean runs
  // over them (criterions.py:19 on a smaller batch) and the other rows get a zero gradient, which every downstream kernel
  // propagates as zero (images are independent through the whole network)
  const int nv = n_valid_dev != nullptr ? min(max(*n_valid_dev, 1), B) : B;
  const float gs = grad_scale / (float)nv;
  const float lam = labels_b == nullptr ? 1.0f : (lam_dev != nullptr ? *lam_dev : lam_host);
  float acc = 0.f;
  if (C <= 16) {
    acc = ls_ce_rows<16, 1, 4>(logits, labels, labels_b, lam, dlogits, B, C, nv, conf, off, gs);
  } else if (C <= 32 * 4) {
    acc = ls_ce_rows<32, 4, 4>(logits, labels, labels_b, lam, dlogits, B, C, nv, conf, off, gs);
  } else if (C <= 32 * kLsMaxV) {
    acc = ls_ce_rows<32, kLsMaxV, 2>(logits, labels, labels_b, lam, dlogits, B, C, nv, conf, off, gs);
  } else {
  for (int r = threadIdx.x; r < B; r += blockDim.x) {
    if (r >= nv) {
      if (dlogits != nullptr)
        for (int j = 0; j < C; ++j) dlogits[(size_t)r * C + j] = 0.f;
      continue;
    }
    const float* z = logits + (size_t)r * C;
    const int y = (int)labels[r];
    const int yb = labels_b != nullptr ? (int)labels_b[r] : y;
    float mx = -INFINITY, sz = 0.f;
    for (int j = 0; j < C; ++j) {
      const float v = z[j];
      mx = fmaxf(mx, v);
      sz += v;
    }
    float se = 0.f;
    for (int j = 0; j < C; ++j) se += expf(z[j] - mx);
    const float lse = ls_ce_lse(mx, se);
    const float zy = z[y], zb = z[yb];
    const float la = ls_ce_row_loss(zy, sz, lse, C, conf, off);
    const float lb = ls_ce_row_loss(zb, sz, lse, C, conf, off);
    acc += lam * la + (1.0f - lam) * lb;
    if (dlogits != nullptr) {
      float* d = dlogits + (size_t)r * C;
      for (int j = 0; j < C; ++j) {
        const float p = expf(z[j] - lse);
        const float q = lam * (j == y ? conf : off) + (1.0f - lam) * (j == yb ? conf : off);
        d[j] = (p - q) * gs;
      }
    }
  }
  }
  acc = warp_sum(acc);
  if (lane == 0) part[warp] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int w = 0; w < nwarps; ++w) s += part[w];
    *loss = s / (float)nv;
  }
}

// The same rows over MANY blocks (a 100-class loss at B = 1024 is 4 M instructions: 57 us on one SM): every block leaves the fixed-order
// sum of its rows in ws[1 + block], the last block to arrive (counter in ws[0], which atomicInc wraps back to zero) adds the partials in
// block order — deterministic, and no second launch.  C <= 256.
constexpr int kLsBlockThreads = 256;
constexpr int kLsMaxBlocks = 256;
__global__ void __launch_bounds__(kLsBlockThreads)
    ls_ce_blocks_kernel(const float* __restrict__ logits, const int64_t* __restrict__ labels, const int64_t* __restrict__ labels_b, float lam_host,
                        const float* __restrict__ lam_dev, const int* __restrict__ n_valid_dev, float* __restrict__ loss, float* __restrict__ dlogits,
                        int B, int C, float smoothing, float grad_scale, float* __restrict__ ws) {
  pdl_trigger();
  pdl_wait();
  __shared__ float part[kLsBlockThreads / 32];
  __shared__ bool last;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const float off = smoothing / (float)(C - 1);
  const float conf = 1.0f - smoothing;
  const int nv = n_valid_dev != nullptr ? min(max(*n_valid_dev, 1), B) : B;
  const float gs = grad_scale / (float)nv;
  const float lam = labels_b == nullptr ? 1.0f : (lam_dev != nullptr ? *lam_dev : lam_host);
  float acc;
  if (C <= 16) acc = ls_ce_rows<16, 1, 2>(logits, labels, labels_b, lam, dlogits, B, C, nv, conf, off, gs);
  else if (C <= 32 * 4) acc = ls_ce_rows<32, 4, 2>(logits, labels, labels_b, lam, dlogits, B, C, nv, conf, off, gs);
  else acc = ls_ce_rows<32, kLsMaxV, 2>(logits, labels, labels_b, lam, dlogits, B, C, nv, conf, off, gs);
  acc = warp_sum(acc);
  if (lane == 0) part[warp] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int w = 0; w < kLsBlockThreads / 32; ++w) s += part[w];
    volatile float* vp = ws + 1;
    vp[blockIdx.x] = s;
    __threadfence();
    const unsigned int done = atomicInc(reinterpret_cast<unsigned int*>(ws), gridDim.x - 1);  // wraps to 0 with the last arrival
    last = done == gridDim.x - 1;
    if (last) {
      __threadfence();
      float t = 0.f;
      for (unsigned int b = 0; b < gridDim.x; ++b) t += vp[b];
      *loss = t / (float)nv;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Validation metrics (network.py:388-395): per row the LS-CE loss above and argmax == label, summed over the batch into a
// [loss_sum, correct, count] record of doubles.  One warp per row, rows gwarp, gwarp + nwarps, ...; a lane walks the columns
// j = lane + 32 i in increasing i, so any C works, and for C <= 256 a row's max, sum and exp-sum come out bit for bit as in
// ls_ce_rows (same per-lane order; the xor tree over 32 lanes equals the 16-lane one when lanes 16..31 hold -inf / 0).
// Per-block partials in fp64, added in block order by the last block to arrive (counter in the first word of ws): deterministic.
// ---------------------------------------------------------------------------------------------
constexpr int kEvalThreads = 256;
constexpr int kEvalMaxBlocks = 256;

// torch.argmax order: NaN above everything, then larger values; equal values -> the smaller index
__device__ __forceinline__ bool argmax_before(float v, int j, float bv, int bj) {
  if (isnan(v) != isnan(bv)) return isnan(v);
  if (isnan(v) || v == bv) return j < bj;
  return v > bv;
}

__global__ void __launch_bounds__(kEvalThreads)
    eval_metrics_kernel(const float* __restrict__ logits, const int64_t* __restrict__ labels, const int* __restrict__ n_valid_dev,
                        int B, int C, float smoothing, double* __restrict__ totals, double* __restrict__ ws) {
  pdl_trigger();
  pdl_wait();
  __shared__ double part[kEvalThreads / 32][2];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const float off = smoothing / (float)(C - 1);
  const float conf = 1.0f - smoothing;
  const int nv = n_valid_dev != nullptr ? min(max(*n_valid_dev, 0), B) : B;
  const int nwarps = (int)gridDim.x * (kEvalThreads / 32);
  double loss_acc = 0.0, corr_acc = 0.0;  // (lane 0's)
  for (int r = (int)blockIdx.x * (kEvalThreads / 32) + warp; r < nv; r += nwarps) {
    const float* z = logits + (size_t)r * C;
    float mx = -INFINITY, sz = 0.f, bv = -INFINITY;
    int bj = C;
    for (int j = lane; j < C; j += 32) {
      const float v = z[j];
      mx = fmaxf(mx, v);
      sz += v;
      if (argmax_before(v, j, bv, bj)) { bv = v; bj = j; }
    }
    mx = group_max<32>(mx);
    sz = group_sum<32>(sz);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const int oj = __shfl_xor_sync(0xffffffffu, bj, o);
      if (argmax_before(ov, oj, bv, bj)) { bv = ov; bj = oj; }
    }
    float se = 0.f;
    for (int j = lane; j < C; j += 32) se += expf(z[j] - mx);
    se = group_sum<32>(se);
    if (lane == 0) {
      const int64_t y = labels[r];
      if (y >= 0 && y < C) {  // a label outside [0, C) is never dereferenced: the row is wrong and its loss NaN
        loss_acc += (double)ls_ce_row_loss(z[y], sz, ls_ce_lse(mx, se), C, conf, off);
        corr_acc += bj == (int)y ? 1.0 : 0.0;
      } else {
        loss_acc += (double)NAN;
      }
    }
  }
  if (lane == 0) {
    part[warp][0] = loss_acc;
    part[warp][1] = corr_acc;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double s0 = 0.0, s1 = 0.0;
    for (int w = 0; w < kEvalThreads / 32; ++w) {
      s0 += part[w][0];
      s1 += part[w][1];
    }
    volatile double* vp = ws + 1;
    vp[2 * blockIdx.x] = s0;
    vp[2 * blockIdx.x + 1] = s1;
    __threadfence();
    const unsigned int done = atomicInc(reinterpret_cast<unsigned int*>(ws), gridDim.x - 1);  // wraps to 0 with the last arrival
    if (done == gridDim.x - 1) {
      __threadfence();
      double t0 = 0.0, t1 = 0.0;
      for (unsigned int b = 0; b < gridDim.x; ++b) {
        t0 += vp[2 * b];
        t1 += vp[2 * b + 1];
      }
      totals[0] += t0;
      totals[1] += t1;
      totals[2] += (double)nv;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Adam (coupled L2), torch.optim.Adam single-tensor arithmetic, over one flat buffer
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
    adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                bf16* __restrict__ shadow, int64_t n, AdamHyper hv, const float* __restrict__ hyper_dev) {
  pdl_trigger();
  pdl_wait();
  AdamHyper h = hv;
  if (hyper_dev != nullptr) h = adam_hyper_from(hyper_dev);
  const int64_t n4 = n >> 2;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 pp = ld4(p + i * 4), gg = ld4(g + i * 4), mm = ld4(m + i * 4), vv = ld4(v + i * 4);
    adam_one(pp.x, gg.x, mm.x, vv.x, h);
    adam_one(pp.y, gg.y, mm.y, vv.y, h);
    adam_one(pp.z, gg.z, mm.z, vv.z, h);
    adam_one(pp.w, gg.w, mm.w, vv.w, h);
    st4(p + i * 4, pp);
    st4(m + i * 4, mm);
    st4(v + i * 4, vv);
    if (shadow != nullptr) st4(shadow + i * 4, pp);
  }
  if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
    const int64_t i = (n4 << 2) + threadIdx.x;
    float pp = p[i], mm = m[i], vv = v[i];
    adam_one(pp, g[i], mm, vv, h);
    p[i] = pp; m[i] = mm; v[i] = vv;
    if (shadow != nullptr) shadow[i] = __float2bfloat16_rn(pp);
  }
}

// SGD with momentum over one flat buffer (the reference's `--optimizer sgd`, network.py:78-84)
__global__ void __launch_bounds__(256)
    sgd_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ buf, bf16* __restrict__ shadow, int64_t n, AdamHyper hv,
               const float* __restrict__ hyper_dev) {
  pdl_trigger();
  pdl_wait();
  AdamHyper h = hv;
  if (hyper_dev != nullptr) h = adam_hyper_from(hyper_dev);
  const int64_t n4 = n >> 2;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 pp = ld4(p + i * 4), gg = ld4(g + i * 4), bb = ld4(buf + i * 4);
    sgd_one(pp.x, gg.x, bb.x, h);
    sgd_one(pp.y, gg.y, bb.y, h);
    sgd_one(pp.z, gg.z, bb.z, h);
    sgd_one(pp.w, gg.w, bb.w, h);
    st4(p + i * 4, pp);
    st4(buf + i * 4, bb);
    if (shadow != nullptr) st4(shadow + i * 4, pp);
  }
  if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
    const int64_t i = (n4 << 2) + threadIdx.x;
    float pp = p[i], bb = buf[i];
    sgd_one(pp, g[i], bb, h);
    p[i] = pp; buf[i] = bb;
    if (shadow != nullptr) shadow[i] = __float2bfloat16_rn(pp);
  }
}

}  // namespace vitb

using namespace vitb;

extern "C" {

int vitb_sgd_multi(float* p, const float* g, float* buf, void* w_shadow, int64_t n, const float* hyper_host, const float* hyper_dev, void* stream) {
  VITB_REQUIRE(p && g && buf, "sgd: null pointer");
  VITB_REQUIRE(hyper_host || hyper_dev, "sgd: need hyper_host or hyper_dev");
  VITB_REQUIRE(((uintptr_t)p | (uintptr_t)g | (uintptr_t)buf) % 16 == 0, "sgd: buffers must be 16-byte aligned");
  VITB_REQUIRE(w_shadow == nullptr || (uintptr_t)w_shadow % 8 == 0, "sgd: shadow must be 8-byte aligned");
  if (n == 0) return 0;
  AdamHyper h = {};
  if (hyper_host) h = adam_hyper_from(hyper_host);
  int blocks = (int)ceil_div64(n / 4 + 1, 256);
  if (blocks > 8 * kNumSMs) blocks = 8 * kNumSMs;
  VITB_LAUNCH((sgd_kernel), blocks, 256, 0, (cudaStream_t)stream, p, g, buf, (bf16*)w_shadow, n, h, hyper_dev);
  VITB_LAUNCH_OK();
  return 0;
}

int vitb_ls_ce_fwd_bwd(const float* logits, const int64_t* labels, float* loss, float* dlogits, int B, int C,
                       float smoothing, float grad_scale, void* stream) {
  return vitb_ls_ce_mix_fwd_bwd(logits, labels, nullptr, 1.0f, nullptr, loss, dlogits, B, C, smoothing, grad_scale, stream);
}

int vitb_ls_ce_mix_fwd_bwd(const float* logits, const int64_t* labels_a, const int64_t* labels_b, float lam, const float* lam_dev, float* loss,
                           float* dlogits, int B, int C, float smoothing, float grad_scale, void* stream) {
  return vitb_ls_ce_batch_fwd_bwd(logits, labels_a, labels_b, lam, lam_dev, nullptr, loss, dlogits, B, C, smoothing, grad_scale, stream);
}

int vitb_ls_ce_batch_fwd_bwd(const float* logits, const int64_t* labels_a, const int64_t* labels_b, float lam, const float* lam_dev,
                             const int* n_valid_dev, float* loss, float* dlogits, int B, int C, float smoothing, float grad_scale, void* stream) {
  VITB_REQUIRE(logits && labels_a && loss, "ls_ce: null pointer");
  VITB_REQUIRE(B > 0 && C > 1, "ls_ce: bad shape B=%d C=%d", B, C);
  VITB_REQUIRE(lam_dev != nullptr || (lam >= 0.0f && lam <= 1.0f), "ls_ce: lam=%f outside [0, 1]", lam);
  VITB_LAUNCH((ls_ce_kernel), 1, 1024, 0, (cudaStream_t)stream, logits, labels_a, labels_b, lam, lam_dev, n_valid_dev, loss, dlogits, B, C, smoothing, grad_scale);
  VITB_LAUNCH_OK();
  return 0;
}

size_t vitb_ls_ce_ws_bytes(void) { return (size_t)(1 + kLsMaxBlocks) * sizeof(float); }

int vitb_ls_ce_blocks_fwd_bwd(const float* logits, const int64_t* labels_a, const int64_t* labels_b, float lam, const float* lam_dev,
                              const int* n_valid_dev, float* loss, float* dlogits, int B, int C, float smoothing, float grad_scale, void* ws,
                              size_t ws_bytes, void* stream) {
  VITB_REQUIRE(logits && labels_a && loss, "ls_ce: null pointer");
  VITB_REQUIRE(B > 0 && C > 1, "ls_ce: bad shape B=%d C=%d", B, C);
  VITB_REQUIRE(lam_dev != nullptr || (lam >= 0.0f && lam <= 1.0f), "ls_ce: lam=%f outside [0, 1]", lam);
  if (ws == nullptr || C > 32 * kLsMaxV)  // no workspace / very wide rows: the single-block kernel
    return vitb_ls_ce_batch_fwd_bwd(logits, labels_a, labels_b, lam, lam_dev, n_valid_dev, loss, dlogits, B, C, smoothing, grad_scale, stream);
  VITB_REQUIRE(ws_bytes >= vitb_ls_ce_ws_bytes() && (uintptr_t)ws % 4 == 0, "ls_ce: workspace too small (%zu < %zu)", ws_bytes, vitb_ls_ce_ws_bytes());
  const int groups_per_block = kLsBlockThreads / (C <= 16 ? 16 : 32);
  int blocks = ceil_div(B, groups_per_block * 2);  // two rows per group and iteration
  if (blocks > kLsMaxBlocks) blocks = kLsMaxBlocks;
  VITB_LAUNCH((ls_ce_blocks_kernel), blocks, kLsBlockThreads, 0, (cudaStream_t)stream, logits, labels_a, labels_b, lam, lam_dev, n_valid_dev, loss, dlogits,
              B, C, smoothing, grad_scale, (float*)ws);
  VITB_LAUNCH_OK();
  return 0;
}

size_t vitb_eval_metrics_ws_bytes(void) { return (size_t)(1 + 2 * kEvalMaxBlocks) * sizeof(double); }

int vitb_eval_metrics(const float* logits, const int64_t* labels, const int* n_valid_dev, int B, int C, float smoothing, double* totals,
                      void* ws, size_t ws_bytes, void* stream) {
  VITB_REQUIRE(logits && labels && totals && ws, "eval_metrics: null pointer");
  VITB_REQUIRE(B > 0 && C > 1, "eval_metrics: bad shape B=%d C=%d", B, C);
  VITB_REQUIRE(ws_bytes >= vitb_eval_metrics_ws_bytes(), "eval_metrics: workspace too small (%zu < %zu)", ws_bytes, vitb_eval_metrics_ws_bytes());
  VITB_REQUIRE(((uintptr_t)ws | (uintptr_t)totals) % 8 == 0, "eval_metrics: ws and totals must be 8-byte aligned");
  int blocks = ceil_div(B, kEvalThreads / 32);
  if (blocks > kEvalMaxBlocks) blocks = kEvalMaxBlocks;
  VITB_LAUNCH((eval_metrics_kernel), blocks, kEvalThreads, 0, (cudaStream_t)stream, logits, labels, n_valid_dev, B, C, smoothing, totals, (double*)ws);
  VITB_LAUNCH_OK();
  return 0;
}

// the epoch record of a training step (network.py:206 logs each step's loss; Lightning averages it weighted by batch size):
// acc[0] += loss * n_valid, in fp64 (exact: a float times an integer below 2^24), with the loss kernels' clamp of n_valid
__global__ void loss_accumulate_kernel(const float* __restrict__ loss, const int* __restrict__ n_valid_dev, int B, double* __restrict__ acc) {
  pdl_trigger();
  pdl_wait();
  const int nv = n_valid_dev != nullptr ? min(max(*n_valid_dev, 1), B) : B;
  acc[0] += (double)loss[0] * (double)nv;
}

int vitb_train_loss_accumulate(const float* loss, const int* n_valid_dev, int B, double* acc, void* stream) {
  VITB_REQUIRE(loss && acc, "train_loss_accumulate: null pointer");
  VITB_REQUIRE(B > 0, "train_loss_accumulate: bad batch size B=%d", B);
  VITB_LAUNCH((loss_accumulate_kernel), 1, 1, 0, (cudaStream_t)stream, loss, n_valid_dev, B, acc);
  VITB_LAUNCH_OK();
  return 0;
}

int vitb_adam_multi(float* p, const float* g, float* m, float* v, void* w_shadow, int64_t n,
                    const float* hyper_host, const float* hyper_dev, void* stream) {
  VITB_REQUIRE(p && g && m && v, "adam: null pointer");
  VITB_REQUIRE(hyper_host || hyper_dev, "adam: need hyper_host or hyper_dev");
  VITB_REQUIRE(((uintptr_t)p | (uintptr_t)g | (uintptr_t)m | (uintptr_t)v) % 16 == 0, "adam: buffers must be 16-byte aligned");
  VITB_REQUIRE(w_shadow == nullptr || (uintptr_t)w_shadow % 8 == 0, "adam: shadow must be 8-byte aligned");
  if (n == 0) return 0;
  AdamHyper h = {};
  if (hyper_host) h = adam_hyper_from(hyper_host);
  int blocks = (int)ceil_div64(n / 4 + 1, 256);
  if (blocks > 8 * kNumSMs) blocks = 8 * kNumSMs;
  VITB_LAUNCH((adam_kernel), blocks, 256, 0, (cudaStream_t)stream, p, g, m, v, (bf16*)w_shadow, n, h, hyper_dev);
  VITB_LAUNCH_OK();
  return 0;
}

}  // extern "C"
