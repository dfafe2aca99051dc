// augment.cu — the reference's AutoAugment sub-policies (autoaugment.py: CIFAR10Policy / SVHNPolicy, applied by utils.get_transform
// between RandomHorizontalFlip and ToTensor) on the device, fused with RandomCrop + flip + ToTensor + Normalize.
//
// One CTA per image: stage the crop / flip into shared memory, run the image's sub-policy (up to two ops, each reading one byte buffer
// and writing the other), write (v / 255 - mean) / std to fp32 NCHW.  Every op reproduces the Pillow call the reference makes, pixel for
// pixel (tests/test_gpu_autoaugment.py compares with oracle/autoaugment_oracle.py, which calls Pillow):
//   LUT ops       invert, posterize, solarize; equalize and autocontrast from per-channel 256-bin histograms (ImageOps, integer / fp64)
//   enhance ops   Image.blend(degenerate, img, (float)factor): fp32 a + alpha * (b - a), truncated and clipped (Blend.c); degenerate =
//                 L (ITU-R 601-2 fixed point), the rounded mean of L, black, or the 3x3 SMOOTH filter with an unfiltered 1-pixel border
//   shear         bicubic affine transform (Geometry.c, generic path): fp64 coordinates, Pillow's cubic and its edge clamping
//   translate     nearest affine of a pure translation (Geometry.c ImagingScaleAffine): fp64 coordinates accumulated pixel by pixel
//   rotate        nearest affine (Geometry.c affine_fixed): 16.16 fixed-point coordinates, computed on the host like Image.rotate
// Out-of-image samples take the reference's fill colour (128, 128, 128).  Floating-point steps use the _rn intrinsics so that the
// compiler cannot contract them into FMAs Pillow does not perform.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"

namespace vitb {
namespace {

// op codes of the table (autoaugment.py / vit-cifar_b200/autoaugment.py OPS: the order of the reference's `ranges`)
enum AaOp {
  AA_SHEAR_X = 0, AA_SHEAR_Y, AA_TRANSLATE_X, AA_TRANSLATE_Y, AA_ROTATE, AA_COLOR, AA_POSTERIZE, AA_SOLARIZE, AA_CONTRAST, AA_SHARPNESS,
  AA_BRIGHTNESS, AA_AUTOCONTRAST, AA_EQUALIZE, AA_INVERT, AA_NUM_OPS
};

constexpr int kAaMaxSub = 32;
constexpr int kAaMaxS = 64;
constexpr int kAaThreads = 256;
constexpr int kAaFill = 128;

struct AaEntry {
  double mag;  // the reference's magnitude for this op and bin
  int op;
  int fx[6];   // rotate: Pillow's 16.16 fixed-point affine for this S (a0, a1, a2', a3, a4, a5'); unused otherwise
};
struct AaTable { AaEntry e[2 * kAaMaxSub]; };

__host__ __device__ inline int align16(int n) { return (n + 15) & ~15; }
inline size_t aa_smem_bytes(int S) { return 2 * (size_t)align16(3 * S * S) + 3 * 256 * sizeof(int) + 3 * 256 + 16; }

__device__ __forceinline__ uint8_t clip_trunc(float t) { return t <= 0.f ? 0 : t >= 255.f ? 255 : (uint8_t)__float2int_rz(t); }
__device__ __forceinline__ uint8_t clip_trunc(double t) { return t <= 0.0 ? 0 : t >= 255.0 ? 255 : (uint8_t)__double2int_rz(t); }

// Image.blend(deg, img, alpha) for one byte (Blend.c: both the interpolation and the extrapolation branch reduce to this)
__device__ __forceinline__ uint8_t blend(int deg, int v, float alpha) {
  return clip_trunc(__fadd_rn((float)deg, __fmul_rn(alpha, (float)(v - deg))));
}

// Pillow's cubic (Geometry.c BICUBIC): p1 + d * (p2 + d * (p3 + d * p4)), evaluated in this order in fp64
__device__ __forceinline__ double cubic(double v1, double v2, double v3, double v4, double d) {
  const double p2 = __dadd_rn(-v1, v3);
  const double p3 = __dsub_rn(__dadd_rn(__dmul_rn(2.0, __dsub_rn(v1, v2)), v3), v4);
  const double p4 = __dadd_rn(__dsub_rn(__dadd_rn(-v1, v2), v3), v4);
  return __dadd_rn(v2, __dmul_rn(d, __dadd_rn(p2, __dmul_rn(d, __dadd_rn(p3, __dmul_rn(d, p4))))));
}

// one output pixel of img.transform(size, AFFINE, a, BICUBIC, fillcolor) (Geometry.c: affine_transform + bicubic_filter32RGB)
__device__ void bicubic_pixel(const uint8_t* in, uint8_t* o, int S, int x, int y, double a0, double a1, double a3, double a4) {
  const double xc = x + 0.5, yc = y + 0.5;
  double xin = __dadd_rn(__dmul_rn(a0, xc), __dmul_rn(a1, yc));  // + a2 = 0
  double yin = __dadd_rn(__dmul_rn(a3, xc), __dmul_rn(a4, yc));  // + a5 = 0
  if (xin < 0.0 || xin >= S || yin < 0.0 || yin >= S) {
    o[0] = o[1] = o[2] = kAaFill;
    return;
  }
  xin = __dsub_rn(xin, 0.5);
  yin = __dsub_rn(yin, 0.5);
  int xi = (int)floor(xin), yi = (int)floor(yin);
  const double fx = __dsub_rn(xin, (double)xi), fy = __dsub_rn(yin, (double)yi);
  xi--; yi--;
  int xs[4];
  for (int k = 0; k < 4; ++k) xs[k] = min(max(xi + k, 0), S - 1);
  for (int c = 0; c < 3; ++c) {
    double v[4];
    const uint8_t* row = in + min(max(yi, 0), S - 1) * S * 3 + c;  // the first row is clamped, the others repeat their predecessor
    for (int k = 0; k < 4; ++k) {
      if (k > 0) {
        if (yi + k < 0 || yi + k >= S) { v[k] = v[k - 1]; continue; }
        row = in + (yi + k) * S * 3 + c;
      }
      // integer p2..p4 in Pillow's first pass are exact, so the fp64 cubic of the bytes gives the same value
      v[k] = cubic(row[xs[0] * 3], row[xs[1] * 3], row[xs[2] * 3], row[xs[3] * 3], fx);
    }
    o[c] = clip_trunc(cubic(v[0], v[1], v[2], v[3], fy));
  }
}

// Python's COORD(v) in Geometry.c
__device__ __forceinline__ int coord(double v) { return v < 0.0 ? -1 : (int)v; }

// ImageOps.equalize / autocontrast LUT of one channel, by one warp (lane l owns bins 8l .. 8l+7)
__device__ void build_lut(int op, const int* h, uint8_t* lut, int lane) {
  int hv[8], sum = 0, nz = 0, lo = 256, hi = -1;
  for (int j = 0; j < 8; ++j) {
    hv[j] = h[lane * 8 + j];
    sum += hv[j];
    if (hv[j]) { ++nz; lo = min(lo, lane * 8 + j); hi = lane * 8 + j; }
  }
  const unsigned full = 0xffffffffu;
  lo = __reduce_min_sync(full, lo);
  hi = __reduce_max_sync(full, hi);
  if (op == AA_AUTOCONTRAST) {
    if (hi <= lo) {
      for (int j = 0; j < 8; ++j) lut[lane * 8 + j] = (uint8_t)(lane * 8 + j);
      return;
    }
    const double scale = __ddiv_rn(255.0, (double)(hi - lo));
    const double offset = __dmul_rn((double)(-lo), scale);
    for (int j = 0; j < 8; ++j) lut[lane * 8 + j] = clip_trunc(__dadd_rn(__dmul_rn((double)(lane * 8 + j), scale), offset));
    return;
  }
  // equalize: step = (count - count of the last occupied bin) // 255; lut[i] = (step // 2 + pixels below i) // step
  const int total = __reduce_add_sync(full, sum);
  nz = __reduce_add_sync(full, nz);
  const int step = nz <= 1 ? 0 : (total - h[hi]) / 255;
  int incl = sum;
  for (int off = 1; off < 32; off <<= 1) {
    const int t = __shfl_up_sync(full, incl, off);
    if (lane >= off) incl += t;
  }
  if (step == 0) {
    for (int j = 0; j < 8; ++j) lut[lane * 8 + j] = (uint8_t)(lane * 8 + j);
    return;
  }
  int n = step / 2 + incl - sum;
  for (int j = 0; j < 8; ++j) {
    lut[lane * 8 + j] = (uint8_t)min(n / step, 255);  // Image.point clips the table to a byte
    n += hv[j];
  }
}

// One op of a sub-policy: in -> o (both S*S*3 HWC bytes in shared memory).  Called by the whole CTA (op is uniform).
__device__ void apply_op(const AaEntry& e, bool neg, const uint8_t* in, uint8_t* o, int S, int* hist, uint8_t* lut, int* red) {
  const int NP = S * S, tid = threadIdx.x;
  const double m = neg ? -e.mag : e.mag;  // the reference draws the sign inside the op: magnitude * random.choice([-1, 1])
  switch (e.op) {
    case AA_INVERT:
    case AA_POSTERIZE:
    case AA_SOLARIZE: {
      const int mask = e.op == AA_POSTERIZE ? ~((1 << (8 - (int)e.mag)) - 1) : 0xff;
      for (int i = tid; i < NP * 3; i += blockDim.x) {
        const int v = in[i];
        o[i] = (uint8_t)(e.op == AA_INVERT ? 255 - v : e.op == AA_POSTERIZE ? (v & mask) : ((double)v < e.mag ? v : 255 - v));
      }
      break;
    }
    case AA_EQUALIZE:
    case AA_AUTOCONTRAST: {
      for (int i = tid; i < 3 * 256; i += blockDim.x) hist[i] = 0;
      __syncthreads();
      for (int p = tid; p < NP; p += blockDim.x)
        for (int c = 0; c < 3; ++c) atomicAdd(&hist[c * 256 + in[p * 3 + c]], 1);
      __syncthreads();
      const int w = tid >> 5;
      if (w < 3) build_lut(e.op, hist + w * 256, lut + w * 256, tid & 31);
      __syncthreads();
      for (int i = tid; i < NP * 3; i += blockDim.x) o[i] = lut[(i % 3) * 256 + in[i]];
      break;
    }
    case AA_COLOR:
    case AA_CONTRAST:
    case AA_BRIGHTNESS:
    case AA_SHARPNESS: {
      const float alpha = __double2float_rn(__dadd_rn(1.0, m));  // ImageEnhance: blend(degenerate, img, 1 + magnitude * sign)
      int mean = 0;
      if (e.op == AA_CONTRAST) {  // solid gray at int(mean(L) + 0.5)
        if (tid == 0) red[0] = 0;
        __syncthreads();
        int s = 0;
        for (int p = tid; p < NP; p += blockDim.x)
          s += (in[p * 3] * 19595 + in[p * 3 + 1] * 38470 + in[p * 3 + 2] * 7471 + 0x8000) >> 16;
        s = __reduce_add_sync(0xffffffffu, s);
        if ((tid & 31) == 0) atomicAdd(red, s);
        __syncthreads();
        mean = (int)__dadd_rn(__ddiv_rn((double)red[0], (double)NP), 0.5);
      }
      const float k1 = __fdiv_rn(1.0f, 13.0f), k5 = __fdiv_rn(5.0f, 13.0f);  // SMOOTH, divided by its scale in fp32 (_imaging.c)
      for (int p = tid; p < NP; p += blockDim.x) {
        const uint8_t* v = in + p * 3;
        const int x = p % S, y = p / S;
        const int L = (v[0] * 19595 + v[1] * 38470 + v[2] * 7471 + 0x8000) >> 16;
        for (int c = 0; c < 3; ++c) {
          int deg = 0;
          if (e.op == AA_COLOR) deg = L;
          else if (e.op == AA_CONTRAST) deg = mean;
          else if (e.op == AA_SHARPNESS) {
            if (x == 0 || y == 0 || x == S - 1 || y == S - 1) {
              deg = v[c];
            } else {  // Filter.c ImagingFilter3x3: 0.5 + row y+1 + row y + row y-1, each (l * k + m * k) + r * k
              float ss = 0.5f;
              for (int dyr = 1; dyr >= -1; --dyr) {
                const uint8_t* r = in + ((y + dyr) * S + x) * 3 + c;
                const float kc = dyr == 0 ? k5 : k1;
                ss = __fadd_rn(ss, __fadd_rn(__fadd_rn(__fmul_rn((float)r[-3], k1), __fmul_rn((float)r[0], kc)), __fmul_rn((float)r[3], k1)));
              }
              deg = clip_trunc(ss);
            }
          }
          o[p * 3 + c] = blend(deg, v[c], alpha);
        }
      }
      break;
    }
    case AA_SHEAR_X:
    case AA_SHEAR_Y:
      for (int p = tid; p < NP; p += blockDim.x)
        bicubic_pixel(in, o + p * 3, S, p % S, p / S, 1.0, e.op == AA_SHEAR_X ? m : 0.0, e.op == AA_SHEAR_Y ? m : 0.0, 1.0);
      break;
    case AA_TRANSLATE_X:
    case AA_TRANSLATE_Y: {
      // ImagingScaleAffine with a = (1, 0, tx, 0, 1, ty): x0 = tx + 0.5, then += 1 per column (the same sums, in the same order)
      const double t = __dmul_rn(e.mag, (double)S);
      const double tx = e.op == AA_TRANSLATE_X ? (neg ? -t : t) : 0.0, ty = e.op == AA_TRANSLATE_Y ? (neg ? -t : t) : 0.0;
      for (int p = tid; p < NP; p += blockDim.x) {
        const int x = p % S, y = p / S;
        double xo = __dadd_rn(tx, 0.5), yo = __dadd_rn(ty, 0.5);
        for (int k = 0; k < x; ++k) xo = __dadd_rn(xo, 1.0);
        for (int k = 0; k < y; ++k) yo = __dadd_rn(yo, 1.0);
        const int xi = coord(xo), yi = coord(yo);
        const bool ok = xi >= 0 && xi < S && yi >= 0 && yi < S;
        for (int c = 0; c < 3; ++c) o[p * 3 + c] = ok ? in[(yi * S + xi) * 3 + c] : (uint8_t)kAaFill;
      }
      break;
    }
    case AA_ROTATE: {  // not signed in the reference: rotate_with_fill(img, magnitude)
      for (int p = tid; p < NP; p += blockDim.x) {
        const int x = p % S, y = p / S;
        const int xx = e.fx[2] + y * e.fx[1] + x * e.fx[0], yy = e.fx[5] + y * e.fx[4] + x * e.fx[3];
        const int xi = xx >> 16, yi = yy >> 16;
        const bool ok = xi >= 0 && xi < S && yi >= 0 && yi < S;
        for (int c = 0; c < 3; ++c) o[p * 3 + c] = ok ? in[(yi * S + xi) * 3 + c] : (uint8_t)kAaFill;
      }
      break;
    }
  }
}

__global__ void __launch_bounds__(kAaThreads)
    augment_autoaugment_kernel(const uint8_t* __restrict__ src, const int32_t* __restrict__ idx, int N, const int64_t* __restrict__ labels_src,
                               int64_t* __restrict__ labels_dst, const int32_t* __restrict__ dx, const int32_t* __restrict__ dy,
                               const uint8_t* __restrict__ flip, const int32_t* __restrict__ code, const __grid_constant__ AaTable tab, int n_sub,
                               float m0, float m1, float m2, float s0, float s1, float s2, float* __restrict__ out, int S, int pad) {
  extern __shared__ __align__(16) uint8_t smem[];
  const int NP = S * S, b = blockIdx.x, tid = threadIdx.x;
  uint8_t* cur = smem;
  uint8_t* nxt = smem + align16(3 * NP);
  int* hist = (int*)(smem + 2 * align16(3 * NP));
  uint8_t* lut = (uint8_t*)(hist + 3 * 256);
  int* red = (int*)(lut + 3 * 256);
  pdl_trigger();
  pdl_wait();

  // 0. the source row: image b of the batch, or row idx[b] of a resident N-image dataset (never read outside [0, N): NaN, label -1)
  const int row = idx ? idx[b] : b;
  const bool oob = idx != nullptr && (row < 0 || row >= N);
  if (idx && tid == 0) labels_dst[b] = oob ? -1 : labels_src[row];

  // 1. stage: RandomCrop + flip, with augment_kernel's index math (black outside the image)
  const int ox = dx ? dx[b] : pad, oy = dy ? dy[b] : pad;
  const bool fl = flip && flip[b];
  const uint8_t* img = src + (int64_t)(oob ? 0 : row) * NP * 3;
  for (int p = oob ? NP : tid; p < NP; p += blockDim.x) {
    const int x = p % S, y = p / S;
    const int sx = (fl ? S - 1 - x : x) + ox - pad, sy = y + oy - pad;
    const bool in = sx >= 0 && sx < S && sy >= 0 && sy < S;
    for (int c = 0; c < 3; ++c) cur[p * 3 + c] = in ? img[(sy * S + sx) * 3 + c] : 0;
  }
  __syncthreads();

  // 2. the sub-policy: code bits 0-7 index, 8/9 apply op 1/2, 10/11 negative sign of op 1/2
  const int cd = code[b], sub = cd & 0xff;
  const bool bad = oob || sub >= n_sub;  // cannot be reported to the host synchronously: the image is written as NaN instead
  if (!bad) {
    for (int k = 0; k < 2; ++k) {
      if (!((cd >> (8 + k)) & 1)) continue;
      apply_op(tab.e[2 * sub + k], (cd >> (10 + k)) & 1, cur, nxt, S, hist, lut, red);
      __syncthreads();
      uint8_t* t = cur; cur = nxt; nxt = t;
    }
  }

  // 3. ToTensor + Normalize, coalesced fp32 NCHW; the same arithmetic as augment_kernel
  float* o = out + (int64_t)b * 3 * NP;
  const float mc[3] = {m0, m1, m2}, sc[3] = {s0, s1, s2};
  for (int c = 0; c < 3; ++c)
    for (int p = tid; p < NP; p += blockDim.x)
      o[(int64_t)c * NP + p] = bad ? __int_as_float(0x7fffffff) : __fdiv_rn(__fsub_rn(__fmul_rn((float)cur[p * 3 + c], 1.0f / 255.0f), mc[c]), sc[c]);
}

// RandomCropPaste (the reference's da.RandomCropPaste, the last transform of get_transform with --rcpaste), in place on normalised
// fp32 (B, 3, S, S).  One CTA per image stages the whole image in shared memory (3 S^2 floats: 48 KB at S = kCpMaxS), because every
// output pixel reads two input pixels: the (flipped) base and, inside the paste box, the front pixel taken before the whole-image flip.
// params[b] = [fx1, fy1, fw, fh, x1, y1, flip_front, flip_img]; a[b] = the blend weight.  The reference blends with a float64 array,
// so torch computes in fp64: out = fp32(fp64(fp32(base * a)) + front * (1 - a)), written with _rn intrinsics so that nothing is
// contracted into an FMA.  Parameters that would read or write outside the image give a NaN image (no synchronous error exists).
constexpr int kCpMaxS = 64;
constexpr int kCpThreads = 256;

__global__ void __launch_bounds__(kCpThreads)
    random_crop_paste_kernel(float* __restrict__ img, const int32_t* __restrict__ params, const double* __restrict__ alpha, int S) {
  extern __shared__ float stage[];
  const int NP = S * S, b = blockIdx.x, tid = threadIdx.x;
  float* im = img + (int64_t)b * 3 * NP;
  pdl_trigger();
  pdl_wait();
  const int32_t* pr = params + b * 8;
  const int fx1 = pr[0], fy1 = pr[1], fw = pr[2], fh = pr[3], x1 = pr[4], y1 = pr[5];
  const bool flip_front = pr[6] != 0, flip_img = pr[7] != 0;
  const double a = alpha[b], na = __dsub_rn(1.0, a);
  const bool bad = fw < 0 || fh < 0 || fx1 < 0 || fy1 < 0 || x1 < 0 || y1 < 0 || fx1 > S - fw || fy1 > S - fh || x1 > S - fw || y1 > S - fh;
  if (bad) {
    for (int i = tid; i < 3 * NP; i += blockDim.x) im[i] = __int_as_float(0x7fffffff);
    return;
  }
  for (int i = tid; i < 3 * NP; i += blockDim.x) stage[i] = im[i];
  __syncthreads();
  for (int i = tid; i < 3 * NP; i += blockDim.x) {
    const int c = i / NP, y = (i % NP) / S, x = i % S;
    const float* ch = stage + c * NP;
    float v = ch[y * S + (flip_img ? S - 1 - x : x)];
    if (x >= x1 && x < x1 + fw && y >= y1 && y < y1 + fh) {
      const int u = flip_front ? fw - 1 - (x - x1) : x - x1;
      const float f = ch[(fy1 + y - y1) * S + fx1 + u];
      const double scaled = (double)__double2float_rn(__dmul_rn((double)v, a));
      v = __double2float_rn(__dadd_rn(scaled, __dmul_rn((double)f, na)));
    }
    im[i] = v;
  }
}

// Python's round(x, 15): the double nearest to x rounded to 15 decimals (both directions correctly rounded)
double round15(double x) {
  char buf[64];
  snprintf(buf, sizeof buf, "%.15f", x);
  return strtod(buf, nullptr);
}

// Image.rotate(deg) of an S x S image as Pillow's affine_fixed sees it: the matrix of Image.rotate (cos / sin rounded to 15 digits,
// centre (S/2, S/2)), then FIX(v) = floor(v * 65536 + 0.5) of a0, a1, a3, a4 and of the pixel-centre offsets a2', a5'
void rotate_fixed(double deg, int S, int fx[6]) {
  double angle = fmod(deg, 360.0);
  if (angle < 0) angle += 360.0;
  const double rad = -(angle * (M_PI / 180.0));
  const double c = S / 2.0;
  const double a = round15(cos(rad)), b = round15(sin(rad)), d = round15(-sin(rad)), e = round15(cos(rad));
  double a2 = a * -c;
  a2 = a2 + b * -c;
  a2 = a2 + 0.0;
  a2 = a2 + c;
  double a5 = d * -c;
  a5 = a5 + e * -c;
  a5 = a5 + 0.0;
  a5 = a5 + c;
  auto FIX = [](double v) { v = v * 65536.0 + 0.5; return v < 0.0 ? (int)floor(v) : (int)v; };
  double t2 = a2 + a * 0.5;
  t2 = t2 + b * 0.5;
  double t5 = a5 + d * 0.5;
  t5 = t5 + e * 0.5;
  fx[0] = FIX(a); fx[1] = FIX(b); fx[2] = FIX(t2); fx[3] = FIX(d); fx[4] = FIX(e); fx[5] = FIX(t5);
}

}  // namespace
}  // namespace vitb

using namespace vitb;

namespace {
int launch_autoaugment(const uint8_t* src, const int32_t* idx, int N, const int64_t* labels_src, int64_t* labels_dst, const int32_t* dx,
                       const int32_t* dy, const uint8_t* flip, const int32_t* code, const int32_t* op_ids, const double* mags, int n_sub,
                       const float* mean3, const float* std3, float* out, int B, int S, int pad, void* stream) {
  VITB_REQUIRE(B > 0 && S > 0 && S <= kAaMaxS && pad >= 0, "augment_autoaugment: bad shape B=%d S=%d pad=%d (S <= %d)", B, S, pad, kAaMaxS);
  VITB_REQUIRE(n_sub >= 1 && n_sub <= kAaMaxSub, "augment_autoaugment: n_sub=%d outside 1..%d", n_sub, kAaMaxSub);
  VITB_REQUIRE(std3[0] != 0.f && std3[1] != 0.f && std3[2] != 0.f, "augment_autoaugment: zero std");
  AaTable tab;
  memset(&tab, 0, sizeof tab);
  for (int i = 0; i < 2 * n_sub; ++i) {
    const int op = op_ids[i];
    const double m = mags[i];
    VITB_REQUIRE(op >= 0 && op < AA_NUM_OPS, "augment_autoaugment: unknown op code %d at table entry %d", op, i);
    VITB_REQUIRE(isfinite(m), "augment_autoaugment: magnitude of table entry %d is not finite", i);
    VITB_REQUIRE(op != AA_POSTERIZE || (m == floor(m) && m >= 0 && m <= 8), "augment_autoaugment: posterize bits %g outside 0..8", m);
    tab.e[i].op = op;
    tab.e[i].mag = m;
    if (op == AA_ROTATE) rotate_fixed(m, S, tab.e[i].fx);
  }
  VITB_LAUNCH((augment_autoaugment_kernel), B, kAaThreads, aa_smem_bytes(S), (cudaStream_t)stream, src, idx, N, labels_src, labels_dst, dx, dy, flip,
              code, tab, n_sub, mean3[0], mean3[1], mean3[2], std3[0], std3[1], std3[2], out, S, pad);
  VITB_LAUNCH_OK();
  return 0;
}
}  // namespace

int vitb_augment_autoaugment(const uint8_t* img_u8, const int32_t* dx, const int32_t* dy, const uint8_t* flip, const int32_t* code,
                             const int32_t* op_ids, const double* mags, int n_sub, const float* mean3, const float* std3, float* out, int B, int S,
                             int pad, void* stream) {
  VITB_REQUIRE(img_u8 && code && op_ids && mags && mean3 && std3 && out, "augment_autoaugment: null pointer");
  return launch_autoaugment(img_u8, nullptr, 0, nullptr, nullptr, dx, dy, flip, code, op_ids, mags, n_sub, mean3, std3, out, B, S, pad, stream);
}

int vitb_augment_autoaugment_gather(const uint8_t* data_u8, const int64_t* labels_src, int N, const int32_t* idx, const int32_t* dx,
                                    const int32_t* dy, const uint8_t* flip, const int32_t* code, const int32_t* op_ids, const double* mags, int n_sub,
                                    const float* mean3, const float* std3, float* out, int64_t* labels_dst, int B, int S, int pad, void* stream) {
  VITB_REQUIRE(data_u8 && labels_src && idx && labels_dst && code && op_ids && mags && mean3 && std3 && out,
               "augment_autoaugment_gather: null pointer");
  VITB_REQUIRE(N > 0, "augment_autoaugment_gather: empty dataset (N=%d)", N);
  return launch_autoaugment(data_u8, idx, N, labels_src, labels_dst, dx, dy, flip, code, op_ids, mags, n_sub, mean3, std3, out, B, S, pad, stream);
}

int vitb_random_crop_paste(float* img, const int32_t* params, const double* alpha, int B, int S, void* stream) {
  VITB_REQUIRE(img && params && alpha, "random_crop_paste: null pointer");
  VITB_REQUIRE(B > 0 && S > 0 && S <= kCpMaxS, "random_crop_paste: bad shape B=%d S=%d (S <= %d)", B, S, kCpMaxS);
  VITB_LAUNCH((random_crop_paste_kernel), B, kCpThreads, (size_t)3 * S * S * sizeof(float), (cudaStream_t)stream, img, params, alpha, S);
  VITB_LAUNCH_OK();
  return 0;
}
