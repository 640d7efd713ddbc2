// HBM-bound kernels of the frame-FID InceptionV3 (cpcsv_b200/frame_fid.py): the stem's resize + im2col and
// the 3x3 max / average pooling.  Both are channel-vectorised like elementwise.cu, never allocate and only
// enqueue on the caller's stream.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.h"

namespace cpcsv {

__device__ __forceinline__ void split16_fid(float v, int dtype, uint16_t& hi, uint16_t& lo) {
  if (dtype == 1) {
    __nv_bfloat16 h = __float2bfloat16_rn(v);
    hi = __bfloat16_as_ushort(h);
    lo = __bfloat16_as_ushort(__float2bfloat16_rn(v - __bfloat162float(h)));
  } else {
    __half h = __float2half_rn(v);
    hi = __half_as_ushort(h);
    lo = __half_as_ushort(__float2half_rn(v - __half2float(h)));
  }
}

static inline int blocks_for(int64_t work, int threads) {
  int64_t b = ceil_div(work, threads);
  const int64_t cap = static_cast<int64_t>(num_sms()) * 16;
  if (b > cap) b = cap;
  return static_cast<int>(b < 1 ? 1 : b);
}

// ------------------------------------------------------------------------- resize + im2col
// source coordinate of output index d for align_corners=False, as PyTorch's upsample_bilinear2d
// (area_pixel_compute_source_index with the float scale in / out, clamped at 0)
__device__ __forceinline__ void bilinear_index(int d, float scale, int in, int& i0, int& i1, float& l1) {
  float r = scale * (static_cast<float>(d) + 0.5f) - 0.5f;
  r = r < 0.f ? 0.f : r;
  i0 = static_cast<int>(r);
  i1 = i0 < in - 1 ? i0 + 1 : i0;
  l1 = r - static_cast<float>(i0);
}

// one thread: 8 consecutive columns of one im2col row (16-B stores of hi and lo)
__global__ void resize_im2col_kernel(const float* __restrict__ x, int N, int H, int W, int64_t sn, int64_t sc,
                                     int64_t sh, int64_t sw, int S, int OH, float scale_h, float scale_w, float a,
                                     float b, uint16_t* __restrict__ hi, uint16_t* __restrict__ lo, int ldp,
                                     int dtype) {
  const int groups = ldp / 8;
  const int64_t total = static_cast<int64_t>(N) * OH * OH * groups;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int g = static_cast<int>(i % groups);
    const int64_t row = i / groups;
    const int ow = static_cast<int>(row % OH);
    const int oh = static_cast<int>((row / OH) % OH);
    const int n = static_cast<int>(row / (static_cast<int64_t>(OH) * OH));
    const float* xn = x + n * sn;
    uint16_t hv[8], lv[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int j = g * 8 + e;
      float v = 0.f;
      if (j < 27) {
        const int tap = j / 3, c = j - tap * 3;
        const int ky = tap / 3, kx = tap - ky * 3;
        int y0, y1, x0, x1;
        float ly, lx;
        bilinear_index(2 * oh + ky, scale_h, H, y0, y1, ly);
        bilinear_index(2 * ow + kx, scale_w, W, x0, x1, lx);
        const float* p = xn + c * sc;
        const float top = (1.f - lx) * p[y0 * sh + x0 * sw] + lx * p[y0 * sh + x1 * sw];
        const float bot = (1.f - lx) * p[y1 * sh + x0 * sw] + lx * p[y1 * sh + x1 * sw];
        v = a * ((1.f - ly) * top + ly * bot) + b;
      }
      split16_fid(v, dtype, hv[e], lv[e]);
    }
    uint4 h4, l4;
    h4.x = hv[0] | (static_cast<uint32_t>(hv[1]) << 16);
    h4.y = hv[2] | (static_cast<uint32_t>(hv[3]) << 16);
    h4.z = hv[4] | (static_cast<uint32_t>(hv[5]) << 16);
    h4.w = hv[6] | (static_cast<uint32_t>(hv[7]) << 16);
    reinterpret_cast<uint4*>(hi + row * ldp)[g] = h4;
    if (lo) {
      l4.x = lv[0] | (static_cast<uint32_t>(lv[1]) << 16);
      l4.y = lv[2] | (static_cast<uint32_t>(lv[3]) << 16);
      l4.z = lv[4] | (static_cast<uint32_t>(lv[5]) << 16);
      l4.w = lv[6] | (static_cast<uint32_t>(lv[7]) << 16);
      reinterpret_cast<uint4*>(lo + row * ldp)[g] = l4;
    }
  }
}

// ------------------------------------------------------------------------- 3x3 pooling
// one thread: 4 channels of one output pixel.  mode 0: max, 1: average over the window taps inside the input
// (count_include_pad=False).  stride 1 pad 1 (Ho = H) or stride 2 pad 0 (Ho = (H - 3) / 2 + 1).
__global__ void pool3x3_kernel(const float* __restrict__ x, int N, int H, int W, int C, int64_t sn, int64_t sh,
                               int64_t sw, int mode, int stride, int Ho, int Wo, float* __restrict__ y,
                               int64_t ysn, int64_t ysh, int64_t ysw, uint16_t* __restrict__ hi,
                               uint16_t* __restrict__ lo, int64_t psn, int64_t psh, int64_t psw, int dtype) {
  const int cq = C / 4;
  const int pad = stride == 1 ? 1 : 0;
  const int64_t total = static_cast<int64_t>(N) * Ho * Wo * cq;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % cq) * 4;
    int64_t q = i / cq;
    const int ow = static_cast<int>(q % Wo);
    q /= Wo;
    const int oh = static_cast<int>(q % Ho);
    const int n = static_cast<int>(q / Ho);
    const int h0 = oh * stride - pad, w0 = ow * stride - pad;
    float4 acc = mode == 0 ? make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY) : make_float4(0.f, 0.f, 0.f, 0.f);
    int cnt = 0;
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
      const int h = h0 + ky;
      if (h < 0 || h >= H) continue;
#pragma unroll
      for (int kx = 0; kx < 3; ++kx) {
        const int w = w0 + kx;
        if (w < 0 || w >= W) continue;
        const float4 v = *reinterpret_cast<const float4*>(x + n * sn + h * sh + w * sw + c);
        if (mode == 0) {
          acc.x = fmaxf(acc.x, v.x); acc.y = fmaxf(acc.y, v.y); acc.z = fmaxf(acc.z, v.z); acc.w = fmaxf(acc.w, v.w);
        } else {
          acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
        }
        ++cnt;
      }
    }
    if (mode == 1) {
      const float inv = 1.f / static_cast<float>(cnt);
      acc.x *= inv; acc.y *= inv; acc.z *= inv; acc.w *= inv;
    }
    if (y) *reinterpret_cast<float4*>(y + n * ysn + oh * ysh + ow * ysw + c) = acc;
    if (hi) {
      uint16_t h[4], l[4];
      split16_fid(acc.x, dtype, h[0], l[0]);
      split16_fid(acc.y, dtype, h[1], l[1]);
      split16_fid(acc.z, dtype, h[2], l[2]);
      split16_fid(acc.w, dtype, h[3], l[3]);
      const int64_t off = n * psn + oh * psh + ow * psw + c;
      *reinterpret_cast<uint2*>(hi + off) =
          make_uint2(h[0] | (static_cast<uint32_t>(h[1]) << 16), h[2] | (static_cast<uint32_t>(h[3]) << 16));
      if (lo)
        *reinterpret_cast<uint2*>(lo + off) =
            make_uint2(l[0] | (static_cast<uint32_t>(l[1]) << 16), l[2] | (static_cast<uint32_t>(l[3]) << 16));
    }
  }
}

}  // namespace cpcsv

using namespace cpcsv;
#define STREAM(s) static_cast<cudaStream_t>(s)

static bool aligned(const void* p, uintptr_t a) { return (reinterpret_cast<uintptr_t>(p) & (a - 1)) == 0; }

extern "C" int cpcsv_resize_im2col(const float* x, int32_t N, int32_t H, int32_t W, int64_t sn, int64_t sc,
                                   int64_t sh, int64_t sw, int32_t S, float a, float b, void* hi, void* lo,
                                   int32_t ldp, int32_t dtype, cpcsv_stream_t stream) {
  CPCSV_REQUIRE(x && hi && N > 0 && H > 0 && W > 0 && S >= 3, "resize_im2col: args");
  CPCSV_REQUIRE(ldp >= 32 && ldp % 8 == 0 && aligned(hi, 16) && (!lo || aligned(lo, 16)),
                "resize_im2col: ldp must be a multiple of 8 >= 32 and the planes 16-B aligned");
  CPCSV_REQUIRE(dtype == 0 || dtype == 1, "resize_im2col: dtype %d", dtype);
  const int OH = (S - 3) / 2 + 1;
  const int64_t work = static_cast<int64_t>(N) * OH * OH * (ldp / 8);
  resize_im2col_kernel<<<blocks_for(work, 256), 256, 0, STREAM(stream)>>>(
      x, N, H, W, sn, sc, sh, sw, S, OH, static_cast<float>(H) / static_cast<float>(S),
      static_cast<float>(W) / static_cast<float>(S), a, b, static_cast<uint16_t*>(hi), static_cast<uint16_t*>(lo),
      ldp, dtype);
  return launched("resize_im2col");
}

extern "C" int cpcsv_pool3x3(const float* x, int32_t N, int32_t H, int32_t W, int32_t C, int64_t sn, int64_t sh,
                             int64_t sw, int32_t mode, int32_t stride, float* y, int64_t ysn, int64_t ysh,
                             int64_t ysw, void* hi, void* lo, int64_t psn, int64_t psh, int64_t psw, int32_t dtype,
                             cpcsv_stream_t stream) {
  CPCSV_REQUIRE(x && N > 0 && H >= 3 && W >= 3 && C > 0 && C % 4 == 0, "pool3x3: args");
  CPCSV_REQUIRE(mode == 0 || mode == 1, "pool3x3: mode %d", mode);
  CPCSV_REQUIRE(stride == 1 || stride == 2, "pool3x3: stride %d", stride);
  CPCSV_REQUIRE(y || hi, "pool3x3: no output");
  CPCSV_REQUIRE(!lo || hi, "pool3x3: lo without hi");
  CPCSV_REQUIRE(dtype == 0 || dtype == 1, "pool3x3: dtype %d", dtype);
  CPCSV_REQUIRE(aligned(x, 16) && sn % 4 == 0 && sh % 4 == 0 && sw % 4 == 0, "pool3x3: x alignment / pitches");
  CPCSV_REQUIRE(!y || (aligned(y, 16) && ysn % 4 == 0 && ysh % 4 == 0 && ysw % 4 == 0),
                "pool3x3: y alignment / pitches");
  CPCSV_REQUIRE(!hi || (aligned(hi, 8) && (!lo || aligned(lo, 8)) && psn % 4 == 0 && psh % 4 == 0 && psw % 4 == 0),
                "pool3x3: plane alignment / pitches");
  const int Ho = stride == 1 ? H : (H - 3) / 2 + 1;
  const int Wo = stride == 1 ? W : (W - 3) / 2 + 1;
  const int64_t work = static_cast<int64_t>(N) * Ho * Wo * (C / 4);
  pool3x3_kernel<<<blocks_for(work, 256), 256, 0, STREAM(stream)>>>(
      x, N, H, W, C, sn, sh, sw, mode, stride, Ho, Wo, y, ysn, ysh, ysw, static_cast<uint16_t*>(hi),
      static_cast<uint16_t*>(lo), psn, psh, psw, dtype);
  return launched("pool3x3");
}
