// Frame SSIM (cpcsv_b200/ssim.py): pytorch_ssim.ssim(x, y, size_average=False) -- 11-tap Gaussian window
// (sigma 1.5) per channel, zero padding 5, moments in fp32 -- as one CTA per frame.  A frame's value depends only
// on its own pixels: the CTA walks the frame's 32 x 32 output tiles and channels in a fixed order, every thread
// accumulates its pixels in fp64, and a fixed-order block reduction finishes.  No atomics, no allocation.
#include "common.h"

namespace cpcsv {

constexpr int kTaps = 11;
constexpr int kHalo = kTaps / 2;
constexpr int kTile = 32;                  // outputs per tile side
constexpr int kIn = kTile + 2 * kHalo;     // input tile side (42)
constexpr int kRun = 4;                    // consecutive outputs one thread computes in each pass
constexpr int kThreads = kTile * (kTile / kRun);
static_assert(kThreads == 256, "the vertical pass maps one thread to each run of kRun rows of one column");

// exp(-(k - 5)^2 / (2 * 1.5^2)) normalised to sum 1 (computed in double, rounded to float)
__constant__ float kGauss[kTaps] = {1.028380084e-03f, 7.598758135e-03f, 3.600077213e-02f, 1.093606895e-01f,
                                    2.130055377e-01f, 2.660117249e-01f, 2.130055377e-01f, 1.093606895e-01f,
                                    3.600077213e-02f, 7.598758135e-03f, 1.028380084e-03f};

// the five windowed moments, in this order: E[x], E[y], E[x^2], E[y^2], E[xy]
constexpr int kMoments = 5;

__device__ __forceinline__ float ssim_pixel(float mx, float my, float exx, float eyy, float exy) {
  const float C1 = 1e-4f, C2 = 9e-4f;      // 0.01^2, 0.03^2: dynamic range 1
  const float mxx = mx * mx, myy = my * my, mxy = mx * my;
  const float sxx = exx - mxx, syy = eyy - myy, sxy = exy - mxy;
  return ((2.f * mxy + C1) * (2.f * sxy + C2)) / ((mxx + myy + C1) * (sxx + syy + C2));
}

__global__ void __launch_bounds__(kThreads) ssim_kernel(
    const float* __restrict__ x, const float* __restrict__ y, int T, int C, int H, int W, int64_t xsb, int64_t xst,
    int64_t xsc, int64_t xsh, int64_t xsw, int64_t ysb, int64_t yst, int64_t ysc, int64_t ysh, int64_t ysw, float a,
    float b, double* __restrict__ out) {
  __shared__ float sx[kIn][kIn], sy[kIn][kIn];
  __shared__ __align__(16) float sh[kMoments][kIn][kTile];   // the horizontal pass of each moment
  __shared__ double red[kThreads / 32];

  const int frame = blockIdx.x;
  const int bi = frame / T, ti = frame - bi * T;
  const float* xf = x + bi * xsb + ti * xst;
  const float* yf = y + bi * ysb + ti * yst;
  const int tid = threadIdx.x;
  double acc = 0.0;

  for (int r0 = 0; r0 < H; r0 += kTile) {
    for (int c0 = 0; c0 < W; c0 += kTile) {
      for (int c = 0; c < C; ++c) {
        // input tile with its halo; outside the frame the mapped value is 0 (zero padding after the affine)
        const float* xc = xf + c * xsc;
        const float* yc = yf + c * ysc;
        for (int e = tid; e < kIn * kIn; e += kThreads) {
          const int i = e / kIn, j = e - i * kIn;
          const int gr = r0 - kHalo + i, gc = c0 - kHalo + j;
          float vx = 0.f, vy = 0.f;
          if (gr >= 0 && gr < H && gc >= 0 && gc < W) {
            vx = a * __ldg(xc + gr * xsh + gc * xsw) + b;
            vy = a * __ldg(yc + gr * ysh + gc * ysw) + b;
          }
          sx[i][j] = vx;
          sy[i][j] = vy;
        }
        __syncthreads();

        // horizontal pass: every input row, kRun consecutive output columns per item
        for (int e = tid; e < kIn * (kTile / kRun); e += kThreads) {
          const int i = e / (kTile / kRun), j0 = (e % (kTile / kRun)) * kRun;
          float m[kMoments][kRun];
#pragma unroll
          for (int q = 0; q < kMoments; ++q)
#pragma unroll
            for (int o = 0; o < kRun; ++o) m[q][o] = 0.f;
#pragma unroll
          for (int k = 0; k < kRun + kTaps - 1; ++k) {
            const float vx = sx[i][j0 + k], vy = sy[i][j0 + k];
            const float v[kMoments] = {vx, vy, vx * vx, vy * vy, vx * vy};
#pragma unroll
            for (int o = 0; o < kRun; ++o) {
              const int t = k - o;
              if (t >= 0 && t < kTaps) {
#pragma unroll
                for (int q = 0; q < kMoments; ++q) m[q][o] = fmaf(kGauss[t], v[q], m[q][o]);
              }
            }
          }
#pragma unroll
          for (int q = 0; q < kMoments; ++q)
            *reinterpret_cast<float4*>(&sh[q][i][j0]) = make_float4(m[q][0], m[q][1], m[q][2], m[q][3]);
        }
        __syncthreads();

        // vertical pass: column j, kRun consecutive output rows; then the SSIM map of the pixels in the frame.
        // (The next tile's loads may overwrite sx / sy at once; sh is rewritten only after its first barrier.)
        {
          const int j = tid % kTile, i0 = (tid / kTile) * kRun;
          float m[kMoments][kRun];
#pragma unroll
          for (int q = 0; q < kMoments; ++q)
#pragma unroll
            for (int o = 0; o < kRun; ++o) m[q][o] = 0.f;
#pragma unroll
          for (int k = 0; k < kRun + kTaps - 1; ++k) {
            float v[kMoments];
#pragma unroll
            for (int q = 0; q < kMoments; ++q) v[q] = sh[q][i0 + k][j];
#pragma unroll
            for (int o = 0; o < kRun; ++o) {
              const int t = k - o;
              if (t >= 0 && t < kTaps) {
#pragma unroll
                for (int q = 0; q < kMoments; ++q) m[q][o] = fmaf(kGauss[t], v[q], m[q][o]);
              }
            }
          }
          if (c0 + j < W) {
#pragma unroll
            for (int o = 0; o < kRun; ++o)
              if (r0 + i0 + o < H)
                acc += static_cast<double>(ssim_pixel(m[0][o], m[1][o], m[2][o], m[3][o], m[4][o]));
          }
        }
      }
    }
  }

  // fixed-order block reduction
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, off);
  if ((tid & 31) == 0) red[tid >> 5] = acc;
  __syncthreads();
  if (tid == 0) {
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < kThreads / 32; ++w) s += red[w];
    out[frame] = s / (static_cast<double>(C) * H * W);
  }
}

}  // namespace cpcsv

using namespace cpcsv;

extern "C" int cpcsv_ssim(const float* x, const float* y, int32_t B, int32_t T, int32_t C, int32_t H, int32_t W,
                          int64_t xsb, int64_t xst, int64_t xsc, int64_t xsh, int64_t xsw, int64_t ysb, int64_t yst,
                          int64_t ysc, int64_t ysh, int64_t ysw, float a, float b, double* out,
                          cpcsv_stream_t stream) {
  CPCSV_REQUIRE(x && y && out, "ssim: null pointer");
  CPCSV_REQUIRE(B > 0 && T > 0 && C > 0 && H > 0 && W > 0, "ssim: B %d T %d C %d H %d W %d must be >= 1", B, T, C,
                H, W);
  const int64_t frames = static_cast<int64_t>(B) * T;
  CPCSV_REQUIRE(frames <= 0x7fffffff, "ssim: %lld frames exceed one grid", static_cast<long long>(frames));
  ssim_kernel<<<static_cast<unsigned>(frames), kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      x, y, T, C, H, W, xsb, xst, xsc, xsh, xsw, ysb, yst, ysc, ysh, ysw, a, b, out);
  return launched("ssim");
}
