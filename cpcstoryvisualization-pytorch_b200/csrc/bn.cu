// BatchNorm (batch statistics) + activation + segmentation modulation + operand split, forward
// and backward: the HBM-bound kernels between the tcgen05 GEMMs.
//
// Layout: x is fp32 [rows, C] (NHWC flattened), C a multiple of 4.  Every thread owns ONE channel
// quad for its whole lifetime, so the per-channel constants (scale/shift/mean/invstd, gradient
// means) sit in registers and the row loop is pure streaming: 16-byte loads, a few FMAs, 8/16-byte
// stores.  Thread block = `qpb` quads x (256 / qpb) row lanes; grid.x walks the channel quads,
// grid.y the rows.  Reductions: fp64 in registers, a tree over the row lanes of the block in shared
// memory, then ONE fp64 red.add per channel and block into the caller-zeroed [2C] accumulator (at
// most a few hundred adds per address, fire-and-forget).  The same accumulator can be filled by the
// tcgen05 GEMM's epilogue instead (conv_gemm.cu: per-tile column sums), in which case the statistics
// pass over the conv output disappears.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.h"

namespace cpcsv {
namespace {

__device__ __forceinline__ float apply_act(float v, int act) {
  if (act == 1) return v > 0.f ? v : 0.f;
  if (act == 2) return v > 0.f ? v : 0.2f * v;
  return v;
}
__device__ __forceinline__ float act_grad(float pre, int act) {
  if (act == 1) return pre > 0.f ? 1.f : 0.f;
  if (act == 2) return pre > 0.f ? 1.f : 0.2f;
  return 1.f;
}
__device__ __forceinline__ uint32_t pack2(float a, float b, int dtype) {
  if (dtype == 1) {
    return static_cast<uint32_t>(__bfloat16_as_ushort(__float2bfloat16_rn(a))) |
           (static_cast<uint32_t>(__bfloat16_as_ushort(__float2bfloat16_rn(b))) << 16);
  }
  return static_cast<uint32_t>(__half_as_ushort(__float2half_rn(a))) |
         (static_cast<uint32_t>(__half_as_ushort(__float2half_rn(b))) << 16);
}
__device__ __forceinline__ float round16(float a, int dtype) {
  return dtype == 1 ? __bfloat162float(__float2bfloat16_rn(a)) : __half2float(__float2half_rn(a));
}

struct Tiling {
  int qpb;   // channel quads per block
  int rpb;   // row lanes per block
  dim3 grid;
};

// quads per block: a power of two <= 256 that does not overshoot the channel count much
inline Tiling make_tiling(int64_t rows, int C, int blocks_per_sm, int min_rows_per_thread = 1) {
  const int cq = C / 4;
  int qpb = 1;
  while (qpb < cq && qpb < 256) qpb <<= 1;
  Tiling t;
  t.qpb = qpb;
  t.rpb = 256 / qpb;
  const int64_t gx = ceil_div(cq, qpb);
  int64_t gy = ceil_div(static_cast<int64_t>(num_sms()) * blocks_per_sm, gx);
  const int64_t max_gy = ceil_div(rows, static_cast<int64_t>(t.rpb) * min_rows_per_thread);
  if (gy > max_gy) gy = max_gy;
  if (gy < 1) gy = 1;
  if (gy > 65535) gy = 65535;
  t.grid = dim3(static_cast<unsigned>(gx), static_cast<unsigned>(gy));
  return t;
}


// Sum the 8 per-thread fp64 values v[0..8) over the rpb row lanes of each channel quad and ADD
// the totals (lanes rl == 0) to `dst` (dst[c + j] += v[j] totals, dst[C + c + j] += v[4 + j]
// totals).  Two passes through an 8 KB buffer: with 16 KB these kernels would not fit next to a
// resident tensor-core GEMM block (which leaves ~15 KB of shared memory per SM), and the step's
// parallel branches could not overlap.
__device__ __forceinline__ void reduce_rows_to(double (*sh)[4], const double* v, int qpb, int rpb,
                                               int ql, int rl, bool active, double* __restrict__ dst,
                                               int C, int c) {
#pragma unroll
  for (int half = 0; half < 2; ++half) {
    if (half) __syncthreads();
#pragma unroll
    for (int j = 0; j < 4; ++j) sh[threadIdx.x][j] = v[4 * half + j];
    __syncthreads();
    if (rl == 0 && active) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        double t = 0;
        for (int k = 0; k < rpb; ++k) t += sh[k * qpb + ql][j];
        atomicAdd(dst + half * C + c + j, t);
      }
    }
  }
}

// ------------------------------------------------------------------------- statistics
// ws[0..C) += sum x, ws[C..2C) += sum x^2  (fp64)
__global__ void __launch_bounds__(256)
stats_kernel(const float* __restrict__ x, int64_t rows, int C, int64_t ldx, double* __restrict__ ws,
             int qpb, int rpb) {
  const int ql = threadIdx.x % qpb, rl = threadIdx.x / qpb;
  const int c = (blockIdx.x * qpb + ql) * 4;
  double s[4] = {0, 0, 0, 0}, ss[4] = {0, 0, 0, 0};
  if (c < C) {
    const int64_t step = static_cast<int64_t>(gridDim.y) * rpb;
    int64_t r = static_cast<int64_t>(blockIdx.y) * rpb + rl;
    for (; r + 3 * step < rows; r += 4 * step) {
      float4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = *reinterpret_cast<const float4*>(x + (r + u * step) * ldx + c);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        s[0] += v[u].x; ss[0] += static_cast<double>(v[u].x) * v[u].x;
        s[1] += v[u].y; ss[1] += static_cast<double>(v[u].y) * v[u].y;
        s[2] += v[u].z; ss[2] += static_cast<double>(v[u].z) * v[u].z;
        s[3] += v[u].w; ss[3] += static_cast<double>(v[u].w) * v[u].w;
      }
    }
    for (; r < rows; r += step) {
      const float4 v = *reinterpret_cast<const float4*>(x + r * ldx + c);
      s[0] += v.x; ss[0] += static_cast<double>(v.x) * v.x;
      s[1] += v.y; ss[1] += static_cast<double>(v.y) * v.y;
      s[2] += v.z; ss[2] += static_cast<double>(v.z) * v.z;
      s[3] += v.w; ss[3] += static_cast<double>(v.w) * v.w;
    }
  }
  __shared__ double sh[256][4];
  const double v8[8] = {s[0], s[1], s[2], s[3], ss[0], ss[1], ss[2], ss[3]};
  reduce_rows_to(sh, v8, qpb, rpb, ql, rl, c < C, ws, C, c);
}

__global__ void finalize_kernel(const double* __restrict__ stats, int64_t rows, int C,
                                const float* __restrict__ gamma, const float* __restrict__ beta,
                                float* running_mean, float* running_var,
                                const int32_t* __restrict__ chan_map, int C_valid, float eps,
                                float momentum, float* mean, float* invstd, float* scale, float* shift) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  if (c >= C_valid || (chan_map && chan_map[c] < 0)) {  // padding channel
    mean[c] = 0.f; invstd[c] = 0.f; scale[c] = 0.f; shift[c] = 0.f;
    return;
  }
  const double n = static_cast<double>(rows);
  const double m = stats[c] / n;
  double var = stats[C + c] / n - m * m;
  if (var < 0) var = 0;
  const float is = static_cast<float>(1.0 / sqrt(var + static_cast<double>(eps)));
  const int p = chan_map ? chan_map[c] : c;
  const float g = gamma[p], b = beta[p];
  mean[c] = static_cast<float>(m);
  invstd[c] = is;
  scale[c] = g * is;
  shift[c] = b - static_cast<float>(m) * g * is;
  if (running_mean) {
    const double unbiased = rows > 1 ? var * n / (n - 1.0) : var;
    running_mean[p] = (1.f - momentum) * running_mean[p] + momentum * static_cast<float>(m);
    running_var[p] = (1.f - momentum) * running_var[p] + momentum * static_cast<float>(unbiased);
  }
}

// ------------------------------------------------------------------------- forward apply
// Batch statistics -> per-channel constants, done by the apply kernel itself (no finalize launch):
// every block derives scale / shift of its own channels from the fp64 sums; the blocks of row 0
// also publish [mean | invstd | scale | shift] for the backward pass and update the running statistics.
struct BnNorm {
  const double* stats;   // [2C] sum, sum of squares (nullptr: use scale / shift as given)
  const float* gamma;
  const float* beta;
  float* running_mean;
  float* running_var;
  const int32_t* chan_map;
  float* vec;            // [4C]
  double inv_rows;       // 1 / rows
  float unbias;          // rows / (rows - 1)
  int C_valid;
  float eps, momentum;
};

template <bool kMod, bool kY, bool kHi, bool kLo>
__global__ void __launch_bounds__(256)
act_pack_kernel(const float* __restrict__ x, int64_t rows, int C, int64_t ldx,
                const float* __restrict__ scale, const float* __restrict__ shift, int act,
                const float* __restrict__ mod, int64_t ldmod, float* __restrict__ y, int64_t ldy,
                uint16_t* __restrict__ hi, uint16_t* __restrict__ lo, int64_t ldp, int dtype, int qpb,
                int rpb, const BnNorm nb) {
  const int ql = threadIdx.x % qpb, rl = threadIdx.x / qpb;
  const int c = (blockIdx.x * qpb + ql) * 4;
  if (c >= C) return;
  float sc[4] = {1.f, 1.f, 1.f, 1.f}, sf[4] = {0.f, 0.f, 0.f, 0.f};
  if (nb.stats) {
    // mean and variance from the fp64 sums with three fp64 multiplies (1 / rows comes from the host);
    // everything after the cancellation-prone difference is fp32 -- every thread of every block runs
    // this prologue, so it must stay a handful of instructions
    const bool writer = blockIdx.y == 0 && rl == 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int cc = c + j;
      const int p = nb.chan_map ? nb.chan_map[cc] : cc;
      float m_ = 0.f, is_ = 0.f, sc_ = 0.f, sf_ = 0.f;
      if (cc < nb.C_valid && p >= 0) {
        const double m = nb.stats[cc] * nb.inv_rows;
        double var = fma(-m, m, nb.stats[C + cc] * nb.inv_rows);
        if (var < 0) var = 0;
        const float varf = static_cast<float>(var);
        is_ = 1.f / sqrtf(varf + nb.eps);
        m_ = static_cast<float>(m);
        sc_ = nb.gamma[p] * is_;
        sf_ = nb.beta[p] - m_ * sc_;
        if (writer && nb.running_mean) {
          nb.running_mean[p] = (1.f - nb.momentum) * nb.running_mean[p] + nb.momentum * m_;
          nb.running_var[p] = (1.f - nb.momentum) * nb.running_var[p] + nb.momentum * (varf * nb.unbias);
        }
      }
      sc[j] = sc_;
      sf[j] = sf_;
      if (writer) {
        nb.vec[cc] = m_; nb.vec[C + cc] = is_; nb.vec[2 * C + cc] = sc_; nb.vec[3 * C + cc] = sf_;
      }
    }
  } else if (scale) {
#pragma unroll
    for (int j = 0; j < 4; ++j) { sc[j] = scale[c + j]; sf[j] = shift[c + j]; }
  }
  const int64_t step = static_cast<int64_t>(gridDim.y) * rpb;
  for (int64_t r = static_cast<int64_t>(blockIdx.y) * rpb + rl; r < rows; r += step) {
    const float4 xv = *reinterpret_cast<const float4*>(x + r * ldx + c);
    float v[4] = {xv.x, xv.y, xv.z, xv.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) v[j] = apply_act(fmaf(v[j], sc[j], sf[j]), act);
    if (kMod) {
      const float4 mv = *reinterpret_cast<const float4*>(mod + r * ldmod + c);
      v[0] *= 1.f + mv.x; v[1] *= 1.f + mv.y; v[2] *= 1.f + mv.z; v[3] *= 1.f + mv.w;
    }
    if (kY) *reinterpret_cast<float4*>(y + r * ldy + c) = make_float4(v[0], v[1], v[2], v[3]);
    if (kHi) {
      uint2 hv;
      hv.x = pack2(v[0], v[1], dtype);
      hv.y = pack2(v[2], v[3], dtype);
      *reinterpret_cast<uint2*>(hi + r * ldp + c) = hv;
      if (kLo) {
        uint2 lv;
        lv.x = pack2(v[0] - round16(v[0], dtype), v[1] - round16(v[1], dtype), dtype);
        lv.y = pack2(v[2] - round16(v[2], dtype), v[3] - round16(v[3], dtype), dtype);
        *reinterpret_cast<uint2*>(lo + r * ldp + c) = lv;
      }
    }
  }
}

// ------------------------------------------------------------------------- residual epilogue
// y = act(x*scale + shift + (r*rscale + rshift)): the last BatchNorm of a residual block, the BatchNorm of
// its projected shortcut (kRS; identity shortcut: r as is), the add and the activation in one pass.
template <bool kRS, bool kY, bool kHi, bool kLo>
__global__ void __launch_bounds__(256)
act_add_pack_kernel(const float* __restrict__ x, int64_t rows, int C, int64_t ldx,
                    const float* __restrict__ scale, const float* __restrict__ shift,
                    const float* __restrict__ r, int64_t ldr, const float* __restrict__ rscale,
                    const float* __restrict__ rshift, int act, float* __restrict__ y, int64_t ldy,
                    uint16_t* __restrict__ hi, uint16_t* __restrict__ lo, int64_t ldp, int dtype, int qpb,
                    int rpb) {
  const int ql = threadIdx.x % qpb, rl = threadIdx.x / qpb;
  const int c = (blockIdx.x * qpb + ql) * 4;
  if (c >= C) return;
  float sc[4], sf[4], rsc[4] = {1.f, 1.f, 1.f, 1.f}, rsf[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    sc[j] = scale[c + j];
    sf[j] = shift[c + j];
    if (kRS) { rsc[j] = rscale[c + j]; rsf[j] = rshift[c + j]; }
  }
  const int64_t step = static_cast<int64_t>(gridDim.y) * rpb;
  for (int64_t row = static_cast<int64_t>(blockIdx.y) * rpb + rl; row < rows; row += step) {
    const float4 xv = *reinterpret_cast<const float4*>(x + row * ldx + c);
    const float4 rv = *reinterpret_cast<const float4*>(r + row * ldr + c);
    const float xs[4] = {xv.x, xv.y, xv.z, xv.w}, rs[4] = {rv.x, rv.y, rv.z, rv.w};
    float v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float res = kRS ? fmaf(rs[j], rsc[j], rsf[j]) : rs[j];
      v[j] = apply_act(fmaf(xs[j], sc[j], sf[j]) + res, act);
    }
    if (kY) *reinterpret_cast<float4*>(y + row * ldy + c) = make_float4(v[0], v[1], v[2], v[3]);
    if (kHi) {
      uint2 hv;
      hv.x = pack2(v[0], v[1], dtype);
      hv.y = pack2(v[2], v[3], dtype);
      *reinterpret_cast<uint2*>(hi + row * ldp + c) = hv;
      if (kLo) {
        uint2 lv;
        lv.x = pack2(v[0] - round16(v[0], dtype), v[1] - round16(v[1], dtype), dtype);
        lv.y = pack2(v[2] - round16(v[2], dtype), v[3] - round16(v[3], dtype), dtype);
        *reinterpret_cast<uint2*>(lo + row * ldp + c) = lv;
      }
    }
  }
}

// ------------------------------------------------------------------------- backward
struct ChanConst {
  float sc[4], sf[4], mean[4], invstd[4];
};
__device__ __forceinline__ ChanConst load_const(const float* scale, const float* shift, const float* mean,
                                                const float* invstd, int c) {
  ChanConst k;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    k.sc[j] = scale ? scale[c + j] : 1.f;
    k.sf[j] = scale ? shift[c + j] : 0.f;
    k.mean[j] = mean ? mean[c + j] : 0.f;
    k.invstd[j] = mean ? invstd[c + j] : 0.f;
  }
  return k;
}

// g = dL/d(pre-activation), xhat, a = activation (before modulation) for one row / 4 channels
__device__ __forceinline__ void bwd_row(const float* __restrict__ x, const float* __restrict__ dy,
                                        const float* __restrict__ mod, int64_t r, int c, int64_t ldx,
                                        int64_t lddy, int64_t ldmod, const ChanConst& k, int act,
                                        float (&g)[4], float (&xhat)[4], float (&a)[4], float (&d)[4]) {
  const float4 xv = *reinterpret_cast<const float4*>(x + r * ldx + c);
  const float4 dv = *reinterpret_cast<const float4*>(dy + r * lddy + c);
  const float xs[4] = {xv.x, xv.y, xv.z, xv.w};
  d[0] = dv.x; d[1] = dv.y; d[2] = dv.z; d[3] = dv.w;
  float ms[4] = {0.f, 0.f, 0.f, 0.f};
  if (mod) {
    const float4 mv = *reinterpret_cast<const float4*>(mod + r * ldmod + c);
    ms[0] = mv.x; ms[1] = mv.y; ms[2] = mv.z; ms[3] = mv.w;
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float pre = fmaf(xs[j], k.sc[j], k.sf[j]);
    a[j] = apply_act(pre, act);
    g[j] = d[j] * (1.f + ms[j]) * act_grad(pre, act);
    xhat[j] = (xs[j] - k.mean[j]) * k.invstd[j];
  }
}

__global__ void __launch_bounds__(256)
bwd_reduce_kernel(const float* __restrict__ x, const float* __restrict__ dy, int64_t rows, int C,
                  int64_t ldx, int64_t lddy, const float* __restrict__ scale,
                  const float* __restrict__ shift, const float* __restrict__ mean,
                  const float* __restrict__ invstd, int act, const float* __restrict__ mod,
                  int64_t ldmod, double* __restrict__ ws, int qpb, int rpb) {
  const int ql = threadIdx.x % qpb, rl = threadIdx.x / qpb;
  const int c = (blockIdx.x * qpb + ql) * 4;
  double s[4] = {0, 0, 0, 0}, sx[4] = {0, 0, 0, 0};
  if (c < C) {
    const ChanConst k = load_const(scale, shift, mean, invstd, c);
    const int64_t step = static_cast<int64_t>(gridDim.y) * rpb;
    int64_t r = static_cast<int64_t>(blockIdx.y) * rpb + rl;
    for (; r + step < rows; r += 2 * step) {
      float g0[4], h0[4], a0[4], d0[4], g1[4], h1[4], a1[4], d1[4];
      bwd_row(x, dy, mod, r, c, ldx, lddy, ldmod, k, act, g0, h0, a0, d0);
      bwd_row(x, dy, mod, r + step, c, ldx, lddy, ldmod, k, act, g1, h1, a1, d1);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        s[j] += static_cast<double>(g0[j]) + g1[j];
        sx[j] += static_cast<double>(g0[j]) * h0[j] + static_cast<double>(g1[j]) * h1[j];
      }
    }
    for (; r < rows; r += step) {
      float g0[4], h0[4], a0[4], d0[4];
      bwd_row(x, dy, mod, r, c, ldx, lddy, ldmod, k, act, g0, h0, a0, d0);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        s[j] += g0[j];
        sx[j] += static_cast<double>(g0[j]) * h0[j];
      }
    }
  }
  __shared__ double sh[256][4];
  const double v8[8] = {s[0], s[1], s[2], s[3], sx[0], sx[1], sx[2], sx[3]};
  reduce_rows_to(sh, v8, qpb, rpb, ql, rl, c < C, ws, C, c);
}

__global__ void __launch_bounds__(256)
bwd_apply_kernel(const float* __restrict__ x, const float* __restrict__ dy, int64_t rows, int C,
                 int64_t ldx, int64_t lddy, const float* __restrict__ scale,
                 const float* __restrict__ shift, const float* __restrict__ mean,
                 const float* __restrict__ invstd, const int32_t* __restrict__ chan_map, int C_valid,
                 int act, const float* __restrict__ mod, int64_t ldmod, const double* __restrict__ sums,
                 int has_bn, float* __restrict__ dx, int64_t lddx, uint16_t* __restrict__ dx16,
                 int64_t ld16, float* __restrict__ dmod, int64_t lddmod, uint16_t* __restrict__ dmod16,
                 int64_t lddmod16, float* __restrict__ dgamma, float* __restrict__ dbeta, int qpb,
                 int rpb) {
  const int ql = threadIdx.x % qpb, rl = threadIdx.x / qpb;
  const int c = (blockIdx.x * qpb + ql) * 4;
  if (c >= C) return;
  const ChanConst k = load_const(scale, shift, has_bn ? mean : nullptr, invstd, c);
  float mg[4] = {0.f, 0.f, 0.f, 0.f}, mgx[4] = {0.f, 0.f, 0.f, 0.f};
  if (has_bn) {
    const float inv_rows = 1.f / static_cast<float>(rows);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      mg[j] = static_cast<float>(sums[c + j]) * inv_rows;
      mgx[j] = static_cast<float>(sums[C + c + j]) * inv_rows;
    }
    if (dgamma && blockIdx.y == 0 && rl == 0) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (c + j < C_valid) {
          const int p = chan_map ? chan_map[c + j] : c + j;
          if (p >= 0) {
            dgamma[p] = static_cast<float>(sums[C + c + j]);
            dbeta[p] = static_cast<float>(sums[c + j]);
          }
        }
      }
    }
  }
  const int64_t step = static_cast<int64_t>(gridDim.y) * rpb;
  for (int64_t r = static_cast<int64_t>(blockIdx.y) * rpb + rl; r < rows; r += step) {
    float g[4], xhat[4], a[4], dv[4], d[4];
    bwd_row(x, dy, mod, r, c, ldx, lddy, ldmod, k, act, g, xhat, a, dv);
#pragma unroll
    for (int j = 0; j < 4; ++j)
      d[j] = has_bn ? k.sc[j] * (g[j] - mg[j] - xhat[j] * mgx[j]) : g[j];   // sc = gamma * invstd
    if (dx) *reinterpret_cast<float4*>(dx + r * lddx + c) = make_float4(d[0], d[1], d[2], d[3]);
    if (dx16) {
      uint2 v;
      v.x = pack2(d[0], d[1], 1);
      v.y = pack2(d[2], d[3], 1);
      *reinterpret_cast<uint2*>(dx16 + r * ld16 + c) = v;
    }
    if (dmod || dmod16) {
      const float m[4] = {dv[0] * a[0], dv[1] * a[1], dv[2] * a[2], dv[3] * a[3]};
      if (dmod) *reinterpret_cast<float4*>(dmod + r * lddmod + c) = make_float4(m[0], m[1], m[2], m[3]);
      if (dmod16) {
        uint2 v;
        v.x = pack2(m[0], m[1], 1);
        v.y = pack2(m[2], m[3], 1);
        *reinterpret_cast<uint2*>(dmod16 + r * lddmod16 + c) = v;
      }
    }
  }
}

}  // namespace
}  // namespace cpcsv

using namespace cpcsv;
#define STREAM(s) static_cast<cudaStream_t>(s)

extern "C" int64_t cpcsv_bn_workspace_doubles(int64_t rows, int32_t C) {
  (void)rows;
  return static_cast<int64_t>(2 * C);
}

extern "C" int cpcsv_bn_stats(const float* x, int64_t rows, int32_t C, int64_t ldx, double* stats,
                              cpcsv_stream_t stream) {
  CPCSV_REQUIRE(x && stats && rows > 0 && C > 0 && C % 4 == 0 && ldx % 4 == 0, "bn_stats: args");
  // every block ends with one fp64 red.add per channel: at least 16 rows per thread
  const Tiling t = make_tiling(rows, C, 4, 16);
  stats_kernel<<<t.grid, 256, 0, STREAM(stream)>>>(x, rows, C, ldx, stats, t.qpb, t.rpb);
  return launched("bn_stats");
}

extern "C" int cpcsv_bn_finalize(const double* stats, int64_t rows, int32_t C, const float* gamma,
                                 const float* beta, float* running_mean, float* running_var,
                                 const int32_t* chan_map, int32_t C_valid, float eps, float momentum,
                                 float* mean, float* invstd, float* scale, float* shift,
                                 cpcsv_stream_t stream) {
  CPCSV_REQUIRE(stats && gamma && beta && mean && invstd && scale && shift && C > 0 && C_valid <= C,
                "bn_finalize: args");
  finalize_kernel<<<static_cast<unsigned>(ceil_div(C, 256)), 256, 0, STREAM(stream)>>>(
      stats, rows, C, gamma, beta, running_mean, running_var, chan_map, C_valid, eps, momentum, mean,
      invstd, scale, shift);
  return launched("bn_finalize");
}

static int launch_act_pack(const float* x, int64_t rows, int32_t C, int64_t ldx, const float* scale,
                           const float* shift, int32_t act, const float* mod, int64_t ldmod, float* y,
                           int64_t ldy, void* hi, void* lo, int64_t ldp, int32_t dtype, const BnNorm& nb,
                           cudaStream_t stream, const char* what) {
  const Tiling t = make_tiling(rows, C, 8, 4);
  uint16_t* h = static_cast<uint16_t*>(hi);
  uint16_t* l = static_cast<uint16_t*>(lo);
#define LAUNCH(M, Y, H, L)                                                                     \
  act_pack_kernel<M, Y, H, L><<<t.grid, 256, 0, stream>>>(x, rows, C, ldx, scale, shift, act, mod, \
                                                           ldmod, y, ldy, h, l, ldp, dtype, t.qpb, \
                                                           t.rpb, nb)
  const int key = (mod ? 8 : 0) | (y ? 4 : 0) | (hi ? 2 : 0) | (lo ? 1 : 0);
  switch (key) {
    case 2: LAUNCH(false, false, true, false); break;
    case 3: LAUNCH(false, false, true, true); break;
    case 4: LAUNCH(false, true, false, false); break;
    case 6: LAUNCH(false, true, true, false); break;
    case 7: LAUNCH(false, true, true, true); break;
    case 10: LAUNCH(true, false, true, false); break;
    case 11: LAUNCH(true, false, true, true); break;
    case 12: LAUNCH(true, true, false, false); break;
    case 14: LAUNCH(true, true, true, false); break;
    case 15: LAUNCH(true, true, true, true); break;
    default: return fail(-1, "%s: unsupported output combination %d", what, key);
  }
#undef LAUNCH
  return launched(what);
}

extern "C" int cpcsv_bn_act_pack(const float* x, int64_t rows, int32_t C, int64_t ldx,
                                 const float* scale, const float* shift, int32_t act,
                                 const float* mod, int64_t ldmod, float* y, int64_t ldy, void* hi,
                                 void* lo, int64_t ldp, int32_t dtype, cpcsv_stream_t stream) {
  CPCSV_REQUIRE(x && rows > 0 && C > 0 && C % 4 == 0 && ldx % 4 == 0, "bn_act_pack: args");
  CPCSV_REQUIRE((!mod || ldmod % 4 == 0) && (!y || ldy % 4 == 0) && (!hi || ldp % 4 == 0),
                "bn_act_pack: pitches must be multiples of 4");
  CPCSV_REQUIRE(hi || y, "bn_act_pack: no output");
  CPCSV_REQUIRE(!lo || hi, "bn_act_pack: lo without hi");
  BnNorm nb = {};
  return launch_act_pack(x, rows, C, ldx, scale, shift, act, mod, ldmod, y, ldy, hi, lo, ldp, dtype, nb,
                         STREAM(stream), "bn_act_pack");
}

extern "C" int cpcsv_bn_norm_act_pack(const float* x, int64_t rows, int32_t C, int64_t ldx,
                                      const double* stats, const float* gamma, const float* beta,
                                      float* running_mean, float* running_var, const int32_t* chan_map,
                                      int32_t C_valid, float eps, float momentum, float* vec, int32_t act,
                                      const float* mod, int64_t ldmod, float* y, int64_t ldy, void* hi,
                                      void* lo, int64_t ldp, int32_t dtype, cpcsv_stream_t stream) {
  CPCSV_REQUIRE(x && stats && gamma && beta && vec && rows > 0 && C > 0 && C % 4 == 0 && ldx % 4 == 0 &&
                    C_valid <= C,
                "bn_norm_act_pack: args");
  CPCSV_REQUIRE((!mod || ldmod % 4 == 0) && (!y || ldy % 4 == 0) && (!hi || ldp % 4 == 0) && (hi || y) &&
                    (!lo || hi) && (!running_mean == !running_var),
                "bn_norm_act_pack: outputs");
  BnNorm nb;
  nb.stats = stats; nb.gamma = gamma; nb.beta = beta;
  nb.running_mean = running_mean; nb.running_var = running_var; nb.chan_map = chan_map; nb.vec = vec;
  nb.inv_rows = 1.0 / static_cast<double>(rows);
  nb.unbias = rows > 1 ? static_cast<float>(static_cast<double>(rows) / static_cast<double>(rows - 1)) : 1.f;
  nb.C_valid = C_valid; nb.eps = eps; nb.momentum = momentum;
  return launch_act_pack(x, rows, C, ldx, nullptr, nullptr, act, mod, ldmod, y, ldy, hi, lo, ldp, dtype, nb,
                         STREAM(stream), "bn_norm_act_pack");
}

extern "C" int cpcsv_bn_add_act_pack(const float* x, int64_t rows, int32_t C, int64_t ldx, const float* scale,
                                     const float* shift, const float* r, int64_t ldr, const float* rscale,
                                     const float* rshift, int32_t act, float* y, int64_t ldy, void* hi, void* lo,
                                     int64_t ldp, int32_t dtype, cpcsv_stream_t stream) {
  CPCSV_REQUIRE(x && r && scale && shift && rows > 0 && C > 0 && C % 4 == 0 && ldx % 4 == 0 && ldr % 4 == 0,
                "bn_add_act_pack: args");
  CPCSV_REQUIRE(!rscale == !rshift, "bn_add_act_pack: rscale and rshift go together");
  CPCSV_REQUIRE((!y || ldy % 4 == 0) && (!hi || ldp % 4 == 0), "bn_add_act_pack: pitches must be multiples of 4");
  CPCSV_REQUIRE(hi || y, "bn_add_act_pack: no output");
  CPCSV_REQUIRE(!lo || hi, "bn_add_act_pack: lo without hi");
  const Tiling t = make_tiling(rows, C, 8, 4);
  uint16_t* h = static_cast<uint16_t*>(hi);
  uint16_t* l = static_cast<uint16_t*>(lo);
#define LAUNCH(RS, Y, H, L)                                                                                   \
  act_add_pack_kernel<RS, Y, H, L><<<t.grid, 256, 0, STREAM(stream)>>>(x, rows, C, ldx, scale, shift, r, ldr, \
                                                                        rscale, rshift, act, y, ldy, h, l,    \
                                                                        ldp, dtype, t.qpb, t.rpb)
  const int key = (rscale ? 8 : 0) | (y ? 4 : 0) | (hi ? 2 : 0) | (lo ? 1 : 0);
  switch (key) {
    case 2: LAUNCH(false, false, true, false); break;
    case 3: LAUNCH(false, false, true, true); break;
    case 4: LAUNCH(false, true, false, false); break;
    case 6: LAUNCH(false, true, true, false); break;
    case 7: LAUNCH(false, true, true, true); break;
    case 10: LAUNCH(true, false, true, false); break;
    case 11: LAUNCH(true, false, true, true); break;
    case 12: LAUNCH(true, true, false, false); break;
    case 14: LAUNCH(true, true, true, false); break;
    case 15: LAUNCH(true, true, true, true); break;
    default: return fail(-1, "bn_add_act_pack: unsupported output combination %d", key);
  }
#undef LAUNCH
  return launched("bn_add_act_pack");
}

extern "C" int cpcsv_bn_bwd_reduce(const float* x, const float* dy, int64_t rows, int32_t C,
                                   int64_t ldx, int64_t lddy, const float* scale, const float* shift,
                                   const float* mean, const float* invstd, int32_t act,
                                   const float* mod, int64_t ldmod, double* sums,
                                   cpcsv_stream_t stream) {
  CPCSV_REQUIRE(x && dy && sums && mean && invstd && rows > 0 && C > 0 && C % 4 == 0 &&
                    ldx % 4 == 0 && lddy % 4 == 0,
                "bn_bwd_reduce: args");
  const Tiling t = make_tiling(rows, C, 4, 16);
  bwd_reduce_kernel<<<t.grid, 256, 0, STREAM(stream)>>>(x, dy, rows, C, ldx, lddy, scale, shift, mean,
                                                        invstd, act, mod, ldmod, sums, t.qpb, t.rpb);
  return launched("bn_bwd_reduce");
}

extern "C" int cpcsv_bn_bwd_apply(const float* x, const float* dy, int64_t rows, int32_t C,
                                  int64_t ldx, int64_t lddy, const float* scale, const float* shift,
                                  const float* mean, const float* invstd, const float* gamma,
                                  const int32_t* chan_map, int32_t C_valid, int32_t act,
                                  const float* mod, int64_t ldmod, const double* sums, int32_t has_bn,
                                  float* dx, int64_t lddx, void* dx16, int64_t ld16, float* dmod,
                                  int64_t lddmod, void* dmod16, int64_t lddmod16, float* dgamma,
                                  float* dbeta, cpcsv_stream_t stream) {
  (void)gamma;
  CPCSV_REQUIRE(x && dy && rows > 0 && C > 0 && C % 4 == 0 && ldx % 4 == 0 && lddy % 4 == 0,
                "bn_bwd_apply: args");
  CPCSV_REQUIRE(!has_bn || (sums && scale && mean && invstd), "bn_bwd_apply: BN tensors missing");
  const Tiling t = make_tiling(rows, C, 8, 4);
  bwd_apply_kernel<<<t.grid, 256, 0, STREAM(stream)>>>(
      x, dy, rows, C, ldx, lddy, scale, shift, mean, invstd, chan_map, C_valid, act, mod, ldmod, sums,
      has_bn, dx, lddx, static_cast<uint16_t*>(dx16), ld16, dmod, lddmod, static_cast<uint16_t*>(dmod16),
      lddmod16, dgamma, dbeta, t.qpb, t.rpb);
  return launched("bn_bwd_apply");
}
