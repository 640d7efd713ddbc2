"""Tensor-level wrappers: one Python function per C-ABI entry point of libcpcsv.so.

Each function takes torch CUDA tensors, extracts raw pointers / pitches and enqueues the
kernel on the current CUDA stream.  Nothing here computes with PyTorch: a CPU tensor or a
missing library raises (no fallback).  Outputs are preallocated by the caller (the library
never allocates).
"""
import ctypes as C

import torch

from . import _lib

ACT_NONE, ACT_RELU, ACT_LRELU = 0, 1, 2
FP16, BF16 = 0, 1
TORCH16 = {FP16: torch.float16, BF16: torch.bfloat16}
MAX_PLANES = _lib.MAX_PLANES


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t, dtype=None):
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("cpcsv ops need CUDA tensors (no CPU fallback); got a %s tensor" % t.device)
    if dtype is not None and t.dtype != dtype:
        raise RuntimeError("expected %s, got %s" % (dtype, t.dtype))
    return C.c_void_p(t.data_ptr())


def _rows2d(t):
    """[rows, C] view with unit column stride -> (rows, C, pitch)."""
    assert t.dim() == 2 and (t.stride(1) == 1 or t.shape[1] == 1), (t.shape, t.stride())
    return t.shape[0], t.shape[1], t.stride(0)


class View:
    """5-D strided view (c, w, p, h, n) of a 16-bit tensor; strides in BYTES (dim 0 = 2)."""

    __slots__ = ("tensor", "dims", "strides")

    def __init__(self, tensor, dims, strides):
        assert tensor.element_size() == 2
        self.tensor, self.dims, self.strides = tensor, tuple(int(d) for d in dims), tuple(int(s) for s in strides)

    @staticmethod
    def nhwc(t):
        """t: [N, H, W, C] (last dim contiguous)."""
        N, H, W, Cc = t.shape
        sn, sh, sw, sc = (s * 2 for s in t.stride())
        assert sc == 2
        return View(t, (Cc, W, 1, H, N), (2, sw, sh, sh, sn))

    @staticmethod
    def nhwc_parity(t):
        """t: [N, H, W, C] viewed as (2C, W/2, 2, H/2, N): element (c + C*wp, ww, hp, hh, n) is
        t[n, 2*hh + hp, 2*ww + wp, c].  Requires the pixel pitch to equal C."""
        N, H, W, Cc = t.shape
        sn, sh, sw, sc = (s * 2 for s in t.stride())
        assert sc == 2 and sw == Cc * 2 and H % 2 == 0 and W % 2 == 0
        return View(t, (2 * Cc, W // 2, 2, H // 2, N), (2, 2 * sw, sh, 2 * sh, sn))

    @staticmethod
    def matrix(t):
        """t: [rows, K] row-major."""
        rows, K = t.shape
        assert t.stride(1) == 1
        pitch = t.stride(0) * 2
        return View(t, (K, rows, 1, 1, 1), (2, pitch, pitch * rows, pitch * rows, pitch * rows))

    def to_c(self):
        v = _lib.View5()
        v.ptr = _ptr(self.tensor).value
        for i in range(5):
            v.dims[i] = self.dims[i]
            v.strides[i] = self.strides[i]
        return v


class GemmJob:
    """Mirror of cpcsv_gemm_t (include/cpcsv.h).  ``taps``: list of (a4, b4, out_off)."""

    def __init__(self, mode, planes, grid, tile, groups, taps_per_group, k_blocks, taps, a, b, out,
                 n_valid, block_n, n_tiles, m_valid=0, splits=1, accumulate=False,
                 out_strides=(0, 0, 0), ldc=0, alpha=None, dtype=BF16, pair=False, stats=None):
        self.mode, self.planes, self.dtype = mode, planes, dtype
        self.grid, self.tile = tuple(grid), tuple(tile)      # (N, H, W), (tile_n, tile_h, tile_w)
        self.groups, self.taps_per_group, self.k_blocks = groups, taps_per_group, k_blocks
        self.taps = list(taps)
        self.a, self.b = list(a), list(b)                    # [hi, lo?] Views
        self.out = out
        self.n_valid, self.block_n, self.n_tiles, self.m_valid = n_valid, block_n, n_tiles, m_valid
        self.splits, self.accumulate = splits, bool(accumulate)
        self.out_strides, self.ldc, self.alpha = tuple(out_strides), ldc, alpha
        self.pair = bool(pair)      # mode 0: cta_group::2 pairs (see conv.use_pair)
        # mode 0, no split-K: fp64 [2, n_valid] accumulator the epilogue adds the per-column sum and
        # sum of squares of the stored values into (BatchNorm batch statistics of the conv output)
        self.stats = stats


def conv_gemm(job):
    g = _lib.Gemm()
    g.mode, g.dtype, g.planes = job.mode, job.dtype, job.planes
    g.N, g.H, g.W = job.grid
    g.tile_n, g.tile_h, g.tile_w = job.tile
    g.groups, g.taps_per_group, g.k_blocks = job.groups, job.taps_per_group, job.k_blocks
    g.m_valid, g.n_valid, g.block_n, g.n_tiles = job.m_valid, job.n_valid, job.block_n, job.n_tiles
    g.splits, g.accumulate, g.cta_pair = job.splits, int(job.accumulate), int(job.pair)
    g.out_stride_n, g.out_stride_h, g.out_stride_w = job.out_strides
    g.ldc = job.ldc
    g.alpha = _ptr(job.alpha, torch.float32).value if job.alpha is not None else None
    g.out = _ptr(job.out, torch.float32).value
    if job.stats is not None:
        assert job.mode == 0 and job.splits == 1 and not job.accumulate and job.stats.dim() == 2
        g.stats, g.stats_ld = _ptr(job.stats, torch.float64).value, job.stats.stride(0)
    for i in range(job.planes):
        g.a[i] = job.a[i].to_c()
        g.b[i] = job.b[i].to_c()
    assert len(job.taps) <= _lib.MAX_TAPS
    for i, (a4, b4, off) in enumerate(job.taps):
        for j in range(4):
            g.taps[i].a[j] = a4[j]
            g.taps[i].b[j] = b4[j]
        g.taps[i].out_off = off
    if (job.splits > 1) and not job.accumulate:
        job.out.zero_()  # split-K partial tiles are combined with red.add
    _lib.check(_lib.load().cpcsv_conv_gemm(C.byref(g), _stream()), "cpcsv_conv_gemm")


# ------------------------------------------------------------------ BatchNorm / packing
def bn_workspace(rows, channels, device):
    """zeroed fp64 [2C] accumulator for bn_stats / bn_bwd_reduce (sum | sum of squares)"""
    n = _lib.load().cpcsv_bn_workspace_doubles(rows, channels)
    return torch.zeros(n, device=device, dtype=torch.float64)


def bn_stats(x, stats):
    rows, Cc, ld = _rows2d(x)
    assert stats.numel() >= 2 * Cc
    _lib.check(_lib.load().cpcsv_bn_stats(_ptr(x, torch.float32), rows, Cc, ld,
                                          _ptr(stats, torch.float64), _stream()), "cpcsv_bn_stats")


def bn_finalize(stats, rows, gamma, beta, running_mean, running_var, chan_map, c_valid,
                mean, invstd, scale, shift, eps=1e-5, momentum=0.1):
    Cc = mean.numel()
    _lib.check(_lib.load().cpcsv_bn_finalize(
        _ptr(stats, torch.float64), rows, Cc, _ptr(gamma, torch.float32), _ptr(beta, torch.float32),
        _ptr(running_mean, torch.float32), _ptr(running_var, torch.float32),
        _ptr(chan_map, torch.int32), c_valid, eps, momentum, _ptr(mean), _ptr(invstd), _ptr(scale),
        _ptr(shift), _stream()), "cpcsv_bn_finalize")


def bn_act_pack(x, scale, shift, act, mod=None, y=None, hi=None, lo=None, dtype=BF16):
    rows, Cc, ld = _rows2d(x)
    ldmod = mod.stride(0) if mod is not None else 0
    ldy = y.stride(0) if y is not None else 0
    ldp = hi.stride(0) if hi is not None else 0
    if lo is not None:
        assert lo.stride(0) == ldp
    _lib.check(_lib.load().cpcsv_bn_act_pack(
        _ptr(x, torch.float32), rows, Cc, ld, _ptr(scale), _ptr(shift), act, _ptr(mod), ldmod,
        _ptr(y), ldy, _ptr(hi), _ptr(lo), ldp, dtype, _stream()), "cpcsv_bn_act_pack")


def bn_add_act_pack(x, scale, shift, r, rscale, rshift, act, y=None, hi=None, lo=None, dtype=BF16):
    """y = act(x*scale + shift + (r*rscale + rshift)); rscale / rshift None: identity shortcut (r as is)"""
    rows, Cc, ld = _rows2d(x)
    rr, rc, ldr = _rows2d(r)
    assert (rr, rc) == (rows, Cc), (r.shape, x.shape)
    ldy = y.stride(0) if y is not None else 0
    ldp = hi.stride(0) if hi is not None else 0
    if lo is not None:
        assert lo.stride(0) == ldp
    _lib.check(_lib.load().cpcsv_bn_add_act_pack(
        _ptr(x, torch.float32), rows, Cc, ld, _ptr(scale, torch.float32), _ptr(shift, torch.float32),
        _ptr(r, torch.float32), ldr, _ptr(rscale, torch.float32), _ptr(rshift, torch.float32), act,
        _ptr(y, torch.float32), ldy, _ptr(hi), _ptr(lo), ldp, dtype, _stream()), "cpcsv_bn_add_act_pack")


def bn_bwd_reduce(x, dy, scale, shift, mean, invstd, act, mod, sums):
    rows, Cc, ld = _rows2d(x)
    _lib.check(_lib.load().cpcsv_bn_bwd_reduce(
        _ptr(x, torch.float32), _ptr(dy, torch.float32), rows, Cc, ld, dy.stride(0), _ptr(scale),
        _ptr(shift), _ptr(mean), _ptr(invstd), act, _ptr(mod), mod.stride(0) if mod is not None else 0,
        _ptr(sums, torch.float64), _stream()), "cpcsv_bn_bwd_reduce")


def bn_bwd_apply(x, dy, scale, shift, mean, invstd, chan_map, c_valid, act, mod, sums, has_bn,
                 dx=None, dx16=None, dmod=None, dmod16=None, dgamma=None, dbeta=None):
    rows, Cc, ld = _rows2d(x)
    _lib.check(_lib.load().cpcsv_bn_bwd_apply(
        _ptr(x, torch.float32), _ptr(dy, torch.float32), rows, Cc, ld, dy.stride(0), _ptr(scale),
        _ptr(shift), _ptr(mean), _ptr(invstd), None, _ptr(chan_map, torch.int32), c_valid, act,
        _ptr(mod), mod.stride(0) if mod is not None else 0, _ptr(sums), int(has_bn),
        _ptr(dx), dx.stride(0) if dx is not None else 0,
        _ptr(dx16), dx16.stride(0) if dx16 is not None else 0,
        _ptr(dmod), dmod.stride(0) if dmod is not None else 0,
        _ptr(dmod16), dmod16.stride(0) if dmod16 is not None else 0,
        _ptr(dgamma), _ptr(dbeta), _stream()), "cpcsv_bn_bwd_apply")


def bn_norm_act_pack(x, stats, gamma, beta, running_mean, running_var, chan_map, c_valid, vec, act, mod=None,
                     y=None, hi=None, lo=None, dtype=BF16, eps=1e-5, momentum=0.1):
    """batch-statistics BatchNorm (sums in `stats`) + activation [+ modulation] + operand split in one
    launch; vec [4, C] receives mean / invstd / scale / shift, the running statistics are updated"""
    rows, Cc, ld = _rows2d(x)
    assert stats.numel() >= 2 * Cc and vec.numel() == 4 * Cc and vec.is_contiguous()
    ldp = hi.stride(0) if hi is not None else 0
    if lo is not None:
        assert lo.stride(0) == ldp
    _lib.check(_lib.load().cpcsv_bn_norm_act_pack(
        _ptr(x, torch.float32), rows, Cc, ld, _ptr(stats, torch.float64), _ptr(gamma, torch.float32),
        _ptr(beta, torch.float32), _ptr(running_mean, torch.float32), _ptr(running_var, torch.float32),
        _ptr(chan_map, torch.int32), c_valid, eps, momentum, _ptr(vec, torch.float32), act, _ptr(mod),
        mod.stride(0) if mod is not None else 0, _ptr(y), y.stride(0) if y is not None else 0, _ptr(hi), _ptr(lo),
        ldp, dtype, _stream()), "cpcsv_bn_norm_act_pack")


# ------------------------------------------------------------------ frame FID (InceptionV3)
POOL_MAX, POOL_AVG = 0, 1


def resize_im2col(x, S, a, b, hi, lo, dtype=BF16):
    """x fp32 [N, 3, H, W] (any strides) -> im2col rows [N * OH * OH, ldp] of the 3x3 stride-2 pad-0 conv on the
    bilinear S x S resize of a * x + b, OH = (S - 3) // 2 + 1 (include/cpcsv.h cpcsv_resize_im2col)"""
    N, Cc, H, W = x.shape
    assert Cc == 3
    ldp = hi.shape[-1]
    OH = (S - 3) // 2 + 1
    assert hi.is_contiguous() and hi.numel() == N * OH * OH * ldp
    assert lo is None or (lo.is_contiguous() and lo.shape == hi.shape)
    sn, sc, sh, sw = x.stride()
    _lib.check(_lib.load().cpcsv_resize_im2col(
        _ptr(x, torch.float32), N, H, W, sn, sc, sh, sw, S, float(a), float(b), _ptr(hi, TORCH16[dtype]),
        _ptr(lo, TORCH16[dtype]), ldp, dtype, _stream()), "cpcsv_resize_im2col")


def pool3x3(x, mode, stride, y=None, hi=None, lo=None, dtype=BF16):
    """3x3 max (POOL_MAX) / average without the padding (POOL_AVG) pooling, stride 1 pad 1 or stride 2 pad 0, of
    x fp32 [N, H, W, C] (channels contiguous, any pixel pitches) into fp32 y and / or 16-bit hi / lo planes
    [N, Ho, Wo, C] (channel slices of wider buffers allowed)"""
    N, H, W, Cc = x.shape
    Ho = H if stride == 1 else (H - 3) // 2 + 1
    Wo = W if stride == 1 else (W - 3) // 2 + 1
    for t in (y, hi, lo):
        assert t is None or (tuple(t.shape) == (N, Ho, Wo, Cc) and t.stride(3) == 1), (None if t is None else t.shape)
    assert x.stride(3) == 1 and (lo is None or lo.stride() == hi.stride())
    ys = y.stride()[:3] if y is not None else (0, 0, 0)
    ps = hi.stride()[:3] if hi is not None else (0, 0, 0)
    _lib.check(_lib.load().cpcsv_pool3x3(
        _ptr(x, torch.float32), N, H, W, Cc, x.stride(0), x.stride(1), x.stride(2), mode, stride,
        _ptr(y, torch.float32), ys[0], ys[1], ys[2], _ptr(hi, TORCH16[dtype]), _ptr(lo, TORCH16[dtype]), ps[0],
        ps[1], ps[2], dtype, _stream()), "cpcsv_pool3x3")


# ------------------------------------------------------------------ frame SSIM
def ssim(x, y, a, b, out):
    """out fp64 [B * T] = per-frame SSIM of a * x + b against a * y + b; x, y fp32 [B, T, C, H, W] of the same shape,
    any strides (include/cpcsv.h cpcsv_ssim)"""
    B, T, Cc, H, W = x.shape
    assert tuple(y.shape) == tuple(x.shape), (x.shape, y.shape)
    assert out.is_contiguous() and out.numel() == B * T, (out.shape, B * T)
    _lib.check(_lib.load().cpcsv_ssim(
        _ptr(x, torch.float32), _ptr(y, torch.float32), B, T, Cc, H, W, *x.stride(), *y.stride(), float(a), float(b),
        _ptr(out, torch.float64), _stream()), "cpcsv_ssim")


# ------------------------------------------------------------------ layout kernels
def images_to_u8(x, out):
    """x [C, H, W] fp32 in [-1, 1] (any strides) -> out uint8 [H, W, C] (contiguous)"""
    Cc, H, W = x.shape
    assert out.dtype == torch.uint8 and out.is_contiguous() and tuple(out.shape) == (H, W, Cc)
    sc, sh, sw = x.stride()
    _lib.check(_lib.load().cpcsv_images_to_u8(_ptr(x, torch.float32), Cc, H, W, sc, sh, sw, _ptr(out), _stream()),
               "cpcsv_images_to_u8")


def pack_nchw(x, bcast, hi, lo, cpad, dtype=BF16):
    N, Cc, H, W = x.shape
    sn, sc, sh, sw = x.stride()
    cb = bcast.shape[1] if bcast is not None else 0
    ldb = bcast.stride(0) if bcast is not None else 0
    _lib.check(_lib.load().cpcsv_pack_nchw(
        _ptr(x, torch.float32), N, Cc, H, W, sn, sc, sh, sw, _ptr(bcast, torch.float32), cb, ldb,
        _ptr(hi), _ptr(lo), cpad, dtype, _stream()), "cpcsv_pack_nchw")


def im2col_small(x, k, s, p, hi, lo, ldp, dtype=BF16):
    N, Cc, H, W = x.shape
    sn, sc, sh, sw = x.stride()
    _lib.check(_lib.load().cpcsv_im2col_small(
        _ptr(x, torch.float32), N, Cc, H, W, sn, sc, sh, sw, k, s, p, _ptr(hi), _ptr(lo), ldp, dtype,
        _stream()), "cpcsv_im2col_small")


def enc0_lrelu_fwd(x, w, alpha, slope, hi, lo, ldp, dtype=BF16):
    """first discriminator layer: conv4x4 s2 p1 (raw weight w [Co, C, 4, 4]) * alpha -> LeakyReLU -> NHWC planes"""
    N, Cc, H, W = x.shape
    sn, sc, sh, sw = x.stride()
    assert w.is_contiguous() and tuple(w.shape[1:]) == (Cc, 4, 4)
    _lib.check(_lib.load().cpcsv_enc0_lrelu_fwd(
        _ptr(x, torch.float32), N, Cc, H, W, sn, sc, sh, sw, _ptr(w, torch.float32), w.shape[0],
        _ptr(alpha, torch.float32), slope, _ptr(hi), _ptr(lo), ldp, dtype, _stream()), "cpcsv_enc0_lrelu_fwd")


def lrelu_bwd16(dy, a_hi, slope, dz):
    """dz (bf16) = dy * (a_hi > 0 ? 1 : slope)"""
    assert dy.is_contiguous() and a_hi.is_contiguous() and dz.is_contiguous() and dz.dtype == torch.bfloat16
    assert dy.numel() == a_hi.numel() == dz.numel()
    _lib.check(_lib.load().cpcsv_lrelu_bwd16(_ptr(dy, torch.float32), _ptr(a_hi), dy.numel(), slope, _ptr(dz),
                                             _stream()), "cpcsv_lrelu_bwd16")


def col2im_small(dcol, N, Cc, H, W, k, s, p, dx):
    assert dx.is_contiguous()
    _lib.check(_lib.load().cpcsv_col2im_small(
        _ptr(dcol, torch.float32), dcol.stride(0), N, Cc, H, W, k, s, p, _ptr(dx, torch.float32),
        _stream()), "cpcsv_col2im_small")


def head_gather_tanh(z, N, H, W, Co, y):
    """y[n, co, h, w] = tanh(sum_{ky,kx} z[(n, h+ky-1, w+kx-1), (ky*3+kx)*Co + co]); z [N*H*W, ld] fp32"""
    assert z.dim() == 2 and z.stride(1) == 1 and z.shape[0] == N * H * W and y.is_contiguous()
    assert tuple(y.shape) == (N, Co, H, W)
    _lib.check(_lib.load().cpcsv_head_gather_tanh(_ptr(z, torch.float32), z.stride(0), N, H, W, Co,
                                                  _ptr(y, torch.float32), _stream()), "cpcsv_head_gather_tanh")


def tanh_bwd_im2col(dy, y, col, dtype=BF16):
    N, Cc, H, W = y.shape
    assert y.is_contiguous()
    sn, sc, sh, sw = dy.stride()
    _lib.check(_lib.load().cpcsv_tanh_bwd_im2col(
        _ptr(dy, torch.float32), sn, sc, sh, sw, _ptr(y, torch.float32), N, Cc, H, W, _ptr(col),
        col.stride(0), dtype, _stream()), "cpcsv_tanh_bwd_im2col")


def pack_matrix(w, rows_out, cols_out, cols_valid, ld_r, ld_c, row_map, hi, lo, dtype=BF16, col_map=None):
    _lib.check(_lib.load().cpcsv_pack_matrix(
        _ptr(w, torch.float32), rows_out, cols_out, cols_valid, ld_r, ld_c, _ptr(row_map, torch.int32),
        _ptr(col_map, torch.int32), _ptr(hi), _ptr(lo), hi.stride(0), dtype, _stream()), "cpcsv_pack_matrix")


def scatter_rows_f32(src, row_map, dst, rows, cols):
    _lib.check(_lib.load().cpcsv_scatter_rows_f32(
        _ptr(src, torch.float32), src.stride(0), _ptr(row_map, torch.int32), _ptr(dst, torch.float32),
        dst.stride(0), rows, cols, _stream()), "cpcsv_scatter_rows_f32")


def pack_conv_weight(w, kind, rows_pad, cols_pad, hi, lo, dtype=BF16):
    Cout, Cin, kh, kw = w.shape
    assert w.is_contiguous()
    _lib.check(_lib.load().cpcsv_pack_conv_weight(
        _ptr(w, torch.float32), Cout, Cin, kh, kw, kind, rows_pad, cols_pad, _ptr(hi), _ptr(lo), dtype,
        _stream()), "cpcsv_pack_conv_weight")


def unpack_conv_wgrad(dwt, mat_stride, ldc, kind, alpha, dw):
    Cout, Cin, kh, kw = dw.shape
    assert dw.is_contiguous()
    _lib.check(_lib.load().cpcsv_unpack_conv_wgrad(
        _ptr(dwt, torch.float32), mat_stride, ldc, Cout, Cin, kh, kw, kind, _ptr(alpha),
        _ptr(dw, torch.float32), _stream()), "cpcsv_unpack_conv_wgrad")


def unpack_conv_wgrad_dot(dwt, mat_stride, ldc, kind, alpha, dw, w, dot):
    """unpack_conv_wgrad (kinds 0 / 2) + dot[0] += sum(dw * w)"""
    Cout, Cin, kh, kw = dw.shape
    assert dw.is_contiguous() and w.is_contiguous() and tuple(w.shape) == tuple(dw.shape)
    _lib.check(_lib.load().cpcsv_unpack_conv_wgrad_dot(
        _ptr(dwt, torch.float32), mat_stride, ldc, Cout, Cin, kh, kw, kind, _ptr(alpha),
        _ptr(dw, torch.float32), _ptr(w, torch.float32), _ptr(dot, torch.float32), _stream()),
        "cpcsv_unpack_conv_wgrad_dot")


# ------------------------------------------------------------------ conditioning path (fp32)
def linear_f32(x, w, bias, y, accumulate=False):
    """y[M,N] = x[M,K] @ w[N,K]^T + bias."""
    M, K = x.shape
    N = w.shape[0]
    assert w.shape[1] == K and y.shape == (M, N)
    _lib.check(_lib.load().cpcsv_linear_f32(
        _ptr(x, torch.float32), x.stride(0), _ptr(w, torch.float32), w.stride(0), _ptr(bias),
        _ptr(y, torch.float32), y.stride(0), M, N, K, int(accumulate), _stream()), "cpcsv_linear_f32")


def linear_tn_f32(a, b, y, accumulate=False):
    """y[M,N] = a[K,M]^T @ b[K,N]."""
    K, M = a.shape
    N = b.shape[1]
    assert b.shape[0] == K and y.shape == (M, N)
    _lib.check(_lib.load().cpcsv_linear_tn_f32(
        _ptr(a, torch.float32), a.stride(0), _ptr(b, torch.float32), b.stride(0),
        _ptr(y, torch.float32), y.stride(0), M, N, K, int(accumulate), _stream()), "cpcsv_linear_tn_f32")


def linear_nn_f32(x, w, y, accumulate=False):
    """y[M,N] = x[M,K] @ w[K,N]."""
    M, K = x.shape
    N = w.shape[1]
    assert w.shape[0] == K and y.shape == (M, N)
    _lib.check(_lib.load().cpcsv_linear_nn_f32(
        _ptr(x, torch.float32), x.stride(0), _ptr(w, torch.float32), w.stride(0),
        _ptr(y, torch.float32), y.stride(0), M, N, K, int(accumulate), _stream()), "cpcsv_linear_nn_f32")


def gru_gates_fwd(gi, gh, h, hnew, save):
    B, H = h.shape
    _lib.check(_lib.load().cpcsv_gru_gates_fwd(_ptr(gi), _ptr(gh), _ptr(h), B, H, _ptr(hnew), _ptr(save),
                                               _stream()), "cpcsv_gru_gates_fwd")


def gru_gates_bwd(dhnew, h, save, dgi, dgh, dh):
    B, H = h.shape
    _lib.check(_lib.load().cpcsv_gru_gates_bwd(_ptr(dhnew), _ptr(h), _ptr(save), B, H, _ptr(dgi),
                                               _ptr(dgh), _ptr(dh), _stream()), "cpcsv_gru_gates_bwd")


def ca_fwd(pre, eps, mu, logvar, code):
    B, Cc = mu.shape
    _lib.check(_lib.load().cpcsv_ca_fwd(_ptr(pre), _ptr(eps), B, Cc, _ptr(mu), _ptr(logvar), _ptr(code),
                                        _stream()), "cpcsv_ca_fwd")


def ca_bwd(pre, eps, dmu, dlogvar, dcode, dpre):
    B, Cc = eps.shape
    _lib.check(_lib.load().cpcsv_ca_bwd(_ptr(pre), _ptr(eps), _ptr(dmu), _ptr(dlogvar), _ptr(dcode), B, Cc,
                                        _ptr(dpre), _stream()), "cpcsv_ca_bwd")


def dfn1d_fwd(img, filt, out):
    N, Cc, L = img.shape
    K = filt.shape[-1]
    _lib.check(_lib.load().cpcsv_dfn1d_fwd(_ptr(img), _ptr(filt), N, Cc, L, K, _ptr(out), _stream()),
               "cpcsv_dfn1d_fwd")


def dfn1d_bwd(img, filt, dout, dimg, dfilt):
    N, Cc, L = img.shape
    K = filt.shape[-1]
    _lib.check(_lib.load().cpcsv_dfn1d_bwd(_ptr(img), _ptr(filt), _ptr(dout), N, Cc, L, K, _ptr(dimg),
                                           _ptr(dfilt), _stream()), "cpcsv_dfn1d_bwd")


def tanh_fwd(x, y):
    _lib.check(_lib.load().cpcsv_tanh_fwd(_ptr(x), _ptr(y), x.numel(), _stream()), "cpcsv_tanh_fwd")


def tanh_bwd(y, dy, dx):
    _lib.check(_lib.load().cpcsv_tanh_bwd(_ptr(y), _ptr(dy), _ptr(dx), y.numel(), _stream()),
               "cpcsv_tanh_bwd")


def affine_sigmoid_fwd(t, alpha, bias, out):
    _lib.check(_lib.load().cpcsv_affine_sigmoid_fwd(_ptr(t), _ptr(alpha), _ptr(bias), _ptr(out), t.numel(),
                                                    _stream()), "cpcsv_affine_sigmoid_fwd")


def affine_sigmoid_bwd(dout, out, alpha, dt, dz):
    _lib.check(_lib.load().cpcsv_affine_sigmoid_bwd(_ptr(dout), _ptr(out), _ptr(alpha), _ptr(dt), _ptr(dz),
                                                    out.numel(), _stream()), "cpcsv_affine_sigmoid_bwd")


# ------------------------------------------------------------------ spectral norm
def spectral_sigma(w2d, u, v, power_iteration, sigma, inv_sigma, scratch, eps=1e-12):
    R, Cc = w2d.shape
    assert w2d.is_contiguous() and scratch.numel() >= R + Cc
    _lib.check(_lib.load().cpcsv_spectral_sigma(
        _ptr(w2d, torch.float32), R, Cc, _ptr(u), _ptr(v), int(power_iteration), eps, _ptr(sigma),
        _ptr(inv_sigma), _ptr(scratch), _stream()), "cpcsv_spectral_sigma")


def spectral_bwd(g2d, w2d, u, v, sigma, dw2d, scratch):
    R, Cc = w2d.shape
    assert g2d.is_contiguous() and w2d.is_contiguous() and dw2d.is_contiguous()
    _lib.check(_lib.load().cpcsv_spectral_bwd(
        _ptr(g2d, torch.float32), _ptr(w2d, torch.float32), _ptr(u), _ptr(v), _ptr(sigma), R, Cc,
        _ptr(dw2d, torch.float32), _ptr(scratch), _stream()), "cpcsv_spectral_bwd")


# ------------------------------------------------------------------ optimiser (Adam fused with the re-layout)
class AdamHyper:
    """device-resident hyper-parameters of one optimiser: lr [1], bc [2] (bias corrections written
    by ``adam_tick``), and the host constants"""

    def __init__(self, lr, bc, beta1, beta2, eps):
        self.lr, self.bc, self.beta1, self.beta2, self.eps = lr, bc, float(beta1), float(beta2), float(eps)

    def to_c(self):
        h = _lib.AdamHyper()
        h.lr, h.bc = _ptr(self.lr, torch.float32).value, _ptr(self.bc, torch.float32).value
        h.beta1, h.beta2, h.eps = self.beta1, self.beta2, self.eps
        return h


def adam_tick(step, beta1, beta2, bc):
    """step += 1; bc = [1 / (1 - beta1^step), 1 / sqrt(1 - beta2^step)]"""
    _lib.check(_lib.load().cpcsv_adam_tick(_ptr(step, torch.float32), beta1, beta2, _ptr(bc, torch.float32),
                                           _stream()), "cpcsv_adam_tick")


def adam_multi(tensors, hyper):
    """Adam step on a list of (p, g, m, v) fp32 tensors (contiguous, same numel each)"""
    n = len(tensors)
    if n == 0:
        return
    arr = (_lib.AdamTensor * n)()
    for i, (p, g, m, v) in enumerate(tensors):
        assert p.is_contiguous() and g.is_contiguous() and m.is_contiguous() and v.is_contiguous()
        assert g.numel() == p.numel() == m.numel() == v.numel()
        arr[i].p, arr[i].g = _ptr(p, torch.float32).value, _ptr(g, torch.float32).value
        arr[i].m, arr[i].v = _ptr(m, torch.float32).value, _ptr(v, torch.float32).value
        arr[i].n = p.numel()
    h = hyper.to_c()
    _lib.check(_lib.load().cpcsv_adam_multi(arr, n, C.byref(h), _stream()), "cpcsv_adam_multi")


def adam_pack_conv(w, g, m, v, planes, hyper=None):
    """[Adam step on the conv weight w [Cout, Cin, kh, kw] (g None: no step), then] every plane of
    ``planes`` = [(kind, dtype, rows_pad, cols_pad, hi, lo-or-None)] rewritten from w"""
    Cout, Cin, kh, kw = w.shape
    assert w.is_contiguous() and (g is None or g.is_contiguous())
    n = len(planes)
    arr = (_lib.Plane * max(n, 1))()
    for i, (kind, dtype, rows_pad, cols_pad, hi, lo) in enumerate(planes):
        arr[i].kind, arr[i].dtype, arr[i].rows_pad, arr[i].cols_pad = kind, dtype, rows_pad, cols_pad
        arr[i].hi, arr[i].lo = _ptr(hi, TORCH16[dtype]).value, (_ptr(lo, TORCH16[dtype]).value if lo is not None else None)
    h = hyper.to_c() if g is not None else None
    _lib.check(_lib.load().cpcsv_adam_pack_conv(
        _ptr(w, torch.float32), _ptr(g, torch.float32), _ptr(m, torch.float32), _ptr(v, torch.float32), Cout, Cin,
        kh, kw, C.byref(h) if h is not None else None, arr, n, _stream()), "cpcsv_adam_pack_conv")


def adam_pack_fc(w, g, m, v, C_, P, Cp, Kp, fwd16=None, fwd_hi=None, fwd_lo=None, bwd=None, hyper=None):
    """fc / fc_seg weight w [C*P, K]: [Adam step, then] the NHWC-ordered planes fwd16 fp16 [P*Cp, Kp],
    fwd_hi / fwd_lo bf16 [P*Cp, Kp], bwd bf16 [Kp, P*Cp]"""
    rows, K = w.shape
    assert rows == C_ * P and w.is_contiguous() and (g is None or g.is_contiguous())
    for t, shape in ((fwd16, (P * Cp, Kp)), (fwd_hi, (P * Cp, Kp)), (fwd_lo, (P * Cp, Kp)), (bwd, (Kp, P * Cp))):
        assert t is None or (tuple(t.shape) == shape and t.is_contiguous()), (shape, None if t is None else t.shape)
    h = hyper.to_c() if g is not None else None
    _lib.check(_lib.load().cpcsv_adam_pack_fc(
        _ptr(w, torch.float32), _ptr(g, torch.float32), _ptr(m, torch.float32), _ptr(v, torch.float32), C_, K, P,
        Cp, Kp, C.byref(h) if h is not None else None, _ptr(fwd16, torch.float16), _ptr(fwd_hi, torch.bfloat16),
        _ptr(fwd_lo, torch.bfloat16), _ptr(bwd, torch.bfloat16), _stream()), "cpcsv_adam_pack_fc")


def spectral_bwd_apply(g2d, u, v, sigma, dot, dw2d):
    """dW = (G - (dot / sigma) u v^T) / sigma with dot = sum(G * W) given; dw2d may be g2d"""
    R, Cc = g2d.shape
    assert g2d.is_contiguous() and dw2d.is_contiguous()
    _lib.check(_lib.load().cpcsv_spectral_bwd_apply(
        _ptr(g2d, torch.float32), _ptr(u), _ptr(v), _ptr(sigma), _ptr(dot, torch.float32), R, Cc,
        _ptr(dw2d, torch.float32), _stream()), "cpcsv_spectral_bwd_apply")
