"""Builders of tcgen05 GEMM jobs (``ops.GemmJob``) for every convolution on the path.

Pure index arithmetic: which TMA coordinates each filter tap reads, which weight rows it
multiplies, where each sub-pixel phase lands in the output.  No tensor math happens here.

Notation: activations are NHWC 16-bit planes ``[N, H, W, C]`` (C a multiple of 64), conv
outputs are fp32 ``[N, H, W, Cpad]``.  ``delta_t = (ky - pad, kx - pad)``.

Sub-pixel identity used for upBlock (nearest x2 then conv3x3, reference model.py:26-34;
SURVEY.md Appendix A): output pixel (2y+a, 2x+b) is a 2x2 conv of the LOW-RES input with
taps (i, j) at offsets (i-1+a, j-1+b) and merged weights -- 16 instead of 36 MACs per
low-res pixel and the up-sampled tensor is never materialised.
"""
from .ops import GemmJob, View, BF16

NUM_SMS = 148


def pixel_tile(N, H, W, rows):
    """Box (tile_n, tile_h, tile_w) of `rows` pixels.  W is a power of two; H usually is -- for any other H (an odd
    number of frames of the temporal convolutions) the box height is the next power of two: the kernel masks rows
    outside the grid and TMA zero-fills their loads.  A grid this rule cannot tile (a W that is no power of two,
    the 147 / 73 / 35 / 17 grids of InceptionV3) gets the box with the fewest masked rows (_min_waste_tile)."""
    tw = min(W, rows)
    th = 1
    while th < H and th * 2 <= rows // tw:
        th *= 2
    tn = rows // (tw * th)
    if tn * th * tw != rows:
        return _min_waste_tile(N, H, W, rows)
    return tn, th, tw


def _min_waste_tile(N, H, W, rows):
    """the power-of-two box of `rows` pixels whose tiles cover the (N, H, W) grid with the fewest masked rows; ties
    go to the wider, then the taller box.  Any such box is legal: every pixel row of the A tile is one 128-B
    channel segment whatever the box shape, and the epilogue masks rows outside the grid."""
    best = None
    tw = 1
    while tw <= rows:
        th = 1
        while tw * th <= rows:
            tn = rows // (tw * th)
            cover = -(-N // tn) * tn * (-(-H // th) * th) * (-(-W // tw) * tw)
            key = (cover, -tw, -th)
            if best is None or key < best[0]:
                best = (key, (tn, th, tw))
            th *= 2
        tw *= 2
    return best[1]


def pick_block_n(npad):
    assert npad % 16 == 0
    for bn in (256, 128, 64, 32, 16):
        if npad % bn == 0:
            return bn
    raise AssertionError(npad)


def pick_splits(tiles, iters, penalty=0.04):
    """Split-K factor that fills the last wave of the persistent grid: with `tiles` work items on
    148 SMs the efficiency is tiles / (ceil(tiles / 148) * 148); splitting the reduction s ways
    multiplies the tile count.  Each extra split costs a red.add pass over the output, so a
    split is only taken when it buys > 4 % per step of s."""
    if iters < 8:
        return 1
    if tiles * 8 < NUM_SMS:
        # a handful of output tiles with a very long reduction (first-layer / head weight gradients,
        # K = all pixels; the 16-tap weight gradients of the 64x64 layers): as many splits as fill ONE wave
        # (rounding up gave 160 work items on 148 SMs, i.e. a second wave with 12 of them: 0.54 wave efficiency,
        # profiles/r01_gemm_bounds_single.txt)
        return max(1, min(NUM_SMS // tiles, iters // 4))
    best, best_score = 1, -1.0
    for s in range(1, min(8, iters // 4) + 1):
        n = tiles * s
        eff = n / (-(-n // NUM_SMS) * NUM_SMS)
        score = eff - penalty * (s - 1)
        if score > best_score + 1e-9:
            best, best_score = s, score
    return best


def use_pair(grid, tile, block_n):
    """Run a fprop / dgrad job as cta_group::2 pairs?  Measured on B200 at every job shape of the
    step (tools/sweep_pair.py, profiles/r01_sweep_pair.txt: median of 9, L2 flushed): 0.79-0.87x the
    time with hi/lo split operands, 0.91-1.00x single-plane, never slower -- so whenever there are
    two 128-row tiles to pair and the B tile can be halved."""
    return _m_tiles(grid, tile) >= 2 and block_n >= 32 and (block_n // 2) % 8 == 0


def _m_tiles(grid, tile):
    n = 1
    for g, t in zip(grid, tile):
        n *= -(-g // t)
    return n


def _fwd_job(a_planes, b_planes, grid, groups, taps_per_group, taps, k_blocks, out, npad,
             out_strides, alpha=None, accumulate=False, dtype=BF16, splits=None, n_valid=None):
    """`npad`: weight rows per tap (the N extent of the GEMM); `n_valid`: output columns stored (default npad), less
    when the output is a channel slice of a wider buffer"""
    tile = pixel_tile(*grid, 128)
    block_n = pick_block_n(npad)
    n_tiles = npad // block_n
    if n_valid is None:
        n_valid = npad
    assert n_valid <= npad, (n_valid, npad)
    if splits is None:
        splits = pick_splits(groups * _m_tiles(grid, tile) * n_tiles, taps_per_group * k_blocks)
    return GemmJob(mode=0, planes=len(a_planes), grid=grid, tile=tile, groups=groups,
                   taps_per_group=taps_per_group, k_blocks=k_blocks, taps=taps, a=a_planes,
                   b=b_planes, out=out, n_valid=n_valid, block_n=block_n, n_tiles=n_tiles,
                   splits=splits, accumulate=accumulate, out_strides=out_strides, alpha=alpha,
                   dtype=dtype, pair=use_pair(grid, tile, block_n))


def _wgrad_job(a_view, b_view, grid, taps, m_valid, npad, out, ldc, dtype=BF16, splits=None, accumulate=False):
    tile = pixel_tile(*grid, 64)
    block_n = 256 if npad % 256 == 0 else (128 if npad % 128 == 0 else 64)
    assert npad % 64 == 0
    n_tiles = npad // block_n
    iters = _m_tiles(grid, tile)
    if splits is None:
        splits = pick_splits(len(taps) * (-(-m_valid // 128)) * n_tiles, iters, penalty=0.10)
    return GemmJob(mode=1, planes=1, grid=grid, tile=tile, groups=len(taps), taps_per_group=1,
                   k_blocks=0, taps=taps, a=[a_view], b=[b_view], out=out, n_valid=npad,
                   block_n=block_n, n_tiles=n_tiles, m_valid=m_valid, splits=splits, ldc=ldc,
                   dtype=dtype, accumulate=accumulate,
                   # cta_group::2 pairs (two 128-channel M tiles share the x tile): the single-CTA kernel is bound by
                   # the L2 -> SM feed at 42 % tensor-pipe activity (profiles/r02_stress512_tensor_pipe_table.txt)
                   pair=m_valid > 128 and block_n % 128 == 0)


def _planes(ts, fn):
    return [fn(t) for t in ts if t is not None]


def _plain_out_strides(out):
    """element strides of an [N, H, W, C] output (C contiguous); `out` may be a strided view, e.g. every second
    frame of a [B, T, HW, C] tensor"""
    assert out.stride(3) == 1
    return (out.stride(0), out.stride(1), out.stride(2))


# ------------------------------------------------------------------ k x k, stride 1
def conv_s1_fwd(x_planes, w_planes, out, k=3, alpha=None, dtype=BF16, splits=None):
    """out[N,H,W,Co] = conv(x[N,H,W,Ci], w), stride 1, pad k//2.  w_planes: packed kind 0
    ``[k*k * Co_pad, Ci]``.  ``splits``: split-K factor (None: pick_splits)."""
    N, H, W, Ci = x_planes[0].shape
    npad = out.shape[-1]
    pad = k // 2
    taps = [((0, kx - pad, 0, ky - pad), ((ky * k + kx) * npad, 0, 0, 0), 0)
            for ky in range(k) for kx in range(k)]
    return _fwd_job(_planes(x_planes, View.nhwc), _planes(w_planes, View.matrix), (N, H, W), 1,
                    k * k, taps, Ci // 64, out, npad, _plain_out_strides(out), alpha, dtype=dtype, splits=splits)


def conv_s1_dgrad(dy, wt, dx, k=3, alpha=None, accumulate=False):
    """dx[N,H,W,Ci] (+)= sum_t dy[p - delta_t] W_t^T.  wt: packed kind 1 ``[k*k * Ci_pad, Co]``."""
    N, H, W, Co = dy.shape
    npad = dx.shape[-1]
    pad = k // 2
    taps = [((0, -(kx - pad), 0, -(ky - pad)), ((ky * k + kx) * npad, 0, 0, 0), 0)
            for ky in range(k) for kx in range(k)]
    return _fwd_job([View.nhwc(dy)], [View.matrix(wt)], (N, H, W), 1, k * k, taps, Co // 64, dx, npad,
                    _plain_out_strides(dx), alpha, accumulate)


def conv_s1_wgrad(dy, x_hi, dwt, k=3):
    """dwt[t][co][ci] = sum_p dy[p, co] x[p + delta_t, ci]  (fp32 ``[k*k, Co, Ci]``)."""
    N, H, W, Co = dy.shape
    Ci = x_hi.shape[-1]
    pad = k // 2
    taps = [((0, 0, 0, 0), (0, kx - pad, 0, ky - pad), (ky * k + kx) * Co * Ci)
            for ky in range(k) for kx in range(k)]
    return _wgrad_job(View.nhwc(dy), View.nhwc(x_hi), (N, H, W), taps, Co, Ci, dwt, Ci)


# ------------------------------------------------------------------ nearest x2 + 3x3 (upBlock)
def _sub_taps():
    """(a, b, i, j, oy, ox) for the 16 merged taps, in packing order."""
    return [(a, b, i, j, i - 1 + a, j - 1 + b)
            for a in range(2) for b in range(2) for i in range(2) for j in range(2)]


def upconv_fwd(x_planes, wm_planes, out, dtype=BF16):
    """out[N,2H,2W,Co] = conv3x3(nearest_x2(x)).  wm_planes: packed kind 2 ``[16 * Co_pad, Ci]``."""
    N, H, W, Ci = x_planes[0].shape
    npad = out.shape[-1]
    assert out.shape[1] == 2 * H and out.shape[2] == 2 * W
    taps = []
    for t, (a, b, i, j, oy, ox) in enumerate(_sub_taps()):
        taps.append(((0, ox, 0, oy), (t * npad, 0, 0, 0), (a * 2 * W + b) * npad))
    strides = (4 * H * W * npad, 4 * W * npad, 2 * npad)
    return _fwd_job(_planes(x_planes, View.nhwc), _planes(wm_planes, View.matrix), (N, H, W), 4, 4,
                    taps, Ci // 64, out, npad, strides, dtype=dtype)


def upconv_dgrad(dz, wmt, dx, accumulate=False):
    """dx[N,H,W,Ci] = sum_{a,b,i,j} dz[2(p - o) + (a,b)] Wm^T.  dz: [N,2H,2W,Co] bf16;
    wmt: packed kind 3 ``[16 * Ci_pad, Co]``."""
    N, H2, W2, Co = dz.shape
    npad = dx.shape[-1]
    taps = [((b * Co, -ox, a, -oy), (t * npad, 0, 0, 0), 0)
            for t, (a, b, i, j, oy, ox) in enumerate(_sub_taps())]
    return _fwd_job([View.nhwc_parity(dz)], [View.matrix(wmt)], (N, H2 // 2, W2 // 2), 1, 16, taps,
                    Co // 64, dx, npad, _plain_out_strides(dx), None, accumulate)


def upconv_wgrad(dz, x_hi, dwt):
    """dwt[(a,b,i,j)][co][ci] = sum_q dz[2q + (a,b), co] x[q + o, ci]."""
    N, H2, W2, Co = dz.shape
    Ci = x_hi.shape[-1]
    taps = [((b * Co, 0, a, 0), (0, ox, 0, oy), t * Co * Ci)
            for t, (a, b, i, j, oy, ox) in enumerate(_sub_taps())]
    return _wgrad_job(View.nhwc_parity(dz), View.nhwc(x_hi), (N, H2 // 2, W2 // 2), taps, Co, Ci, dwt, Ci)


# ------------------------------------------------------------------ 4x4, stride 2, pad 1
def _s2_split(kk):
    """kernel index -> (parity, block offset) of input coordinate 2*o + kk - 1."""
    d = kk - 1
    return d % 2, d // 2


def conv_s2_fwd(x_planes, w_planes, out, alpha=None, dtype=BF16, splits=None):
    """out[N,H/2,W/2,Co] = conv4x4 s2 p1 (x[N,H,W,Ci]).  w_planes: kind 0 ``[16 * Co_pad, Ci]``."""
    N, H, W, Ci = x_planes[0].shape
    npad = out.shape[-1]
    taps = []
    for ky in range(4):
        hp, dh = _s2_split(ky)
        for kx in range(4):
            wp, dw = _s2_split(kx)
            taps.append(((wp * Ci, dw, hp, dh), ((ky * 4 + kx) * npad, 0, 0, 0), 0))
    return _fwd_job(_planes(x_planes, View.nhwc_parity), _planes(w_planes, View.matrix),
                    (N, H // 2, W // 2), 1, 16, taps, Ci // 64, out, npad, _plain_out_strides(out),
                    alpha, dtype=dtype, splits=splits)


def conv_s2_dgrad(dy, wt, dx, alpha=None):
    """dx[N,H,W,Ci] = transposed conv of dy[N,H/2,W/2,Co]: 4 output parities x 2x2 taps.
    wt: packed kind 1 ``[16 * Ci_pad, Co]``."""
    N, Ho, Wo, Co = dy.shape
    npad = dx.shape[-1]
    W = 2 * Wo

    def par_taps(par):      # kernel indices contributing to output parity `par` and their shift
        return [(1, 0), (3, -1)] if par == 0 else [(0, 1), (2, 0)]

    taps = []
    for a in range(2):
        for b in range(2):
            for ky, dh in par_taps(a):
                for kx, dw in par_taps(b):
                    taps.append(((0, dw, 0, dh), ((ky * 4 + kx) * npad, 0, 0, 0), (a * W + b) * npad))
    strides = (4 * Ho * Wo * npad, 2 * W * npad, 2 * npad)
    return _fwd_job([View.nhwc(dy)], [View.matrix(wt)], (N, Ho, Wo), 4, 4, taps, Co // 64, dx, npad,
                    strides, alpha)


def conv_s2_wgrad(dy, x_hi, dwt):
    """dwt[t][co][ci] = sum_q dy[q, co] x[2q + delta_t, ci]."""
    N, Ho, Wo, Co = dy.shape
    Ci = x_hi.shape[-1]
    taps = []
    for ky in range(4):
        hp, dh = _s2_split(ky)
        for kx in range(4):
            wp, dw = _s2_split(kx)
            taps.append(((0, 0, 0, 0), (wp * Ci, dw, hp, dh), (ky * 4 + kx) * Co * Ci))
    return _wgrad_job(View.nhwc(dy), View.nhwc_parity(x_hi), (N, Ho, Wo), taps, Co, Ci, dwt, Ci)


# ------------------------------------------------------------------ plain GEMMs (Linear, im2col'd convs)
def _rows_as_nhwc(t):
    return t.view(t.shape[0], 1, 1, t.shape[1])


def gemm_nt(a_planes, b_planes, out, alpha=None, accumulate=False, dtype=BF16, splits=None):
    """out[M, Npad] = a[M, K] @ b[Npad, K]^T  (K multiple of 64)."""
    M, K = a_planes[0].shape
    npad = out.shape[-1]
    assert b_planes[0].shape == (npad, K), (b_planes[0].shape, npad, K)
    taps = [((0, 0, 0, 0), (0, 0, 0, 0), 0)]
    av = [View.nhwc(_rows_as_nhwc(t)) for t in a_planes if t is not None]
    return _fwd_job(av, _planes(b_planes, View.matrix), (M, 1, 1), 1, 1, taps, K // 64, out, npad,
                    (out.stride(0), 0, 0), alpha, accumulate, dtype=dtype, splits=splits)


def gemm_tn(a, b, out):
    """out[Ma, Nb] = a[R, Ma]^T @ b[R, Nb]  (reduction over rows; operands MN-major)."""
    R, Ma = a.shape
    Nb = b.shape[1]
    taps = [((0, 0, 0, 0), (0, 0, 0, 0), 0)]
    return _wgrad_job(View.nhwc(_rows_as_nhwc(a)), View.nhwc(_rows_as_nhwc(b)), (R, 1, 1), taps, Ma, Nb,
                      out, out.stride(0))


# ------------------------------------------------------------------ temporal 3-tap, stride 2, pad 1
# Conv3d(kernel (3, 1, 1), stride (2, 1, 1), padding (1, 0, 0)) of the order-consistency critic (reference
# model.py:160-189).  Activations are [B, T, HW, C] (NHWC with H = T, W = H*W of the frame); output frame t_out
# reads input frames 2*t_out + kt - 1.  The EVEN input frames (kt = 1) and the ODD ones (kt = 0, 2) are two
# strided views x[:, 0::2] / x[:, 1::2] of the same buffer, so a tap is a plain coordinate offset and TMA's
# zero fill outside a view is exactly the temporal zero padding, for odd and even T alike.
def _even_odd(t5):
    return t5[:, 0::2], t5[:, 1::2]


def conv_t3_fwd(x_planes, w_planes, out, alpha=None, dtype=BF16):
    """out[B, T_out, HW, Co] = temporal conv of x[B, T, HW, Ci]; w_planes: packed kind 0 ``[3 * Co_pad, Ci]``
    (tap kt at rows [kt * Co_pad, ...)).  Two jobs: even frames (overwrite), odd frames (accumulate)."""
    B, T, HW, Ci = x_planes[0].shape
    To, npad = out.shape[1], out.shape[-1]
    assert To == (T - 1) // 2 + 1
    ev = [_even_odd(t)[0] for t in x_planes if t is not None]
    od = [_even_odd(t)[1] for t in x_planes if t is not None]
    wv = _planes(w_planes, View.matrix)
    jobs = [_fwd_job([View.nhwc(t) for t in ev], wv, (B, To, HW), 1, 1, [((0, 0, 0, 0), (1 * npad, 0, 0, 0), 0)],
                     Ci // 64, out, npad, _plain_out_strides(out), alpha, False, dtype=dtype, splits=1)]
    if T > 1:
        taps = [((0, 0, 0, -1), (0 * npad, 0, 0, 0), 0), ((0, 0, 0, 0), (2 * npad, 0, 0, 0), 0)]
        jobs.append(_fwd_job([View.nhwc(t) for t in od], wv, (B, To, HW), 1, 2, taps, Ci // 64, out, npad,
                             _plain_out_strides(out), alpha, True, dtype=dtype, splits=1))
    return jobs


def conv_t3s1_fwd(x_planes, w_planes, out, alpha=None, dtype=BF16, splits=None):
    """Conv3d (3, 1, 1) stride 1 pad (1, 0, 0) of R(2+1)D-18 (torchvision Conv2Plus1D / R2Plus1dStem, the
    reference's fid/residual2p1.py): out[B, T, HW, Co] = sum_kt x[B, t + kt - 1, HW, Ci] W_kt.  One job, three
    taps; the zero fill of frames -1 and T is the temporal padding.  w_planes: kind 0 ``[3 * Co_pad, Ci]``."""
    B, T, HW, Ci = x_planes[0].shape
    npad = out.shape[-1]
    assert tuple(out.shape[:3]) == (B, T, HW)
    taps = [((0, 0, 0, kt - 1), (kt * npad, 0, 0, 0), 0) for kt in range(3)]
    return _fwd_job(_planes(x_planes, View.nhwc), _planes(w_planes, View.matrix), (B, T, HW), 1, 3, taps,
                    Ci // 64, out, npad, _plain_out_strides(out), alpha, dtype=dtype, splits=splits)


def conv_p2_fwd(x_planes, w_planes, out, dtype=BF16, splits=None):
    """Conv3d (1, 1, 1) stride (2, 2, 2) (the projected shortcut of a downsampling R(2+1)D-18 block):
    out[B, To, H/2, W/2, Co] = x[B, 2 t, 2 y, 2 x, Ci] W, To = (T - 1) // 2 + 1.  The even frames of a [B, T, H,
    W, C] tensor are no single uniform-stride batch dimension when B > 1, but ONE frame x[:, 2 t] is (batch stride
    T*H*W*C, pixel pitch C): one single-tap parity-view job per output frame.  w_planes: kind 0 ``[Co_pad, Ci]``."""
    B, T, H, W, Ci = x_planes[0].shape
    To, npad = out.shape[1], out.shape[-1]
    assert To == (T - 1) // 2 + 1 and tuple(out.shape[2:4]) == (H // 2, W // 2)
    wv = _planes(w_planes, View.matrix)
    taps = [((0, 0, 0, 0), (0, 0, 0, 0), 0)]
    return [_fwd_job([View.nhwc_parity(p[:, 2 * t]) for p in x_planes if p is not None], wv, (B, H // 2, W // 2),
                     1, 1, taps, Ci // 64, out[:, t], npad, _plain_out_strides(out[:, t]), dtype=dtype,
                     splits=splits)
            for t in range(To)]


def conv_t3_dgrad(dy, wt, dx, alpha=None):
    """dx[B, T, HW, Ci] = transposed temporal conv of dy[B, T_out, HW, Co]; wt: packed kind 1
    ``[3 * Ci_pad, Co]``.  Even input frames receive tap 1, odd ones taps 0 (from t_out = hh + 1) and 2 (hh)."""
    B, To, HW, Co = dy.shape
    T, npad = dx.shape[1], dx.shape[-1]
    dxe, dxo = _even_odd(dx)
    jobs = [_fwd_job([View.nhwc(dy)], [View.matrix(wt)], (B, dxe.shape[1], HW), 1, 1,
                     [((0, 0, 0, 0), (1 * npad, 0, 0, 0), 0)], Co // 64, dxe, npad, _plain_out_strides(dxe), alpha,
                     splits=1)]
    if T > 1:
        taps = [((0, 0, 0, 1), (0 * npad, 0, 0, 0), 0), ((0, 0, 0, 0), (2 * npad, 0, 0, 0), 0)]
        jobs.append(_fwd_job([View.nhwc(dy)], [View.matrix(wt)], (B, dxo.shape[1], HW), 1, 2, taps, Co // 64, dxo,
                             npad, _plain_out_strides(dxo), alpha, splits=1))
    return jobs


def conv_t3_wgrad(dy, x_hi, dwt):
    """dwt[kt][co][ci] += sum dy[b, t_out, p, co] * x[b, 2 t_out + kt - 1, p, ci]  (fp32 ``[3, Co, Ci]``, ZEROED by
    the caller: the two jobs share the tensor, so neither may clear it for its split-K partial sums)"""
    B, To, HW, Co = dy.shape
    T, Ci = x_hi.shape[1], x_hi.shape[-1]
    xe, xo = _even_odd(x_hi)
    jobs = [_wgrad_job(View.nhwc(dy), View.nhwc(xe), (B, To, HW), [((0, 0, 0, 0), (0, 0, 0, 0), 1 * Co * Ci)],
                       Co, Ci, dwt, Ci, accumulate=True)]
    if T > 1:
        taps = [((0, 0, 0, 0), (0, 0, 0, -1), 0 * Co * Ci), ((0, 0, 0, 0), (0, 0, 0, 0), 2 * Co * Ci)]
        jobs.append(_wgrad_job(View.nhwc(dy), View.nhwc(xo), (B, To, HW), taps, Co, Ci, dwt, Ci, accumulate=True))
    return jobs


# ------------------------------------------------------------------ InceptionV3 geometries (frame FID)
def conv_kxl_fwd(x_planes, w_planes, out, kh, kw, ph, pw, dtype=BF16, splits=None):
    """out[N, Ho, Wo, :n] = conv(x[N, H, W, Ci], w), stride 1, kernel kh x kw, padding (ph, pw): Ho = H + 2 ph - kh + 1
    (smaller than H for an unpadded 3x3).  Tap (ky, kx) reads x[h + ky - ph, w + kx - pw]; TMA's zero fill outside
    the view is the padding.  w_planes: packed kind 0 ``[kh*kw * Co_pad, Ci]`` (tap ky*kw + kx at rows
    [tap * Co_pad, ...)).  ``out`` may be a channel slice ``buf[..., c0:c0 + n]`` of a wider fp32 buffer (c0 and
    the pitches multiples of 4): n <= Co_pad columns are stored.  More than CPCSV_MAX_TAPS = 16 taps (5x5) run as
    two jobs on the same output: the first 16 taps overwrite, the rest add with one red.add per element
    (``splits`` 1 for both), so the result stays bit-reproducible.  Returns the list of jobs."""
    N, H, W, Ci = x_planes[0].shape
    Ho, Wo = H + 2 * ph - kh + 1, W + 2 * pw - kw + 1
    assert tuple(out.shape[:3]) == (N, Ho, Wo), (tuple(out.shape), (N, Ho, Wo))
    ntap = kh * kw
    npad = w_planes[0].shape[0] // ntap
    assert npad * ntap == w_planes[0].shape[0] and npad % 64 == 0
    taps = [((0, kx - pw, 0, ky - ph), ((ky * kw + kx) * npad, 0, 0, 0), 0) for ky in range(kh) for kx in range(kw)]
    chunks = [taps[i:i + 16] for i in range(0, ntap, 16)]
    if len(chunks) > 1:
        splits = 1
    av, bv = _planes(x_planes, View.nhwc), _planes(w_planes, View.matrix)
    return [_fwd_job(av, bv, (N, Ho, Wo), 1, len(ch), ch, Ci // 64, out, npad, _plain_out_strides(out),
                     accumulate=i > 0, dtype=dtype, splits=splits, n_valid=out.shape[-1])
            for i, ch in enumerate(chunks)]


def conv_s2v_fwd(x_planes, w_planes, out, dtype=BF16, splits=None):
    """out[N, So, So, :n] = conv3x3 stride 2 pad 0 (x), So = (S - 3) // 2 + 1, as one 9-tap job on the parity view:
    tap k of a row / column reads parity k % 2 at block offset k // 2 (input index 2 o + k).

    Layout of an odd-sized input (S = 35, 17): ``x_planes`` are the WHOLE buffers ``[N, S + 1, S + 1, Ci]``, one
    extra row and column that a valid output never reads (its largest index is 2 (So - 1) + 2 = S - 1), so
    ``View.nhwc_parity`` applies to them; stride-1 consumers of the same activation read the ``[:, :S, :S]``
    slice, whose view dims are S, so TMA zero-fills exactly the padding.  Rows of the pixel box beyond the output
    grid may read the extra row / column; the kernel masks them.  Even S needs no extra row.
    w_planes: kind 0 ``[9 * Co_pad, Ci]``; ``out`` may be a channel slice as in conv_kxl_fwd."""
    N, P, P2, Ci = x_planes[0].shape
    So = out.shape[1]
    assert P == P2 and P % 2 == 0 and out.shape[2] == So and 2 * So + 1 <= P, (tuple(x_planes[0].shape), So)
    npad = w_planes[0].shape[0] // 9
    assert npad * 9 == w_planes[0].shape[0] and npad % 64 == 0
    taps = []
    for ky in range(3):
        for kx in range(3):
            taps.append((((kx % 2) * Ci, kx // 2, ky % 2, ky // 2), ((ky * 3 + kx) * npad, 0, 0, 0), 0))
    return _fwd_job(_planes(x_planes, View.nhwc_parity), _planes(w_planes, View.matrix), (N, So, So), 1, 9, taps,
                    Ci // 64, out, npad, _plain_out_strides(out), dtype=dtype, splits=splits, n_valid=out.shape[-1])
