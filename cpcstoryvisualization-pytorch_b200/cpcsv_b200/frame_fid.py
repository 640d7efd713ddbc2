"""Frame-level FID (the frame metric of the paper, reference ``fid/fid_score_v.py`` with the InceptionV3 of
``fid/inception.py``): pool3 features of single frames from the FID InceptionV3 run on the kernels of libcpcsv.so.
The Gaussian statistics and the Frechet distance are ``fsd.FeatureStats`` / ``fsd.frechet_distance``.

The contract is pytorch-fid's ``InceptionV3([pool3])``: torchvision's ``Inception3`` trunk (``transform_input``
False, BatchNorm eps 1e-3) with the FID blocks -- the branch pool of Mixed_5b..5d, 6b..6e and 7b is
``avg_pool2d(3, 1, 1, count_include_pad=False)``, that of Mixed_7c ``max_pool2d(3, 1, 1)`` -- and the 2048
features after the global average pool, in eval mode.  On channels-last activations every convolution is an
implicit GEMM of the tcgen05 kernel with bf16 hi/lo split operands:

* Conv2d_1a_3x3 (3x3 stride 2 pad 0 on the resized frame): ``cpcsv_resize_im2col`` computes the bilinear 299 x 299
  samples on the fly and writes the conv's im2col rows (K = 27 -> 64); one ``conv.gemm_nt``;
* every stride-1 convolution (1x1, 1x3 / 3x1, 1x7 / 7x1, 3x3 pad 0 or 1, 5x5 pad 2): ``conv.conv_kxl_fwd``, the 5x5
  as an overwriting 16-tap job plus an accumulating 9-tap job;
* 3x3 stride 2 pad 0 on the odd grids 35 and 17: ``conv.conv_s2v_fwd`` on the parity view.  Its input lives in a
  buffer with one extra (never read) row and column, [N, S + 1, S + 1, C]; stride-1 consumers read the
  [:, :S, :S] slice (see conv_s2v_fwd);
* pooling (maxpool1 / maxpool2, the stride-2 max-pool branches of Mixed_6a / 7a, the branch pools):
  ``cpcsv_pool3x3``.

Channel concatenation: every branch's last GEMM writes its slice [c0, c0 + Co) of one fp32 block buffer (output
pointer + pitches; every offset is a multiple of 4; the 288-channel outputs of Mixed_5c / 5d are padded to 320
zeroed channels, as the next GEMM's K must be a multiple of 64), and ONE
``cpcsv_bn_act_pack`` applies the concatenated eval BatchNorm + ReLU (a max-pooled branch that enters the
concatenation directly gets scale 1, shift 0: its values are ReLU outputs already).  Inner branch layers use
engine.BnActNode.  The tape runs with ``split_k=False``: a frame's features are bit-for-bit reproducible and do
not depend on the other frames of its chunk.
"""
import torch
import torch.nn as nn

from . import conv, ops
from .engine import T4, BnActNode, Tape, eval_affine, pack_im2col_weight, pack_taps, rup, _e
from .fsd import FeatureStats
from .nets import _CACHE, _bn_tuple

FEATURE_DIM = 2048
RESIZE = 299


# ------------------------------------------------------------------------------------------ modules
class BasicConv2d(nn.Module):
    """torchvision.models.inception.BasicConv2d: conv (no bias), BatchNorm (eps 1e-3), ReLU"""

    def __init__(self, cin, cout, kernel_size, stride=1, padding=0):
        super().__init__()
        self.conv = nn.Conv2d(cin, cout, kernel_size, stride, padding, bias=False)
        self.bn = nn.BatchNorm2d(cout, eps=0.001)


class InceptionA(nn.Module):
    def __init__(self, cin, pool_features):
        super().__init__()
        self.branch1x1 = BasicConv2d(cin, 64, 1)
        self.branch5x5_1 = BasicConv2d(cin, 48, 1)
        self.branch5x5_2 = BasicConv2d(48, 64, 5, padding=2)
        self.branch3x3dbl_1 = BasicConv2d(cin, 64, 1)
        self.branch3x3dbl_2 = BasicConv2d(64, 96, 3, padding=1)
        self.branch3x3dbl_3 = BasicConv2d(96, 96, 3, padding=1)
        self.branch_pool = BasicConv2d(cin, pool_features, 1)


class InceptionB(nn.Module):
    def __init__(self, cin):
        super().__init__()
        self.branch3x3 = BasicConv2d(cin, 384, 3, stride=2)
        self.branch3x3dbl_1 = BasicConv2d(cin, 64, 1)
        self.branch3x3dbl_2 = BasicConv2d(64, 96, 3, padding=1)
        self.branch3x3dbl_3 = BasicConv2d(96, 96, 3, stride=2)


class InceptionC(nn.Module):
    def __init__(self, cin, c7):
        super().__init__()
        self.branch1x1 = BasicConv2d(cin, 192, 1)
        self.branch7x7_1 = BasicConv2d(cin, c7, 1)
        self.branch7x7_2 = BasicConv2d(c7, c7, (1, 7), padding=(0, 3))
        self.branch7x7_3 = BasicConv2d(c7, 192, (7, 1), padding=(3, 0))
        self.branch7x7dbl_1 = BasicConv2d(cin, c7, 1)
        self.branch7x7dbl_2 = BasicConv2d(c7, c7, (7, 1), padding=(3, 0))
        self.branch7x7dbl_3 = BasicConv2d(c7, c7, (1, 7), padding=(0, 3))
        self.branch7x7dbl_4 = BasicConv2d(c7, c7, (7, 1), padding=(3, 0))
        self.branch7x7dbl_5 = BasicConv2d(c7, 192, (1, 7), padding=(0, 3))
        self.branch_pool = BasicConv2d(cin, 192, 1)


class InceptionD(nn.Module):
    def __init__(self, cin):
        super().__init__()
        self.branch3x3_1 = BasicConv2d(cin, 192, 1)
        self.branch3x3_2 = BasicConv2d(192, 320, 3, stride=2)
        self.branch7x7x3_1 = BasicConv2d(cin, 192, 1)
        self.branch7x7x3_2 = BasicConv2d(192, 192, (1, 7), padding=(0, 3))
        self.branch7x7x3_3 = BasicConv2d(192, 192, (7, 1), padding=(3, 0))
        self.branch7x7x3_4 = BasicConv2d(192, 192, 3, stride=2)


class InceptionE(nn.Module):
    def __init__(self, cin):
        super().__init__()
        self.branch1x1 = BasicConv2d(cin, 320, 1)
        self.branch3x3_1 = BasicConv2d(cin, 384, 1)
        self.branch3x3_2a = BasicConv2d(384, 384, (1, 3), padding=(0, 1))
        self.branch3x3_2b = BasicConv2d(384, 384, (3, 1), padding=(1, 0))
        self.branch3x3dbl_1 = BasicConv2d(cin, 448, 1)
        self.branch3x3dbl_2 = BasicConv2d(448, 384, 3, padding=1)
        self.branch3x3dbl_3a = BasicConv2d(384, 384, (1, 3), padding=(0, 1))
        self.branch3x3dbl_3b = BasicConv2d(384, 384, (3, 1), padding=(1, 0))
        self.branch_pool = BasicConv2d(cin, 192, 1)


class FrameFeatureNet(nn.Module):
    """FID InceptionV3 pool3 features on the kernel path: fp32 frames ``[N, 3, H, W]`` of any size in
    ``input_range`` (the generator's [-1, 1]) -> fp32 ``[N, 2048]``.

    Parameter and buffer names are those of ``torchvision.models.inception_v3`` (and of the pytorch-fid
    checkpoint), so either ``state_dict()`` loads directly; ``fc.*`` and ``AuxLogits.*`` entries are dropped.
    Preprocessing, as pytorch-fid: map ``input_range`` to [0, 1], resize bilinearly to 299 x 299
    (align_corners=False, no antialias), map [0, 1] to [-1, 1].  Both maps are per-element affine and the bilinear
    weights sum to 1, so the kernel resizes the raw frame and applies the ONE composed affine to each sample.
    Frames go through the network ``chunk`` at a time (about 20 MB of activations per frame, an estimate).
    Eval mode and ``torch.no_grad()`` only; the module starts in eval mode."""

    def __init__(self, input_range=(-1.0, 1.0), chunk=128):
        super().__init__()
        self.input_range = (float(input_range[0]), float(input_range[1]))
        assert self.input_range[1] > self.input_range[0]
        self.chunk = int(chunk)
        self.Conv2d_1a_3x3 = BasicConv2d(3, 32, 3, stride=2)
        self.Conv2d_2a_3x3 = BasicConv2d(32, 32, 3)
        self.Conv2d_2b_3x3 = BasicConv2d(32, 64, 3, padding=1)
        self.Conv2d_3b_1x1 = BasicConv2d(64, 80, 1)
        self.Conv2d_4a_3x3 = BasicConv2d(80, 192, 3)
        self.Mixed_5b = InceptionA(192, 32)
        self.Mixed_5c = InceptionA(256, 64)
        self.Mixed_5d = InceptionA(288, 64)
        self.Mixed_6a = InceptionB(288)
        self.Mixed_6b = InceptionC(768, 128)
        self.Mixed_6c = InceptionC(768, 160)
        self.Mixed_6d = InceptionC(768, 160)
        self.Mixed_6e = InceptionC(768, 192)
        self.Mixed_7a = InceptionD(768)
        self.Mixed_7b = InceptionE(1280)
        self.Mixed_7c = InceptionE(2048)
        self.register_load_state_dict_pre_hook(_drop_heads)
        self.eval()

    def forward(self, frames):
        if self.training:
            raise RuntimeError("cpcsv_b200: FrameFeatureNet runs in eval mode only (BatchNorm with the running "
                               "statistics of the checkpoint); call .eval() before extracting features")
        if torch.is_grad_enabled():
            raise RuntimeError("cpcsv_b200: FrameFeatureNet is forward-only; call it under torch.no_grad()")
        if frames.dim() != 4 or frames.shape[1] != 3:
            raise ValueError("FrameFeatureNet: expected frames [N, 3, H, W], got %s" % (tuple(frames.shape),))
        lo, hi = self.input_range
        a, b = 2.0 / (hi - lo), -2.0 * lo / (hi - lo) - 1.0
        out = torch.empty(frames.shape[0], FEATURE_DIM, device=frames.device)
        for s in range(0, frames.shape[0], self.chunk):
            x = frames[s:s + self.chunk].float()
            out[s:s + x.shape[0]] = FrameRunner(self).run(x, a, b)
        return out


def _drop_heads(module, state_dict, prefix, *args):
    for k in [k for k in state_dict if k.startswith(prefix + "fc.") or k.startswith(prefix + "AuxLogits.")]:
        del state_dict[k]


# ------------------------------------------------------------------------------------------ runner
class Act:
    """an activation of S x S pixels: fp32 values and / or 16-bit planes in [N, P, P, C] buffers, P = S, or S + 1
    for an odd S that a stride-2 convolution reads (conv.conv_s2v_fwd)"""

    __slots__ = ("S", "f32", "hi", "lo")

    def __init__(self, S, f32=None, hi=None, lo=None):
        self.S, self.f32, self.hi, self.lo = S, f32, hi, lo

    @property
    def C(self):
        return (self.hi if self.hi is not None else self.f32).shape[-1]

    def planes(self, full=False):
        return [p if full or p is None else p[:, :self.S, :self.S] for p in (self.hi, self.lo)]

    def values(self):
        return self.f32[:, :self.S, :self.S]


def _pool_out(S, stride):
    return S if stride == 1 else (S - 3) // 2 + 1


class FrameRunner:
    """one chunk of frames through the FID InceptionV3; intermediate buffers are freed as soon as Python drops
    them (the nodes are not kept on the tape)"""

    def __init__(self, net):
        self.net = net
        self.tape = Tape(_CACHE, training=False, need_grad=False, planes=2, dtype=ops.BF16, split_k=False)

    # ---------------------------------------------------------------- helpers
    def _zbuf(self, S, C, pad):
        """fp32 conv output buffer; a padded one is zeroed so its extra row / column stays finite"""
        P = S + (S & 1) if pad else S
        if pad and P != S:
            return torch.zeros((self.N, P, P, C), device=self.dev)
        return _e((self.N, P, P, C), self.dev)

    def _block_buf(self, S, width, pad=False):
        """fp32 buffer of a concatenated block output: channels padded to a multiple of 64 (288 -> 320) for the next
        layer's K.  No job writes the padding channels, and zero weight columns do not cancel a NaN: zero them."""
        buf = self._zbuf(S, rup(width, 64), pad)
        if buf.shape[-1] > width:
            buf[..., width:].zero_()
        return buf

    def _planes(self, shape):
        t16 = ops.TORCH16[self.tape.dtype]
        return _e(shape, self.dev, t16), _e(shape, self.dev, t16)

    def conv(self, x, bc, out=None, pad=False):
        """the convolution of BasicConv2d `bc` on Act x, into `out` (an fp32 [N, So, So, Co] channel slice of a block
        buffer) or, when None, into a new buffer -> (T4 of that buffer, So)"""
        t = self.tape
        w = bc.conv.weight
        Co, Ci, kh, kw = w.shape
        assert rup(Ci, 64) == x.C, (Ci, x.C)
        stride = bc.conv.stride[0]
        ph, pw = bc.conv.padding
        So = x.S + 2 * ph - kh + 1 if stride == 1 else (x.S - 3) // 2 + 1
        z = None
        if out is None:
            buf = self._zbuf(So, rup(Co, 64), pad)
            z = T4(self.N, buf.shape[1], buf.shape[2], buf.shape[3])
            z.f32 = buf
            out = buf[:, :So, :So]
        wp = pack_taps(t.cache, w, w.detach, 0, rup(Co, 64), x.C, t.planes, t.dtype)
        if stride == 1:
            jobs = conv.conv_kxl_fwd(x.planes(), wp, out, kh, kw, ph, pw, dtype=t.dtype, splits=t.splits)
        else:
            assert (kh, kw, ph, pw) == (3, 3, 0, 0) and stride == 2
            jobs = [conv.conv_s2v_fwd(x.planes(full=True), wp, out, dtype=t.dtype, splits=t.splits)]
        for job in jobs:
            ops.conv_gemm(job)
        return z, So

    def basic(self, x, bc, pad=False, want_f32=False, want_planes=True):
        """BasicConv2d: conv, then eval BatchNorm + ReLU (engine.BnActNode) -> Act"""
        z, So = self.conv(x, bc, pad=pad)
        node = BnActNode(self.tape, z, _bn_tuple(bc.bn), ops.ACT_RELU, "fid", want_f32=want_f32,
                         want_planes=want_planes, eps=bc.bn.eps)
        node.forward()
        o = node.out
        return Act(So, o.f32, o.hi, o.lo)

    def pool(self, x, mode, stride, y=None, planes=False, channels=None):
        """3x3 pooling of x's fp32 values (the first `channels`; default all) into `y` (fp32 view) and / or new
        hi / lo planes -> planes Act or None"""
        So = _pool_out(x.S, stride)
        xv = x.values() if channels is None else x.values()[..., :channels]
        hi = lo = None
        if planes:
            hi, lo = self._planes((self.N, So, So, xv.shape[-1]))
        ops.pool3x3(xv, mode, stride, y, hi, lo, self.tape.dtype)
        return Act(So, y, hi, lo) if planes else None

    def finish(self, buf, S, parts, want_f32=True, want_planes=True):
        """ONE eval BatchNorm + ReLU over a concatenated block buffer; parts: [(bn or None, width)] in channel order
        (None: a pooled branch, scale 1 / shift 0)"""
        C = buf.shape[-1]
        width = sum(w for _, w in parts)
        parts = parts + [(None, C - width)] if C > width else parts
        sc, sh = [], []
        for bn, w in parts:
            if bn is None:     # a pooled branch (ReLU outputs already) or the zeroed padding channels
                sc.append(torch.ones(w, device=self.dev))
                sh.append(torch.zeros(w, device=self.dev))
            else:
                a, b = eval_affine(_bn_tuple(bn), w, None, w, bn.eps)
                sc.append(a)
                sh.append(b)
        assert sum(w for _, w in parts) == C, (parts, C)
        scale, shift = torch.cat(sc).contiguous(), torch.cat(sh).contiguous()
        y = _e(buf.shape, self.dev) if want_f32 else None
        hi, lo = self._planes(buf.shape) if want_planes else (None, None)
        rows = buf.numel() // C
        ops.bn_act_pack(buf.view(rows, C), scale, shift, ops.ACT_RELU, None,
                        y.view(rows, C) if y is not None else None, hi.view(rows, C) if hi is not None else None,
                        lo.view(rows, C) if lo is not None else None, self.tape.dtype)
        return Act(S, y, hi, lo)

    # ---------------------------------------------------------------- blocks
    def block_a(self, m, x, pad_out):
        cp = m.branch_pool.conv.out_channels
        buf = self._block_buf(x.S, 224 + cp, pad_out)
        v = buf[:, :x.S, :x.S]
        self.conv(x, m.branch1x1, v[..., 0:64])
        self.conv(self.basic(x, m.branch5x5_1), m.branch5x5_2, v[..., 64:128])
        d = self.basic(self.basic(x, m.branch3x3dbl_1), m.branch3x3dbl_2)
        self.conv(d, m.branch3x3dbl_3, v[..., 128:224])
        self.conv(self.pool(x, ops.POOL_AVG, 1, planes=True), m.branch_pool, v[..., 224:224 + cp])
        return self.finish(buf, x.S, [(m.branch1x1.bn, 64), (m.branch5x5_2.bn, 64), (m.branch3x3dbl_3.bn, 96),
                                      (m.branch_pool.bn, cp)])

    def block_b(self, m, x):
        So = (x.S - 3) // 2 + 1
        C = m.branch3x3.conv.in_channels      # the real channels of x (its buffer may be padded)
        buf = self._block_buf(So, 480 + C)
        self.conv(x, m.branch3x3, buf[..., 0:384])
        d = self.basic(self.basic(x, m.branch3x3dbl_1), m.branch3x3dbl_2, pad=True)
        self.conv(d, m.branch3x3dbl_3, buf[..., 384:480])
        self.pool(x, ops.POOL_MAX, 2, y=buf[..., 480:480 + C], channels=C)
        return self.finish(buf, So, [(m.branch3x3.bn, 384), (m.branch3x3dbl_3.bn, 96), (None, C)])

    def block_c(self, m, x):
        buf = self._block_buf(x.S, 768)
        self.conv(x, m.branch1x1, buf[..., 0:192])
        b = self.basic(self.basic(x, m.branch7x7_1), m.branch7x7_2)
        self.conv(b, m.branch7x7_3, buf[..., 192:384])
        d = x
        for bc in (m.branch7x7dbl_1, m.branch7x7dbl_2, m.branch7x7dbl_3, m.branch7x7dbl_4):
            d = self.basic(d, bc)
        self.conv(d, m.branch7x7dbl_5, buf[..., 384:576])
        self.conv(self.pool(x, ops.POOL_AVG, 1, planes=True), m.branch_pool, buf[..., 576:768])
        return self.finish(buf, x.S, [(m.branch1x1.bn, 192), (m.branch7x7_3.bn, 192), (m.branch7x7dbl_5.bn, 192),
                                      (m.branch_pool.bn, 192)])

    def block_d(self, m, x):
        So = (x.S - 3) // 2 + 1
        C = m.branch3x3_1.conv.in_channels
        buf = self._block_buf(So, 512 + C)
        self.conv(self.basic(x, m.branch3x3_1, pad=True), m.branch3x3_2, buf[..., 0:320])
        b = self.basic(self.basic(x, m.branch7x7x3_1), m.branch7x7x3_2)
        self.conv(self.basic(b, m.branch7x7x3_3, pad=True), m.branch7x7x3_4, buf[..., 320:512])
        self.pool(x, ops.POOL_MAX, 2, y=buf[..., 512:512 + C], channels=C)
        return self.finish(buf, So, [(m.branch3x3_2.bn, 320), (m.branch7x7x3_4.bn, 192), (None, C)])

    def block_e(self, m, x, pool_mode, last):
        buf = self._block_buf(x.S, 2048)
        self.conv(x, m.branch1x1, buf[..., 0:320])
        b = self.basic(x, m.branch3x3_1)
        self.conv(b, m.branch3x3_2a, buf[..., 320:704])
        self.conv(b, m.branch3x3_2b, buf[..., 704:1088])
        d = self.basic(self.basic(x, m.branch3x3dbl_1), m.branch3x3dbl_2)
        self.conv(d, m.branch3x3dbl_3a, buf[..., 1088:1472])
        self.conv(d, m.branch3x3dbl_3b, buf[..., 1472:1856])
        self.conv(self.pool(x, pool_mode, 1, planes=True), m.branch_pool, buf[..., 1856:2048])
        return self.finish(buf, x.S, [(m.branch1x1.bn, 320), (m.branch3x3_2a.bn, 384), (m.branch3x3_2b.bn, 384),
                                      (m.branch3x3dbl_3a.bn, 384), (m.branch3x3dbl_3b.bn, 384),
                                      (m.branch_pool.bn, 192)], want_planes=not last)

    # ---------------------------------------------------------------- network
    def run(self, frames, a, b):
        """frames fp32 [N, 3, H, W]; a, b: the composed input affine -> fp32 [N, 2048]"""
        net, t = self.net, self.tape
        self.N, self.dev = frames.shape[0], frames.device
        OH = (RESIZE - 3) // 2 + 1
        stem = net.Conv2d_1a_3x3
        Kp = rup(27, 64)
        col_hi, col_lo = self._planes((self.N * OH * OH, Kp))
        ops.resize_im2col(frames, RESIZE, a, b, col_hi, col_lo, t.dtype)
        z = T4(self.N, OH, OH, rup(stem.conv.out_channels, 64))
        z.f32 = _e((z.N, z.H, z.W, z.C), self.dev)
        ops.conv_gemm(conv.gemm_nt([col_hi, col_lo], pack_im2col_weight(t.cache, stem.conv.weight, "fwd", Kp, t.planes,
                                                                        t.dtype),
                                   z.f32.view(-1, z.C), dtype=t.dtype, splits=t.splits))
        del col_hi, col_lo
        node = BnActNode(t, z, _bn_tuple(stem.bn), ops.ACT_RELU, "fid", eps=stem.bn.eps)
        node.forward()
        x = Act(OH, None, node.out.hi, node.out.lo)
        x = self.basic(x, net.Conv2d_2a_3x3)
        x = self.basic(x, net.Conv2d_2b_3x3, want_f32=True, want_planes=False)
        x = self.pool(x, ops.POOL_MAX, 2, planes=True)                                      # maxpool1
        x = self.basic(x, net.Conv2d_3b_1x1)
        x = self.basic(x, net.Conv2d_4a_3x3, want_f32=True, want_planes=False)
        S = _pool_out(x.S, 2)
        y = _e((self.N, S, S, x.C), self.dev)
        x = self.pool(x, ops.POOL_MAX, 2, y=y, planes=True)                                 # maxpool2
        x = self.block_a(net.Mixed_5b, x, False)
        x = self.block_a(net.Mixed_5c, x, False)
        x = self.block_a(net.Mixed_5d, x, True)
        x = self.block_b(net.Mixed_6a, x)
        for m in (net.Mixed_6b, net.Mixed_6c, net.Mixed_6d, net.Mixed_6e):
            x = self.block_c(m, x)
        x = self.block_d(net.Mixed_7a, x)
        x = self.block_e(net.Mixed_7b, x, ops.POOL_AVG, False)
        x = self.block_e(net.Mixed_7c, x, ops.POOL_MAX, True)
        t.release()
        # the global average pool
        return x.values().reshape(self.N, -1, FEATURE_DIM).mean(1)


# ------------------------------------------------------------------------------------------ statistics
def frame_statistics(batches, net, stats=None):
    """add the features of every frame of an iterable of batches -- frames ``[N, 3, H, W]`` or stories
    ``[B, 3, T, H, W]`` (flattened to B * T frames) -- to ``stats`` (a new ``fsd.FeatureStats(dim=2048)`` when
    None) and return it"""
    stats = stats if stats is not None else FeatureStats(dim=FEATURE_DIM)
    with torch.no_grad():
        for x in batches:
            if x.dim() == 5:
                x = x.transpose(1, 2).reshape(-1, x.shape[1], x.shape[3], x.shape[4])
            stats.update(net(x))
    return stats
