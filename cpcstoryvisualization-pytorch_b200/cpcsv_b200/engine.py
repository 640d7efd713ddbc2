"""Layer-level execution engine: a tiny reverse-mode tape over NHWC buffers whose every
arithmetic step is a libcpcsv.so kernel (``ops``).  ``model.py`` builds one tape per network
call (generator trunk, discriminator encoder, logits head) and exposes it to PyTorch autograd
as a single ``torch.autograd.Function``.

Precision recipe (SURVEY.md Appendix E): forward convolutions whose result feeds a backward
pass run with hi/lo split bf16 operands (3 MMAs, ~16-bit significand); backward GEMMs (dgrad,
wgrad) are single-pass bf16; statistics, normalisation and all gradients are fp32.
"""
import weakref

import torch
import torch.nn.functional as F

from . import conv, ops
from .ops import ACT_NONE, ACT_RELU, ACT_LRELU, BF16  # noqa: F401


# BatchNorm batch statistics come out of the producing GEMM's epilogue (cpcsv_gemm_t.stats) whenever that
# GEMM runs without split-K; otherwise from one statistics pass.  Either way the per-channel constants are
# derived inside the apply kernel (cpcsv_bn_norm_act_pack): at most 2 launches between consecutive GEMMs.
EPILOGUE_STATS = True

# Operand precision of NO-GRAD network calls (the fakes for the discriminator update, inference).  Default:
# single-pass fp16 (SURVEY.md Appendix E recipe R*), which leaves ~1.5e-3 relative error on the images and is
# what bounds the discriminator-gradient parity (cosine 0.9998 at the cfg/final.yml batch, 0.9990-0.9995 per
# tensor on reduced-width models).  CPCSV_NOGRAD_SPLIT=1: bf16 hi/lo planes (3 MMAs) there as well -- images
# to 2e-5, discriminator gradients to 0.99997 -- at 3x the tensor-core work of those calls (+2.4 TFLOP per step
# at cfg/final.yml).
import os as _os  # noqa: E402
NOGRAD_SPLIT = _os.environ.get("CPCSV_NOGRAD_SPLIT", "0") == "1"


def rup(x, m):
    return (x + m - 1) // m * m


class T4:
    """NHWC tensor record: fp32 values and/or 16-bit operand planes, plus gradient slots."""

    __slots__ = ("N", "H", "W", "C", "f32", "hi", "lo", "grad", "grad16", "needs_grad", "stats", "stats_done")

    def __init__(self, N, H, W, C):
        self.N, self.H, self.W, self.C = N, H, W, C
        self.f32 = self.hi = self.lo = self.grad = self.grad16 = None
        self.needs_grad = False
        self.stats = None           # zeroed fp64 [2, C]: per-channel sum / sum of squares of f32
        self.stats_done = False     # filled by the producing GEMM's epilogue

    @property
    def rows(self):
        return self.N * self.H * self.W

    def mat(self, t):
        return t.view(self.rows, self.C)

    def planes(self, n):
        return [self.hi, self.lo if n == 2 else None]


class CacheEntry:
    """one packed form of a parameter: ``val`` (operand planes), the validity ``tag``, the stream / event
    of the kernel that last wrote it, a weak reference to the parameter, and -- for planes that live in
    PERSISTENT buffers kept current by the optimiser -- their ``spec`` and the ``fill`` closure that
    re-packs them in place"""

    __slots__ = ("tag", "val", "stream", "event", "ref", "spec", "fill", "in_capture")

    def __init__(self, tag, val, stream, event, ref, spec=None, fill=None, in_capture=False):
        self.tag, self.val, self.stream, self.event, self.ref, self.spec, self.fill = \
            tag, val, stream, event, ref, spec, fill
        self.in_capture = in_capture     # the event was recorded while a CUDA graph was being captured


class WeightCache:
    """16-bit operand planes of parameters.

    Two kinds of entries:
      * MAINTAINED (``spec`` given): the planes of the tensor-core convolutions and of fc / fc_seg live in
        persistent buffers.  ``optim.PackedAdam`` rewrites them in the same kernel that updates the fp32
        weight, so they are always current -- inside replayed CUDA graphs too -- and nothing is re-packed
        between an optimiser step and the next forward pass.  A parameter changed in any other way
        (``load_state_dict``, another optimiser, ``invalidate``) is re-packed IN PLACE at its next use.
      * plain: small derived forms (first discriminator layer, head gradients); rebuilt when the parameter
        changed (``_version``), after every optimiser step (global post-step hook in nets.py, because fused
        optimisers do not bump ``_version``) or when the capture state differs."""

    def __init__(self):
        self.d = {}
        self.epoch = 0
        self.replays = 0

    def invalidate(self):
        self.epoch += 1

    def note_replay(self):
        """a captured CUDA graph that contains optimiser steps has been replayed: the weights moved without any
        Python-side trace (no ``_version`` bump, no optimiser hook).  Plain entries packed EAGERLY are stale from
        here on and are rebuilt at their next eager use; maintained planes were rewritten by the graph itself and
        entries packed inside the capture belong to the graph."""
        self.replays += 1

    def invalidate_params(self, param_ids, keep_maintained=False):
        """drop the entries of the given parameters (keys start with id(param)); maintained planes are
        marked stale (re-packed into the same buffers at the next use) unless the optimiser that
        just stepped keeps them current itself"""
        for key in [k for k in self.d if k[0] in param_ids]:
            ent = self.d[key]
            if ent.spec is None:
                del self.d[key]
            elif not keep_maintained:
                ent.tag = None

    def maintained(self, param):
        """[(key, entry)] of the persistent planes of `param`"""
        pid = id(param)
        return [(k, e) for k, e in self.d.items() if k[0] == pid and e.spec is not None and e.ref() is param]

    def refreshed(self, ent, param):
        """the optimiser has just rewritten the planes of `ent` on the current stream; every later
        consumer is ordered after it by the step's fork / join structure"""
        ent.tag = self._tag(param, True, False)
        ent.stream = ent.event = None

    def mark_synced(self, streams=None):
        """after packing streams have been joined into the current one: later consumers need no
        event wait (and must not wait on an event of an earlier graph capture).  `streams` = the
        streams that were joined (None: every stream)"""
        for ent in self.d.values():
            if ent.stream is not None and (streams is None or ent.stream in streams):
                ent.stream = ent.event = None

    def _tag(self, param, maintained, capturing):
        # planes packed while a CUDA graph is being captured only exist once that graph replays,
        # and planes packed eagerly must not be waited on from inside a capture: for plain entries
        # the capture state is part of the validity tag.  Maintained planes sit in persistent buffers
        # that the (captured or eager) optimiser step keeps current: valid in both states.
        if maintained:
            return (param._version, param.data_ptr(), self.epoch)
        return (param._version, param.data_ptr(), self.epoch, capturing, 0 if capturing else self.replays)

    def get(self, key, param, build, spec=None, fill=None):
        """Entries remember the stream that packed them and an event recorded after the pack
        kernel: a consumer on another stream (concurrent network calls, pack prefetching) waits
        on the event instead of racing with the pack.  ``spec`` / ``fill(val)``: maintained entry
        (``build`` allocates AND fills; ``fill`` re-packs into the existing buffers)."""
        on_gpu = param.is_cuda
        capturing = on_gpu and torch.cuda.is_current_stream_capturing()
        tag = self._tag(param, spec is not None, capturing)
        ent = self.d.get(key)
        cur = torch.cuda.current_stream() if on_gpu else None
        # keys carry id(param): an entry only counts while THAT parameter object is alive (a freed
        # parameter's id, address and version can all be recycled by a later one)
        alive = ent is not None and ent.ref() is param
        if alive and ent.tag == tag:
            if on_gpu and ent.stream is not None and ent.in_capture != capturing:
                # (maintained planes only: plain entries carry the capture state in their tag.)  An event
                # recorded outside a capture cannot be waited on inside one, and vice versa.  Packed eagerly,
                # read inside a capture: torch.cuda.graph() synchronises the device before capturing, so the
                # pack is complete.  Packed inside a capture, read eagerly: the reader is enqueued after the
                # replay that produced the planes.
                ent.stream = ent.event = None
            if on_gpu and ent.stream is not None and ent.stream != cur:
                cur.wait_event(ent.event)
                if ent.spec is None:
                    for tns in (ent.val if isinstance(ent.val, (list, tuple)) else [ent.val]):
                        if tns is not None:
                            tns.record_stream(cur)     # keep the allocator from recycling it early
            return ent.val
        if alive and spec is not None and ent.spec == spec:
            # stale persistent planes (the parameter was modified outside PackedAdam): re-pack in place.
            # Earlier readers of the old contents may still be running on other streams.
            if on_gpu and not capturing:
                torch.cuda.synchronize(param.device)
            fill(ent.val)
            val = ent.val
        else:
            val = build()
        ev = None
        if on_gpu:
            ev = torch.cuda.Event()
            ev.record(cur)
        # the entry (and the operand planes it keeps alive) goes away with the parameter
        self.d[key] = CacheEntry(tag, val, cur, ev, weakref.ref(param, lambda _r, k=key, d=self.d: d.pop(k, None)),
                                 spec, fill, capturing)
        return val


def _e(shape, dev, dtype=torch.float32):
    return torch.empty(shape, device=dev, dtype=dtype)


def _row_pad_map(rows, rows_pad, dev):
    m = torch.full((rows_pad,), -1, dtype=torch.int32, device=dev)
    m[:rows] = torch.arange(rows, dtype=torch.int32, device=dev)
    return m


class StateOrder:
    """In-place module state that several network calls update (BatchNorm running statistics,
    num_batches_tracked) must be updated in program order even when the calls run on different
    CUDA streams (trainer runs sample_videos / sample_images concurrently).  Every update of a
    state tensor records an event; an update issued later from another stream waits on it."""

    _last = {}

    @classmethod
    def reset(cls):
        """all streams have been joined: nothing issued later needs the recorded events"""
        cls._last.clear()

    @classmethod
    def before(cls, tensor):
        if tensor is None or not tensor.is_cuda:
            return
        ent = cls._last.get(tensor.data_ptr())
        if ent is not None:
            cur = torch.cuda.current_stream()
            capturing = torch.cuda.is_current_stream_capturing()
            if ent[0] != cur and ent[2] == capturing:
                cur.wait_event(ent[1])

    @classmethod
    def after(cls, tensor):
        if tensor is None or not tensor.is_cuda:
            return
        cur = torch.cuda.current_stream()
        ev = torch.cuda.Event()
        ev.record(cur)
        cls._last[tensor.data_ptr()] = (cur, ev, torch.cuda.is_current_stream_capturing())


# ------------------------------------------------------------------------------ gradient sink
# An optimiser that wants parameter gradients the moment a tape has computed them (optim.PackedAdam with
# ``overlap_with_backward(..., buckets=...)``): the generator trunk is ONE autograd Function, so autograd hands all of
# its parameter gradients over together, at the very end of its backward pass -- the sink gets each layer's
# gradients right after that layer's weight-gradient GEMM instead.
_GRAD_SINK = [None]


def set_grad_sink(sink):
    _GRAD_SINK[0] = sink


def grad_sink():
    return _GRAD_SINK[0]


# ------------------------------------------------------------------------------ aux branch
WGRAD_ON_AUX_STREAM = True
_AUX_STREAMS = {}


class AuxBranch:
    """Side stream of one tape's backward pass for work nothing later in the same pass waits for:
    the weight-gradient GEMM of a layer (+ its un-packing and spectral-norm backward) runs there
    while the data-gradient chain (dgrad -> BN backward -> dgrad ...) continues on the tape's own
    stream.  ``run`` forks after everything issued so far; ``join`` makes the tape's stream wait
    for the branch (call it before handing the gradients back to autograd)."""

    def __init__(self):
        self.stream = None
        self.keep = []

    def run(self, fn, *keep):
        """`keep`: tensors the branch reads that the caller is about to drop -- held until
        ``join`` so the allocator cannot recycle them under the branch's kernels"""
        if not (WGRAD_ON_AUX_STREAM and torch.cuda.is_available()):
            fn()
            return
        cur = torch.cuda.current_stream()
        if self.stream is None:
            key = (cur.device, cur.cuda_stream)
            st = _AUX_STREAMS.get(key)
            if st is None:
                st = _AUX_STREAMS[key] = torch.cuda.Stream(device=cur.device, priority=cur.priority)
            self.stream = st
        ev = torch.cuda.Event()
        ev.record(cur)
        self.stream.wait_event(ev)
        self.keep.extend(keep)
        with torch.cuda.stream(self.stream):
            fn()

    def join(self):
        if self.stream is not None:
            torch.cuda.current_stream().wait_stream(self.stream)
            self.stream = None
        self.keep = []


# ------------------------------------------------------------------------------ conv nodes
CONV_GEOM = {
    # kind: (job kernel, fwd pack kind, dgrad pack kind, wgrad taps, unpack kind)
    "s1": (3, 0, 1, 9, 0),
    "up": (3, 2, 3, 16, 2),
    "s2": (4, 0, 1, 16, 0),
    # 3x3 stride 2 pad 1 as the 4x4 "s2" job: the same input coordinate 2*o + k - 1, with the 4th row and
    # column of the packed weight zero
    "s2k3": (4, 0, 1, 16, 0),
}
# geometries whose weight kernel is smaller than the job's (zero-padded to it): kind -> weight kernel
WEIGHT_KERNEL = {"s2k3": 3}


def pack_taps(cache, w, w4, kindcode, rows_pad, cols_pad, planes, dtype):
    """(cached) tap-major operand planes of ``w4()``, a 4-D ``[Co, Ci, kh, kw]`` view of parameter ``w``
    (cpcsv_pack_conv_weight handles any kh x kw); a plain entry, re-packed when the parameter changed"""
    def build():
        ntap = w4().shape[2] * w4().shape[3]
        t16 = ops.TORCH16[dtype]
        hi = _e((ntap * rows_pad, cols_pad), w.device, t16)
        lo = _e((ntap * rows_pad, cols_pad), w.device, t16) if planes == 2 else None
        ops.pack_conv_weight(w4(), kindcode, rows_pad, cols_pad, hi, lo, dtype)
        return [hi, lo]
    return cache.get((id(w), "taps", kindcode, planes, dtype), w, build)


def pack_im2col_weight(cache, w, kind, K_pad, planes=1, dtype=BF16):
    """(cached) weight of an im2col'd convolution, columns k = tap * Ci + c (the order of cpcsv_im2col_small):
    ``"fwd"``: the B operand of the forward GEMM, ``[hi, lo]`` planes ``[Co_pad, K_pad]``; ``"bwd"``: the B operand
    of the data-gradient GEMM (into the im2col matrix), one bf16 plane ``[K_pad, Co_pad]``"""
    Co = w.shape[0]
    K, Cop = w.shape[1:].numel(), rup(Co, 64)
    if kind == "bwd":
        planes, dtype = 1, BF16

    def build():
        w2 = w.detach().reshape(Co, w.shape[1], -1).permute(0, 2, 1).reshape(Co, K).contiguous()
        t16 = ops.TORCH16[dtype]
        if kind == "fwd":
            hi = _e((Cop, K_pad), w.device, t16)
            lo = _e((Cop, K_pad), w.device, t16) if planes == 2 else None
            ops.pack_matrix(w2, Cop, K_pad, K, K, 1, _row_pad_map(Co, Cop, w.device), hi, lo, dtype)
        else:
            hi, lo = _e((K_pad, Cop), w.device, t16), None
            ops.pack_matrix(w2, K_pad, Cop, Co, 1, K, _row_pad_map(K, K_pad, w.device), hi, None)
        return [hi, lo]
    return cache.get((id(w), "im2col", kind, planes, dtype), w, build)


def pack_conv(cache, w, geom, kindcode, rows_pad, cols_pad, planes, dtype=BF16):
    """(cached, persistent) tap-major 16-bit operand planes of a conv weight; kinds as
    cpcsv_pack_conv_weight.  Filled here at first use, afterwards kept current by optim.PackedAdam."""
    ntap = CONV_GEOM[geom][3]

    def fill(val):
        ops.adam_pack_conv(w.detach(), None, None, None, [(kindcode, dtype, rows_pad, cols_pad, val[0], val[1])])

    def build():
        dev = w.device
        t16 = ops.TORCH16[dtype]
        hi = _e((ntap * rows_pad, cols_pad), dev, t16)
        lo = _e((ntap * rows_pad, cols_pad), dev, t16) if planes == 2 else None
        fill([hi, lo])
        return [hi, lo]
    return cache.get((id(w), kindcode, planes, dtype), w, build,
                     spec=("conv", kindcode, dtype, rows_pad, cols_pad, planes), fill=fill)


def prefetch_conv(cache, w, geom, forward=True, backward=True):
    """pack the training-time operand planes of one conv weight ahead of use: forward = bf16
    hi/lo split [Co_pad, Ci_pad] taps, backward = single-plane transposed taps (dgrad)"""
    Co_pad, Ci_pad = rup(w.shape[0], 64), rup(w.shape[1], 64)
    _k, fkind, bkind, _nt, _uk = CONV_GEOM[geom]
    if forward:
        pack_conv(cache, w, geom, fkind, Co_pad, Ci_pad, 2, BF16)
    if backward:
        pack_conv(cache, w, geom, bkind, Ci_pad, Co_pad, 1, BF16)


def prefetch_conv_nograd(cache, w, geom):
    """the single-plane fp16 forward taps a no-grad generator call uses"""
    Co_pad, Ci_pad = rup(w.shape[0], 64), rup(w.shape[1], 64)
    pack_conv(cache, w, geom, CONV_GEOM[geom][1], Co_pad, Ci_pad, 1, ops.FP16)


def attach_stats(tape, job, out, wanted):
    """BatchNorm batch statistics of a GEMM's output from its epilogue (no split-K, training mode)"""
    if wanted and tape.training:
        out.stats = tape.stat_slot(out.C, out.f32.device)
        if EPILOGUE_STATS and job.mode == 0 and job.splits == 1 and not job.accumulate and job.block_n % 32 == 0:
            job.stats = out.stats
            out.stats_done = True


class ConvNode:
    """3x3 s1 / nearest-x2+3x3 / 4x4 s2 / 3x3 s2 (``s2k3``) convolution, optionally spectrally normalised
    (weight = weight_orig / sigma applied as the epilogue scalar alpha).

    A 4-D weight whose kernel is the job's gets the persistent operand planes optim.PackedAdam keeps
    current (pack_conv); any other weight -- a Conv3d ``[Co, Ci, 1, k, k]``, a 3x3 weight run as the 4x4 job
    -- is packed from its 4-D (zero-padded) tap view into a plain cache entry (pack_taps)."""

    def __init__(self, tape, kind, x, weight, name, sn=None, alpha=None, bn_stats=False):
        self.tape, self.kind, self.x, self.w, self.name, self.sn = tape, kind, x, weight, name, sn
        self.bn_stats = bn_stats    # a batch-statistics BatchNorm consumes the output
        Co, Ci = weight.shape[0], weight.shape[1]
        self.Co, self.Ci = Co, Ci
        self.Co_pad, self.Ci_pad = rup(Co, 64), x.C
        assert rup(Ci, 64) == x.C, (name, Ci, x.C)
        N, H, W = x.N, x.H, x.W
        if kind == "up":
            H, W = 2 * H, 2 * W
        elif kind != "s1":
            H, W = H // 2, W // 2
        self.out = T4(N, H, W, self.Co_pad)
        self.alpha = alpha          # 1/sigma of a spectral norm whose power iteration already ran
        self.dW = None

    def _w4(self):
        k = CONV_GEOM[self.kind][0]
        wk = WEIGHT_KERNEL.get(self.kind, k)
        w = self.w.detach()
        w4 = w.view(w.shape[0], w.shape[1], wk, wk)
        return w4 if wk == k else F.pad(w4, (0, k - wk, 0, k - wk)).contiguous()

    def _pack(self, kindcode, rows_pad, cols_pad, planes, dtype=BF16):
        w, k = self.w, CONV_GEOM[self.kind][0]
        if w.dim() == 4 and w.shape[2] == w.shape[3] == k:
            return pack_conv(self.tape.cache, w, self.kind, kindcode, rows_pad, cols_pad, planes, dtype)
        return pack_taps(self.tape.cache, w, self._w4, kindcode, rows_pad, cols_pad, planes, dtype)

    def forward(self):
        t, x, out = self.tape, self.x, self.out
        dev = x.hi.device
        if self.sn is not None and self.alpha is None:     # not already computed ahead of the chain
            self.alpha = self.sn.forward(self.w, t.training, t.need_grad)
        wp = self._pack(CONV_GEOM[self.kind][1], self.Co_pad, self.Ci_pad, t.planes, t.dtype)
        out.f32 = _e((out.N, out.H, out.W, out.C), dev)
        xp = x.planes(t.planes)
        if self.kind == "s1":
            job = conv.conv_s1_fwd(xp, wp, out.f32, 3, self.alpha, dtype=t.dtype, splits=t.splits)
        elif self.kind == "up":
            job = conv.upconv_fwd(xp, wp, out.f32, dtype=t.dtype)
        else:
            job = conv.conv_s2_fwd(xp, wp, out.f32, self.alpha, dtype=t.dtype, splits=t.splits)
        attach_stats(t, job, out, self.bn_stats)
        ops.conv_gemm(job)

    def backward(self, need_wgrad=True):
        x, out = self.x, self.out
        dz = out.grad16
        assert dz is not None, self.name
        dev = dz.device
        dkind = CONV_GEOM[self.kind][2]
        if x.needs_grad:
            # data gradient first: it is what the rest of the backward chain waits for
            wt = self._pack(dkind, self.Ci_pad, self.Co_pad, 1)[0]
            acc = x.grad is not None
            if not acc:
                x.grad = _e((x.N, x.H, x.W, x.C), dev)
            if self.kind == "s1":
                job = conv.conv_s1_dgrad(dz, wt, x.grad, 3, self.alpha, acc)
            elif self.kind == "up":
                job = conv.upconv_dgrad(dz, wt, x.grad, acc)
            else:
                assert not acc
                job = conv.conv_s2_dgrad(dz, wt, x.grad, self.alpha)
            ops.conv_gemm(job)
        if need_wgrad:
            self.tape.aux.run(lambda: self._wgrad(dz), dz)
        out.grad16 = None

    def _wgrad(self, dz):
        x = self.x
        dev = dz.device
        k, _f, _d, ntap, ukind = CONV_GEOM[self.kind]
        wk = WEIGHT_KERNEL.get(self.kind, k)
        dwt = _e((ntap, self.Co_pad, self.Ci_pad), dev)
        if self.kind == "s1":
            job = conv.conv_s1_wgrad(dz, x.hi, dwt, 3)
        elif self.kind == "up":
            job = conv.upconv_wgrad(dz, x.hi, dwt)
        else:
            job = conv.conv_s2_wgrad(dz, x.hi, dwt)
        ops.conv_gemm(job)
        if self.sn is not None and wk == k:
            # spectral norm: sum(dW_eff .* W_orig) comes out of the same pass that un-packs the gradient
            g = _e(tuple(self.w.shape), dev)
            dot = torch.zeros(1, device=dev)
            ops.unpack_conv_wgrad_dot(dwt, self.Co_pad * self.Ci_pad, self.Ci_pad, ukind, None, g,
                                      self.w.detach(), dot)
            self.dW = self.sn.backward(g, self.w, dot)
            return
        g = _e((self.Co, self.Ci, k, k) if wk != k else tuple(self.w.shape), dev)
        ops.unpack_conv_wgrad(dwt, self.Co_pad * self.Ci_pad, self.Ci_pad, ukind, None, g)
        if wk != k:     # zero-padded kernel: keep the taps the weight has
            g = g[:, :, :wk, :wk].contiguous().view(self.w.shape)
        self.dW = self.sn.backward(g, self.w) if self.sn is not None else g


class TemporalNode:
    """Conv3d (3, 1, 1) stride (s, 1, 1) pad (1, 0, 0), s = 1 or 2, optionally spectrally normalised (alpha =
    1/sigma): [B, T, HW, Ci] -> [B, To, HW, Co] on ``[B * T, H, W, C]`` activations.  Backward: stride 2 only."""

    def __init__(self, tape, x, B, weight, name, stride, sn=None, alpha=None):
        self.tape, self.x, self.B, self.w, self.name, self.stride = tape, x, B, weight, name, stride
        self.sn, self.alpha = sn, alpha
        self.Co, self.Ci = weight.shape[0], weight.shape[1]
        self.Co_pad, self.Ci_pad = rup(self.Co, 64), x.C
        assert rup(self.Ci, 64) == x.C and x.N % B == 0 and stride in (1, 2), name
        self.T = x.N // B
        self.To = self.T if stride == 1 else (self.T - 1) // 2 + 1
        self.out = T4(B * self.To, x.H, x.W, self.Co_pad)
        self.dW = None

    def _w4(self):
        w = self.w.detach()
        return w.view(w.shape[0], w.shape[1], 3, 1)

    def _pack(self, kindcode, rows_pad, cols_pad, planes, dtype=BF16):
        return pack_taps(self.tape.cache, self.w, self._w4, kindcode, rows_pad, cols_pad, planes, dtype)

    def _v(self, t, frames):
        return t.view(self.B, frames, self.x.H * self.x.W, t.shape[-1]) if t is not None else None

    def forward(self):
        t, x, out = self.tape, self.x, self.out
        wp = self._pack(0, self.Co_pad, self.Ci_pad, t.planes, t.dtype)
        out.f32 = _e((out.N, out.H, out.W, out.C), x.hi.device)
        xp = [self._v(p, self.T) for p in x.planes(t.planes)]
        if self.stride == 1:
            jobs = [conv.conv_t3s1_fwd(xp, wp, self._v(out.f32, self.To), self.alpha, dtype=t.dtype,
                                       splits=t.splits)]
        else:
            jobs = conv.conv_t3_fwd(xp, wp, self._v(out.f32, self.To), self.alpha, dtype=t.dtype)
        for job in jobs:
            ops.conv_gemm(job)

    def backward(self, need_wgrad=True):
        x, out = self.x, self.out
        dz = out.grad16
        assert dz is not None and self.stride == 2, self.name
        dz5 = self._v(dz, self.To)
        if x.needs_grad:
            assert x.grad is None
            wt = self._pack(1, self.Ci_pad, self.Co_pad, 1)[0]
            x.grad = _e((x.N, x.H, x.W, x.C), dz.device)
            for job in conv.conv_t3_dgrad(dz5, wt, self._v(x.grad, self.T), self.alpha):
                ops.conv_gemm(job)
        if need_wgrad:
            self.tape.aux.run(lambda: self._wgrad(dz5), dz)
        out.grad16 = None

    def _wgrad(self, dz5):
        dev = dz5.device
        # zeroed: the even- and odd-frame jobs accumulate into it (and for T == 1 taps 0 / 2 have no job at all)
        dwt = torch.zeros((3, self.Co_pad, self.Ci_pad), device=dev)
        for job in conv.conv_t3_wgrad(dz5, self._v(self.x.hi, self.T), dwt):
            ops.conv_gemm(job)
        g = _e((self.Co, self.Ci, 3, 1), dev)
        ops.unpack_conv_wgrad(dwt, self.Co_pad * self.Ci_pad, self.Ci_pad, 0, None, g)
        g = g.view(self.w.shape)
        self.dW = self.sn.backward(g, self.w) if self.sn is not None else g


class Im2colNode:
    """k x k convolution (stride, pad, no bias) of a few-channel NCHW fp32 image ``img`` as im2col + one GEMM,
    K = k*k*Ci padded to a multiple of 64, optionally spectrally normalised (alpha = 1/sigma, the epilogue
    scalar).  Output: T4 with the fp32 conv output; ``backward`` returns d(img) [n, Ci, H, W] fp32."""

    def __init__(self, tape, img, weight, name, stride, pad, sn=None, alpha=None):
        self.tape, self.img, self.w, self.name, self.stride, self.pad = tape, img, weight, name, stride, pad
        self.sn, self.alpha = sn, alpha
        n, Ci, H, W = img.shape
        self.Co, self.k = weight.shape[0], weight.shape[-1]
        assert weight.shape[1] == Ci, name
        self.K_pad = rup(self.k * self.k * Ci, 64)
        Ho, Wo = (H + 2 * pad - self.k) // stride + 1, (W + 2 * pad - self.k) // stride + 1
        self.out = T4(n, Ho, Wo, rup(self.Co, 64))
        self.col = self.dW = None

    def forward(self):
        t, out, Kp = self.tape, self.out, self.K_pad
        dev = self.img.device
        t16 = ops.TORCH16[t.dtype]
        col = T4(out.N, out.H, out.W, Kp)
        col.hi = _e((out.N, out.H, out.W, Kp), dev, t16)
        col.lo = _e((out.N, out.H, out.W, Kp), dev, t16) if t.planes == 2 else None
        ops.im2col_small(self.img.detach(), self.k, self.stride, self.pad, col.hi, col.lo, Kp, t.dtype)
        if self.sn is not None and self.alpha is None:
            self.alpha = self.sn.forward(self.w, t.training, t.need_grad)
        out.f32 = _e((out.N, out.H, out.W, out.C), dev)
        ops.conv_gemm(conv.gemm_nt([col.hi.view(-1, Kp), col.lo.view(-1, Kp) if col.lo is not None else None],
                                   pack_im2col_weight(t.cache, self.w, "fwd", Kp, t.planes, t.dtype),
                                   out.f32.view(-1, out.C), alpha=self.alpha, dtype=t.dtype, splits=t.splits))
        col.lo = None
        if t.need_grad:
            self.col = col      # the weight gradient multiplies with it

    def backward(self, need_wgrad=True, need_dx=True):
        """consumes out.grad16"""
        dz = self.out.grad16.view(-1, self.out.C)
        dev = dz.device
        Kp = self.K_pad
        if need_wgrad:
            def wgrad():
                d = _e((self.out.C, Kp), dev)
                ops.conv_gemm(conv.gemm_tn(dz, self.col.hi.view(-1, Kp), d))
                Ci = self.w.shape[1]
                g = d[:self.Co, :self.k * self.k * Ci].reshape(self.Co, -1, Ci).permute(0, 2, 1).contiguous()
                g = g.view(self.w.shape)
                self.dW = self.sn.backward(g, self.w) if self.sn is not None else g
            self.tape.aux.run(wgrad, dz)
        dx = None
        if need_dx:
            n, Ci, H, W = self.img.shape
            dcol = _e((dz.shape[0], Kp), dev)
            ops.conv_gemm(conv.gemm_nt([dz, None], pack_im2col_weight(self.tape.cache, self.w, "bwd", Kp), dcol,
                                       alpha=self.alpha))
            dx = _e((n, Ci, H, W), dev)
            ops.col2im_small(dcol, n, Ci, H, W, self.k, self.stride, self.pad, dx)
        self.out.grad16 = None
        return dx


class SpectralNorm:
    """Legacy torch spectral_norm semantics (1 power iteration per forward call in train mode,
    u/v buffers updated in place; reference model.py:5,19,79; SURVEY.md Appendix A)."""

    def __init__(self, u, v):
        self.u, self.v = u, v
        self.saved = None

    def forward(self, w_orig, training, need_grad):
        dev = w_orig.device
        R = w_orig.shape[0]
        w2d = w_orig.detach().view(R, -1)
        sig = _e((2,), dev)
        scratch = _e((R + w2d.shape[1],), dev)
        # u / v are updated in place once per call: calls of the same module that run on parallel
        # streams (real / fake / wrong-pair passes) iterate in issue order
        StateOrder.before(self.u)
        ops.spectral_sigma(w2d, self.u, self.v, training, sig[0:1], sig[1:2], scratch)
        if need_grad:
            # one cat kernel instead of two clone()s: device-to-device memcpy NODES of parallel
            # CUDA-graph branches execute in one shared order (like memset nodes), kernels do not
            uv = torch.cat((self.u.detach().reshape(-1), self.v.detach().reshape(-1)))
            self.saved = (uv[:R], uv[R:], sig)
        StateOrder.after(self.u)
        return sig[1:2]

    def backward(self, g, w_orig, dot=None):
        """``dot``: sum(g * w_orig) already accumulated by the caller -> one in-place pass"""
        u, v, sig = self.saved
        R = w_orig.shape[0]
        if dot is not None:
            ops.spectral_bwd_apply(g.view(R, -1), u, v, sig[0:1], dot, g.view(R, -1))
            return g
        dw = torch.empty_like(g)
        ops.spectral_bwd(g.view(R, -1), w_orig.detach().view(R, -1), u, v, sig[0:1], dw.view(R, -1),
                         _e((4,), g.device))
        return dw


class GemmNode:
    """out[rows, Npad] = x[rows, K] @ W^T for a Linear whose packed weight is supplied by
    ``pack(planes) -> [hi, lo]`` (row re-ordering / padding is the packer's business)."""

    def __init__(self, tape, x, n_out_pad, pack_fwd, pack_bwd, name, bn_stats=False):
        self.tape, self.x, self.name = tape, x, name
        self.bn_stats = bn_stats
        self.pack_fwd, self.pack_bwd = pack_fwd, pack_bwd
        self.out = T4(x.N, x.H, x.W, n_out_pad)
        self.npad = n_out_pad
        self.dwt = None

    def forward(self):
        t, x, out = self.tape, self.x, self.out
        dev = x.hi.device
        out.f32 = _e((out.N, out.H, out.W, out.C), dev)
        a = [p.view(x.rows, x.C) if p is not None else None for p in x.planes(t.planes)]
        job = conv.gemm_nt(a, self.pack_fwd(t.planes, t.dtype), out.f32.view(x.rows, self.npad), dtype=t.dtype,
                           splits=t.splits)
        attach_stats(t, job, out, self.bn_stats)
        ops.conv_gemm(job)

    def backward(self, need_wgrad=True):
        x, out = self.x, self.out
        dz = out.grad16.view(x.rows, self.npad)
        dev = dz.device
        if x.needs_grad:
            acc = x.grad is not None
            if not acc:
                x.grad = _e((x.N, x.H, x.W, x.C), dev)
            ops.conv_gemm(conv.gemm_nt([dz, None], [self.pack_bwd(), None], x.grad.view(x.rows, x.C),
                                       accumulate=acc))
        if need_wgrad:
            def wgrad():
                self.dwt = _e((self.npad, x.C), dev)
                ops.conv_gemm(conv.gemm_tn(dz, x.hi.view(x.rows, x.C), self.dwt))
            self.tape.aux.run(wgrad, dz)
        out.grad16 = None


# ------------------------------------------------------------------------------ BN / act node
def eval_affine(bn, C, chan_map, c_valid, eps=1e-5):
    """per-channel (scale, shift) of an eval-mode BatchNorm over the C (padded / re-ordered) channels
    of a kernel tensor: scale = gamma / sqrt(running_var + eps), shift = beta - running_mean * scale;
    channels beyond c_valid or mapped to -1 (padding) get 0 / 0, like cpcsv_bn_finalize."""
    gamma, beta, rmean, rvar, _ = bn
    dev = gamma.device
    sc = gamma.detach() / torch.sqrt(rvar + eps)
    sh = beta.detach() - rmean * sc
    pos = torch.arange(C, device=dev)
    idx = chan_map.long() if chan_map is not None else pos
    valid = (pos < c_valid) & (idx >= 0)
    src = idx.clamp(0, sc.numel() - 1)
    zero = torch.zeros((), device=dev)
    return (torch.where(valid, sc[src], zero).contiguous(), torch.where(valid, sh[src], zero).contiguous())


class BnActNode:
    """[BatchNorm (batch statistics)] -> activation -> [* (1 + mod)] -> operand planes / fp32."""

    def __init__(self, tape, z, bn, act, name, mod=None, want_f32=False, want_planes=True,
                 chan_map=None, c_valid=None, pre_bias=None, eps=1e-5):
        self.tape, self.z, self.bn, self.act, self.name, self.mod = tape, z, bn, act, name, mod
        self.eps = eps      # of the eval-mode normalisation (InceptionV3's BasicConv2d: 1e-3)
        # bias of the producing conv that was NOT added to z (a batch-statistics BatchNorm removes it;
        # only the eval-mode normalisation with running statistics has to account for it)
        self.pre_bias = pre_bias
        self.want_f32, self.want_planes, self.chan_map = want_f32, want_planes, chan_map
        self.c_valid = c_valid if c_valid is not None else (bn[0].numel() if bn else z.C)
        self.out = T4(z.N, z.H, z.W, z.C)
        self.stat = None
        self.dgamma = self.dbeta = None

    def forward(self):
        t, z, out = self.tape, self.z, self.out
        dev = z.f32.device
        zm = z.mat(z.f32)
        if self.want_f32:
            out.f32 = _e((z.N, z.H, z.W, z.C), dev)
        if self.want_planes:
            t16 = ops.TORCH16[t.dtype]
            out.hi = _e((z.N, z.H, z.W, z.C), dev, t16)
            out.lo = _e((z.N, z.H, z.W, z.C), dev, t16) if t.planes == 2 else None
        modm = z.mat(self.mod.f32) if self.mod is not None else None
        ym = z.mat(out.f32) if out.f32 is not None else None
        him = z.mat(out.hi) if out.hi is not None else None
        lom = z.mat(out.lo) if out.lo is not None else None
        scale = shift = None
        if self.bn is not None and not t.training:
            # eval mode (reference inference.py:88, trainer.py:161,177 call netG.eval() for the FID / SSIM
            # loops): normalise with the running statistics, no batch statistics, no state update
            if t.need_grad:
                raise NotImplementedError("cpcsv_b200: backward through eval-mode BatchNorm is not implemented "
                                          "(the reference only evaluates under torch.no_grad())")
            scale, shift = eval_affine(self.bn, z.C, self.chan_map, self.c_valid, self.eps)
            if self.pre_bias is not None:
                b = torch.zeros(z.C, device=dev)
                b[:self.pre_bias.numel()].copy_(self.pre_bias.detach())
                shift = shift + scale * b
        elif self.bn is not None:
            gamma, beta, rmean, rvar, nbt = self.bn
            if nbt is not None:
                t.counters.append(nbt)
            vec = _e((4, z.C), dev)
            self.stat = vec
            if z.stats is None:
                z.stats = t.stat_slot(z.C, dev)
            if not z.stats_done:
                ops.bn_stats(zm, z.stats.view(-1))
            StateOrder.before(rmean)
            ops.bn_norm_act_pack(zm, z.stats.view(-1), gamma.detach(), beta.detach(), rmean, rvar, self.chan_map,
                                 self.c_valid, vec, self.act, modm, ym, him, lom, t.dtype)
            StateOrder.after(rmean)
            if not t.need_grad and self.mod is None:
                z.f32 = None        # nothing reads the raw conv output again: release it early
            return
        ops.bn_act_pack(zm, scale, shift, self.act, modm, ym, him, lom, t.dtype)
        if not t.need_grad and self.mod is None:
            z.f32 = None        # nothing reads the raw conv output again: release it early

    def backward(self, need_param_grad=True):
        z, out = self.z, self.out
        dy = out.grad
        assert dy is not None, self.name
        dev = dy.device
        zm, dym = z.mat(z.f32), z.mat(dy)
        has_bn = self.bn is not None
        modm = z.mat(self.mod.f32) if self.mod is not None else None
        z.grad16 = _e((z.N, z.H, z.W, z.C), dev, torch.bfloat16)
        dmod16 = None
        if self.mod is not None:
            m = self.mod
            dmod16 = _e((m.N, m.H, m.W, m.C), dev, torch.bfloat16)
            m.grad16 = dmod16
        dmod16m = z.mat(dmod16) if dmod16 is not None else None
        sums = None
        if has_bn:
            vec = self.stat
            sums = self.tape.stat_slot(z.C, dev).view(-1)
            if need_param_grad:
                # every entry is written by the apply stage (all real channels are mapped)
                self.dgamma = torch.empty_like(self.bn[0])
                self.dbeta = torch.empty_like(self.bn[1])
            ops.bn_bwd_reduce(zm, dym, vec[2], vec[3], vec[0], vec[1], self.act, modm, sums)
        vec = self.stat if has_bn else (None, None, None, None)
        ops.bn_bwd_apply(zm, dym, vec[2], vec[3], vec[0], vec[1], self.chan_map, self.c_valid, self.act,
                         modm, sums, has_bn, dx=None, dx16=z.mat(z.grad16), dmod=None, dmod16=dmod16m,
                         dgamma=self.dgamma, dbeta=self.dbeta)
        out.grad = None


class Tape:
    """One network call.  With ``need_grad`` the forward GEMMs use bf16 hi/lo split operands
    (3 MMAs); a no-grad call (the fakes for the discriminator update, inference) uses single-pass
    fp16 operands -- SURVEY.md Appendix E: fp16, not bf16, keeps the discriminator gradients that
    are computed on those fakes within tolerance.

    ``split_k=False``: no forward GEMM splits its reduction (the nearest-x2 "up" convolution of the generator
    always picks its own split).  Split-K partial sums meet in fp32 atomics in
    whatever order they arrive; without them every output is bit-for-bit reproducible."""

    STAT_CHUNK = 1 << 15       # fp64 slots per zero-filled arena chunk (override per network call)

    def __init__(self, cache, training=True, need_grad=True, planes=None, dtype=None, stat_chunk=None,
                 split_k=True):
        self.cache, self.training, self.need_grad = cache, training, need_grad
        self.splits = None if split_k else 1    # the forward job builders' `splits` (None: conv.pick_splits)
        self._arena, self._arena_used = None, 0
        self._chunk = stat_chunk if stat_chunk is not None else self.STAT_CHUNK
        split = need_grad or NOGRAD_SPLIT
        self.planes = planes if planes is not None else (2 if split else 1)
        self.dtype = dtype if dtype is not None else (ops.BF16 if split else ops.FP16)
        self.nodes = []
        self.counters = []      # num_batches_tracked buffers to bump once the forward is done
        self.aux = AuxBranch()  # weight-gradient side branch of the backward pass

    def stat_slot(self, C, dev):
        """a zeroed fp64 [2, C] accumulator (BatchNorm sums of the forward / backward pass): slices of
        arena chunks that are zero-filled with ONE launch each, instead of one fill per layer"""
        n = 2 * C
        if self._arena is None or self._arena_used + n > self._arena.numel():
            self._arena = torch.zeros(max(self._chunk, n), device=dev, dtype=torch.float64)
            self._arena_used = 0
        s = self._arena[self._arena_used:self._arena_used + n].view(2, C)
        self._arena_used += n
        return s

    def finish_forward(self):
        """one multi-tensor launch for all `num_batches_tracked += 1` of this call"""
        if self.counters:
            StateOrder.before(self.counters[0])
            torch._foreach_add_(self.counters, 1)
            StateOrder.after(self.counters[0])
            self.counters = []
        if not self.need_grad:
            self.release()
        else:
            # the lo operand planes are only read by the forward GEMMs (backward GEMMs are
            # single-pass on the hi plane): give their memory back now
            for n in self.nodes:
                for t4 in (getattr(n, "out", None), getattr(n, "x", None)):
                    if t4 is not None:
                        t4.lo = None

    def release(self):
        """break the tape <-> node reference cycle so the activations are freed by reference
        counting right away instead of whenever Python's cycle collector runs"""
        self.aux.join()
        for n in self.nodes:
            n.tape = None
        self.nodes = []

    def add(self, node):
        self.nodes.append(node)
        node.forward()
        return node.out if hasattr(node, "out") else None
