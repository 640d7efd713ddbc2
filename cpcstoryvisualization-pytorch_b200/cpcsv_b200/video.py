"""Kernel tape of the order-consistency critic ``VideoEncoder`` (reference model.py:99-113, 150-210; the
``seq_consisten_model`` of ``STAGE1_D_STY_V2`` when ``cfg.USE_SEQ_CONSISTENCY``; SURVEY.md section 8 row f4).

Every Conv3d of the reference is (1, k, k) or (k, 1, 1), so on channels-last activations
``[B * T, H, W, C]`` each one is an implicit GEMM the tcgen05 kernel already runs:

* stem conv (1, 7, 7) stride (1, 2, 2), 3 input channels: im2col (K = 147 -> 192) + one GEMM
  (engine.Im2colNode);
* stem conv (1, 1, 1) with TEMPORAL padding 1 (model.py:109-111; T -> T + 2, the two new frames are zero
  before the BatchNorm and relu(beta) after it): a 1-tap GEMM written into frames 1..T of a zero-filled
  ``[B, T + 2, HW, C]`` tensor through the job's output strides;
* (1, 3, 3) stride (1, 2, 2) pad (0, 1, 1): engine.ConvNode's ``s2k3`` geometry, the 4x4 / stride-2 parity-view
  job with a zero 4th row / column (the cascade generator's downBlock geometry), frames folded into the batch
  dimension;
* (3, 1, 1) stride (2, 1, 1) pad (1, 0, 0): engine.TemporalNode, conv.conv_t3_* on ``[B, T, HW, C]`` views
  (even / odd frames).

All convs are spectrally normalised (1 / sigma is the GEMM's epilogue scalar), followed by a batch-statistics
BatchNorm3d (= per-channel statistics over all B*T*H*W rows) and ReLU / LeakyReLU(0.2): engine.BnActNode.
AdaptiveAvgPool3d(1) and the 4-layer detector (two spectral-norm Linears around a BatchNorm1d) are a few
hundred floats per story: fp32 kernels of cpcsv_b200.functions.
"""
import torch

from . import conv, ops
from .engine import T4, BnActNode, ConvNode, Im2colNode, SpectralNorm, Tape, TemporalNode, pack_taps, rup, _e
from .nets import _CACHE, TapeFn, _bn_tuple, _eval_bn_unsupported

# (index inside story_encoder, geometry) after the stem; model.py:155-189
LAYERS = ((1, "spatial"), (4, "temporal"), (7, "spatial"), (10, "temporal"), (13, "spatial"), (16, "temporal"),
          (19, "spatial"), (22, "temporal"))


class PointwiseNode:
    """Conv3d (1, 1, 1) with padding (1, 0, 0) (model.py:109-111): output frames 1..T = x W^T, frames 0 and
    T + 1 = 0"""

    def __init__(self, tape, x, B, weight, name, sn, alpha):
        self.tape, self.x, self.B, self.w, self.name, self.sn, self.alpha = tape, x, B, weight, name, sn, alpha
        self.Co, self.Ci = weight.shape[0], weight.shape[1]
        self.Co_pad, self.Ci_pad = rup(self.Co, 64), x.C
        assert rup(self.Ci, 64) == x.C and x.N % B == 0
        self.T = x.N // B
        self.out = T4(B * (self.T + 2), x.H, x.W, self.Co_pad)
        self.dW = None

    def _w4(self):
        w = self.w.detach()
        return w.view(w.shape[0], w.shape[1], 1, 1)

    def _pack(self, kindcode, rows_pad, cols_pad, planes, dtype=ops.BF16):
        return pack_taps(self.tape.cache, self.w, self._w4, kindcode, rows_pad, cols_pad, planes, dtype)

    def _v(self, t, frames):
        return t.view(self.B, frames, self.x.H * self.x.W, t.shape[-1]) if t is not None else None

    def _inner(self, t):
        return self._v(t, self.T + 2)[:, 1:self.T + 1]

    def forward(self):
        t, x, out = self.tape, self.x, self.out
        wp = self._pack(0, self.Co_pad, self.Ci_pad, t.planes, t.dtype)
        out.f32 = torch.zeros((out.N, out.H, out.W, out.C), device=x.hi.device)
        ops.conv_gemm(conv.conv_s1_fwd([self._v(p, self.T) for p in x.planes(t.planes)], wp,
                                       self._inner(out.f32), 1, self.alpha, dtype=t.dtype))

    def backward(self, need_wgrad=True):
        x, out = self.x, self.out
        dz = out.grad16
        assert dz is not None, self.name
        dzi = self._inner(dz)
        if x.needs_grad:
            assert x.grad is None
            wt = self._pack(1, self.Ci_pad, self.Co_pad, 1)[0]
            x.grad = _e((x.N, x.H, x.W, x.C), dz.device)
            ops.conv_gemm(conv.conv_s1_dgrad(dzi, wt, self._v(x.grad, self.T), 1, self.alpha))
        if need_wgrad:
            self.tape.aux.run(lambda: self._wgrad(dzi), dz)
        out.grad16 = None

    def _wgrad(self, dzi):
        dev = dzi.device
        dwt = _e((1, self.Co_pad, self.Ci_pad), dev)
        ops.conv_gemm(conv.conv_s1_wgrad(dzi, self._v(self.x.hi, self.T), dwt, 1))
        g = _e((self.Co, self.Ci, 1, 1), dev)
        ops.unpack_conv_wgrad(dwt, self.Co_pad * self.Ci_pad, self.Ci_pad, 0, None, g)
        self.dW = self.sn.backward(g.view(self.w.shape), self.w)


class VideoEncoderRunner:
    """story_encoder + pool of one VideoEncoder call: story [B, 3, T, 64, 64] fp32 -> latents [B, 512] fp32"""

    def __init__(self, V, need_grad):
        self.V, self.need_grad = V, need_grad
        names = ["story_encoder.0.0.weight_orig", "story_encoder.0.1.weight", "story_encoder.0.1.bias",
                 "story_encoder.0.3.weight_orig", "story_encoder.0.4.weight", "story_encoder.0.4.bias"]
        for idx, _geom in LAYERS:
            names += ["story_encoder.%d.weight_orig" % idx, "story_encoder.%d.weight" % (idx + 1),
                      "story_encoder.%d.bias" % (idx + 1)]
        self.names = names
        self.params = dict(V.named_parameters())

    def apply(self, story):
        return TapeFn.apply(self, story, *[self.params[n] for n in self.names])[0]

    def run_forward(self, story, *plist):
        V = self.V
        _eval_bn_unsupported(V)
        enc = V.story_encoder
        stem = enc[0]
        B, Cin, T, H, W = story.shape
        assert Cin == 3 and H % 32 == 0 and W % 32 == 0, "VideoEncoder: 3-channel frames, sides multiple of 32"
        # hi/lo split operands also without grad: the logits of a no-grad call are the regression TARGET of the
        # generator-side loss (miscc/utils.py:165-167), and the critic is a small part of the step
        tape = Tape(_CACHE, training=V.training, need_grad=self.need_grad, planes=2, dtype=ops.BF16)
        self.tape, self.shape = tape, (B, Cin, T, H, W)
        tr, ng = V.training, self.need_grad

        def sn_of(mod):
            s = SpectralNorm(mod.weight_u, mod.weight_v)
            return s, s.forward(mod.weight_orig, tr, ng)

        # frames as batch entries: n = b * T + t
        frames = story.detach().permute(0, 2, 1, 3, 4).contiguous().view(B * T, Cin, H, W)
        self.stem = Im2colNode(tape, frames, stem[0].weight_orig, "vstem.conv", 2, 3,
                               sn=SpectralNorm(stem[0].weight_u, stem[0].weight_v))
        z0 = tape.add(self.stem)
        bn0 = BnActNode(tape, z0, _bn_tuple(stem[1]), ops.ACT_RELU, "vstem.bn0")
        a = tape.add(bn0)
        sn, alpha = sn_of(stem[3])
        pw = PointwiseNode(tape, a, B, stem[3].weight_orig, "vstem.point", sn, alpha)
        z = tape.add(pw)
        bn1 = BnActNode(tape, z, _bn_tuple(stem[4]), ops.ACT_RELU, "vstem.bn1")
        a = tape.add(bn1)
        self.stem_nodes = (bn0, pw, bn1)
        self.layers = []
        for li, (idx, geom) in enumerate(LAYERS):
            sn, alpha = sn_of(enc[idx])
            if geom == "spatial":
                cn = ConvNode(tape, "s2k3", a, enc[idx].weight_orig, "venc%d" % idx, sn=sn, alpha=alpha,
                              bn_stats=True)
            else:
                cn = TemporalNode(tape, a, B, enc[idx].weight_orig, "venc%d" % idx, 2, sn=sn, alpha=alpha)
            z = tape.add(cn)
            last = li == len(LAYERS) - 1
            bn = BnActNode(tape, z, _bn_tuple(enc[idx + 1]), ops.ACT_LRELU, "venc%d.bn" % idx, want_f32=last,
                           want_planes=not last)
            a = tape.add(bn)
            self.layers.append((cn, bn, idx))
        self.feat = a
        tape.finish_forward()
        Cf = enc[LAYERS[-1][0]].weight_orig.shape[0]
        # AdaptiveAvgPool3d(1) (model.py:191,208): mean over the remaining frames and pixels of every story
        return a.f32.view(B, -1, a.C)[:, :, :Cf].mean(1)

    def run_backward(self, grads, needs):
        (dlat,) = grads
        pg = {}
        need_w = any(needs[1:])
        feat = self.feat
        B = self.shape[0]
        dev = dlat.device
        per = feat.N // B * feat.H * feat.W
        Cf = dlat.shape[1]
        g = torch.zeros(B, per, feat.C, device=dev)
        g[:, :, :Cf].copy_((dlat / per).unsqueeze(1).expand(B, per, Cf))
        feat.grad = g.view(feat.N, feat.H, feat.W, feat.C)
        for nd in self.tape.nodes:
            if hasattr(nd, "x"):
                nd.x.needs_grad = True
        for cn, bn, idx in reversed(self.layers):
            bn.backward(need_w)
            pg["story_encoder.%d.weight" % (idx + 1)] = bn.dgamma
            pg["story_encoder.%d.bias" % (idx + 1)] = bn.dbeta
            cn.backward(need_w)
            pg["story_encoder.%d.weight_orig" % idx] = cn.dW
        bn0, pw, bn1 = self.stem_nodes
        bn1.backward(need_w)
        pg["story_encoder.0.4.weight"], pg["story_encoder.0.4.bias"] = bn1.dgamma, bn1.dbeta
        pw.backward(need_w)
        bn0.backward(need_w)
        pg["story_encoder.0.1.weight"], pg["story_encoder.0.1.bias"] = bn0.dgamma, bn0.dbeta
        dx = self.stem.backward(need_w, bool(needs[0]))
        dstory = None
        if dx is not None:
            Bb, Cin, T, H, W = self.shape
            dstory = dx.view(Bb, T, Cin, H, W).permute(0, 2, 1, 3, 4)
        self.tape.aux.join()
        pg["story_encoder.0.0.weight_orig"] = self.stem.dW
        pg["story_encoder.0.3.weight_orig"] = pw.dW
        for cn, _bn, idx in self.layers:
            pg["story_encoder.%d.weight_orig" % idx] = cn.dW
        out = [dstory]
        for nme, need in zip(self.names, needs[1:]):
            out.append(pg.get(nme) if need else None)
        self.tape.release()
        self.tape = self.layers = self.stem_nodes = self.stem = self.feat = None
        return out
