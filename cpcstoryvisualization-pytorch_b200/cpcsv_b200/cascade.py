"""Kernel tapes of the CASCADE generator (reference ``cascade_model.py``; SURVEY.md section 8
row f2): the segmentation trunk runs first, its 1-channel mask is re-encoded by ``presample``
(conv3x3 1 -> nseg/16 + BN + ReLU) and four ``downBlock`` s (conv3x3 stride 2 WITH bias + BN +
ReLU), and the re-encoded features modulate the image trunk (``cascade_model.py:399-437``);
``train_autoencoder`` (``cascade_model.py:528-540``) is the mask auto-encoder built from the same
layers.  Every arithmetic step is one of the libcpcsv.so kernels the plain generator already uses:

* downBlock conv = engine.ConvNode's ``s2k3`` geometry: the 4x4 / stride-2 / pad-1 implicit GEMM of the
  discriminators with the 3x3 kernel embedded in the upper-left taps (same input coordinate
  ``2*o + k - 1``; the 4th row and column of the packed weight are zero), so forward, dgrad and wgrad
  reuse the parity-view jobs;
* its bias is directly followed by a batch-statistics BatchNorm, which removes it from the
  output: it is not added at all, its gradient is identically zero, and only the BatchNorm
  running mean sees it (``running_mean += momentum * bias`` after the statistics kernel);
* presample (1 input channel) = im2col'd K = 64 GEMM (engine.Im2colNode).

The intermediate activations the reference returns as ``latents`` (``cascade_model.py:441-445``)
are outputs of the autograd Function; their incoming gradients (latent-MSE losses,
``trainer.py:369-376``) are injected into the tape's gradient slots.
"""
import torch

from . import ops
from .engine import BnActNode, ConvNode, Im2colNode, StateOrder, Tape, rup
from .nets import _CACHE, TapeFn, TrunkRunner, _alias, _bn_tuple, _eval_needs_no_grad

BN_MOMENTUM = 0.1


class SegEncoder:
    """presample + downsample1..4_seg on one tape (cascade_model.py:312-320, 413-418)."""

    PARAM_NAMES = ["presample.0.weight", "presample.1.weight", "presample.1.bias"] + [
        "downsample%d_seg.%s" % (i, s) for i in range(1, 5) for s in ("0.weight", "0.bias", "1.weight", "1.bias")]

    def __init__(self, tape, G):
        self.tape, self.G = tape, G
        self.pre = self.pre_bn = None
        self.downs = []          # [(conv node, bn node, index)] for downsample1..4_seg

    def forward(self, seg, want_f32=True):
        """seg [n, 1, 64, 64] fp32 -> activations (g_seg1 4x4, g_seg2 8x8, g_seg3 16x16, g_seg4 32x32)"""
        tape, G = self.tape, self.G
        self.pre = Im2colNode(tape, seg, G.presample[0].weight, "presample", 1, 1)
        z = tape.add(self.pre)
        self.pre_bn = BnActNode(tape, z, _bn_tuple(G.presample[1]), ops.ACT_RELU, "presample.bn")
        a = tape.add(self.pre_bn)
        outs = []
        for i in range(1, 5):
            blk = getattr(G, "downsample%d_seg" % i)
            cn = ConvNode(tape, "s2k3", a, blk[0].weight, "downsample%d_seg" % i)
            zc = tape.add(cn)
            bn = BnActNode(tape, zc, _bn_tuple(blk[1]), ops.ACT_RELU, "downsample%d_seg.bn" % i,
                           want_f32=want_f32, pre_bias=blk[0].bias)
            a = tape.add(bn)
            if tape.training:
                # the conv bias only shifts the batch mean BatchNorm subtracts again
                rm = blk[1].running_mean
                StateOrder.before(rm)
                rm.add_(blk[0].bias.detach(), alpha=BN_MOMENTUM)
                StateOrder.after(rm)
            self.downs.append((cn, bn, i))
            outs.append(a)
        g4, g3, g2, g1 = outs
        return g1, g2, g3, g4

    def backward_level(self, i, need_w, pg):
        """BatchNorm + conv backward of downsample{i}_seg; False when its output has no gradient"""
        cn, bn, _ = self.downs[i - 1]
        if bn.out.grad is None:
            return False
        bn.backward(need_w)
        cn.backward(need_w)
        if need_w:
            pre = "downsample%d_seg." % i
            pg[pre + "1.weight"], pg[pre + "1.bias"] = bn.dgamma, bn.dbeta
            pg[pre + "0.bias"] = torch.zeros_like(getattr(self.G, "downsample%d_seg" % i)[0].bias)
            pg[pre + "0.weight"] = cn      # resolved to cn.dW after the aux branch joined
        return True

    def backward_presample(self, need_w, need_dx, pg):
        if self.pre_bn.out.grad is None:
            return None
        self.pre_bn.backward(need_w)
        dx = self.pre.backward(need_w, need_dx)
        if need_w:
            pg["presample.1.weight"], pg["presample.1.bias"] = self.pre_bn.dgamma, self.pre_bn.dbeta
            pg["presample.0.weight"] = self.pre
        return dx


def _resolve(pg):
    """weight gradients produced on the aux branch are read from their nodes after the join"""
    for k, v in list(pg.items()):
        if isinstance(v, (ConvNode, Im2colNode)):
            pg[k] = v.dW


def _nchw(t4, C):
    return t4.f32.permute(0, 3, 1, 2)[:, :C]


def _inject(t4, g, C):
    """add an incoming NCHW gradient of a latent output to the activation's fp32 NHWC gradient slot"""
    if g is None:
        return
    gn = g.permute(0, 2, 3, 1)
    if t4.grad is None:
        t4.grad = torch.zeros(t4.N, t4.H, t4.W, t4.C, device=g.device)
        t4.grad[..., :C].copy_(gn)
    else:
        t4.grad[..., :C].add_(gn)


class CascadeTrunkRunner(TrunkRunner):
    """fc_seg -> 4 seg up-blocks -> img_seg -> presample + 4 downBlocks -> image trunk modulated by
    seg_c(g_seg1) / seg_c1(g_seg2) -> img.

    Outputs: img [N,3,64,64], seg [N,1,64,64], then the latents (zmc_seg, h_seg1, h_seg2, h_seg3,
    g_seg1, g_seg2, g_seg3, g_seg4) as NCHW fp32 views."""

    def __init__(self, G, need_grad, want_seg):
        super().__init__(G, need_grad, want_seg)
        self.names = self.names + SegEncoder.PARAM_NAMES

    def apply(self, zmc_all):
        return TapeFn.apply(self, zmc_all, *[self.params[n] for n in self.names])

    def run_forward(self, zmc_all, *plist):
        G = self.G
        _eval_needs_no_grad(G, self.need_grad)
        N = zmc_all.shape[0]
        # Split bf16 operands (3 MMAs) also for the no-grad call: the image depends on the mask
        # through tanh -> re-encoder -> modulation, twice the depth of the plain generator, and
        # single-pass fp16 fakes (rel. error 4e-3 here vs 1.5e-3 there) push the discriminator
        # gradients computed on them below the 0.999 cosine bound (measured on the emulator).
        tape = Tape(_CACHE, training=G.training, need_grad=self.need_grad, planes=2, dtype=ops.BF16)
        self.tape = tape
        ngf, nseg = G.gf_dim, G.gf_dim_seg
        x0 = self._latent_planes(tape, zmc_all)
        nodes = {}

        def bn_of(seq_name, idx):
            return _bn_tuple(getattr(G, seq_name)[idx])

        fc_img, perm_img = self._fc_node(tape, x0, G.fc[0], ngf, "fc")
        z_fc = tape.add(fc_img)
        fc_seg, perm_seg = self._fc_node(tape, x0, G.fc_seg[0], nseg, "fc_seg")
        z_fs = tape.add(fc_seg)
        nodes["fc"], nodes["fc_seg"] = fc_img, fc_seg
        # segmentation trunk first (cascade_model.py:403-410)
        bn_fs = BnActNode(tape, z_fs, bn_of("fc_seg", 1), ops.ACT_RELU, "fc_seg.bn", chan_map=perm_seg,
                          c_valid=z_fs.C, want_f32=True)
        a_seg = _alias(tape.add(bn_fs), N, 4, 4, rup(nseg, 64))
        nodes["fc_seg.bn"] = bn_fs
        seg_acts = [a_seg]
        for i in range(1, 5):
            up_s = getattr(G, "upsample%d_seg" % i)
            cs = ConvNode(tape, "up", a_seg, up_s[1].weight, "upsample%d_seg" % i)
            z_s = tape.add(cs)
            bs = BnActNode(tape, z_s, _bn_tuple(up_s[2]), ops.ACT_RELU, "upsample%d_seg.bn" % i,
                           want_planes=True, want_f32=(i < 4))
            a_seg = tape.add(bs)
            seg_acts.append(a_seg)
            nodes.update({cs.name: cs, bs.name: bs})
        seg = self._head_fwd(a_seg, G.img_seg[0].weight, 1, "img_seg")
        # mask re-encoder (cascade_model.py:412-418)
        enc = SegEncoder(tape, G)
        g1, g2, g3, g4 = enc.forward(seg)
        # image trunk (cascade_model.py:420-437)
        c_segc = ConvNode(tape, "s1", g1, G.seg_c.weight, "seg_c")
        s0 = tape.add(c_segc)
        bn_fc = BnActNode(tape, z_fc, bn_of("fc", 1), ops.ACT_RELU, "fc.bn", mod=s0, chan_map=perm_img,
                          c_valid=z_fc.C)
        a_img = _alias(tape.add(bn_fc), N, 4, 4, rup(ngf, 64))
        self.alias = {"fc": a_img, "fc_seg": seg_acts[0]}
        nodes.update({"seg_c": c_segc, "fc.bn": bn_fc})
        for i in range(1, 5):
            up_i = getattr(G, "upsample%d" % i)
            ci = ConvNode(tape, "up", a_img, up_i[1].weight, "upsample%d" % i)
            z_i = tape.add(ci)
            mod = None
            if i == 1:
                c1 = ConvNode(tape, "s1", g2, G.seg_c1.weight, "seg_c1")
                mod = tape.add(c1)
                nodes["seg_c1"] = c1
            bi = BnActNode(tape, z_i, _bn_tuple(up_i[2]), ops.ACT_RELU, "upsample%d.bn" % i, mod=mod)
            a_img = tape.add(bi)
            nodes.update({ci.name: ci, bi.name: bi})
        img = self._head_fwd(a_img, G.img[0].weight, 3, "img")
        self.nodes, self.enc = nodes, enc
        self.a_img, self.a_seg, self.seg_acts, self.g_acts = a_img, a_seg, seg_acts, (g1, g2, g3, g4)
        self.img, self.seg = img, seg
        self.lat_channels = [nseg, nseg // 2, nseg // 4, nseg // 8, nseg, nseg // 2, nseg // 4, nseg // 8]
        lat_t4 = seg_acts[:4] + [g1, g2, g3, g4]
        latents = tuple(_nchw(t, c) for t, c in zip(lat_t4, self.lat_channels))
        tape.finish_forward()
        return (img, seg) + latents

    def run_backward(self, grads, needs):
        d_img, d_seg = grads[0], grads[1]
        d_h, d_g = grads[2:6], grads[6:10]
        G, nodes, enc = self.G, self.nodes, self.enc
        g1, g2, g3, g4 = self.g_acts
        ch = self.lat_channels
        pg = {}
        need_w = any(needs[1:])
        for t in self._all_acts():
            t.needs_grad = True

        def bn_conv_bwd(bn_name, conv_name, prefix_bn, prefix_conv):
            bn, cv = nodes[bn_name], nodes[conv_name]
            if bn.out.grad is None:
                return False
            bn.backward(need_w)
            pg[prefix_bn + ".weight"], pg[prefix_bn + ".bias"] = bn.dgamma, bn.dbeta
            cv.backward(need_w)
            pg[prefix_conv] = cv
            return True

        # image trunk, top down
        if d_img is not None:
            self._head_bwd(self.a_img, G.img[0].weight, self.img, d_img, need_w, pg, "img.0.weight")
        for i in (4, 3, 2, 1):
            bn_conv_bwd("upsample%d.bn" % i, "upsample%d" % i, "upsample%d.2" % i, "upsample%d.1.weight" % i)
        self._fc_bwd("fc", need_w, pg)
        # mask re-encoder, bottom (4x4) up.  The stride-2 data gradients overwrite their target, so
        # each of them is issued before the other contributions to the same activation.
        if nodes["seg_c"].out.grad16 is not None:
            nodes["seg_c"].backward(need_w)
            pg["seg_c.weight"] = nodes["seg_c"]
        _inject(g1, d_g[0], ch[4])
        enc.backward_level(4, need_w, pg)                 # -> g2.grad
        if nodes["seg_c1"].out.grad16 is not None:
            nodes["seg_c1"].backward(need_w)
            pg["seg_c1.weight"] = nodes["seg_c1"]
        _inject(g2, d_g[1], ch[5])
        enc.backward_level(3, need_w, pg)                 # -> g3.grad
        _inject(g3, d_g[2], ch[6])
        enc.backward_level(2, need_w, pg)                 # -> g4.grad
        _inject(g4, d_g[3], ch[7])
        enc.backward_level(1, need_w, pg)                 # -> presample activation
        d_mask = enc.backward_presample(need_w, True, pg)
        if d_mask is not None:
            d_seg = d_mask if d_seg is None else d_seg + d_mask
        # segmentation trunk, top down
        if d_seg is not None:
            self._head_bwd(self.a_seg, G.img_seg[0].weight, self.seg, d_seg, need_w, pg, "img_seg.0.weight")
        for i in (4, 3, 2, 1):
            if i < 4:
                _inject(self.seg_acts[i], d_h[i], ch[i])
            bn_conv_bwd("upsample%d_seg.bn" % i, "upsample%d_seg" % i, "upsample%d_seg.2" % i,
                        "upsample%d_seg.1.weight" % i)
        _inject(self.seg_acts[0], d_h[0], ch[0])
        self._fc_bwd("fc_seg", need_w, pg)
        self.tape.aux.join()
        _resolve(pg)
        dz = None
        if needs[0] and self.x0.grad is not None:
            dz = self.x0.grad.view(self.x0.N, self.x0.C)[:, :self.K]
        out = [dz]
        for n, need in zip(self.names, needs[1:]):
            out.append(pg.get(n) if need else None)
        self.tape.release()
        self.tape = self.nodes = self.alias = self.a_img = self.a_seg = self.x0 = None
        self.enc = self.seg_acts = self.g_acts = None
        return out


class AutoencoderRunner(TrunkRunner):
    """StoryGAN.train_autoencoder (cascade_model.py:528-540): mask [n,1,64,64] -> presample + 4
    downBlocks -> upsample1..4_seg -> img_seg -> reconstructed mask [n,1,64,64]."""

    def __init__(self, G, need_grad):
        self.G, self.need_grad = G, need_grad
        names = list(SegEncoder.PARAM_NAMES)
        for i in range(1, 5):
            names += ["upsample%d_seg.1.weight" % i, "upsample%d_seg.2.weight" % i, "upsample%d_seg.2.bias" % i]
        names += ["img_seg.0.weight"]
        self.names = names
        self.params = dict(G.named_parameters())

    def apply(self, mask):
        return TapeFn.apply(self, mask, *[self.params[n] for n in self.names])[0]

    def run_forward(self, mask, *plist):
        G = self.G
        _eval_needs_no_grad(G, self.need_grad)
        tape = Tape(_CACHE, training=G.training, need_grad=self.need_grad)
        self.tape = tape
        enc = SegEncoder(tape, G)
        g1, _g2, _g3, _g4 = enc.forward(mask, want_f32=False)
        a = g1
        self.ups = []
        for i in range(1, 5):
            up_s = getattr(G, "upsample%d_seg" % i)
            cs = ConvNode(tape, "up", a, up_s[1].weight, "upsample%d_seg" % i)
            z_s = tape.add(cs)
            bs = BnActNode(tape, z_s, _bn_tuple(up_s[2]), ops.ACT_RELU, "upsample%d_seg.bn" % i)
            a = tape.add(bs)
            self.ups.append((cs, bs, i))
        self.enc, self.a_top = enc, a
        self.rec = self._head_fwd(a, G.img_seg[0].weight, 1, "img_seg")
        tape.finish_forward()
        return self.rec

    def run_backward(self, grads, needs):
        (d_rec,) = grads
        G, enc = self.G, self.enc
        pg = {}
        need_w = any(needs[1:])
        for t in self._all_acts():
            t.needs_grad = True
        self._head_bwd(self.a_top, G.img_seg[0].weight, self.rec, d_rec, need_w, pg, "img_seg.0.weight")
        for cs, bs, i in reversed(self.ups):
            bs.backward(need_w)
            pg["upsample%d_seg.2.weight" % i], pg["upsample%d_seg.2.bias" % i] = bs.dgamma, bs.dbeta
            cs.backward(need_w)
            pg["upsample%d_seg.1.weight" % i] = cs
        for i in (4, 3, 2, 1):
            enc.backward_level(i, need_w, pg)
        dx = enc.backward_presample(need_w, bool(needs[0]), pg)
        self.tape.aux.join()
        _resolve(pg)
        out = [dx if needs[0] else None]
        for n, need in zip(self.names, needs[1:]):
            out.append(pg.get(n) if need else None)
        self.tape.release()
        self.tape = self.enc = self.ups = self.a_top = None
        return out
