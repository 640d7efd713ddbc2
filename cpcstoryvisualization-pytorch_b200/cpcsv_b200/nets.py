"""Network-level runners: build the kernel tape (engine.py) for one call of the generator
trunk, a discriminator encoder or the conditional-logits head, and expose it to autograd as
ONE ``torch.autograd.Function`` whose inputs are the activations plus every parameter.

Reference call sites: generator trunk ``model.py:379-407 / 445-470``; encoders
``model.py:498-514, 540-556, 582-598``; ``D_GET_LOGITS.forward`` ``model.py:86-97``.
"""
import torch

from . import conv, engine, ops
from .engine import T4, BnActNode, ConvNode, GemmNode, SpectralNorm, Tape, pack_im2col_weight, rup, _e, _row_pad_map

_CACHE = engine.WeightCache()


def weight_cache():
    return _CACHE


def invalidate_weight_cache():
    """Mark every packed operand plane stale (re-packed at its next use).  The cache validates
    entries against ``Tensor._version``; ``optim.PackedAdam`` keeps the planes current itself, and
    every other ``torch.optim`` step (fused optimisers do not bump ``_version``) invalidates the
    stepped parameters through the global post-step hook registered below.  Call this by hand after
    modifying parameters through any other path that bypasses the version counter (``.data``
    edits; ``miscc.utils.weights_init`` does it for you)."""
    _CACHE.invalidate()


def _install_optimizer_hook():
    try:
        from torch.optim.optimizer import register_optimizer_step_post_hook
    except ImportError as e:  # pragma: no cover - every supported torch has it
        raise RuntimeError("cpcsv_b200 needs torch.optim global step hooks (torch >= 2.0)") from e
    def hook(opt, args, kwargs):
        ids = {id(p) for g in opt.param_groups for p in g["params"]}
        # optim.PackedAdam has just rewritten the persistent planes itself
        _CACHE.invalidate_params(ids, keep_maintained=getattr(opt, "maintains_planes", False))

    register_optimizer_step_post_hook(hook)


_install_optimizer_hook()


def _conv_weights(module):
    """(weight, geometry) of the tensor-core convolutions of a StoryGAN or a discriminator"""
    out = []
    if hasattr(module, "upsample1"):
        for i in range(1, 5):
            out.append((getattr(module, "upsample%d" % i)[1].weight, "up"))
            out.append((getattr(module, "upsample%d_seg" % i)[1].weight, "up"))
        out += [(module.seg_c.weight, "s1"), (module.seg_c1.weight, "s1")]
    if hasattr(module, "encode_img"):
        for idx in (2, 5, 8):
            out.append((module.encode_img[idx].weight_orig, "s2"))
        out.append((module.get_cond_logits.outlogits[0].weight_orig, "s1"))
    return out


def fc_maps(G, C, dev):
    """fc emits feature j = c*16 + p (``view(-1, C, 4, 4)``, model.py:379); the trunk wants NHWC
    order j' = p*Cp + c with Cp = C rounded up to 64.  perm[j'] = j, or -1 for the padding
    channels (zero weight rows, zero BN scale)."""
    key = ("fcperm", C, str(dev))
    m = G._cpcsv_maps.get(key)
    if m is None:
        Cp = rup(C, 64)
        jp = torch.arange(16 * Cp, device=dev)
        c, p = jp % Cp, jp // Cp
        m = torch.where(c < C, c * 16 + p, torch.full_like(jp, -1)).to(torch.int32)
        G._cpcsv_maps[key] = m
    return m


def pack_fc_fwd(cache, G, lin, C, Kp, planes, dtype):
    """(cached) operand planes [16*Cp, Kp] of fc / fc_seg for the forward GEMM (rows re-ordered to NHWC).
    The two forms the step uses -- single-plane fp16 (no-grad pass) and bf16 hi/lo -- are persistent and
    kept current by optim.PackedAdam (cpcsv_adam_pack_fc)."""
    w = lin.weight
    K, Cp = w.shape[1], rup(C, 64)
    t16 = ops.TORCH16[dtype]
    if (planes, dtype) in ((1, ops.FP16), (2, ops.BF16)):
        def fill(val):
            if planes == 1:
                ops.adam_pack_fc(w.detach(), None, None, None, C, 16, Cp, Kp, fwd16=val[0])
            else:
                ops.adam_pack_fc(w.detach(), None, None, None, C, 16, Cp, Kp, fwd_hi=val[0], fwd_lo=val[1])

        def build():
            val = [_e((16 * Cp, Kp), w.device, t16), _e((16 * Cp, Kp), w.device, t16) if planes == 2 else None]
            fill(val)
            return val
        return cache.get((id(w), "fc_fwd", planes, dtype), w, build,
                         spec=("fc", "fwd16" if planes == 1 else "fwd", C, Cp, Kp), fill=fill)
    perm = fc_maps(G, C, w.device)

    def build_generic():
        hi = _e((16 * Cp, Kp), w.device, t16)
        lo = _e((16 * Cp, Kp), w.device, t16) if planes == 2 else None
        ops.pack_matrix(w.detach(), 16 * Cp, Kp, K, K, 1, perm, hi, lo, dtype)
        return [hi, lo]
    return cache.get((id(w), "fc_fwd", planes, dtype), w, build_generic)


def pack_fc_bwd(cache, G, lin, C, Kp):
    """(cached, persistent) transposed bf16 plane [Kp, 16*Cp] for the data-gradient GEMM"""
    w = lin.weight
    Cp = rup(C, 64)

    def fill(val):
        ops.adam_pack_fc(w.detach(), None, None, None, C, 16, Cp, Kp, bwd=val)

    def build():
        hi = _e((Kp, 16 * Cp), w.device, torch.bfloat16)
        fill(hi)
        return hi
    return cache.get((id(w), "fc_bwd", 1), w, build, spec=("fc", "bwd", C, Cp, Kp), fill=fill)


def _prefetch_fc(G, no_grad_forward, forward, backward):
    for lin, C in ((G.fc[0], G.gf_dim), (G.fc_seg[0], G.gf_dim_seg)):
        Kp = rup(lin.weight.shape[1], 64)
        if no_grad_forward:
            pack_fc_fwd(_CACHE, G, lin, C, Kp, 1, ops.FP16)
        if forward:
            pack_fc_fwd(_CACHE, G, lin, C, Kp, 2, ops.BF16)
        if backward:
            pack_fc_bwd(_CACHE, G, lin, C, Kp)


_PREFETCH_STREAMS = {}


def prefetch_weights(modules, forward=True, backward=True, no_grad_forward=False):
    """Re-pack the conv weights of `modules` (StoryGAN / discriminators) into their bf16 operand
    planes on a side stream, concurrently with whatever the current stream does next; consumers
    synchronise through the cache entries' events.  Returns a handle for ``join_prefetch`` (call
    it before the enclosing CUDA-graph capture / stage ends), or None on CPU."""
    mods = [m for m in modules if m is not None]
    if not mods or not next(mods[0].parameters()).is_cuda:
        return None
    main = torch.cuda.current_stream()
    side = _PREFETCH_STREAMS.get(main.device)
    if side is None:
        # lowest priority: the re-layout kernels are many small blocks that would otherwise fill
        # every SM's block slots and delay the latency-bound kernels of the critical path
        side = _PREFETCH_STREAMS[main.device] = torch.cuda.Stream(device=main.device, priority=0)
    side.wait_stream(main)
    with torch.cuda.stream(side):
        # in the order the step consumes them: no-grad generator pass, forward planes, backward planes
        gens = [m for m in mods if hasattr(m, "fc_seg")]
        if no_grad_forward:
            for G in gens:
                if hasattr(G, "presample"):     # cascade generator: its no-grad call uses the split planes
                    continue
                _prefetch_fc(G, True, False, False)
                for w, geom in _conv_weights(G):
                    engine.prefetch_conv_nograd(_CACHE, w, geom)
        for fwd, bwd in ((forward, False), (False, backward)):
            if not (fwd or bwd):
                continue
            for m in mods:
                if m in gens:
                    _prefetch_fc(m, False, fwd, bwd)
                for w, geom in _conv_weights(m):
                    engine.prefetch_conv(_CACHE, w, geom, fwd, bwd)
    return side


def sync_point(streams=None, reset_state_order=True):
    """side streams (`streams`; None = all of them) have been joined into the current one:
    forget their cross-stream events.  `reset_state_order=False` while other streams that touch
    ordered module state are still running detached."""
    if reset_state_order:
        engine.StateOrder.reset()
        # Only then may the cache forget who packed what: "joined into the current stream" orders the pack before
        # every LATER consumer only if that consumer descends from the current stream.  A detached branch (it waits
        # for the stage's start event, not for this join) or a later branch of an enclosing fork does not -- found by
        # tests/streamcheck.py on the cascade generator: the early generator forward read head / mask-conv planes that
        # the no-grad call had packed on another stream, without waiting for the pack.
        _CACHE.mark_synced(streams)


def join_prefetch(handle):
    if handle is not None:
        torch.cuda.current_stream().wait_stream(handle)
        _CACHE.mark_synced([handle])


class TapeFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, runner, *tensors):
        ctx.runner = runner
        # outputs nothing downstream uses (the mask of a sample_videos call, unused latents) come
        # back as None, not as zero tensors: their branch of the backward pass is skipped
        ctx.set_materialize_grads(False)
        outs = runner.run_forward(*tensors)
        return outs if isinstance(outs, tuple) else (outs,)

    @staticmethod
    def backward(ctx, *grads):
        runner = ctx.runner
        ctx.runner = None
        return (None,) + tuple(runner.run_backward(grads, ctx.needs_input_grad[1:]))


def _bn_tuple(bn):
    return (bn.weight, bn.bias, bn.running_mean, bn.running_var, bn.num_batches_tracked)


def _eval_bn_unsupported(mod):
    """discriminators: the reference never calls .eval() on them (only on netG, for the FID / SSIM loops)"""
    if not mod.training:
        raise RuntimeError("cpcsv_b200: eval-mode discriminators (running statistics, frozen spectral-norm "
                           "vectors) are not part of the accelerated path; the reference only ever calls "
                           ".eval() on the generator (inference.py:88, trainer.py:161,177)")


def _eval_needs_no_grad(G, need_grad):
    """generator in eval mode (running statistics): forward only"""
    if not G.training and need_grad:
        raise RuntimeError("cpcsv_b200: the eval-mode generator runs under torch.no_grad() only "
                           "(reference inference.py:88-89, trainer.py:161-162)")


# =============================================================================== generator trunk
class TrunkRunner:
    """fc / fc_seg -> 4 up-blocks per branch with seg_c / seg_c1 modulation -> img / img_seg.

    Inputs of the Function: zmc_all [N, ninput] and the parameters in ``self.names`` order.
    Outputs: img [N,3,64,64], seg [N,1,64,64] (NCHW fp32, tanh range)."""

    @staticmethod
    def parameter_names():
        names = ["fc.0.weight", "fc.1.weight", "fc.1.bias"]
        for i in range(1, 5):
            names += ["upsample%d.1.weight" % i, "upsample%d.2.weight" % i, "upsample%d.2.bias" % i]
        names += ["img.0.weight", "seg_c.weight", "seg_c1.weight",
                  "fc_seg.0.weight", "fc_seg.1.weight", "fc_seg.1.bias"]
        for i in range(1, 5):
            names += ["upsample%d_seg.1.weight" % i, "upsample%d_seg.2.weight" % i,
                      "upsample%d_seg.2.bias" % i]
        names += ["img_seg.0.weight"]
        return names

    def __init__(self, G, need_grad, want_seg):
        self.G, self.need_grad, self.want_seg = G, need_grad, want_seg
        self.names = self.parameter_names()
        self.params = dict(G.named_parameters())

    def apply(self, zmc_all):
        return TapeFn.apply(self, zmc_all, *[self.params[n] for n in self.names])

    # ---------------------------------------------------------------- helpers
    def _fc_node(self, tape, x0, lin, C, name):
        G, Kp = self.G, x0.C
        perm = fc_maps(G, C, lin.weight.device)
        node = GemmNode(tape, x0, 16 * rup(C, 64),
                        lambda planes, dtype: pack_fc_fwd(tape.cache, G, lin, C, Kp, planes, dtype),
                        lambda: pack_fc_bwd(tape.cache, G, lin, C, Kp), name, bn_stats=True)
        return node, perm

    def _latent_planes(self, tape, zmc_all):
        """latent [N, K] fp32 -> operand planes (zero padded to a multiple of 64 columns)"""
        dev = zmc_all.device
        N, K = zmc_all.shape
        Kp = rup(K, 64)
        t16 = ops.TORCH16[tape.dtype]
        x0 = T4(N, 1, 1, Kp)
        x0.hi = torch.zeros(N, 1, 1, Kp, device=dev, dtype=t16)
        x0.lo = torch.zeros(N, 1, 1, Kp, device=dev, dtype=t16) if tape.planes == 2 else None
        zc = zmc_all.detach().contiguous()
        ops.bn_act_pack(_pad4(zc), None, None, ops.ACT_NONE, hi=x0.hi.view(N, Kp)[:, :rup(K, 4)],
                        lo=x0.lo.view(N, Kp)[:, :rup(K, 4)] if x0.lo is not None else None,
                        dtype=tape.dtype)
        x0.needs_grad = self.need_grad
        self.x0, self.K = x0, K
        return x0

    # ---------------------------------------------------------------- forward
    def run_forward(self, zmc_all, *plist):
        G = self.G
        _eval_needs_no_grad(G, self.need_grad)
        N, K = zmc_all.shape
        tape = Tape(_CACHE, training=G.training, need_grad=self.need_grad, stat_chunk=1 << 18)
        self.tape = tape
        self.sink = engine.grad_sink() if self.need_grad else None
        if self.sink is not None:
            # this call's backward pass will offer one contribution per parameter (see run_backward)
            self.sink.announce([self.params[n] for n in self.names])
        ngf, nseg = G.gf_dim, G.gf_dim_seg
        x0 = self._latent_planes(tape, zmc_all)

        nodes = {}

        def bn_of(seq_name, idx):
            return _bn_tuple(getattr(G, seq_name)[idx])

        # image branch head of the trunk
        fc_img, perm_img = self._fc_node(tape, x0, G.fc[0], ngf, "fc")
        z_fc = tape.add(fc_img)
        fc_seg, perm_seg = self._fc_node(tape, x0, G.fc_seg[0], nseg, "fc_seg")
        z_fs = tape.add(fc_seg)
        nodes["fc"], nodes["fc_seg"] = fc_img, fc_seg
        bn_fs = BnActNode(tape, z_fs, bn_of("fc_seg", 1), ops.ACT_RELU, "fc_seg.bn", chan_map=perm_seg,
                          c_valid=z_fs.C)
        a_seg = _alias(tape.add(bn_fs), N, 4, 4, rup(nseg, 64))
        c_segc = ConvNode(tape, "s1", a_seg, G.seg_c.weight, "seg_c")
        s0 = tape.add(c_segc)
        bn_fc = BnActNode(tape, z_fc, bn_of("fc", 1), ops.ACT_RELU, "fc.bn", mod=s0, chan_map=perm_img,
                          c_valid=z_fc.C)
        a_img = _alias(tape.add(bn_fc), N, 4, 4, rup(ngf, 64))
        self.alias = {"fc": a_img, "fc_seg": a_seg}
        nodes.update({"fc_seg.bn": bn_fs, "seg_c": c_segc, "fc.bn": bn_fc})
        for i in range(1, 5):
            up_s = getattr(G, "upsample%d_seg" % i)
            cs = ConvNode(tape, "up", a_seg, up_s[1].weight, "upsample%d_seg" % i, bn_stats=True)
            z_s = tape.add(cs)
            bs = BnActNode(tape, z_s, _bn_tuple(up_s[2]), ops.ACT_RELU, "upsample%d_seg.bn" % i,
                           want_planes=True)
            a_seg = tape.add(bs)
            up_i = getattr(G, "upsample%d" % i)
            ci = ConvNode(tape, "up", a_img, up_i[1].weight, "upsample%d" % i, bn_stats=True)
            z_i = tape.add(ci)
            mod = None
            if i == 1:
                c1 = ConvNode(tape, "s1", a_seg, G.seg_c1.weight, "seg_c1")
                mod = tape.add(c1)
                nodes["seg_c1"] = c1
            bi = BnActNode(tape, z_i, _bn_tuple(up_i[2]), ops.ACT_RELU, "upsample%d.bn" % i, mod=mod)
            a_img = tape.add(bi)
            nodes.update({cs.name: cs, bs.name: bs, ci.name: ci, bi.name: bi})
        self.nodes = nodes
        self.a_img, self.a_seg = a_img, a_seg
        img = self._head_fwd(a_img, G.img[0].weight, 3, "img")
        seg = self._head_fwd(a_seg, G.img_seg[0].weight, 1, "img_seg")
        self.img, self.seg = img, seg
        tape.finish_forward()
        return img, seg

    def _head_pack(self, w):
        """3x3 head conv weight as the B operand of the im2col'd-gradient GEMM: [Ci_pad, 64] with
        column tap*Co + co"""
        Co, Ci = w.shape[0], w.shape[1]
        Cip = rup(Ci, 64)

        def build():
            w2 = w.detach().permute(1, 2, 3, 0).reshape(Ci, 9 * Co).contiguous()   # [ci, tap*Co+co]
            hi = _e((Cip, 64), w.device, torch.bfloat16)
            ops.pack_matrix(w2, Cip, 64, 9 * Co, 9 * Co, 1, None if Cip == Ci else _row_pad_map(Ci, Cip, w.device),
                            hi, None)
            return hi
        return _CACHE.get((id(w), "head_bwd", 1, ops.BF16), w, build)

    def _head_pack_fwd(self, w, planes, dtype):
        """3x3 head conv weight as the B operand of the pixel-major forward GEMM: [Npad, Ci_pad] with row
        tap*Co + co = w[co, :, tap] (Npad = 9*Co rounded up to 16)"""
        Co, Ci = w.shape[0], w.shape[1]
        Cip, Np = rup(Ci, 64), rup(9 * Co, 16)

        def build():
            w2 = w.detach().permute(2, 3, 0, 1).reshape(9 * Co, Ci).contiguous()    # [tap*Co + co, ci]
            t16 = ops.TORCH16[dtype]
            hi = _e((Np, Cip), w.device, t16)
            lo = _e((Np, Cip), w.device, t16) if planes == 2 else None
            ops.pack_matrix(w2, Np, Cip, Ci, Ci, 1, _row_pad_map(9 * Co, Np, w.device), hi, lo, dtype)
            return [hi, lo]
        return _CACHE.get((id(w), "head_fwd", planes, dtype), w, build)

    def _head_fwd(self, a, w, Co, name):
        """img / img_seg: conv3x3 -> tanh with 3 / 1 output channels (reference model.py:272-274, 298-300):
        one pixel-major tensor-core GEMM Z[p, tap*Co + co] (the activation is read once, N = 9*Co padded to
        16 / 32) and a gather-tanh kernel over the L2-resident Z.  In the step 21.33 vs 21.47 ms against the
        direct CUDA-core kernel of round 1 (gpurun_out r02_c6)."""
        dev = a.hi.device
        tp = self.tape
        y = _e((a.N, Co, a.H, a.W), dev)
        wp = self._head_pack_fwd(w, tp.planes, tp.dtype)
        z = _e((a.rows, wp[0].shape[0]), dev)
        planes = [a.hi.view(a.rows, a.C), a.lo.view(a.rows, a.C) if tp.planes == 2 else None]
        ops.conv_gemm(conv.gemm_nt(planes, wp, z, dtype=tp.dtype))
        ops.head_gather_tanh(z, a.N, a.H, a.W, Co, y)
        return y

    def _head_bwd(self, a, w, y, dy, need_w, pg, name):
        """accumulates d(a) into a.grad; the weight gradient goes to pg[name] (aux branch)"""
        dev = y.device
        Co, Ci = w.shape[0], w.shape[1]
        col = _e((a.rows, 64), dev, torch.bfloat16)
        ops.tanh_bwd_im2col(dy, y, col)
        acc = a.grad is not None
        if not acc:
            a.grad = _e((a.N, a.H, a.W, a.C), dev)
        ops.conv_gemm(conv.gemm_nt([col, None], [self._head_pack(w), None], a.grad.view(a.rows, a.C),
                                   accumulate=acc))
        if need_w:
            def wgrad():
                d = _e((a.C, 64), dev)
                ops.conv_gemm(conv.gemm_tn(a.hi.view(a.rows, a.C), col, d))
                pg[name] = d[:Ci, :9 * Co].reshape(Ci, 3, 3, Co).permute(3, 0, 1, 2).contiguous()
            self.tape.aux.run(wgrad, col)

    # ---------------------------------------------------------------- backward
    def run_backward(self, grads, needs):
        d_img, d_seg = grads
        G, nodes = self.G, self.nodes
        pg = {}
        need_w = any(needs[1:])
        for t in self._all_acts():
            t.needs_grad = True
        if d_img is not None:
            self._head_bwd(self.a_img, G.img[0].weight, self.img, d_img, need_w, pg, "img.0.weight")
        seg_tail = d_seg is not None
        if seg_tail:
            self._head_bwd(self.a_seg, G.img_seg[0].weight, self.seg, d_seg, need_w, pg, "img_seg.0.weight")

        taken, offered = set(), set()
        need_of = dict(zip(self.names, needs[1:]))

        def offer(*names):
            """hand finished parameter gradients to the optimiser's gradient sink (engine.grad_sink) on the weight-
            gradient side branch, i.e. after the kernels that produce them"""
            if self.sink is None:
                return

            def run():
                for n in names:
                    if n not in offered and need_of.get(n):
                        offered.add(n)
                        if self.sink.offer(self.params[n], pg.get(n)):
                            taken.add(n)
            self.tape.aux.run(run)

        if d_img is not None:
            offer("img.0.weight")

        def bn_conv_bwd(bn_name, conv_name, prefix_bn, prefix_conv):
            bn, cv = nodes[bn_name], nodes[conv_name]
            if bn.out.grad is None:
                return False
            bn.backward(need_w)
            pg[prefix_bn + ".weight"], pg[prefix_bn + ".bias"] = bn.dgamma, bn.dbeta
            cv.backward(need_w)
            pg[prefix_conv] = cv.dW
            offer(prefix_bn + ".weight", prefix_bn + ".bias", prefix_conv)
            return True

        # image branch, top down; level 1 also emits the seg_c1 gradient, level 0 seg_c's
        for i in (4, 3, 2, 1):
            bn_conv_bwd("upsample%d.bn" % i, "upsample%d" % i, "upsample%d.2" % i, "upsample%d.1.weight" % i)
            if i == 1 and nodes["seg_c1"].out.grad16 is not None:
                nodes["seg_c1"].backward(need_w)
                pg["seg_c1.weight"] = nodes["seg_c1"].dW
                offer("seg_c1.weight")
        self._fc_bwd("fc", need_w, pg)
        offer("fc.1.weight", "fc.1.bias", "fc.0.weight")
        if nodes["seg_c"].out.grad16 is not None:
            nodes["seg_c"].backward(need_w)
            pg["seg_c.weight"] = nodes["seg_c"].dW
            offer("seg_c.weight")
        if seg_tail:
            offer("img_seg.0.weight")
        for i in (4, 3, 2, 1):
            bn_conv_bwd("upsample%d_seg.bn" % i, "upsample%d_seg" % i, "upsample%d_seg.2" % i,
                        "upsample%d_seg.1.weight" % i)
        self._fc_bwd("fc_seg", need_w, pg)
        offer(*self.names)        # whatever is left (layers without a gradient in this call offer None)
        self.tape.aux.join()
        dz = None
        if needs[0] and self.x0.grad is not None:
            dz = self.x0.grad.view(self.x0.N, self.x0.C)[:, :self.K]
        out = [dz]
        for n, need in zip(self.names, needs[1:]):
            out.append(pg.get(n) if need and n not in taken else None)
        self.tape.release()
        self.tape = self.nodes = self.alias = self.a_img = self.a_seg = self.x0 = self.sink = None
        return out

    def _all_acts(self):
        seen = []
        for nd in self.tape.nodes:
            if hasattr(nd, "x"):
                seen.append(nd.x)
        return seen

    def _fc_bwd(self, name, need_w, pg):
        bn, fc = self.nodes[name + ".bn"], self.nodes[name]
        al = self.alias[name]
        if al.grad is None:
            return
        bn.out.grad = al.grad.view(bn.out.N, 1, 1, bn.out.C)
        bn.backward(need_w)
        pg[name + ".1.weight"], pg[name + ".1.bias"] = bn.dgamma, bn.dbeta
        fc.backward(need_w)
        if need_w:
            lin = getattr(self.G, name)[0]
            C = lin.weight.shape[0] // 16
            perm = fc_maps(self.G, C, lin.weight.device)

            def scatter():      # after the weight-gradient GEMM, on the same branch
                dw = torch.empty_like(lin.weight)
                ops.scatter_rows_f32(fc.dwt, perm, dw, fc.npad, lin.weight.shape[1])
                pg[name + ".0.weight"] = dw
            self.tape.aux.run(scatter)


def _alias(t, N, H, W, C):
    """the same buffers seen with another NHWC shape (fc output [N, 16C] -> [N, 4, 4, C])"""
    a = T4(N, H, W, C)
    for f in ("f32", "hi", "lo"):
        v = getattr(t, f)
        if v is not None:
            setattr(a, f, v.view(N, H, W, C))
    return a


def _pad4(x):
    """[M, K] fp32 -> same values with K padded to a multiple of 4 (zero columns)."""
    M, K = x.shape
    Kp = rup(K, 4)
    if Kp == K:
        return x
    out = torch.zeros(M, Kp, device=x.device)
    out[:, :K].copy_(x)
    return out


# =============================================================================== D encoder
class EncoderRunner:
    """encode_img: conv4x4 s2 -> LeakyReLU (one direct kernel, csrc/enc0.cu), then 3 x
    [SN conv4x4 s2 -> BN -> LeakyReLU].  Input x [n, C, 64, 64] fp32 (any strides); output
    features [n, 8*ndf, 4, 4] fp32 as a channels-last view."""

    def __init__(self, D, need_grad):
        self.D, self.need_grad = D, need_grad
        enc = D.encode_img
        self.sn0 = hasattr(enc[0], "weight_orig")
        names = ["encode_img.0.weight_orig" if self.sn0 else "encode_img.0.weight"]
        for idx in (2, 5, 8):
            names += ["encode_img.%d.weight_orig" % idx, "encode_img.%d.weight" % (idx + 1),
                      "encode_img.%d.bias" % (idx + 1)]
        self.names = names
        self.params = dict(D.named_parameters())

    def apply(self, x):
        return TapeFn.apply(self, x, *[self.params[n] for n in self.names])[0]

    def _w0(self):
        enc0 = self.D.encode_img[0]
        return enc0.weight_orig if self.sn0 else enc0.weight

    def run_forward(self, x, *plist):
        D = self.D
        n, Cin, H, W = x.shape
        w0 = self._w0()
        Cop = rup(w0.shape[0], 64)
        if not (Cop <= 128 and Cin in (1, 3) and H % 4 == 0 and W % 64 == 0):
            raise NotImplementedError(
                "cpcsv_b200: the first discriminator layer (csrc/enc0.cu) takes at most 128 output channels "
                "(DF_DIM <= 128) and 1- or 3-channel images with H %% 4 == 0 and W %% 64 == 0; got %d output "
                "channels, %d x %d x %d images" % (w0.shape[0], Cin, H, W))
        _eval_bn_unsupported(D)
        enc = D.encode_img
        dev = x.device
        tape = Tape(_CACHE, training=D.training, need_grad=self.need_grad, planes=2, dtype=ops.BF16)
        self.tape = tape
        self.x_shape = (n, Cin, H, W)
        xd = x.detach()
        Ho, Wo = H // 2, W // 2
        sns = [SpectralNorm(enc[idx].weight_u, enc[idx].weight_v) for idx in (2, 5, 8)]
        self.sn_first = SpectralNorm(enc[0].weight_u, enc[0].weight_v) if self.sn0 else None
        alpha0 = self.sn_first.forward(w0, D.training, self.need_grad) if self.sn_first is not None else None
        self.alpha0, self.x0 = alpha0, xd
        alphas = [sn.forward(enc[idx].weight_orig, D.training, self.need_grad) for sn, idx in zip(sns, (2, 5, 8))]
        # layer 0 in ONE launch: conv + 1/sigma + LeakyReLU + hi/lo planes
        a = T4(n, Ho, Wo, Cop)
        a.hi = _e((n, Ho, Wo, Cop), dev, torch.bfloat16)
        a.lo = _e((n, Ho, Wo, Cop), dev, torch.bfloat16)
        ops.enc0_lrelu_fwd(xd, w0.detach(), alpha0, 0.2, a.hi, a.lo, Cop)
        self.a0 = a
        self.layers = []
        for li, idx in enumerate((2, 5, 8)):
            cmod, bmod = enc[idx], enc[idx + 1]
            cn = ConvNode(tape, "s2", a, cmod.weight_orig, "enc%d" % idx, sn=sns[li], alpha=alphas[li],
                          bn_stats=True)
            z = tape.add(cn)
            last = (li == 2)
            bn = BnActNode(tape, z, _bn_tuple(bmod), ops.ACT_LRELU, "enc%d.bn" % idx, want_f32=last,
                           want_planes=not last)
            a = tape.add(bn)
            self.layers.append((cn, bn, idx))
        self.feat = a
        Cf = enc[8].weight_orig.shape[0]
        tape.finish_forward()
        self.a0.lo = None
        return a.f32.permute(0, 3, 1, 2)[:, :Cf]

    def run_backward(self, grads, needs):
        (dfeat,) = grads
        D = self.D
        pg = {}
        need_w = any(needs[1:])
        feat = self.feat
        dev = dfeat.device
        Cf = D.encode_img[8].weight_orig.shape[0]
        g = torch.zeros(feat.N, feat.H, feat.W, feat.C, device=dev)
        g[..., :Cf].copy_(dfeat.permute(0, 2, 3, 1))
        feat.grad = g
        for nd in self.tape.nodes:
            if hasattr(nd, "x"):
                nd.x.needs_grad = True
        w0 = self._w0()
        Co, Ci = w0.shape[0], w0.shape[1]
        K = 16 * Ci
        a0 = self.a0
        a0.needs_grad = True
        col_hi = None
        if need_w:
            # the im2col matrix the layer-0 weight gradient multiplies with: built on the side branch at the START
            # of the backward pass (it only needs the input image), consumed there at the end
            n, Cin, H, W = self.x_shape
            col_hi = _e((n * (H // 2) * (W // 2), 64), dev, torch.bfloat16)
            self.tape.aux.run(lambda: ops.im2col_small(self.x0, 4, 2, 1, col_hi, None, 64))
        for cn, bn, idx in reversed(self.layers):
            bn.backward(need_w)
            pg["encode_img.%d.weight" % (idx + 1)] = bn.dgamma
            pg["encode_img.%d.bias" % (idx + 1)] = bn.dbeta
            cn.backward(need_w)
            pg["encode_img.%d.weight_orig" % idx] = cn.dW
        # layer 0
        dz0 = _e((a0.N, a0.H, a0.W, a0.C), dev, torch.bfloat16)
        ops.lrelu_bwd16(a0.grad, a0.hi, 0.2, dz0)
        a0.grad = None
        Cop = a0.C
        dz0m = dz0.view(-1, Cop)
        if need_w:
            def wgrad0():
                d = _e((Cop, 64), dev)
                ops.conv_gemm(conv.gemm_tn(dz0m, col_hi, d))
                gw = d[:Co, :K].reshape(Co, 4, 4, Ci).permute(0, 3, 1, 2).contiguous()
                if self.sn_first is not None:
                    gw = self.sn_first.backward(gw, w0)
                pg[self.names[0]] = gw
            self.tape.aux.run(wgrad0, dz0)
        dx = None
        if needs[0]:
            n, Cin, H, W = self.x_shape
            dcol = _e((dz0m.shape[0], 64), dev)
            # layer-0 weight as the B operand: [64, Co_pad] with row tap*Ci + c
            ops.conv_gemm(conv.gemm_nt([dz0m, None], pack_im2col_weight(_CACHE, w0, "bwd", 64), dcol,
                                       alpha=self.alpha0))
            dx = _e((n, Cin, H, W), dev)
            ops.col2im_small(dcol, n, Cin, H, W, 4, 2, 1, dx)
        out = [dx]
        for nme, need in zip(self.names, needs[1:]):
            out.append(pg.get(nme) if need else None)
        self.tape.release()
        self.tape = self.layers = self.feat = self.a0 = self.x0 = None
        return out


# =============================================================================== logits head
class LogitsRunner:
    """D_GET_LOGITS: [h_code | c_code tiled 4x4] -> SN conv3x3 -> BN -> LeakyReLU ->
    SN conv4x4 s4 (+bias) -> sigmoid -> [n]."""

    def __init__(self, L, need_grad):
        self.L, self.need_grad = L, need_grad
        self.names = ["outlogits.0.weight_orig", "outlogits.1.weight", "outlogits.1.bias",
                      "outlogits.3.weight_orig", "outlogits.3.bias"]
        self.params = dict(L.named_parameters())

    def apply(self, h_code, c_code):
        return TapeFn.apply(self, h_code, c_code, *[self.params[n] for n in self.names])[0]

    def _w3_perm(self, Cp):
        """final 4x4 conv weight [1, C, 4, 4] -> row vector over the NHWC-flattened features
        [(y*4+x)*Cp + c]."""
        w = self.L.outlogits[3].weight_orig
        C = w.shape[1]
        out = torch.zeros(1, 16, Cp, device=w.device)
        out[0, :, :C] = w.detach()[0].permute(1, 2, 0).reshape(16, C)
        return out.view(1, 16 * Cp)

    def run_forward(self, h_code, c_code, *plist):
        L = self.L
        _eval_bn_unsupported(L)
        seq = L.outlogits
        dev = h_code.device
        n, Cf, H, W = h_code.shape
        Ce = c_code.shape[1]
        Cc = rup(Cf + Ce, 64)
        tape = Tape(_CACHE, training=L.training, need_grad=self.need_grad, planes=2, dtype=ops.BF16)
        self.tape = tape
        x = T4(n, H, W, Cc)
        sn = SpectralNorm(seq[0].weight_u, seq[0].weight_v)
        self.sn3 = SpectralNorm(seq[3].weight_u, seq[3].weight_v)
        alpha = sn.forward(seq[0].weight_orig, L.training, self.need_grad)
        inv_sigma = self.sn3.forward(seq[3].weight_orig, L.training, self.need_grad)
        x.hi = _e((n, H, W, Cc), dev, torch.bfloat16)
        x.lo = _e((n, H, W, Cc), dev, torch.bfloat16)
        ops.pack_nchw(h_code.detach(), c_code.detach().contiguous().view(n, Ce), x.hi, x.lo, Cc)
        self.x, self.Cf = x, Cf
        cn = ConvNode(tape, "s1", x, seq[0].weight_orig, "logits.conv", sn=sn, alpha=alpha, bn_stats=True)
        z = tape.add(cn)
        bn = BnActNode(tape, z, _bn_tuple(seq[1]), ops.ACT_LRELU, "logits.bn", want_f32=True,
                       want_planes=False)
        a = tape.add(bn)
        self.cn, self.bn, self.a = cn, bn, a
        # final layer: dot product over the 4x4 x C features, spectral norm on a [1, 16C] matrix
        feat = a.f32.view(n, H * W * a.C)
        wrow = self._w3_perm(a.C)
        t = _e((n, 1), dev)
        ops.linear_f32(feat, wrow, None, t)
        out = _e((n,), dev)
        ops.affine_sigmoid_fwd(t.view(n), inv_sigma, seq[3].bias.detach(), out)
        self.wrow, self.inv_sigma, self.out = wrow, inv_sigma, out
        tape.finish_forward()
        return out

    def run_backward(self, grads, needs):
        (dout,) = grads
        L, a = self.L, self.a
        seq = L.outlogits
        dev = dout.device
        n = a.N
        need_w = any(needs[2:])
        pg = {}
        dout = dout.contiguous()
        dt, dz = _e((n, 1), dev), _e((n, 1), dev)
        ops.affine_sigmoid_bwd(dout, self.out, self.inv_sigma, dt.view(n), dz.view(n))
        feat = a.f32.view(n, -1)
        a.grad = _e((a.N, a.H, a.W, a.C), dev)
        ops.linear_nn_f32(dt, self.wrow, a.grad.view(n, -1))          # d feat = dt (x) w_row
        if need_w:
            gw = _e((1, feat.shape[1]), dev)
            ops.linear_tn_f32(dz, feat, gw)                           # dL/dW_eff (NHWC-flattened)
            w3 = seq[3].weight_orig
            C = w3.shape[1]
            g4 = gw.view(16, a.C)[:, :C].reshape(4, 4, C).permute(2, 0, 1).reshape(1, C, 4, 4).contiguous()
            pg["outlogits.3.weight_orig"] = self.sn3.backward(g4, w3)
            ones = torch.ones(n, 1, device=dev)
            db = _e((1, 1), dev)
            ops.linear_tn_f32(dz, ones, db)
            pg["outlogits.3.bias"] = db.view(1)
        self.x.needs_grad = bool(needs[0])
        self.bn.backward(need_w)
        pg["outlogits.1.weight"], pg["outlogits.1.bias"] = self.bn.dgamma, self.bn.dbeta
        self.cn.backward(need_w)
        pg["outlogits.0.weight_orig"] = self.cn.dW
        dh = None
        if needs[0]:
            dh = self.x.grad.permute(0, 3, 1, 2)[:, :self.Cf]
        out = [dh, None]
        for nme, need in zip(self.names, needs[2:]):
            out.append(pg.get(nme) if need else None)
        self.tape.release()
        self.tape = self.cn = self.bn = self.a = self.x = None
        return out


# =============================================================================== cate_classify
def cate_classify_weight_rows(w, Cp):
    """conv(ndf*8 -> L, k4 s4 p1) on a 4x4 map = dot product with the kernel's lower-right 3x3
    taps (padding rows/cols hit zeros).  Returns [L, 16*Cp] over NHWC-flattened features; built
    with differentiable torch slicing so the weight gradient flows back through autograd."""
    Lc, C = w.shape[0], w.shape[1]
    k = torch.nn.functional.pad(w[:, :, 1:, 1:], (0, 1, 0, 1))          # [L, C, 4, 4] aligned to pixels
    k = k.permute(0, 2, 3, 1)                                           # [L, 4, 4, C]
    if Cp > C:
        k = torch.nn.functional.pad(k, (0, Cp - C))
    return k.reshape(Lc, 16 * Cp)
