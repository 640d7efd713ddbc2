"""Drop-in for the reference's ``trainer.py``: ``GANTrainer(output_dir, args, ratio).train(
imageloader, storyloader, testloader, stage)`` with the same batch-dict contract, optimiser
settings, LR schedule, checkpoint files and step sequence (reference trainer.py:187-485), on
top of the CUDA-kernel modules in ``model.py``.

What is different from the reference, deliberately:
  * the body of the hot loop lives in ``train_step`` (the reference has one monolithic
    ``train``); ``train`` calls it once per story batch;
  * one process drives one GPU.  Multi-GPU = one process per GPU (torchrun), each with its own
    ``cfg.TRAIN.*_BATCH_SIZE`` shard (weak scaling, like the reference's batch x num_gpus);
    gradients are averaged with one NCCL all-reduce per optimiser step (``GradSync``);
  * the never-stepped ReduceLROnPlateau schedulers (reference l.224-228, broken on torch>=2.7)
    are not created; tensorboard logging is optional and lazy (no per-step host sync unless a
    logger is attached);
  * while the generator is updated the discriminators' parameters have requires_grad off, so the
    weight gradients the reference computes and then discards (zeroed by the next
    ``zero_grad``) are not computed.
"""
import os
import time

import numpy as np
import torch
import torch.distributed as dist
import torch.optim as optim

from miscc.config import cfg
from miscc.utils import (KL_loss, compute_discriminator_loss, compute_generator_loss, count_param,
                         mkdir_p, save_image_results, save_model, save_story_results, weights_init)
from cpcsv_b200 import nets as knets
from cpcsv_b200 import streams


class GradSync:
    """Average gradients across ranks: per network ONE copy of its gradients into a flat buffer
    (a single multi-tensor launch), ONE all-reduce (NCCL: averaging inside the collective), and
    the parameters' ``.grad`` re-pointed at slices of the reduced buffer (no copy back).
    Capturable into the step's CUDA graph together with the kernels around it."""

    ALIGN = 64      # elements: every slice starts 256-byte aligned (vectorised optimiser loads)

    def __init__(self, enabled=None):
        self.enabled = dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1 \
            if enabled is None else enabled
        self.world = dist.get_world_size() if self.enabled else 1
        self.avg_in_collective = self.enabled and dist.is_initialized() and dist.get_backend() == "nccl"

    def __call__(self, params, inplace=False):
        """``inplace``: write the averaged values back into the existing ``.grad`` tensors instead of
        re-pointing ``.grad`` at the reduced buffer.  Required when the optimiser step that follows is a
        REPLAYED CUDA graph: it reads the gradient memory it saw at capture time (the addresses the
        replayed backward pass writes), not whatever ``.grad`` points at afterwards."""
        if not self.enabled:
            return
        owners = [p for p in params if p.grad is not None]
        if not owners:
            return
        grads = [p.grad for p in owners]
        offs, total = [], 0
        for g in grads:
            offs.append(total)
            total += (g.numel() + self.ALIGN - 1) // self.ALIGN * self.ALIGN
        flat = torch.empty(total, device=grads[0].device, dtype=grads[0].dtype)     # alignment gaps stay unread
        views = [flat[o:o + g.numel()].view(g.shape) for o, g in zip(offs, grads)]
        torch._foreach_copy_(views, grads)
        if self.world > 1:
            if self.avg_in_collective:
                dist.all_reduce(flat, op=dist.ReduceOp.AVG)
            else:
                dist.all_reduce(flat)
                flat.div_(self.world)
        if inplace:
            torch._foreach_copy_(grads, views)
            return
        for p, v in zip(owners, views):
            p.grad = v


def broadcast_initial_state(nets, src=0):
    """data parallel: every rank starts from rank `src`'s parameters and buffers (the reference has one
    process and one set of weights; with one process per GPU the initialisation RNG may differ per rank)"""
    if not (dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1):
        return
    for net in nets.values():
        for t in list(net.parameters()) + list(net.buffers()):
            dist.broadcast(t.data, src)


def build_networks(video_len=None):
    """StoryGAN + the three discriminators, initialised like reference trainer.py:87-97."""
    if cfg.CASCADE_MODEL:      # reference trainer.py:83-86
        from cascade_model import StoryGAN, STAGE1_D_IMG, STAGE1_D_STY_V2, STAGE1_D_SEG
    else:
        from model import StoryGAN, STAGE1_D_IMG, STAGE1_D_STY_V2, STAGE1_D_SEG
    nets = {"G": StoryGAN(video_len if video_len is not None else cfg.VIDEO_LEN),
            "D_im": STAGE1_D_IMG(), "D_st": STAGE1_D_STY_V2(), "D_se": STAGE1_D_SEG()}
    for n in nets.values():
        n.apply(weights_init)
    return nets


def build_optimizers(nets, fused=None, lr_tensor_device=None):
    """Adam(betas=(0.5, 0.999)); lr from cfg (reference trainer.py:212-220).  On a GPU (``fused``) this is
    ``cpcsv_b200.optim.PackedAdam``: the same arithmetic as ``torch.optim.Adam`` in hand-written
    multi-tensor kernels that also rewrite the 16-bit operand planes of the updated weights.
    ``fused=False``: stock ``torch.optim.Adam`` (CPU tests of the host logic).  ``lr_tensor_device``: hold the
    learning rate in a device tensor (CUDA-graph replays see later changes, ``set_lr``)."""
    fused = torch.cuda.is_available() if fused is None else fused
    opts = {}
    for k, net in nets.items():
        lr = cfg.TRAIN.GENERATOR_LR if k == "G" else cfg.TRAIN.DISCRIMINATOR_LR
        params = [p for p in net.parameters() if p.requires_grad]
        if fused:
            from cpcsv_b200.optim import PackedAdam
            if lr_tensor_device is not None:
                lr = torch.tensor(float(lr), device=lr_tensor_device)
            opts[k] = PackedAdam(params, lr=lr, betas=(0.5, 0.999))
            if k == "G" and not hasattr(net, "presample"):
                # the trunk's Adam + re-layout kernels are issued as soon as its gradients are complete,
                # overlapping the backward pass of the conditioning path (armed per step in train_step)
                # -- layer by layer: one bucket per trunk module (conv / Linear weight + its BatchNorm)
                named = dict(net.named_parameters())
                early = [n for n in knets.TrunkRunner.parameter_names() if n in named and named[n].requires_grad]
                buckets = {}
                for n in early:
                    buckets.setdefault(n.split(".")[0], []).append(named[n])
                # (one rank only: with a gradient exchange every bucket costs a flat copy + a small all-reduce, measured
                # 22.15 vs 21.68 ms / step at 2 GPUs -- there the whole trunk is exchanged and updated at once)
                layerwise = LAYERWISE_G_ADAM and not (dist.is_available() and dist.is_initialized()
                                                      and dist.get_world_size() > 1)
                opts[k].overlap_with_backward([named[n] for n in early],
                                              buckets=list(buckets.values()) if layerwise else None)
        else:
            opts[k] = optim.Adam(params, lr=lr, betas=(0.5, 0.999))
    return opts


def _set_requires_grad(net, flag):
    for p in net.parameters():
        p.requires_grad_(flag)


def prepare_inputs(st_batch, im_batch):
    """reference trainer.py:252-288: slice text to cfg.TEXT.DIMENSION, append labels."""
    T = cfg.TEXT.DIMENSION
    im_labels, st_labels = im_batch["labels"], st_batch["labels"]
    return dict(
        st_real=st_batch["images"], im_real=im_batch["images"], se_real=im_batch["images_seg"],
        st_labels=st_labels, im_labels=im_labels,
        im_motion=torch.cat((im_batch["description"][:, :T], im_labels), 1),
        im_content=im_batch["content"][:, :, :T],
        st_motion=torch.cat((st_batch["description"][:, :, :T], st_labels), 2),
        st_content=st_batch["description"][:, :, :T])


def _cond_vectors(x, c_mu, cim_mu):
    """reference trainer.py:303-307 / 386-389 (without the FloatTensor host round trip)."""
    T = cfg.TEXT.DIMENSION
    chars = (x["st_labels"].mean(1) > 0).to(c_mu.dtype)
    st_mu = torch.cat((c_mu, x["st_motion"][:, :, :T].mean(1).squeeze(), chars), 1)
    im_mu = torch.cat((x["im_motion"], cim_mu), 1)
    return st_mu, im_mu


def _latent_loss(latents):
    """sum of MSE(g_seg_k, h_k) over the four (decoder, re-encoder) pairs, reference trainer.py:371-375"""
    hs, gs = latents
    return sum(torch.nn.functional.mse_loss(g, h) for g, h in zip(gs, hs))


D_NETS = ("D_se", "D_im", "D_st")
CONCURRENT_D = True     # run the three discriminators on parallel CUDA streams
CONCURRENT_G = True     # run sample_videos / sample_images of one phase on two streams
EARLY_G = True          # issue the generator-update forward alongside the discriminator update
LAYERWISE_G_ADAM = os.environ.get("CPCSV_LAYERWISE_ADAM", "1") != "0"   # trunk Adam per layer, under the backward pass
# Issue the discriminators' real-image encoder passes before the fakes exist, on detached streams.  OFF: together with
# EARLY_G it made the STORY discriminator's losses of a graph-replayed step deviate intermittently (tools/diag_run.sh,
# 'small' preset, zero learning rates: about 1 step in 12 with st_errD or st_errG off by 1-10 %, every other loss
# exact; with either switch off 60 of 60 steps agree to 1e-5).  The race was not found; the early passes bought no
# measurable time any more (20.07 / 20.03 ms without vs 20.08 ms with them), so they are opt-in (CPCSV_EARLY_D_REAL=1).
EARLY_D_REAL = os.environ.get("CPCSV_EARLY_D_REAL", "0") == "1"
step_stream = streams.step_stream
Detached = streams.Detached


def _concurrently(*thunks, enabled=None):
    return streams.concurrently(*thunks, enabled=CONCURRENT_D if enabled is None else enabled)


def stage_discriminators(nets, x, labels, early_generator=False, opts=None, grad_sync=None):
    """reference trainer.py:290-343 minus the optimiser steps: no-grad fakes, the three
    discriminator losses and their backward passes.  The three discriminators are independent
    networks, so running all backward passes before any of their Adam steps (instead of the
    reference's se.step() between se.backward() and im.backward()) gives identical results.

    ``early_generator``: also issue the forward pass of the generator update (reference
    trainer.py:365-368) on detached streams.  It reads only the generator's weights (updated at
    the very end of the step) and fresh noise, so it does not depend on the discriminator update
    and fills the tensor cores while the discriminators' many small kernels run.  It is issued
    after the no-grad calls, so noise is drawn and BatchNorm running statistics are updated in
    the reference's order.  The handle comes back under ``out['early_generator']``.

    ``opts``: when given, every discriminator's Adam step (which also rewrites the operand planes of its
    weights for the generator stage) is issued on that discriminator's own stream right after its backward
    pass, so it overlaps with the other discriminators still running instead of forming a
    tensor-core-idle gap after the join.  ``grad_sync`` (with ``opts``): the gradient exchange of each
    discriminator is issued there as well, between its backward pass and its Adam step: the all-reduce of
    the first two discriminators runs under the remaining compute of the others."""
    netG, netD_im, netD_st, netD_se = nets["G"], nets["D_im"], nets["D_st"], nets["D_se"]
    im_ones, im_zeros, st_ones, st_zeros = labels
    gpus = None
    out = {}
    start = None
    if (early_generator or EARLY_D_REAL) and torch.cuda.is_available():
        start = torch.cuda.Event()
        start.record()
    # The real-image encoder passes (reference miscc/utils.py:58: netD(real_imgs)) depend on the
    # discriminators' weights and the data only: they are issued first, on detached streams, and fill the
    # tensor cores while the generator's conditioning path (GRUs, small Linears: latency-bound, no GEMM)
    # runs.  Module state (BatchNorm running statistics, spectral-norm vectors) is still updated real
    # pass first, fake pass second, as in the reference.
    real_pass = None
    if EARLY_D_REAL:
        reals = {"D_se": x["se_real"], "D_im": x["im_real"], "D_st": x["st_real"]}
        real_pass = Detached([lambda k=k: nets[k](reals[k]) for k in D_NETS], after=start)
    # weight re-layout for this stage's discriminator passes and for the next stage's generator
    # passes runs on a side stream, overlapped with the no-grad generator forward below
    prefetch = knets.prefetch_weights([netG, netD_se, netD_im, netD_st], no_grad_forward=True)
    # (2) fakes for the discriminator update
    def no_grad(fn, *a, **kw):
        with torch.no_grad():      # grad mode is thread-local state, so set it inside the thunk
            return fn(*a, **kw)

    if early_generator:
        streams.hold_state_order()     # keep the ordered-state events alive across the join below
    (_, st_fake, _, _, c_mu, _, _), (_, im_fake, _, _, cim_mu, _, se_fake) = _concurrently(
        lambda: no_grad(netG.sample_videos, x["st_motion"], x["st_content"]),
        lambda: no_grad(netG.sample_images, x["im_motion"], x["im_content"], seg=True),
        enabled=CONCURRENT_G)
    if early_generator:
        streams.release_state_order()
        out["early_generator"] = generator_forward(nets, x, after=start)
    st_mu, im_mu = _cond_vectors(x, c_mu, cim_mu)
    out["p1_st_fake"], out["p1_im_fake"], out["p1_se_fake"] = st_fake, im_fake, se_fake
    # (3) discriminators
    for k in ("D_im", "D_st", "D_se"):
        nets[k].zero_grad(set_to_none=True)
    # the three discriminators are independent networks made of many small kernels at this
    # batch size: run them on three concurrent streams (fork / join around the block)
    real_feats = dict(zip(D_NETS, real_pass.join())) if real_pass is not None else {}

    def d_update(key, real, fake, ones, zeros, cate, cond):
        netD = nets[key]
        err = compute_discriminator_loss(netD, real, fake, ones, zeros, cate, cond, gpus,
                                         real_features=real_feats.get(key))[0]
        err.backward()
        if opts is not None:
            if grad_sync is not None:
                grad_sync(list(netD.parameters()))
            opts[key].step()
        return err

    se_errD, im_errD, st_errD = _concurrently(
        lambda: d_update("D_se", x["se_real"], se_fake, im_ones, im_zeros, x["im_labels"], im_mu),
        lambda: d_update("D_im", x["im_real"], im_fake, im_ones, im_zeros, x["im_labels"], im_mu),
        lambda: d_update("D_st", x["st_real"], st_fake, st_ones, st_zeros, x["st_labels"], st_mu))
    out.update(se_errD=se_errD.detach(), im_errD=im_errD.detach(), st_errD=st_errD.detach())
    knets.join_prefetch(prefetch)
    return out


def generator_forward(nets, x, after=None):
    """the two generator calls of the generator update (reference trainer.py:365-368), issued on
    detached streams; ``.join()`` gives the two 7-tuples"""
    netG = nets["G"]
    netG.zero_grad(set_to_none=True)
    return Detached([lambda: netG.sample_videos(x["st_motion"], x["st_content"]),
                     lambda: netG.sample_images(x["im_motion"], x["im_content"], seg=True)], after=after)


def stage_generator(nets, x, labels, ratio=1.0, skip_d_wgrad=True, forward=None):
    """reference trainer.py:365-415: generator forward with fresh noise (or the already issued
    ``forward`` handle of ``generator_forward``), the three adversarial losses + KL terms,
    backward."""
    netG, netD_im, netD_st, netD_se = nets["G"], nets["D_im"], nets["D_st"], nets["D_se"]
    im_ones, im_zeros, st_ones, st_zeros = labels
    gpus = None
    out = {}
    # the discriminators were just updated: re-pack their weights while the generator runs
    prefetch = knets.prefetch_weights([netD_se, netD_im, netD_st])
    if forward is None:
        netG.zero_grad(set_to_none=True)
    if skip_d_wgrad:
        for k in ("D_im", "D_st", "D_se"):
            _set_requires_grad(nets[k], False)
    try:
        if forward is not None:
            g_vid, g_img = forward.join()
        else:
            g_vid, g_img = _concurrently(
                lambda: netG.sample_videos(x["st_motion"], x["st_content"]),
                lambda: netG.sample_images(x["im_motion"], x["im_content"], seg=True),
                enabled=CONCURRENT_G)
        (video_latents, st_fake, _, _, c_mu, c_logvar, _) = g_vid
        (image_latents, im_fake, _, _, cim_mu, cim_logvar, se_fake) = g_img
        st_mu, im_mu = _cond_vectors(x, c_mu, cim_mu)
        if video_latents is not None:
            # cascade generator, reference trainer.py:369-384 (the tuples are paired by position)
            video_latent_loss, image_latent_loss = _latent_loss(video_latents), _latent_loss(image_latents)
            rec_real = netG.train_autoencoder(x["se_real"])
            rec_fake = netG.train_autoencoder(se_fake)
            reconstruct_loss = (torch.nn.functional.mse_loss(rec_real, x["se_real"])
                                + torch.nn.functional.mse_loss(rec_fake, se_fake)) / 2.0
            out.update(video_latent_loss=video_latent_loss.detach(), image_latent_loss=image_latent_loss.detach(),
                       reconstruct_loss=reconstruct_loss.detach())
        se_errG, im_errG, st_errG = _concurrently(
            lambda: compute_generator_loss(netD_se, se_fake, x["se_real"], im_ones, x["im_labels"], im_mu, gpus)[0],
            lambda: compute_generator_loss(netD_im, im_fake, x["im_real"], im_ones, x["im_labels"], im_mu, gpus)[0],
            lambda: compute_generator_loss(netD_st, st_fake, x["st_real"], st_ones, x["st_labels"], st_mu, gpus)[0])
        im_kl = KL_loss(cim_mu, cim_logvar)
        st_kl = KL_loss(c_mu, c_logvar)
        kl_w = cfg.TRAIN.COEFF.KL
        total = im_errG + im_kl * kl_w + ratio * (se_errG * cfg.SEGMENT_RATIO + st_errG * cfg.IMAGE_RATIO
                                                  + st_kl * kl_w)
        if video_latents is not None:      # reference trainer.py:412-413
            total = total + (video_latent_loss + reconstruct_loss) * cfg.RECONSTRUCT_LOSS
        total.backward()
    finally:
        if skip_d_wgrad:
            for k in ("D_im", "D_st", "D_se"):
                _set_requires_grad(nets[k], True)
    out.update(se_errG=se_errG.detach(), im_errG=im_errG.detach(), st_errG=st_errG.detach(),
               im_kl=im_kl.detach(), st_kl=st_kl.detach(), errG_total=total.detach())
    out["p3_st_fake"], out["p3_im_fake"], out["p3_se_fake"] = st_fake.detach(), im_fake.detach(), se_fake.detach()
    knets.join_prefetch(prefetch)
    return out


def _early_g(nets):
    """EARLY_G, except for the cascade generator: with its two generator calls running concurrently AND issued early
    the story branch's generator loss of a graph-replayed step deviated intermittently (tools/diag_run.sh
    small_cascade: 2 of 15 steps, st_errG only; 60 of 60 clean with EARLY_G or CONCURRENT_G off).  Not root-caused:
    the cascade step keeps the generator forward inside the generator stage."""
    return EARLY_G and not hasattr(nets["G"], "presample")


def sync_grads(nets, names, grad_sync, inplace=False):
    """the one exchange step of the data-parallel job: average gradients across ranks"""
    if grad_sync:
        for k in names:
            if inplace:
                grad_sync(list(nets[k].parameters()), inplace=True)
            else:
                grad_sync(list(nets[k].parameters()))


def train_step(nets, opts, x, labels, ratio=1.0, grad_sync=None, apply_optim=True, skip_d_wgrad=True,
               after_discriminators=None):
    """One iteration of the reference's hot loop (trainer.py:290-416).  ``x`` from
    ``prepare_inputs`` (device tensors), ``labels`` = (im_ones, im_zeros, st_ones, st_zeros).
    Returns a dict of loss tensors (no host sync)."""
    exchange = grad_sync is not None and getattr(grad_sync, "enabled", True)
    out = stage_discriminators(nets, x, labels, early_generator=_early_g(nets), opts=opts if apply_optim else None,
                               grad_sync=grad_sync if exchange else None)
    if not apply_optim:
        sync_grads(nets, D_NETS, grad_sync)
    if after_discriminators is not None:
        after_discriminators()      # the real images have been read for the last time (GraphedStep.load_async)
    early = apply_optim and hasattr(opts["G"], "expect_backward")
    if early:
        # the generator's Adam step starts inside the backward pass; with several ranks the gradient
        # exchange of those (trunk) parameters is issued there too, right before their update
        opts["G"].expect_backward(pre_update=(lambda params: grad_sync(params)) if exchange else None)
    try:
        out.update(stage_generator(nets, x, labels, ratio, skip_d_wgrad, forward=out.pop("early_generator", None)))
    finally:
        if hasattr(opts["G"], "disarm"):
            opts["G"].disarm()
    if exchange and early and opts["G"].early_fired:
        done = opts["G"].updated_ids()
        grad_sync([p for p in nets["G"].parameters() if id(p) not in done])
    else:
        sync_grads(nets, ("G",), grad_sync)
    if apply_optim:
        opts["G"].step()
    return out


LOSS_KEYS = ("se_errD", "im_errD", "st_errD", "se_errG", "im_errG", "st_errG", "im_kl", "st_kl", "errG_total")


def build_capturable_optimizers(nets, device):
    """``build_optimizers`` for a step that is replayed as a CUDA graph: ``PackedAdam`` (step count on the
    device) with the learning rate held in a device tensor, so the halving schedule (reference
    trainer.py:447-456) acts on later replays (``set_lr``) instead of being frozen into the captured launches."""
    return build_optimizers(nets, fused=True, lr_tensor_device=device)


def set_lr(opt, lr):
    """works for float and for device-tensor learning rates (capturable optimisers)"""
    for g in opt.param_groups:
        if torch.is_tensor(g["lr"]):
            g["lr"].fill_(lr)
        else:
            g["lr"] = lr


class GraphedStep:
    """``train_step`` on STATIC device buffers, replayed as CUDA graphs: ~1500 kernel launches on a
    dozen streams per step become one graph launch (reference hot loop trainer.py:290-416; SURVEY.md
    section 8 row f1).

    The whole step is ONE graph, with or without a gradient exchange: with ``grad_sync`` enabled (N > 1)
    the NCCL all-reduces are captured inside it -- each discriminator's exchange sits between its backward
    pass and its Adam step on that discriminator's stream, i.e. under the other discriminators' compute
    (measured at 2 GPUs: 22.5 ms / step vs 22.9 ms for the three-graph variant, 21.1 ms on one GPU).
    ``segmented=True`` keeps the three-graph variant -- discriminator stage | discriminator Adam steps +
    generator stage | generator Adam step, the two all-reduces issued eagerly between them.  A process
    that captured collectives should leave with ``close()`` before the process group is destroyed.

    ``dev_st`` / ``dev_im``: dicts of device tensors with the batch-dict contract of the reference's
    loaders (``images``, ``description``, ``labels`` [, ``content``, ``images_seg``]); ``load`` copies
    a new batch into them.  The optimisers must be capturable (``build_capturable_optimizers``) and
    must have taken at least one eager step (state allocated) before ``capture``."""

    def __init__(self, nets, opts, labels, dev_st, dev_im, grad_sync=None, ratio=1.0, use_graph=True,
                 segmented=None):
        self.nets, self.opts, self.labels, self.ratio = nets, opts, labels, ratio
        self._captured_grads = None
        self.dev_st, self.dev_im = dev_st, dev_im
        self.device = labels[0].device
        self.grad_sync = grad_sync
        exchange = grad_sync is not None and getattr(grad_sync, "enabled", True)
        self.segmented = bool(segmented) if segmented is not None else False
        if use_graph and getattr(nets["D_st"], "seq_consisten_model", None) is not None:
            # create_random_shuffle (miscc/utils.py:14-44) permutes the real stories on the HOST from the python /
            # numpy generators every step: a replayed graph would repeat one permutation forever
            raise NotImplementedError("cfg.USE_SEQ_CONSISTENCY draws a host-side shuffle every step; "
                                      "run the eager step (use_graph=False / CPCSV_GRAPH=0)")
        self.use_graph = use_graph
        self.graph = None
        self.graphs = []
        self.loss_keys = LOSS_KEYS
        self.loss_dev = torch.zeros(len(LOSS_KEYS), device=self.device)
        self.loss_host = torch.zeros(len(LOSS_KEYS))
        if self.device.type == "cuda":
            self.loss_host = self.loss_host.pin_memory()
        self._copy_stream = self._staging = None
        self._pending = False
        # recorded INSIDE the step (an external event node of the graph) once the discriminator stage is over:
        # from there on nothing reads the real images, the next batch may be copied over them
        self._inputs_free = None
        self._io_done, self._late, self._pending_direct = None, None, False

    # --- static buffers ----------------------------------------------------------------------
    def fits(self, st_batch, im_batch):
        """True when the batch has the shapes of the static buffers (loaders use drop_last)"""
        for dst, src in ((self.dev_st, st_batch), (self.dev_im, im_batch)):
            for k, t in dst.items():
                if k not in src or tuple(src[k].shape) != tuple(t.shape):
                    return False
        return True

    def load(self, st_batch, im_batch):
        """host (pinned) or device batch dicts -> static device buffers, on the current stream"""
        for dst, src in ((self.dev_st, st_batch), (self.dev_im, im_batch)):
            for k, t in dst.items():
                t.copy_(src[k], non_blocking=True)

    def _early_free(self):
        """(static buffer, batch index, key) of the inputs nothing reads after the discriminator stage: every one
        of them -- ``_step_body`` works on private copies of the small text / label tensors, and the real images are
        last read by the discriminators -- except the real masks of the cascade generator (its reconstruction loss
        reads them in the generator stage)"""
        late = {"images_seg"} if hasattr(self.nets["G"], "presample") else set()
        return [(t, bi, k) for bi, d in enumerate((self.dev_st, self.dev_im)) for k, t in d.items()
                if not (bi == 1 and k in late)]

    def load_async(self, st_batch, im_batch):
        """Pipelined ``load`` of step k+1's inputs while step k is still being replayed (call it right after
        ``step()``).  With the whole step in one graph the real images -- 92 % of the bytes -- go STRAIGHT into the
        static buffers on a copy stream, as soon as step k's graph has passed its discriminator stage (an external
        event recorded inside the graph): the copy hides under the generator stage.  So do the small text / label
        tensors (the step works on private copies of them, ``_step_body``); only the cascade generator's real masks
        are copied by the next ``step()`` right before its replay.  Without that event (eager step, three-graph variant) everything goes to a staging set of buffers
        and the next ``step`` moves staging -> static buffers with one multi-tensor device copy."""
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream(device=self.device)
        if self._inputs_free is not None and self.graph is not None and not self.segmented:
            if self._io_done is None:
                self._io_done = torch.cuda.Event()
            batches = (st_batch, im_batch)
            early = self._early_free()
            with torch.cuda.stream(self._copy_stream):
                self._copy_stream.wait_event(self._inputs_free)
                for dst, bi, k in early:
                    dst.copy_(batches[bi][k], non_blocking=True)
                self._io_done.record(self._copy_stream)
            taken = {id(dst) for dst, _bi, _k in early}
            self._late = [(t, src[k]) for d, src in ((self.dev_st, st_batch), (self.dev_im, im_batch))
                          for k, t in d.items() if id(t) not in taken]
            self._pending_direct = True
            return
        if self._staging is None:
            self._staging = [{k: torch.empty_like(t) for k, t in d.items()} for d in (self.dev_st, self.dev_im)]
            self._ready, self._consumed = torch.cuda.Event(), torch.cuda.Event()
        with torch.cuda.stream(self._copy_stream):
            self._copy_stream.wait_event(self._consumed)      # staging free again (no-op the first time)
            for dst, src in zip(self._staging, (st_batch, im_batch)):
                for k, t in dst.items():
                    t.copy_(src[k], non_blocking=True)
            self._ready.record(self._copy_stream)
        self._pending = True

    def _consume_direct(self):
        cur = torch.cuda.current_stream()
        cur.wait_event(self._io_done)
        for dst, src in self._late:
            dst.copy_(src, non_blocking=True)
        self._late, self._pending_direct = None, False

    def _consume_staging(self):
        cur = torch.cuda.current_stream()
        cur.wait_event(self._ready)
        dsts = [t for d in (self.dev_st, self.dev_im) for t in d.values()]
        srcs = [s[k] for d, s in zip((self.dev_st, self.dev_im), self._staging) for k in d]
        torch._foreach_copy_(dsts, srcs)
        self._consumed.record(cur)
        self._pending = False

    def download(self):
        self.loss_host.copy_(self.loss_dev, non_blocking=True)

    def losses(self):
        """dict of the step's losses as Python floats (host sync)"""
        self.download()
        if self.device.type == "cuda":
            torch.cuda.current_stream().synchronize()
        return {k: float(v) for k, v in zip(self.loss_keys, self.loss_host)}

    # --- the step ------------------------------------------------------------------------------
    def _record(self, out):
        self.loss_dev.copy_(torch.stack([out[k].reshape(()) for k in self.loss_keys]))

    def _step_body(self):
        from miscc.utils import accuracy_on_device
        x = prepare_inputs(self.dev_st, self.dev_im)
        for k in ("st_labels", "im_labels", "im_content", "st_content"):
            # views of the static input buffers that the generator stage still reads: private copies, so that the
            # next batch may be copied over the inputs while this step is still running (load_async)
            x[k] = x[k].clone()
        with accuracy_on_device():          # no host round trip inside the step (scoped, not process-wide)
            self._record(train_step(self.nets, self.opts, x, self.labels, self.ratio, self.grad_sync,
                                    after_discriminators=self._mark_inputs_free))

    def _mark_inputs_free(self):
        if self._inputs_free is not None:
            self._inputs_free.record()

    # the step in three segments, with the NCCL gradient exchange between them
    def _seg_d(self):
        from miscc.utils import accuracy_on_device
        self._x = prepare_inputs(self.dev_st, self.dev_im)
        with accuracy_on_device():
            self._out = stage_discriminators(self.nets, self._x, self.labels, early_generator=_early_g(self.nets))
        if "early_generator" in self._out:
            self._out["early_generator"].join()      # every branch joins before the segment ends

    def _seg_g(self):
        from miscc.utils import accuracy_on_device
        for k in D_NETS:
            self.opts[k].step()
        with accuracy_on_device():
            self._out.update(stage_generator(self.nets, self._x, self.labels, self.ratio,
                                             forward=self._out.pop("early_generator", None)))

    def _seg_opt(self):
        self.opts["G"].step()
        self._record(self._out)

    def capture(self, capture_error_mode=None):
        """``capture_error_mode="thread_local"`` when other host threads keep making CUDA calls
        during the capture (DataLoader pin-memory thread, NCCL watchdog)"""
        # everything issued so far has to be complete: planes packed eagerly are read inside the capture
        # without event waits (an event recorded outside a capture cannot be waited on inside it)
        if self.device.type == "cuda":
            torch.cuda.synchronize(self.device)
        knets.sync_point(None)
        stream = step_stream(self.device)
        kw = {}
        if capture_error_mode is not None:
            kw["capture_error_mode"] = capture_error_mode
        if not self.segmented:
            self.graph = torch.cuda.CUDAGraph()
            self._inputs_free = torch.cuda.Event(external=True) if self.device.type == "cuda" else None
            if self.grad_sync is not None and getattr(self.grad_sync, "enabled", False):
                kw["capture_error_mode"] = "thread_local"   # the NCCL watchdog thread keeps running
            with torch.cuda.graph(self.graph, stream=stream, **kw):
                self._step_body()
            return
        self.graphs = []
        pool = None
        for seg in (self._seg_d, self._seg_g, self._seg_opt):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, pool=pool, stream=stream, **kw):
                seg()
            pool = g.pool()
            self.graphs.append(g)
        self.graph = True
        # the replayed backward passes write, and the replayed optimiser steps read, THESE gradient tensors;
        # an eager step in between (a batch of another size) re-points .grad elsewhere
        self._captured_grads = [(p, p.grad) for net in self.nets.values() for p in net.parameters()]

    def close(self):
        """drop the captured graphs (they hold the NCCL kernels of the gradient exchange): call before
        ``torch.distributed.destroy_process_group()``"""
        self.graph, self.graphs = None, []
        if self.device.type == "cuda":
            torch.cuda.synchronize(self.device)

    def _restore_captured_grads(self):
        if self._captured_grads is not None:
            for p, g in self._captured_grads:
                p.grad = g

    def step(self):
        if self._pending_direct:
            self._consume_direct()
        if self._pending:
            self._consume_staging()
        if self.graph is not None:
            knets.weight_cache().note_replay()      # the replay moves the weights behind the cache's back
        if self.graph is None:
            self._step_body()
        elif not self.segmented:
            self.graph.replay()
        else:
            # in place: the captured Adam steps read the gradient memory of the captured backward pass
            self._restore_captured_grads()
            self.graphs[0].replay()
            sync_grads(self.nets, D_NETS, self.grad_sync, inplace=True)
            self.graphs[1].replay()
            sync_grads(self.nets, ("G",), self.grad_sync, inplace=True)
            self.graphs[2].replay()


def snapshot_sources(output_dir, cfg_file=None):
    """reference trainer.py:55-61: keep the settings and the model / trainer sources next to the run
    (``inference.py:61-68`` later re-imports ``<output_dir>/model.py`` under another name; the copy
    finds ``cpcsv_b200`` through ``sys.path`` or ``CPCSV_B200_HOME``).  With ``cfg.CASCADE_MODEL`` the
    cascade file is the one stored as ``model.py``, as in the reference."""
    from shutil import copyfile
    here = os.path.dirname(os.path.abspath(__file__))
    if os.path.exists(os.path.join(output_dir, "Model", "model.py")):      # the reference's (never true) guard
        return
    if cfg_file and os.path.exists(cfg_file):
        copyfile(cfg_file, os.path.join(output_dir, "setting.yml"))
    copyfile(os.path.join(here, "cascade_model.py" if cfg.CASCADE_MODEL else "model.py"),
             os.path.join(output_dir, "model.py"))
    copyfile(os.path.join(here, "trainer.py"), os.path.join(output_dir, "trainer.py"))


class GANTrainer(object):
    world, rank = 1, 0      # one process per GPU; set from the torchrun environment in __init__

    def __init__(self, output_dir, args, ratio=1.0):
        if cfg.TRAIN.FLAG:
            output_dir = "{}/".format(output_dir)
            self.model_dir = os.path.join(output_dir, "Model")
            self.image_dir = os.path.join(output_dir, "Image")
            self.log_dir = os.path.join(output_dir, "log")
            self.test_dir = os.path.join(output_dir, "Test")
            for d in (self.model_dir, self.image_dir, self.log_dir, self.test_dir):
                mkdir_p(d)
            snapshot_sources(output_dir, getattr(args, "cfg_file", None))
        self.video_len = cfg.VIDEO_LEN
        self.max_epoch = cfg.TRAIN.MAX_EPOCH
        self.snapshot_interval = cfg.TRAIN.SNAPSHOT_INTERVAL
        self.gpus = [int(ix) for ix in str(cfg.GPU_ID).split(",")]
        if len(self.gpus) != 1:
            raise RuntimeError("this trainer drives ONE GPU per process; launch one process per GPU with "
                               "torchrun instead of listing several ids in cfg.GPU_ID")
        self.num_gpus = 1
        self.imbatch_size = cfg.TRAIN.IM_BATCH_SIZE
        self.stbatch_size = cfg.TRAIN.ST_BATCH_SIZE
        self.ratio = ratio
        self.con_ckpt = getattr(args, "continue_ckpt", None)
        local_rank = int(os.environ.get("LOCAL_RANK", self.gpus[0]))
        torch.cuda.set_device(local_rank)
        self.device = torch.device("cuda", local_rank)
        # data parallel = one process per GPU (torchrun): join the job's process group here, so that the
        # reference's main_pororo.py / main_clevr.py need no change (they never call init_process_group)
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        if self.world > 1:
            if not dist.is_available():
                raise RuntimeError("WORLD_SIZE > 1 but torch.distributed is not available")
            if not dist.is_initialized():
                dist.init_process_group("nccl", device_id=self.device)
        self._logger = None
        if self.rank == 0:
            try:
                from tensorboardX import SummaryWriter
                self._logger = SummaryWriter(self.log_dir)
            except Exception:
                pass

    def load_network_stageI(self):
        nets = build_networks(self.video_len)
        print("The total parameter is : {}M".format(sum(count_param(n) for n in nets.values()) // 1e6))
        if cfg.NET_G != "":
            nets["G"].load_state_dict(torch.load(cfg.NET_G, map_location="cpu"))
        if self.con_ckpt:
            nets["G"].load_state_dict(torch.load("{}/netG_epoch_{}.pth".format(self.model_dir, self.con_ckpt)))
            for k, tag in (("D_im", "im"), ("D_st", "st"), ("D_se", "se")):
                nets[k].load_state_dict(torch.load("{}/netD_{}_epoch_last.pth".format(self.model_dir, tag)))
        for n in nets.values():
            n.to(self.device)
        return nets["G"], nets["D_im"], nets["D_st"], nets["D_se"]

    def sample_real_image_batch(self, to_device=True):
        if self.imagedataset is None:
            self.imagedataset = enumerate(self.imageloader)
        batch_idx, batch = next(self.imagedataset)
        if to_device:
            batch = {k: (v if k == "text" else v.to(self.device, non_blocking=True)) for k, v in batch.items()}
        if batch_idx == len(self.imageloader) - 1:
            self.imagedataset = enumerate(self.imageloader)
        return batch

    def calculate_vfid(self, netG, epoch, testloader):
        """reference trainer.py:160-174: FID / video-FID of generated test stories with the generator in
        EVAL mode (running BatchNorm statistics; supported by the kernel path under no_grad).  The
        metric code (``fid/`` of the reference: InceptionV3 / R(2+1)D features + Frechet distance) is
        evaluation plumbing outside this package and is imported from the reference tree."""
        try:
            from fid.fid_score_v import fid_score
            from fid.utils import IgnoreLabelDataset, StoryGANDataset
            from fid.vfid_score import fid_score as vfid_score
        except ImportError as e:
            raise RuntimeError("cfg.EVALUATE_FID_SCORE needs the reference's fid/ package on sys.path") from e
        netG.eval()
        try:
            with torch.no_grad():
                generated = StoryGANDataset(netG, len(testloader), testloader.dataset)
                real = IgnoreLabelDataset(testloader.dataset)
                vfid_value = vfid_score(real, generated, cuda=True, normalize=True,
                                        r_cache=".cache/seg_story_vfid_reference_score.npz")
                fid_value = fid_score(real, generated, cuda=True, normalize=True,
                                      r_cache=".cache/seg_story_fid_reference_score.npz")
        finally:
            netG.train()
        if self._logger is not None:
            self._logger.add_scalar("Evaluation/vfid", vfid_value, epoch)
            self._logger.add_scalar("Evaluation/fid", fid_value, epoch)
        return vfid_value, fid_value

    def calculate_fsd(self, netG, testloader, feature_net, real_stats=None, epoch=None, seed=0):
        """Story-level Frechet distance (FSD) of generated test stories on the kernel path (cpcsv_b200.fsd):
        R(2+1)D-18 features (``feature_net``, a ``fsd.StoryFeatureNet``) of the real ``images`` of every test
        batch and of the stories ``netG.sample_videos`` generates for the same batch, whole batches per call,
        with the generator in eval mode under no_grad.  ``real_stats``: a ``fsd.FeatureStats`` of the real
        stories computed (or ``FeatureStats.load``-ed) before; the real images are then not run again.  The
        generator's noise is drawn from a generator seeded with ``seed`` (the global RNG state is restored
        afterwards), so the value is reproducible.  ``netG`` is left in train mode."""
        from cpcsv_b200 import fsd
        real = fsd.FeatureStats() if real_stats is None else None
        fake = fsd.FeatureStats()
        for fake_stories, real_stories in self._sample_test_stories(netG, testloader, seed):
            fake.update(feature_net(fake_stories))
            if real is not None:
                real.update(feature_net(real_stories))
        real = real if real is not None else real_stats
        value = fsd.frechet_distance(real.mu, real.sigma, fake.mu.to(real.mu.device), fake.sigma.to(real.mu.device))
        if self._logger is not None:
            self._logger.add_scalar("Evaluation/fsd", value, epoch)
        return value

    def calculate_fid(self, netG, testloader, feature_net, real_stats=None, epoch=None, seed=0):
        """Frame-level FID of generated test stories on the kernel path (cpcsv_b200.frame_fid), the frame
        counterpart of ``calculate_fsd``: InceptionV3 pool3 features (``feature_net``, a
        ``frame_fid.FrameFeatureNet``) of every frame of the real ``images`` of every test batch and of every frame
        the generator produces for the same batch (eval mode, no_grad, noise seeded with ``seed``, the RNG state
        restored, ``netG`` left in train mode).  ``real_stats``: a ``fsd.FeatureStats(dim=2048)`` of the real
        frames computed (``frame_fid.frame_statistics``) or loaded before.  Logged as ``Evaluation/frame_fid``;
        ``calculate_vfid`` (the reference's ``fid/`` package) is unchanged."""
        from cpcsv_b200 import frame_fid, fsd
        real = fsd.FeatureStats(dim=frame_fid.FEATURE_DIM) if real_stats is None else None
        fake = fsd.FeatureStats(dim=frame_fid.FEATURE_DIM)
        for fake_stories, real_stories in self._sample_test_stories(netG, testloader, seed):
            frame_fid.frame_statistics([fake_stories], feature_net, fake)
            if real is not None:
                frame_fid.frame_statistics([real_stories], feature_net, real)
        real = real if real is not None else real_stats
        value = fsd.frechet_distance(real.mu, real.sigma, fake.mu.to(real.mu.device), fake.sigma.to(real.mu.device))
        if self._logger is not None:
            self._logger.add_scalar("Evaluation/frame_fid", value, epoch)
        return value

    def calculate_ssim(self, netG, testloader, epoch=None, seed=0):
        """Mean SSIM of generated test stories on the kernel path (cpcsv_b200.ssim), the SSIM counterpart of
        ``calculate_fsd`` (reference trainer.py:175-182, through ``pytorch_ssim``): over every frame of every test
        batch, between the story the generator produces for the batch (eval mode, no_grad, noise seeded with
        ``seed``, the RNG state restored, ``netG`` left in train mode) and the batch's real ``images``.  Both are in
        [-1, 1], mapped to [0, 1] inside the kernel.  Logged as ``Evaluation/ssim``."""
        from cpcsv_b200 import ssim
        scores = [ssim.frame_ssim(fake_stories, real_stories, input_range=(-1, 1))
                  for fake_stories, real_stories in self._sample_test_stories(netG, testloader, seed)]
        value = float(torch.cat(scores).mean())
        if self._logger is not None:
            self._logger.add_scalar("Evaluation/ssim", value, epoch)
        return value

    def _sample_test_stories(self, netG, testloader, seed):
        """yields (generated stories, real ``images``) of every test batch: ``netG.sample_videos`` in eval mode under
        no_grad, with noise from a generator seeded with ``seed``; the global RNG state is restored and ``netG``
        is back in train mode once the loop ends"""
        dev = next(netG.parameters()).device
        text_dim = cfg.TEXT.DIMENSION
        netG.eval()
        try:
            with torch.no_grad(), torch.random.fork_rng(devices=[dev] if dev.type == "cuda" else []):
                torch.manual_seed(seed)
                for batch in testloader:
                    description = batch["description"].to(dev)
                    st_content = description[:, :, :text_dim]
                    st_motion = torch.cat((st_content, batch["labels"].to(dev)), 2)
                    _, fake_stories, _, _, _, _, _ = netG.sample_videos(st_motion, st_content)
                    yield fake_stories, batch["images"].to(dev)
        finally:
            netG.train()

    GRAPH_WARMUP_STEPS = 3      # eager steps (optimiser state, weight caches, NCCL) before the capture

    def _shard_loader(self, loader):
        """with several ranks every rank must see its own shard of the data: a loader without a
        DistributedSampler (the reference's main scripts build plain shuffling loaders) is rebuilt around one"""
        from torch.utils.data import DataLoader
        from torch.utils.data.distributed import DistributedSampler
        if self.world <= 1 or loader is None or isinstance(getattr(loader, "sampler", None), DistributedSampler):
            return loader
        sampler = DistributedSampler(loader.dataset, num_replicas=self.world, rank=self.rank, shuffle=True,
                                     drop_last=True)
        return DataLoader(loader.dataset, batch_size=loader.batch_size, sampler=sampler, drop_last=True,
                          num_workers=loader.num_workers, collate_fn=loader.collate_fn,
                          pin_memory=loader.pin_memory)

    def train(self, imageloader, storyloader, testloader, stage=1):
        """reference trainer.py:187-485.  On a GPU the step runs through ``GraphedStep``: batches are
        copied into static device buffers and, after ``GRAPH_WARMUP_STEPS`` eager iterations, every
        iteration is one CUDA-graph replay (``CPCSV_GRAPH=0`` keeps the eager step).  Losses stay on
        the device; they are read back only when a logger is attached, every 20 iterations."""
        imageloader, storyloader = self._shard_loader(imageloader), self._shard_loader(storyloader)
        self.imageloader, self.imagedataset = imageloader, None
        netG, netD_im, netD_st, netD_se = self.load_network_stageI()
        nets = {"G": netG, "D_im": netD_im, "D_st": netD_st, "D_se": netD_se}
        broadcast_initial_state(nets)
        if self.world > 1:
            # identical weights on every rank, but independent noise (the reference's mains seed every
            # process with 0: identical noise would make the averaged gradients equal the local ones)
            seed = torch.initial_seed() + self.rank
            torch.manual_seed(seed)
            torch.cuda.manual_seed(seed)
        dev = self.device
        use_graph = dev.type == "cuda" and os.environ.get("CPCSV_GRAPH", "1") != "0"
        if cfg.USE_SEQ_CONSISTENCY:
            use_graph = False       # per-step host-side story shuffle (see GraphedStep.__init__)
        opts = build_capturable_optimizers(nets, dev) if use_graph else build_optimizers(nets)
        labels = (torch.ones(self.imbatch_size, device=dev), torch.zeros(self.imbatch_size, device=dev),
                  torch.ones(self.stbatch_size, device=dev), torch.zeros(self.stbatch_size, device=dev))
        grad_sync = GradSync()
        graphed, eager_steps = None, 0
        generator_lr, discriminator_lr = cfg.TRAIN.GENERATOR_LR, cfg.TRAIN.DISCRIMINATOR_LR
        lr_decay_step = cfg.TRAIN.LR_DECAY_EPOCH
        start_epoch = int(self.con_ckpt) if self.con_ckpt else 0
        c_time = time.time()

        def tensors(batch):
            return {k: v for k, v in batch.items() if torch.is_tensor(v)}

        for epoch in range(start_epoch, self.max_epoch):
            start_t = time.time()
            num_step = len(storyloader)
            last = None
            for ld in (storyloader, imageloader):
                if self.world > 1 and hasattr(getattr(ld, "sampler", None), "set_epoch"):
                    ld.sampler.set_epoch(epoch)
            # One batch of look-ahead (SURVEY.md section 8 row f3; reference trainer.py:143-158,248): while the
            # graph of step i replays, the host-to-device copy of batch i+1 runs on a copy stream into staging
            # buffers (GraphedStep.load_async); step i+1 starts with one device-to-device multi-tensor copy.
            batches = ((data, tensors(data), tensors(self.sample_real_image_batch(to_device=False)))
                       for data in storyloader)
            pending = next(batches, None)
            staged = False
            i = -1
            while pending is not None:
                i += 1
                data, st_batch, im_batch = pending
                want_log = self._logger is not None and i % 20 == 0
                stats = None
                if use_graph and graphed is None:
                    graphed = GraphedStep(nets, opts, labels, {k: v.to(dev) for k, v in st_batch.items()},
                                          {k: v.to(dev) for k, v in im_batch.items()}, grad_sync, self.ratio)
                async_io = use_graph and dev.type == "cuda"
                if use_graph and graphed.fits(st_batch, im_batch):
                    if not staged:
                        graphed.load(st_batch, im_batch)
                    if graphed.graph is None:
                        if eager_steps >= self.GRAPH_WARMUP_STEPS:
                            graphed.capture(capture_error_mode="thread_local")   # loader threads
                        else:
                            eager_steps += 1
                    graphed.step()                      # consumes a staged batch first
                    pending = next(batches, None)       # the loader works while the GPU runs step i
                    staged = False
                    if async_io and pending is not None and graphed.fits(pending[1], pending[2]):
                        graphed.load_async(pending[1], pending[2])
                        staged = True
                    if want_log:
                        stats = graphed.losses()
                else:
                    pending, staged = next(batches, None), False
                    # the eager step on the same kernels: CPCSV_GRAPH=0, or a batch of another size
                    # (a loader without drop_last)
                    st_dev = {k: v.to(dev, non_blocking=True) for k, v in st_batch.items()}
                    im_dev = {k: v.to(dev, non_blocking=True) for k, v in im_batch.items()}
                    n_st, n_im = st_dev["images"].shape[0], im_dev["images"].shape[0]
                    lab = labels if (n_im, n_st) == (self.imbatch_size, self.stbatch_size) else (
                        torch.ones(n_im, device=dev), torch.zeros(n_im, device=dev),
                        torch.ones(n_st, device=dev), torch.zeros(n_st, device=dev))
                    out = train_step(nets, opts, prepare_inputs(st_dev, im_dev), lab, self.ratio, grad_sync)
                    if want_log:
                        stats = {k: float(out[k]) for k in LOSS_KEYS}
                if stats is not None:
                    step = i + num_step * epoch
                    for key, val in stats.items():
                        self._logger.add_scalar(key, val, step)
                last = (data, st_batch, i)
            # end-of-epoch sample sheet from the last story batch (reference trainer.py:437-444): one more
            # train-mode no-grad generator call (it moves the BatchNorm running statistics, as there)
            if last is not None and self.rank == 0:
                data, st_batch, i = last
                st_dev = {k: v.to(dev, non_blocking=True) for k, v in st_batch.items()}
                T = cfg.TEXT.DIMENSION
                st_content = st_dev["description"][:, :, :T]
                st_motion = torch.cat((st_content, st_dev["labels"]), 2)
                with torch.no_grad():
                    _, fake, _, _, _, _, se_fake = netG.sample_videos(st_motion, st_content, seg=True)
                st_result = save_story_results(st_batch["images"].cpu(), fake, data.get("text"), epoch,
                                               self.image_dir, i)
                se_result = save_image_results(None, se_fake)
                if self._logger is not None and hasattr(self._logger, "add_image"):
                    self._logger.add_image("pororo", st_result.transpose(2, 0, 1) / 255, epoch)
                    self._logger.add_image("segment", se_result.transpose(2, 0, 1) / 255, epoch)
            # learning-rate halving, reference trainer.py:447-456
            if epoch % lr_decay_step == 0 and epoch > 0:
                generator_lr *= 0.5
                discriminator_lr *= 0.5
                set_lr(opts["G"], generator_lr)
                for k in ("D_st", "D_im"):
                    set_lr(opts[k], discriminator_lr)
                lr_decay_step *= 2
            if cfg.EVALUATE_FID_SCORE and self.rank == 0:
                self.calculate_vfid(netG, epoch, testloader)
            print("----[{}/{}] epoch {:.1f} min, total {:.1f} h----".format(
                epoch, self.max_epoch, (time.time() - start_t) / 60, (time.time() - c_time) / 3600))
            if epoch % self.snapshot_interval == 0 and int(os.environ.get("RANK", "0")) == 0:
                save_model(netG, netD_im, netD_st, netD_se, epoch, self.model_dir)
        if int(os.environ.get("RANK", "0")) == 0:
            save_model(netG, netD_im, netD_st, netD_se, self.max_epoch, self.model_dir)
        if graphed is not None:
            graphed.close()
        return nets


def story_rate(ms_per_step, n_gpus=1):
    """stories / s for a measured step time (BASELINE.json metric)."""
    return cfg.TRAIN.ST_BATCH_SIZE * n_gpus / (ms_per_step * 1e-3)


__all__ = ["GANTrainer", "GraphedStep", "train_step", "build_networks", "build_optimizers",
           "build_capturable_optimizers", "set_lr", "prepare_inputs", "GradSync", "broadcast_initial_state", "story_rate", "LOSS_KEYS", "np"]
