"""Cascade generator (reference cascade_model.py; SURVEY.md section 8 row f2).

Node level: the 3x3 / stride-2 downBlock convolution (engine.ConvNode "s2k3": the 4x4 / stride-2 implicit
GEMM with zero 4th taps) and the 1-channel ``presample`` convolution (engine.Im2colNode), forward + dgrad + wgrad
against ``torch.nn.functional`` in fp64 -- on the CPU emulator of the kernel contract and,
``-m gpu``, on libcpcsv.so.  Step level (``-m gpu``): the whole cascade training step on the real
kernels against the fp64 oracle and against the golden outputs of the REAL reference.

(The file sorts last on purpose: these GPU cases were added after the last GPU session of round 1
and ``pytest -x`` must reach every earlier case first.)
"""
import os

import pytest
import torch
import torch.nn.functional as F

import emulator
import harness
from cpcsv_b200 import engine, ops
from oracle import presets
from test_step_parity import (GOLD, _check, _check_against_golden, _check_generator_buffers, _step_pair)


@pytest.fixture(params=["emu", pytest.param("cuda", marks=pytest.mark.gpu)])
def dev(request, monkeypatch):
    if request.param == "emu":
        emulator.install(monkeypatch)
        return torch.device("cpu")
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    return torch.device("cuda")


def rnd(*shape, seed=0, dev="cpu", scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to(dev)


def rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30))


def bf16r(t):
    return t.to(torch.bfloat16).float()


def _planes_t4(x_nchw, cpad):
    """NCHW fp32 -> T4 with hi/lo bf16 NHWC planes, channels zero padded to cpad"""
    N, C, H, W = x_nchw.shape
    v = torch.zeros(N, H, W, cpad, device=x_nchw.device)
    v[..., :C] = x_nchw.permute(0, 2, 3, 1)
    t = engine.T4(N, H, W, cpad)
    t.hi = v.to(torch.bfloat16)
    t.lo = (v - t.hi.float()).to(torch.bfloat16)
    return t


def _sn(Co, K, dev):
    """unit u [Co], v [K] of a spectral norm and an engine.SpectralNorm over copies of them"""
    u = F.normalize(rnd(Co, seed=7), dim=0).to(dev)
    v = F.normalize(rnd(K, seed=8), dim=0).to(dev)
    return u.double(), v.double(), engine.SpectralNorm(u.clone(), v.clone())


def _sigma(w, u, v):
    """legacy torch spectral_norm in fp64: one power iteration from (u, v), then sigma = u^T W v, differentiable
    in w with the iterated u, v held constant"""
    w2 = w.reshape(w.shape[0], -1)
    with torch.no_grad():
        v = F.normalize(w2.t() @ u, dim=0, eps=1e-12)
        u = F.normalize(w2 @ v, dim=0, eps=1e-12)
    return u @ (w2 @ v)


@pytest.mark.parametrize("N,H,Ci,Co,sn", [(3, 8, 60, 128, False), (2, 64, 2, 4, False), (5, 16, 64, 100, False),
                                          # Conv3d (1, 3, 3) weight with a spectral norm (the video critic's layers)
                                          (2, 16, 24, 40, True)])
def test_s2k3_conv_node(dev, N, H, Ci, Co, sn):
    """conv3x3 stride 2 pad 1 (cascade_model.py:36-41) as engine.ConvNode's "s2k3" geometry: forward, data
    gradient, weight gradient"""
    x = rnd(N, Ci, H, H, seed=1, dev=dev)
    shape = (Co, Ci, 1, 3, 3) if sn else (Co, Ci, 3, 3)
    w = torch.nn.Parameter(rnd(*shape, seed=2, dev=dev, scale=0.05))
    tape = engine.Tape(engine.WeightCache(), training=True, need_grad=True)
    a = _planes_t4(x, engine.rup(Ci, 64))
    u, v, snm = _sn(Co, Ci * 9, dev) if sn else (None, None, None)

    def w_eff(wd, wsig):
        """the 4-D weight the convolution applies; wsig: the weight sigma is computed from"""
        w4 = wd.view(Co, Ci, 3, 3)
        return w4 / _sigma(wsig, u, v) if sn else w4
    node = engine.ConvNode(tape, "s2k3", a, w, "down", sn=snm)
    out = tape.add(node)
    ref = F.conv2d(x.double(), w_eff(w.detach().double(), w.detach().double()), stride=2, padding=1)
    got = out.f32.permute(0, 3, 1, 2)
    assert rel(got[:, :Co], ref) < 3e-5
    assert got.shape[1] == Co or float(got[:, Co:].abs().max()) == 0.0
    # backward: single-pass bf16 operands
    dz = torch.zeros(N, H // 2, H // 2, out.C, device=dev)
    dz[..., :Co] = rnd(N, H // 2, H // 2, Co, seed=3, dev=dev)
    out.grad16 = dz.to(torch.bfloat16)
    a.needs_grad = True
    node.backward(True)
    tape.aux.join()
    xd = bf16r(x).double().requires_grad_(True)
    wd = w.detach().double().requires_grad_(True)
    dzr = bf16r(dz)[..., :Co].permute(0, 3, 1, 2).double()
    y = F.conv2d(xd, w_eff(bf16r(w.detach()).double(), w.detach().double()), stride=2, padding=1)
    gx = torch.autograd.grad(y, xd, dzr)[0]
    assert rel(a.grad.permute(0, 3, 1, 2)[:, :Ci], gx) < 1e-5
    gw = torch.autograd.grad(F.conv2d(bf16r(x).double(), w_eff(wd, wd), stride=2, padding=1), wd, dzr)[0]
    assert tuple(node.dW.shape) == shape
    assert rel(node.dW, gw) < 1e-5


@pytest.mark.parametrize("planes,dtype", [(2, ops.BF16), (1, ops.FP16)])
@pytest.mark.parametrize("N,Co,k,stride,pad,Ci,sn", [(3, 2, 3, 1, 1, 1, False), (2, 64, 3, 1, 1, 1, False),
                                                     # the video critic's stem: (1, 7, 7) stride (1, 2, 2)
                                                     # pad (0, 3, 3) on 3 channels with a spectral norm
                                                     (2, 16, 7, 2, 3, 3, True)])
def test_im2col_node(dev, planes, dtype, N, Co, k, stride, pad, Ci, sn):
    """engine.Im2colNode: presample's conv3x3(1 -> Co) on the 1-channel mask (cascade_model.py:312-316), and a
    spectrally normalised 7x7 stride-2 convolution with K = 147 -> 192"""
    x = torch.tanh(rnd(N, Ci, 64, 64, seed=4, dev=dev))
    w = torch.nn.Parameter(rnd(Co, Ci, k, k, seed=5, dev=dev, scale=0.3))
    need_grad = planes == 2
    tape = engine.Tape(engine.WeightCache(), training=True, need_grad=need_grad, planes=planes, dtype=dtype)
    u, v, snm = _sn(Co, Ci * k * k, dev) if sn else (None, None, None)

    def w_eff(wd, wsig):
        return wd / _sigma(wsig, u, v) if sn else wd
    mc = engine.Im2colNode(tape, x, w, "presample", stride, pad, sn=snm)
    z = tape.add(mc)
    ref = F.conv2d(x.double(), w_eff(w.detach().double(), w.detach().double()), stride=stride, padding=pad)
    got = z.f32.permute(0, 3, 1, 2)
    assert rel(got[:, :Co], ref) < (3e-5 if planes == 2 else 1e-3)
    assert got.shape[1] == Co or float(got[:, Co:].abs().max()) == 0.0
    if not need_grad:
        return
    Ho = 64 // stride
    dz = torch.zeros(N, Ho, Ho, z.C, device=dev)
    dz[..., :Co] = rnd(N, Ho, Ho, Co, seed=6, dev=dev)
    z.grad16 = dz.to(torch.bfloat16)
    dx = mc.backward(True, True)
    tape.aux.join()
    xd = bf16r(x).double().requires_grad_(True)
    wd = w.detach().double().requires_grad_(True)
    dzr = bf16r(dz)[..., :Co].permute(0, 3, 1, 2).double()
    gw = torch.autograd.grad(F.conv2d(xd.detach(), w_eff(wd, wd), stride=stride, padding=pad), wd, dzr)[0]
    assert rel(mc.dW, gw) < 1e-5
    wb = w_eff(bf16r(w.detach()).double(), w.detach().double())
    gxr = torch.autograd.grad(F.conv2d(xd, wb, stride=stride, padding=pad), xd, dzr)[0]
    assert rel(dx, gxr) < 1e-5


# ------------------------------------------------------------------------------ whole step on the GPU
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["tiny_cascade", "small_cascade"])
def test_cascade_step_gpu(name):
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    p = presets.get(name)
    dev = torch.device("cuda")
    _, out, grads, ref_out, ref_grads = _step_pair(p, dev)
    res = harness.compare(out, grads, ref_out, ref_grads, verbose=True)
    print(name, res)
    _check(res, small_tensor_cos=0.99 if name.startswith("tiny") else None)


@pytest.mark.gpu
def test_tiny_cascade_step_gpu_vs_reference_golden():
    gold = torch.load(os.path.join(GOLD, "step_tiny_cascade.pt"))
    nets, out, grads = harness.run_product_step(gold["preset"], torch.device("cuda"))
    _check_against_golden(gold, out, grads)
    _check_generator_buffers(gold, nets)


# ------------------------------------------------------------------------------ CUDA-graph step (f1)
@pytest.mark.gpu
@pytest.mark.timeout(300)
def test_graphed_step_replay_matches_eager_gpu():
    """trainer.GraphedStep (the step GANTrainer.train and bench.py replay as ONE CUDA graph): three
    steps as eager-eager-capture+replay give the losses of three eager steps.  Noise is injected
    (static tensors) and the learning rates are ZERO, so both runs compute every step from
    identical weights and inputs and differ by split-K red.add ordering only.  (With the real
    learning rates the first Adam steps are lr * sign(g)-like and amplify that rounding noise to
    2e-3 of the losses after two updates -- measured on B200, profiles/r01_gpu_tests_final.log --
    which says nothing about the graph.)"""
    import copy
    import trainer
    from oracle import params, synth
    p = presets.get("small")
    dev = torch.device("cuda")
    base = harness.build_product(p, params.init_all(p, 0), dev)
    noise = synth.make_noise(p, 2, device=dev)
    batch = synth.make_batch(p, 1, device=dev)
    st = {"images": batch["st_real"], "description": batch["st_desc"], "labels": batch["st_labels"]}
    im = {"images": batch["im_real"], "description": batch["im_desc"], "content": batch["im_content"],
          "labels": batch["im_labels"], "images_seg": batch["se_real"]}
    N, B = p["IM_BATCH"], p["ST_BATCH"]
    labels = (torch.ones(N, device=dev), torch.zeros(N, device=dev), torch.ones(B, device=dev),
              torch.zeros(B, device=dev))
    losses = {}
    for mode in ("eager", "graph"):
        nets = copy.deepcopy(base)
        opts = trainer.build_capturable_optimizers(nets, dev)
        for o in opts.values():
            trainer.set_lr(o, 0.0)
        gs = trainer.GraphedStep(nets, opts, labels, {k: v.clone() for k, v in st.items()},
                                 {k: v.clone() for k, v in im.items()}, grad_sync=None)
        for i in range(3):
            harness.inject_noise(nets["G"], synth.NoiseFeed(noise))
            gs.load(st, im)
            if mode == "graph" and i == 2:
                gs.capture()
            gs.step()
        losses[mode] = gs.losses()
        torch.cuda.synchronize()
    for k, v in losses["eager"].items():
        assert abs(v - losses["graph"][k]) <= 1e-3 * abs(v) + 1e-6, (k, v, losses["graph"][k])
    trainer.set_lr(opts["G"], 5e-5)
    assert float(opts["G"].param_groups[0]["lr"]) == pytest.approx(5e-5)


@pytest.mark.gpu
@pytest.mark.timeout(300)
@pytest.mark.parametrize("name", ["small", pytest.param("small_cascade", marks=pytest.mark.xfail(
    strict=False, reason="open issue (DESIGN.md section 6): intermittent deviation of replayed cascade steps, seen in "
                         "this test once per few runs of the whole GPU suite and never when it runs alone"))])
def test_load_async_feeds_every_replay_its_own_batch_gpu(name):
    """GraphedStep.load_async: batch k+1 is copied from pinned host memory into the static input buffers WHILE the
    graph of step k is still running (behind the external event the graph records after its discriminator stage).
    Three different batches, zero learning rates, injected noise: the pipelined run gives, step by step, the losses
    of a run that loads every batch serially before its replay -- no step sees a half-overwritten batch."""
    import copy
    import trainer
    from oracle import params, synth
    p = presets.get(name)
    dev = torch.device("cuda")
    base = harness.build_product(p, params.init_all(p, 0), dev)
    noise = synth.make_noise(p, 2, device=dev)

    def host_batch(seed):
        b = synth.make_batch(p, seed)
        st = {"images": b["st_real"], "description": b["st_desc"], "labels": b["st_labels"]}
        im = {"images": b["im_real"], "description": b["im_desc"], "content": b["im_content"],
              "labels": b["im_labels"], "images_seg": b["se_real"]}
        return ({k: v.pin_memory() for k, v in st.items()}, {k: v.pin_memory() for k, v in im.items()})
    batches = [host_batch(s) for s in (11, 12, 13, 14)]
    N, B = p["IM_BATCH"], p["ST_BATCH"]
    labels = (torch.ones(N, device=dev), torch.zeros(N, device=dev), torch.ones(B, device=dev),
              torch.zeros(B, device=dev))
    runs = {}
    for mode in ("serial", "pipelined"):
        nets = copy.deepcopy(base)
        opts = trainer.build_capturable_optimizers(nets, dev)
        for o in opts.values():
            trainer.set_lr(o, 0.0)
        st0, im0 = batches[0]
        gs = trainer.GraphedStep(nets, opts, labels, {k: v.to(dev) for k, v in st0.items()},
                                 {k: v.to(dev) for k, v in im0.items()}, grad_sync=None)
        for _ in range(2):                       # eager warm-up on batch 0, then capture
            harness.inject_noise(nets["G"], synth.NoiseFeed(noise))
            gs.step()
        harness.inject_noise(nets["G"], synth.NoiseFeed(noise))
        gs.capture()
        out = []
        if mode == "serial":
            for st, im in batches[1:]:
                gs.load(st, im)
                gs.step()
                out.append(gs.losses())
        else:
            gs.load(*batches[1])
            for i in range(1, 4):
                gs.step()
                if i + 1 < 4:
                    gs.load_async(*batches[i + 1])     # right behind the replay that is still running
                out.append(gs.losses())
            assert gs._inputs_free is not None and gs._io_done is not None     # the direct path was taken
        torch.cuda.synchronize()
        runs[mode] = out
        # the static buffers end up holding the last batch
        assert torch.equal(gs.dev_st["images"].cpu(), batches[3][0]["images"])
        assert torch.equal(gs.dev_im["labels"].cpu(), batches[3][1]["labels"])
    # The story discriminator's losses are subject to the open intermittent deviation of replayed steps (DESIGN.md
    # section 6, tools/diag_run.sh: discrete alternative values within ~15 %, unrelated to the input path -- it shows up
    # between two serial runs as well); a wrong or half-overwritten batch moves EVERY loss by far more than that.
    loose = ("st_errD", "st_errG", "errG_total")
    for a, b in zip(runs["serial"], runs["pipelined"]):
        for k, v in a.items():
            tol = 0.15 if k in loose else 1e-3
            assert abs(v - b[k]) <= tol * abs(v) + 1e-6, (k, v, b[k])
    # and the batches really differ: step 1 and step 2 of one run do not agree
    assert any(abs(runs["serial"][0][k] - runs["serial"][1][k]) > 5e-3 * abs(runs["serial"][0][k])
               for k in ("im_errD", "st_errD", "se_errD"))


# ------------------------------------------------------------------------------ eval-mode generator
@pytest.mark.gpu
@pytest.mark.timeout(300)
@pytest.mark.parametrize("name", ["tiny", "tiny_cascade"])
def test_product_eval_mode_gpu(name):
    """netG.eval() under no_grad (reference inference.py:88-89) on the real kernels vs the golden
    outputs of the REAL reference"""
    from test_eval_mode import run_product_eval
    run_product_eval(name, torch.device("cuda"))
