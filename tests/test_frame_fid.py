"""Frame-level FID on the kernel path (cpcsv_b200.frame_fid; reference fid/fid_score_v.py with the InceptionV3 of
fid/inception.py): the tap tables of the InceptionV3 geometries, the tile choice on non-power-of-two grids, the
whole ``FrameFeatureNet`` against the fp64 oracle (oracle/fid_inception.py), the state-dict names,
``GANTrainer.calculate_fid``, and (``-m gpu``) the kernels ``cpcsv_resize_im2col`` / ``cpcsv_pool3x3``.  The CPU
cases run the product's host logic on the kernel-contract emulator; the emulations of the two new entry points
live here."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import emulator
import harness
from cpcsv_b200 import conv, frame_fid, fsd, ops
from oracle import params, presets, synth

torchvision = pytest.importorskip("torchvision")
from oracle.fid_inception import FIDInception  # noqa: E402
from test_fsd import _trainer  # noqa: E402


# ------------------------------------------------------------------------------------------ emulation
def emu_resize_im2col(x, S, a, b, hi, lo, dtype=1):
    """include/cpcsv.h cpcsv_resize_im2col: im2col rows of the 3x3 stride-2 pad-0 conv on a * resize(x) + b"""
    N = x.shape[0]
    r = F.interpolate(x.float(), size=(S, S), mode="bilinear", align_corners=False) * a + b
    cols = F.unfold(r, 3, stride=2)                                       # [N, 3 * 9, L]
    L = cols.shape[-1]
    cols = cols.view(N, 3, 9, L).permute(0, 3, 2, 1).reshape(N * L, 27)  # column tap * 3 + c
    full = torch.zeros(N * L, hi.shape[-1])
    full[:, :27] = cols
    h, l_ = emulator._split16(full, dtype)
    hi.copy_(h.view_as(hi))
    if lo is not None:
        lo.copy_(l_.view_as(lo))


def emu_pool3x3(x, mode, stride, y=None, hi=None, lo=None, dtype=1):
    """include/cpcsv.h cpcsv_pool3x3"""
    xn = x.permute(0, 3, 1, 2).float()
    pad = 1 if stride == 1 else 0
    if mode == ops.POOL_MAX:
        r = F.max_pool2d(xn, 3, stride, pad)
    else:
        r = F.avg_pool2d(xn, 3, stride, pad, count_include_pad=False)
    r = r.permute(0, 2, 3, 1)
    if y is not None:
        y.copy_(r)
    if hi is not None:
        h, l_ = emulator._split16(r, dtype)
        hi.copy_(h)
        if lo is not None:
            lo.copy_(l_)


def install(monkeypatch):
    emulator.install(monkeypatch)
    monkeypatch.setattr(ops, "resize_im2col", emu_resize_im2col)
    monkeypatch.setattr(ops, "pool3x3", emu_pool3x3)


def _bf16(t):
    return t.to(torch.bfloat16).double()


def _rel(a, b):
    return float((a.double().cpu() - b.double().cpu()).norm() / b.double().cpu().norm())


# ------------------------------------------------------------------------------------------ tap tables
# (kh, kw, ph, pw, input S): every stride-1 geometry of InceptionV3 on a grid of the network's sizes
KXL_CASES = [(1, 1, 0, 0, 73), (1, 1, 0, 0, 8), (3, 3, 0, 0, 149), (3, 3, 1, 1, 147), (3, 3, 0, 0, 73),
             (3, 3, 1, 1, 35), (5, 5, 2, 2, 35), (1, 7, 0, 3, 17), (7, 1, 3, 0, 17), (1, 3, 0, 1, 8), (3, 1, 1, 0, 8)]


@pytest.mark.parametrize("kh,kw,ph,pw,S", KXL_CASES)
def test_conv_kxl_taps(monkeypatch, kh, kw, ph, pw, S):
    """conv_kxl_fwd into a channel slice of a NaN-filled block buffer: the slice is F.conv2d, nothing else changes
    (masked rows of the pixel boxes never show)"""
    install(monkeypatch)
    g = torch.Generator().manual_seed(kh * 100 + kw * 10 + S)
    N, Ci, Co, c0 = 2, 64, 48, 16
    x = _bf16(torch.randn(N, Ci, S, S, generator=g))
    w = _bf16(torch.randn(Co, Ci, kh, kw, generator=g))
    ref = F.conv2d(x, w, padding=(ph, pw)).permute(0, 2, 3, 1)
    So = ref.shape[1]
    xp = x.permute(0, 2, 3, 1).to(torch.bfloat16).contiguous()
    wp = torch.zeros(kh * kw, 64, Ci, dtype=torch.bfloat16)
    wp[:, :Co] = w.view(Co, Ci, kh * kw).permute(2, 0, 1).to(torch.bfloat16)
    buf = torch.full((N, So, So, 128), float("nan"))
    jobs = conv.conv_kxl_fwd([xp, None], [wp.view(-1, Ci), None], buf[..., c0:c0 + Co], kh, kw, ph, pw)
    assert len(jobs) == (2 if kh * kw > 16 else 1)
    if len(jobs) == 2:
        assert not jobs[0].accumulate and jobs[1].accumulate and all(j.splits == 1 for j in jobs)
        assert len(jobs[0].taps) == 16 and len(jobs[1].taps) == kh * kw - 16
    for job in jobs:
        ops.conv_gemm(job)
    assert torch.allclose(buf[..., c0:c0 + Co].double(), ref, rtol=1e-6, atol=1e-5)
    assert torch.isnan(buf[..., :c0]).all() and torch.isnan(buf[..., c0 + Co:]).all()


@pytest.mark.parametrize("S", [17, 35, 299])
def test_conv_s2v_taps(monkeypatch, S):
    """3x3 stride 2 pad 0 on an odd grid through the [N, S + 1, S + 1, C] buffer whose extra row and column hold
    garbage (never read by a valid output)"""
    install(monkeypatch)
    g = torch.Generator().manual_seed(S)
    N, Ci, Co, c0 = 2 if S < 299 else 1, 128, 96, 32
    x = _bf16(torch.randn(N, Ci, S, S, generator=g))
    w = _bf16(torch.randn(Co, Ci, 3, 3, generator=g))
    ref = F.conv2d(x, w, stride=2).permute(0, 2, 3, 1)
    So = ref.shape[1]
    full = torch.full((N, S + 1, S + 1, Ci), 1e30).to(torch.bfloat16)
    full[:, :S, :S] = x.permute(0, 2, 3, 1).to(torch.bfloat16)
    wp = torch.zeros(9, 128, Ci, dtype=torch.bfloat16)
    wp[:, :Co] = w.view(Co, Ci, 9).permute(2, 0, 1).to(torch.bfloat16)
    buf = torch.full((N, So, So, 256), float("nan"))
    ops.conv_gemm(conv.conv_s2v_fwd([full, None], [wp.view(-1, Ci), None], buf[..., c0:c0 + Co]))
    assert torch.allclose(buf[..., c0:c0 + Co].double(), ref, rtol=1e-6, atol=1e-5)
    assert torch.isnan(buf[..., :c0]).all() and torch.isnan(buf[..., c0 + Co:]).all()


def _pixel_tile_parent(N, H, W, rows):
    """pixel_tile of the parent commit (power-of-two W only)"""
    tw = min(W, rows)
    th = 1
    while th < H and th * 2 <= rows // tw:
        th *= 2
    tn = rows // (tw * th)
    assert tn * th * tw == rows, (N, H, W, rows)
    return tn, th, tw


def test_pixel_tile_unchanged_on_power_of_two_grids():
    for rows in (64, 128):
        for N in (1, 2, 3, 5, 8, 12, 64, 96, 1000):
            for H in (1, 2, 3, 4, 5, 8, 16, 32, 64, 128):
                for W in (1, 2, 4, 8, 16, 32, 64, 128, 256, 4096):
                    assert conv.pixel_tile(N, H, W, rows) == _pixel_tile_parent(N, H, W, rows), (N, H, W, rows)


@pytest.mark.parametrize("N", [1, 2, 64, 128])
@pytest.mark.parametrize("S", [147, 73, 71, 35, 17, 149])
def test_pixel_tile_non_power_of_two_grids(N, S):
    """a grid the parent's rule tiles keeps its box (W >= 128); on any other, the box chosen masks no more rows
    than any other power-of-two box of 128 pixels"""
    tn, th, tw = conv.pixel_tile(N, S, S, 128)
    assert tn * th * tw == 128
    if S >= 128:
        assert (tn, th, tw) == _pixel_tile_parent(N, S, S, 128)
        return

    def cover(b):
        return -(-N // b[0]) * b[0] * (-(-S // b[1]) * b[1]) * (-(-S // b[2]) * b[2])
    boxes = [(128 // (h * w), h, w) for h in (1, 2, 4, 8, 16, 32, 64, 128) for w in (1, 2, 4, 8, 16, 32, 64, 128)
             if h * w <= 128]
    assert cover((tn, th, tw)) == min(cover(b) for b in boxes)


# ------------------------------------------------------------------------------------------ emulations
def _bilinear64(x, S):
    """explicit fp64 bilinear resize (align_corners=False, source index clamped at 0)"""
    N, C, H, W = x.shape

    def idx(n_in):
        d = torch.arange(S, dtype=torch.float64)
        r = ((d + 0.5) * (n_in / S) - 0.5).clamp_min(0)
        i0 = r.floor().long()
        i1 = torch.where(i0 < n_in - 1, i0 + 1, i0)
        return i0, i1, r - i0
    y0, y1, ly = idx(H)
    x0, x1, lx = idx(W)
    xd = x.double()
    top = xd[:, :, y0][:, :, :, x0] * (1 - lx) + xd[:, :, y0][:, :, :, x1] * lx
    bot = xd[:, :, y1][:, :, :, x0] * (1 - lx) + xd[:, :, y1][:, :, :, x1] * lx
    return top * (1 - ly).view(-1, 1) + bot * ly.view(-1, 1)


@pytest.mark.parametrize("H,W", [(64, 64), (32, 48), (299, 299)])
def test_resize_im2col_emulation(H, W):
    g = torch.Generator().manual_seed(H + W)
    x = torch.rand(2, 3, H, W, generator=g) * 2 - 1
    a, b = 2.0 / 3.0, 0.25
    OH = 149
    hi = torch.empty(2 * OH * OH, 64, dtype=torch.bfloat16)
    lo = torch.empty_like(hi)
    emu_resize_im2col(x, 299, a, b, hi, lo)
    _check_resize_cols(hi, lo, x, a, b)


def _check_resize_cols(hi, lo, x, a, b):
    """im2col rows of a * resize_299(x) + b against the fp64 restatement, to the precision of a hi / lo pair (a
    16-bit significand: one fp32 ulp of difference in the sample moves the rounding of lo by up to 2^-17 |v|), and
    hi / lo a valid split: |lo| is at most half a bf16 ulp of hi"""
    N, OH = x.shape[0], 149
    r = _bilinear64(x.cpu(), 299) * a + b
    got = (hi.double() + lo.double()).cpu().view(N, OH, OH, 64)
    assert torch.all(got[..., 27:] == 0)
    assert torch.all(lo.double().abs().cpu() <= hi.double().abs().cpu() * 2.0 ** -8)
    for ky in range(3):
        for kx in range(3):
            for c in range(3):
                ref = r[:, c, ky:ky + 2 * OH - 1:2, kx:kx + 2 * OH - 1:2]
                assert torch.allclose(got[..., (ky * 3 + kx) * 3 + c], ref, rtol=0, atol=2e-5)  # hi + lo: 16 bits


@pytest.mark.parametrize("mode,stride,S", [(0, 2, 147), (0, 2, 35), (0, 1, 8), (1, 1, 35), (1, 1, 17), (1, 1, 8)])
def test_pool3x3_emulation(mode, stride, S):
    g = torch.Generator().manual_seed(S + stride)
    N, C = 2, 8
    x = torch.randn(N, S, S, C, generator=g)
    So = S if stride == 1 else (S - 3) // 2 + 1
    y = torch.empty(N, So, So, C)
    emu_pool3x3(x, mode, stride, y)
    pad = 1 if stride == 1 else 0
    xp = F.pad(x.double().permute(0, 3, 1, 2), (pad,) * 4, value=float("nan"))
    for oh in range(0, So, 3):
        for ow in range(0, So, 2):
            win = xp[:, :, oh * stride:oh * stride + 3, ow * stride:ow * stride + 3].reshape(N, C, 9)
            ok = ~torch.isnan(win[0, 0])
            ref = win[..., ok].amax(-1) if mode == 0 else win[..., ok].mean(-1)
            assert torch.allclose(y[:, oh, ow].double(), ref, rtol=1e-6, atol=1e-6)


# ------------------------------------------------------------------------------------------ references
def smooth_frames(n, generator, H=64, W=64):
    """frames in [-1, 1] with structure at several scales"""
    x = torch.rand(n, 3, max(H // 8, 2), max(W // 8, 2), generator=generator) * 2 - 1
    x = F.interpolate(x, size=(H, W), mode="bilinear", align_corners=False)
    return (0.8 * x + 0.2 * (torch.rand(n, 3, H, W, generator=generator) * 2 - 1)).clamp(-1, 1)


_CALIBRATED = {}


def calibrated_reference(seed=0):
    """the oracle with BatchNorm running statistics calibrated by train-mode passes (cumulative averages) over
    smooth synthetic frames, then randomised gamma / beta, in eval mode (random-init statistics blow up over 94
    layers)"""
    if seed not in _CALIBRATED:
        torch.manual_seed(seed)
        net = FIDInception()
        g = torch.Generator().manual_seed(seed + 1)
        bns = [m for m in net.modules() if isinstance(m, torch.nn.BatchNorm2d)]
        for bn in bns:
            bn.momentum = None
            bn.reset_running_stats()
        net.train()
        with torch.no_grad():
            for _ in range(2):
                net.features(smooth_frames(6, g))
            for bn in bns:
                bn.weight.uniform_(0.75, 1.25, generator=g)
                bn.bias.uniform_(-0.1, 0.1, generator=g)
                bn.momentum = 0.1
        _CALIBRATED[seed] = {k: v.clone() for k, v in net.eval().state_dict().items()}
    net = FIDInception()
    net.load_state_dict(_CALIBRATED[seed])
    return net.eval()


def reference_features(ref64, frames, chunk=32):
    with torch.no_grad():
        return torch.cat([ref64.features(frames[i:i + chunk].double()) for i in range(0, frames.shape[0], chunk)])


def product_net(dev, seed=0, chunk=128):
    net = frame_fid.FrameFeatureNet(chunk=chunk)
    net.load_state_dict(calibrated_reference(seed).state_dict())
    return net.to(dev)


# ------------------------------------------------------------------------------------------ feature network
def test_feature_net_emulated_matches_fp64_oracle(monkeypatch):
    """the whole product network on the emulated kernels vs the fp64 oracle (2 frames, 64 x 64)"""
    install(monkeypatch)
    torch.set_num_threads(min(8, os.cpu_count() or 1))
    g = torch.Generator().manual_seed(3)
    frames = smooth_frames(2, g)
    ref = reference_features(calibrated_reference().double(), frames)
    with torch.no_grad():
        feats = product_net(torch.device("cpu"))(frames)
    assert feats.shape == (2, frame_fid.FEATURE_DIM) and feats.dtype == torch.float32
    for i in range(2):
        r = _rel(feats[i], ref[i])
        print("frame %d relL2 %.2e" % (i, r))
        assert r <= 1e-3, (i, r)


def test_state_dict_names_and_refusals():
    """torchvision's inception_v3 state_dict (fc and AuxLogits included) loads strictly; the product's keys are
    torchvision's minus those; the oracle and the product load each other's state strictly; train mode and
    grad-enabled calls raise"""
    tv = torchvision.models.inception_v3(weights=None, aux_logits=True, init_weights=False)
    net = frame_fid.FrameFeatureNet()
    net.load_state_dict(tv.state_dict(), strict=True)
    want = {k for k in tv.state_dict() if not (k.startswith("fc.") or k.startswith("AuxLogits."))}
    assert set(net.state_dict()) == want
    for k, v in net.state_dict().items():
        assert torch.equal(v, tv.state_dict()[k]), k
    ref = calibrated_reference()
    net.load_state_dict(ref.state_dict(), strict=True)
    back = FIDInception()
    back.load_state_dict(dict(net.state_dict(), **{k: v for k, v in ref.state_dict().items() if k.startswith("fc.")}),
                         strict=True)
    for k, v in ref.state_dict().items():
        assert torch.equal(back.state_dict()[k], v), k
    assert not net.training
    x = torch.zeros(1, 3, 64, 64)
    with pytest.raises(RuntimeError, match="torch.no_grad"):
        net(x)
    net.train()
    with torch.no_grad(), pytest.raises(RuntimeError, match="eval mode"):
        net(x)
    net.eval()
    with torch.no_grad(), pytest.raises(ValueError, match="frames"):
        net(torch.zeros(1, 3, 2, 64, 64))


# ------------------------------------------------------------------------------------------ trainer hook
def run_calculate_fid(device, batches):
    """tiny-preset generator and synthetic test batches; calculate_fid twice (same value: seeded noise, reproducible
    features) and once with cached real statistics; returns the FID"""
    p = presets.get("tiny")
    netG = harness.build_product(p, params.init_all(p, 0), device)["G"]
    loader = []
    for seed in range(1, batches + 1):
        b = synth.make_batch(p, seed, device=device)
        loader.append({"images": b["st_real"], "description": b["st_desc"], "labels": b["st_labels"]})
    feature_net = product_net(device)
    t, logged = _trainer()
    before = {k: v.clone() for k, v in netG.state_dict().items() if "running" in k or "tracked" in k}
    v1 = t.calculate_fid(netG, loader, feature_net, epoch=3)
    assert netG.training
    v2 = t.calculate_fid(netG, loader, feature_net, epoch=4)
    tol = 0.0 if device.type == "cpu" else 1e-4 * abs(v1)
    assert np.isfinite(v1) and v1 > 0 and abs(v1 - v2) <= tol, (v1, v2)
    for k, v in netG.state_dict().items():
        if k in before:
            assert torch.equal(v, before[k]), k
    assert logged == [("Evaluation/frame_fid", v1, 3), ("Evaluation/frame_fid", v2, 4)]
    real = frame_fid.frame_statistics([b["images"] for b in loader], feature_net)
    assert real.n == sum(b["images"].shape[0] * b["images"].shape[2] for b in loader)
    v3 = t.calculate_fid(netG, loader, feature_net, real_stats=real)
    assert abs(v3 - v1) <= tol + 1e-9 * abs(v1), (v3, v1)
    return v1


def test_calculate_fid_emulated(monkeypatch):
    install(monkeypatch)
    torch.set_num_threads(min(8, os.cpu_count() or 1))
    run_calculate_fid(torch.device("cpu"), 1)


# ------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("H,W", [(64, 64), (32, 48)])
def test_resize_im2col_kernel(H, W):
    """cpcsv_resize_im2col on a strided input: every row and column written, both planes, against the fp64
    restatement (the fp32 sample may differ from PyTorch's own bilinear kernel in the last bit -- contracted FMAs --
    so the check is to the precision of the hi / lo pair, as for the emulation)"""
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(H * W)
    x = (torch.rand(5, 4, H, W, device=dev, generator=g) * 2 - 1)[:, 1:]
    OH = 149
    hi = torch.full((5 * OH * OH, 64), float("nan"), device=dev).to(torch.bfloat16)
    lo = torch.full_like(hi, float("nan"))
    ops.resize_im2col(x, 299, 1.25, -0.5, hi, lo)
    torch.cuda.synchronize()
    assert not torch.isnan(hi.float()).any() and not torch.isnan(lo.float()).any()
    _check_resize_cols(hi, lo, x, 1.25, -0.5)


@pytest.mark.gpu
@pytest.mark.parametrize("mode,stride,S,C", [(0, 2, 147, 64), (0, 2, 35, 288), (0, 1, 8, 2048), (1, 1, 35, 192),
                                             (1, 1, 17, 768), (1, 1, 8, 1280)])
def test_pool3x3_kernel(mode, stride, S, C):
    """cpcsv_pool3x3 against its emulation: input a slice of a padded buffer, fp32 output a channel slice of a
    wider buffer, planes with their own pitch"""
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(S * C + mode)
    N = 3
    x = torch.randn(N, S + 1, S + 1, C + 8, device=dev, generator=g)[:, :S, :S, 4:4 + C]
    So = S if stride == 1 else (S - 3) // 2 + 1
    res = []
    for fn in (ops.pool3x3, emu_pool3x3):
        ybuf = torch.full((N, So, So, C + 64), float("nan"), device=dev)
        hi = torch.full((N, So + 1, So + 1, C), float("nan"), device=dev).to(torch.bfloat16)
        lo = torch.full_like(hi, float("nan"))
        fn(x, mode, stride, ybuf[..., 32:32 + C], hi[:, :So, :So], lo[:, :So, :So])
        res.append((ybuf, hi, lo))
    torch.cuda.synchronize()
    (y, hi, lo), (ye, hie, loe) = res
    assert torch.isnan(y[..., :32]).all() and torch.isnan(y[..., 32 + C:]).all()
    assert float((y[..., 32:32 + C] - ye[..., 32:32 + C]).abs().max()) <= 1e-6 * float(ye[..., 32:32 + C].abs().max())
    assert torch.equal(hi[:, :So, :So], hi[:, :So, :So].float().to(torch.bfloat16))
    assert float((hi[:, :So, :So].double() + lo[:, :So, :So].double() - y[..., 32:32 + C].double()).abs().max()) \
        <= 2 ** -16 * float(y[..., 32:32 + C].abs().max())
    assert torch.isnan(hi[:, So].float()).all()


# per-frame relL2 max measured on a B200: 3.96e-4 (DESIGN.md section 6.3); bound with 2x headroom
FEATURE_RTOL = 8e-4


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_feature_net_gpu_matches_fp64_oracle():
    dev = torch.device("cuda")
    g = torch.Generator().manual_seed(21)
    frames = smooth_frames(64, g).to(dev)
    ref = reference_features(calibrated_reference().double().to(dev), frames)
    with torch.no_grad():
        feats = product_net(dev, chunk=48)(frames)        # two chunks, the second one partial
    errs = [(feats[i].double() - ref[i]).norm().item() / ref[i].norm().item() for i in range(64)]
    print("per-frame relL2 max %.2e median %.2e" % (max(errs), sorted(errs)[32]))
    assert max(errs) <= FEATURE_RTOL


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_features_do_not_depend_on_the_chunk():
    """the same frames in two different chunks (other neighbours, other tile shapes): bit-identical features"""
    dev = torch.device("cuda")
    g = torch.Generator().manual_seed(5)
    frames = smooth_frames(40, g).to(dev)
    net = product_net(dev, chunk=40)
    with torch.no_grad():
        a = net(frames)
        net.chunk = 7
        b = net(frames[3:40])
    assert torch.equal(a[3:], b)


@pytest.mark.gpu
@pytest.mark.timeout(1800)
def test_fid_gpu_matches_fp64_oracle_features():
    """FID between 512 synthetic frames and a perturbation of them, from product features vs fp64 oracle"""
    dev = torch.device("cuda")
    g = torch.Generator().manual_seed(99)
    a = smooth_frames(512, g)
    b = (0.85 * a + 0.15 * smooth_frames(512, g) + 0.05).clamp(-1, 1)
    ref64 = calibrated_reference().double().to(dev)
    net = product_net(dev)
    vals = {}
    for name, fn in (("product", lambda s: net(s)), ("fp64", lambda s: reference_features(ref64, s, chunk=64))):
        with torch.no_grad():
            sa = fsd.FeatureStats(dim=frame_fid.FEATURE_DIM).update(fn(a.to(dev)))
            sb = fsd.FeatureStats(dim=frame_fid.FEATURE_DIM).update(fn(b.to(dev)))
        vals[name] = fsd.frechet_distance(sa.mu, sa.sigma, sb.mu, sb.sigma)
    print("FID product %.6f fp64 %.6f" % (vals["product"], vals["fp64"]))
    assert vals["fp64"] > 0
    assert abs(vals["product"] - vals["fp64"]) <= 1e-3 * vals["fp64"]


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_calculate_fid_gpu():
    print("FID tiny %.6f" % run_calculate_fid(torch.device("cuda"), 2))
