"""Frame SSIM on the kernel path (cpcsv_b200.ssim; reference ssim_score.py and the SSIM loop of trainer.py, both
through pytorch_ssim): the fp64 oracle (oracle/ssim.py) against a brute-force double loop, ``frame_ssim``'s host
logic, ``GANTrainer.calculate_ssim``, and (``-m gpu``) the kernel ``cpcsv_ssim`` against the oracle.  The CPU cases
run the product's host logic on the kernel-contract emulator; the emulation of ``cpcsv_ssim`` (the oracle in fp32)
lives here."""
import ctypes
import math
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import emulator
import harness
from cpcsv_b200 import _lib, ops, ssim
from oracle import params, presets, synth
from oracle import ssim as ssim_oracle
from test_fsd import _trainer


# ------------------------------------------------------------------------------------------ emulation
def emu_ssim(x, y, a, b, out):
    """include/cpcsv.h cpcsv_ssim: out[b * T + t] = SSIM of frame (b, t) of a * x + b against a * y + b (x, y
    [B, T, C, H, W], fp32 moments)"""
    for t in (x, y):
        if t.dtype != torch.float32:
            raise RuntimeError("expected torch.float32, got %s" % t.dtype)
    assert out.dtype == torch.float64 and x.shape == y.shape and out.numel() == x.shape[0] * x.shape[1]
    Cc, H, W = x.shape[2:]
    xf, yf = (a * t.reshape(-1, Cc, H, W) + b for t in (x, y))
    out.copy_(ssim_oracle.ssim(xf, yf, size_average=False))


def install(monkeypatch):
    emulator.install(monkeypatch)
    monkeypatch.setattr(ops, "ssim", emu_ssim)


def pairs(n, c, h, w, generator, device="cpu"):
    """(name, x, y) in [0, 1]: independent noise, a near-identical copy, a smoothed copy"""
    x = torch.rand(n, c, h, w, generator=generator).to(device)
    noise = torch.rand(n, c, h, w, generator=generator).to(device)
    close = (x + 0.05 * torch.randn(n, c, h, w, generator=generator).to(device)).clamp(0, 1)
    smooth = F.avg_pool2d(x, 5, 1, 2)
    return [("noise", x, noise), ("close", x, close), ("smooth", x, smooth)]


# ------------------------------------------------------------------------------------------ oracle
def brute_force_ssim(x, y):
    """per-frame SSIM by a double loop over every pixel and window tap (numpy, float64)"""
    g = np.array([math.exp(-(k - 5) ** 2 / 4.5) for k in range(11)])
    g /= g.sum()
    N, C, H, W = x.shape
    out = np.zeros(N)
    for n in range(N):
        total = 0.0
        for c in range(C):
            for i in range(H):
                for j in range(W):
                    m = np.zeros(5)       # E[x], E[y], E[x^2], E[y^2], E[xy]
                    for u in range(11):
                        for v in range(11):
                            r, s = i + u - 5, j + v - 5
                            if 0 <= r < H and 0 <= s < W:
                                a, b = x[n, c, r, s], y[n, c, r, s]
                                m += g[u] * g[v] * np.array([a, b, a * a, b * b, a * b])
                    mx, my = m[0], m[1]
                    sxx, syy, sxy = m[2] - mx * mx, m[3] - my * my, m[4] - mx * my
                    total += ((2 * mx * my + 1e-4) * (2 * sxy + 9e-4)) / ((mx * mx + my * my + 1e-4) *
                                                                         (sxx + syy + 9e-4))
        out[n] = total / (C * H * W)
    return out


@pytest.mark.parametrize("H,W", [(7, 9), (3, 5)])
def test_oracle_matches_brute_force(H, W):
    """pins the zero padding (border windows not renormalised), the window and its normalisation, C1 and C2"""
    g = torch.Generator().manual_seed(H * W)
    for name, x, y in pairs(2, 3, H, W, g):
        x, y = x.double(), y.double()
        ref = brute_force_ssim(x.numpy(), y.numpy())
        got = ssim_oracle.ssim(x, y, size_average=False)
        assert np.allclose(got.numpy(), ref, rtol=0, atol=1e-13), (name, got, ref)
        assert abs(float(ssim_oracle.ssim(x, y)) - ref.mean()) <= 1e-13


# ------------------------------------------------------------------------------------------ host logic
def test_frame_ssim_story_view_equals_frames(monkeypatch):
    """stories [B, C, T, H, W] go in without a copy; frame b * T + t of the result is frame (b, t)"""
    install(monkeypatch)
    g = torch.Generator().manual_seed(1)
    x = torch.rand(2, 3, 4, 16, 24, generator=g)
    y = (x + 0.1 * torch.randn(x.shape, generator=g)).clamp(0, 1)
    got = ssim.frame_ssim(x, y)
    want = ssim.frame_ssim(*(t.transpose(1, 2).reshape(-1, 3, 16, 24) for t in (x, y)))
    assert got.shape == (8,) and got.dtype == torch.float64
    assert torch.equal(got, want)
    ref = ssim_oracle.ssim(*(t.transpose(1, 2).reshape(-1, 3, 16, 24).double() for t in (x, y)), size_average=False)
    assert float((got - ref).abs().max()) <= 2e-6


def test_frame_ssim_strided_views_and_input_range(monkeypatch):
    install(monkeypatch)
    g = torch.Generator().manual_seed(2)
    xb = torch.rand(3, 5, 12, 20, generator=g)
    x = xb[:, 1:4, :, ::2]                                                   # channel slice, strided columns
    y = torch.rand(3, 12, 10, 3, generator=g).permute(0, 3, 1, 2)            # channels last
    assert not x.is_contiguous() and not y.is_contiguous()
    got = ssim.frame_ssim(x, y)
    ref = ssim_oracle.ssim(x.double(), y.double(), size_average=False)
    assert float((got - ref).abs().max()) <= 2e-6
    assert torch.equal(got, ssim.frame_ssim(x.contiguous(), y.contiguous()))
    # [-1, 1] inputs with input_range=(-1, 1) score as the same frames in [0, 1]
    got_pm = ssim.frame_ssim(2 * x - 1, 2 * y - 1, input_range=(-1, 1))
    assert float((got_pm - ref).abs().max()) <= 2e-6
    # and without the mapping they would not: C1 / C2 assume a dynamic range of 1
    assert float((ssim.frame_ssim(2 * x - 1, 2 * y - 1) - ref).abs().max()) > 1e-3


def test_frame_ssim_refusals(monkeypatch):
    x = torch.rand(2, 3, 8, 8)
    with pytest.raises(ValueError, match="shape"):
        ssim.frame_ssim(x, x[:1])
    with pytest.raises(ValueError, match="shape"):
        ssim.frame_ssim(x, x.transpose(2, 3)[..., :4])
    with pytest.raises(ValueError, match="frames"):
        ssim.frame_ssim(x[0], x[0])
    with pytest.raises(ValueError, match="input_range"):
        ssim.frame_ssim(x, x, input_range=(1, 1))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ssim.frame_ssim(x, x)                       # the real binding: CPU tensors are refused
    install(monkeypatch)
    for dtype in (torch.float64, torch.float16):
        with pytest.raises(RuntimeError, match="float32"):
            ssim.frame_ssim(x.to(dtype), x.to(dtype))


def test_kernel_argument_errors_do_not_need_a_gpu():
    lib = _lib.load()
    out = torch.zeros(1, dtype=torch.float64)
    p = ctypes.c_void_p(out.data_ptr())
    assert lib.cpcsv_ssim(None, p, 1, 1, 1, 8, 8, 0, 0, 0, 8, 1, 0, 0, 0, 8, 1, 1.0, 0.0, p, None) < 0
    assert b"ssim" in lib.cpcsv_last_error_string()
    assert lib.cpcsv_ssim(p, p, 1, 1, 1, 0, 8, 0, 0, 0, 8, 1, 0, 0, 0, 8, 1, 1.0, 0.0, p, None) < 0
    assert b"H 0" in lib.cpcsv_last_error_string()


# ------------------------------------------------------------------------------------------ trainer hook
def run_calculate_ssim(device, batches):
    """tiny-preset generator and synthetic test batches; calculate_ssim twice -> the value"""
    p = presets.get("tiny")
    netG = harness.build_product(p, params.init_all(p, 0), device)["G"]
    loader = []
    for seed in range(1, batches + 1):
        b = synth.make_batch(p, seed, device=device)
        loader.append({"images": b["st_real"], "description": b["st_desc"], "labels": b["st_labels"]})
    t, logged = _trainer()
    before = {k: v.clone() for k, v in netG.state_dict().items() if "running" in k or "tracked" in k}
    v1 = t.calculate_ssim(netG, loader, epoch=3)
    assert netG.training
    v2 = t.calculate_ssim(netG, loader, epoch=4)
    tol = 0.0 if device.type == "cpu" else 1e-4 * abs(v1)
    assert isinstance(v1, float) and -1.0 <= v1 <= 1.0 and abs(v1 - v2) <= tol, (v1, v2)
    for k, v in netG.state_dict().items():
        if k in before:
            assert torch.equal(v, before[k]), k
    assert logged == [("Evaluation/ssim", v1, 3), ("Evaluation/ssim", v2, 4)]
    return v1


def test_calculate_ssim_emulated(monkeypatch):
    install(monkeypatch)
    torch.set_num_threads(min(8, os.cpu_count() or 1))
    run_calculate_ssim(torch.device("cpu"), 1)


# ------------------------------------------------------------------------------------------ GPU
# per-frame |kernel - fp64 oracle|: torch's fp32 restatement on the CPU is within 4e-7 on 64 x 64 frames
SSIM_ATOL = 2e-6
KERNEL_SHAPES = [(7, 3, 64, 64), (5, 1, 64, 64), (3, 3, 37, 53), (4, 3, 3, 5), (2, 3, 128, 96)]


def _layout(t, kind, generator):
    """frames t [N, C, H, W] -> (tensor handed to frame_ssim, the frames it holds in result order)"""
    N, C, H, W = t.shape
    if kind == "frames":
        return t, t
    if kind == "story":        # [B, C, T, H, W] view of a buffer with wider rows; frame b * T + t
        B = 2
        buf = torch.rand(B, C, N, H, W + 3, generator=generator).to(t.device)
        s = buf[..., 1:W + 1]
        s[1] = t.transpose(0, 1)
        s[0] = t.flip(0).transpose(0, 1)
        return s, s.transpose(1, 2).reshape(-1, C, H, W)
    assert kind == "slice"     # channel slice of a wider channels-last buffer
    buf = torch.rand(N, H, W, C + 2, generator=generator).to(t.device).permute(0, 3, 1, 2)
    v = buf[:, 1:C + 1]
    v.copy_(t)
    return v, v


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["frames", "story", "slice"])
@pytest.mark.parametrize("shape", KERNEL_SHAPES)
def test_ssim_kernel_matches_fp64_oracle(shape, layout):
    dev = torch.device("cuda")
    g = torch.Generator().manual_seed(sum(shape))
    worst = 0.0
    for name, x, y in pairs(*shape, g, dev):
        xa, xf = _layout(x, layout, g)
        ya, yf = _layout(y, layout, g)
        got = ssim.frame_ssim(xa, ya)
        ref = ssim_oracle.ssim(xf.double(), yf.double(), size_average=False)
        err = float((got - ref).abs().max())
        worst = max(worst, err)
        assert got.shape == ref.shape and err <= SSIM_ATOL, (name, err)
    print("%s %s max |d| %.2e" % (shape, layout, worst))


@pytest.mark.gpu
def test_ssim_kernel_input_range():
    dev = torch.device("cuda")
    g = torch.Generator().manual_seed(7)
    for name, x, y in pairs(6, 3, 64, 64, g, dev):
        ref = ssim_oracle.ssim(x.double(), y.double(), size_average=False)
        got = ssim.frame_ssim(2 * x - 1, 2 * y - 1, input_range=(-1, 1))
        assert float((got - ref).abs().max()) <= SSIM_ATOL, name


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(6, 3, 64, 64), (3, 1, 3, 5), (2, 3, 37, 53)])
def test_ssim_kernel_identity(shape):
    x = torch.rand(*shape, generator=torch.Generator().manual_seed(4)).cuda()
    assert float((ssim.frame_ssim(x, x) - 1).abs().max()) <= 1e-6


@pytest.mark.gpu
def test_ssim_kernel_bit_reproducible():
    """a frame's value does not depend on the batch, its index or a repeated call"""
    dev = torch.device("cuda")
    g = torch.Generator().manual_seed(11)
    x = torch.rand(1001, 3, 64, 64, generator=g).to(dev)
    y = (x + 0.05 * torch.randn(x.shape, generator=g).to(dev)).clamp(0, 1)
    alone = ssim.frame_ssim(x[:1], y[:1])
    xs, ys = x.roll(537, 0), y.roll(537, 0)           # frame 0 at index 537 among the 1000 others
    batch = ssim.frame_ssim(xs, ys)
    again = ssim.frame_ssim(xs, ys)
    assert torch.equal(batch[537:538], alone)
    assert torch.equal(batch, again)


@pytest.mark.gpu
def test_ssim_kernel_refuses_other_dtypes():
    x = torch.rand(2, 3, 8, 8, device="cuda")
    for dtype in (torch.float64, torch.float16, torch.bfloat16):
        with pytest.raises(RuntimeError, match="float32"):
            ssim.frame_ssim(x.to(dtype), x.to(dtype))


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_calculate_ssim_gpu():
    print("SSIM tiny %.6f" % run_calculate_ssim(torch.device("cuda"), 2))
