"""tcgen05 GEMM jobs (cpcsv_b200/conv.py) against torch.nn.functional fp32 references.

Every case runs twice: with the CPU emulator of the kernel contract (host index logic, runs
anywhere) and, marked ``gpu``, through libcpcsv.so on the B200 (the kernel itself).
"""
import pytest
import torch
import torch.nn.functional as F

import emulator
from cpcsv_b200 import conv, ops


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


def split(x, planes):
    hi = x.to(torch.bfloat16)
    if planes == 1:
        return [hi, None], hi.float()
    lo = (x - hi.float()).to(torch.bfloat16)
    return [hi, lo], x


def pack_w(w, kind, rows_pad, cols_pad, planes, dev):
    ntap = 16 if kind >= 2 else w.shape[2] * w.shape[3]
    hi = torch.empty(ntap * rows_pad, cols_pad, dtype=torch.bfloat16, device=dev)
    lo = torch.empty_like(hi) if planes == 2 else None
    ops.pack_conv_weight(w.contiguous(), kind, rows_pad, cols_pad, hi, lo)
    return [hi, lo]


def nhwc(x):
    return x.permute(0, 2, 3, 1).contiguous()


def rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30))


def eff_weight(w, planes):
    """the weight values the kernel actually multiplies with"""
    hi = w.to(torch.bfloat16).float()
    if planes == 1:
        return hi
    return hi + (w - hi).to(torch.bfloat16).float()


TOL = {1: 2e-5, 2: 2e-5}


@pytest.mark.parametrize("planes", [1, 2])
@pytest.mark.parametrize("N,H,Ci,Co", [(3, 8, 64, 64), (5, 4, 128, 128), (2, 16, 64, 256)])
def test_conv3x3_fwd(dev, planes, N, H, Ci, Co):
    x = rnd(N, Ci, H, H, seed=1, dev=dev)
    w = rnd(Co - 4, Ci - 3, 3, 3, seed=2, dev=dev, scale=0.05)   # ragged true channel counts
    xp, x_eff = split(nhwc(x), planes)
    x_eff = x_eff.permute(0, 3, 1, 2)
    wp = pack_w(w, 0, Co, Ci, planes, dev)
    out = torch.full((N, H, H, Co), 7.0, device=dev)
    ops.conv_gemm(conv.conv_s1_fwd(xp, wp, out))
    ref = F.conv2d(x_eff[:, :Ci - 3].double(), eff_weight(w, planes).double(), padding=1)
    got = out.permute(0, 3, 1, 2)
    # planes=2 drops the lo*lo term: relative error ~2^-16 of the operand products
    assert rel(got[:, :Co - 4], ref) < (3e-5 if planes == 2 else 1e-5)
    assert float(got[:, Co - 4:].abs().max()) == 0.0


@pytest.mark.parametrize("planes", [1, 2])
@pytest.mark.parametrize("N,H,Ci,Co", [(3, 4, 128, 64), (2, 8, 64, 128), (9, 4, 64, 64)])
def test_upconv_fwd(dev, planes, N, H, Ci, Co):
    x = rnd(N, Ci, H, H, seed=3, dev=dev)
    w = rnd(Co, Ci, 3, 3, seed=4, dev=dev, scale=0.05)
    xp, x_eff = split(nhwc(x), planes)
    wp = pack_w(w, 2, Co, Ci, planes, dev)
    out = torch.zeros(N, 2 * H, 2 * H, Co, device=dev)
    ops.conv_gemm(conv.upconv_fwd(xp, wp, out))
    ref = F.conv2d(F.interpolate(x_eff.permute(0, 3, 1, 2).double(), scale_factor=2, mode="nearest"),
                   w.double(), padding=1)
    # merged weights are rounded after merging -> compare at bf16-weight accuracy
    assert rel(out.permute(0, 3, 1, 2), ref) < (3e-3 if planes == 1 else 3e-5)


@pytest.mark.parametrize("planes", [1, 2])
@pytest.mark.parametrize("N,H,Ci,Co", [(3, 8, 64, 128), (2, 16, 128, 64), (17, 8, 64, 64)])
def test_conv4x4s2_fwd(dev, planes, N, H, Ci, Co):
    x = rnd(N, Ci, H, H, seed=5, dev=dev)
    w = rnd(Co, Ci, 4, 4, seed=6, dev=dev, scale=0.05)
    xp, x_eff = split(nhwc(x), planes)
    wp = pack_w(w, 0, Co, Ci, planes, dev)
    alpha = torch.tensor([0.37], device=dev)
    out = torch.zeros(N, H // 2, H // 2, Co, device=dev)
    ops.conv_gemm(conv.conv_s2_fwd(xp, wp, out, alpha=alpha))
    ref = 0.37 * F.conv2d(x_eff.permute(0, 3, 1, 2).double(), eff_weight(w, planes).double(), stride=2, padding=1)
    assert rel(out.permute(0, 3, 1, 2), ref) < 3e-5


def _grad_refs(fwd, x, w, dy):
    x = x.double().requires_grad_(True)
    w = w.double().requires_grad_(True)
    y = fwd(x, w)
    gx, gw = torch.autograd.grad(y, (x, w), dy.double())
    return gx, gw


def bf16r(t):
    return t.to(torch.bfloat16).float()


@pytest.mark.parametrize("N,H,Ci,Co", [(3, 8, 64, 64), (6, 4, 128, 64)])
def test_conv3x3_backward(dev, N, H, Ci, Co):
    x = bf16r(rnd(N, Ci, H, H, seed=7, dev=dev))
    w = bf16r(rnd(Co, Ci, 3, 3, seed=8, dev=dev, scale=0.05))
    dy = bf16r(rnd(N, Co, H, H, seed=9, dev=dev))
    gx, gw = _grad_refs(lambda a, b: F.conv2d(a, b, padding=1), x, w, dy)
    dy16 = nhwc(dy).to(torch.bfloat16)
    wt = pack_w(w, 1, Ci, Co, 1, dev)[0]
    dx = torch.zeros(N, H, H, Ci, device=dev)
    ops.conv_gemm(conv.conv_s1_dgrad(dy16, wt, dx))
    assert rel(dx.permute(0, 3, 1, 2), gx) < 1e-5
    dwt = torch.zeros(9, Co, Ci, device=dev)
    ops.conv_gemm(conv.conv_s1_wgrad(dy16, nhwc(x).to(torch.bfloat16), dwt))
    dw = torch.empty(Co, Ci, 3, 3, device=dev)
    ops.unpack_conv_wgrad(dwt, Co * Ci, Ci, 0, None, dw)
    assert rel(dw, gw) < 1e-5


@pytest.mark.parametrize("N,H,Ci,Co", [(3, 4, 64, 64), (5, 8, 128, 64)])
def test_upconv_backward(dev, N, H, Ci, Co):
    x = bf16r(rnd(N, Ci, H, H, seed=10, dev=dev))
    w = rnd(Co, Ci, 3, 3, seed=11, dev=dev, scale=0.05)
    dz = bf16r(rnd(N, Co, 2 * H, 2 * H, seed=12, dev=dev))
    gx, gw = _grad_refs(lambda a, b: F.conv2d(F.interpolate(a, scale_factor=2, mode="nearest"), b, padding=1),
                        x, w, dz)
    dz16 = nhwc(dz).to(torch.bfloat16)
    wmt = pack_w(w, 3, Ci, Co, 1, dev)[0]
    dx = torch.zeros(N, H, H, Ci, device=dev)
    ops.conv_gemm(conv.upconv_dgrad(dz16, wmt, dx))
    assert rel(dx.permute(0, 3, 1, 2), gx) < 4e-3        # merged weights rounded to bf16
    dwt = torch.zeros(16, Co, Ci, device=dev)
    ops.conv_gemm(conv.upconv_wgrad(dz16, nhwc(x).to(torch.bfloat16), dwt))
    dw = torch.empty(Co, Ci, 3, 3, device=dev)
    ops.unpack_conv_wgrad(dwt, Co * Ci, Ci, 2, None, dw)
    assert rel(dw, gw) < 1e-5


@pytest.mark.parametrize("N,H,Ci,Co", [(3, 8, 64, 64), (4, 16, 64, 128)])
def test_conv4x4s2_backward(dev, N, H, Ci, Co):
    x = bf16r(rnd(N, Ci, H, H, seed=13, dev=dev))
    w = bf16r(rnd(Co, Ci, 4, 4, seed=14, dev=dev, scale=0.05))
    dy = bf16r(rnd(N, Co, H // 2, H // 2, seed=15, dev=dev))
    gx, gw = _grad_refs(lambda a, b: F.conv2d(a, b, stride=2, padding=1), x, w, dy)
    dy16 = nhwc(dy).to(torch.bfloat16)
    wt = pack_w(w, 1, Ci, Co, 1, dev)[0]
    dx = torch.zeros(N, H, H, Ci, device=dev)
    ops.conv_gemm(conv.conv_s2_dgrad(dy16, wt, dx))
    assert rel(dx.permute(0, 3, 1, 2), gx) < 1e-5
    dwt = torch.zeros(16, Co, Ci, device=dev)
    ops.conv_gemm(conv.conv_s2_wgrad(dy16, nhwc(x).to(torch.bfloat16), dwt))
    dw = torch.empty(Co, Ci, 4, 4, device=dev)
    ops.unpack_conv_wgrad(dwt, Co * Ci, Ci, 0, None, dw)
    assert rel(dw, gw) < 1e-5


@pytest.mark.parametrize("M,K,N_", [(90, 640, 512), (7, 64, 16), (300, 128, 1024)])
def test_gemm_nt_tn(dev, M, K, N_):
    a = rnd(M, K, seed=16, dev=dev)
    b = rnd(N_, K, seed=17, dev=dev, scale=0.05)
    ap, a_eff = split(a, 2)
    bh = b.to(torch.bfloat16)
    bl = (b - bh.float()).to(torch.bfloat16)
    out = torch.zeros(M, N_, device=dev)
    ops.conv_gemm(conv.gemm_nt(ap, [bh, bl], out))
    assert rel(out, a.double() @ b.double().t()) < 3e-5
    # accumulate on top
    ops.conv_gemm(conv.gemm_nt([ap[0], None], [bh, None], out, accumulate=True))
    ref2 = a.double() @ b.double().t() + ap[0].double() @ bh.double().t()
    assert rel(out, ref2) < 3e-5
    if N_ % 64 == 0 and K % 64 == 0:
        c = torch.zeros(K, N_, device=dev)
        a16 = a.to(torch.bfloat16)
        d = rnd(M, N_, seed=18, dev=dev).to(torch.bfloat16)
        ops.conv_gemm(conv.gemm_tn(a16, d, c))
        assert rel(c, a16.double().t() @ d.double()) < 1e-5


def test_split_k_and_many_tiles(dev):
    """forced split-K (red.add epilogue) and a grid with more tiles than SMs"""
    N, H, Ci, Co = (2, 4, 512, 64)
    x = rnd(N, Ci, H, H, seed=19, dev=dev)
    w = rnd(Co, Ci, 3, 3, seed=20, dev=dev, scale=0.05)
    xp, x_eff = split(nhwc(x), 2)
    wp = pack_w(w, 0, Co, Ci, 2, dev)
    out = torch.full((N, H, H, Co), 3.0, device=dev)
    job = conv.conv_s1_fwd(xp, wp, out)
    job.splits = 5
    ops.conv_gemm(job)
    ref = F.conv2d(x.double(), eff_weight(w, 2).double(), padding=1)
    assert rel(out.permute(0, 3, 1, 2), ref) < 3e-5
    if dev.type == "cuda":
        N, H, Ci, Co = (40, 32, 64, 64)       # 320 M-tiles > 148 SMs: persistent loop + 2 TMEM stages
        x = rnd(N, Ci, H, H, seed=21, dev=dev)
        w = rnd(Co, Ci, 3, 3, seed=22, dev=dev, scale=0.05)
        xp, x_eff = split(nhwc(x), 2)
        wp = pack_w(w, 0, Co, Ci, 2, dev)
        out = torch.zeros(N, H, H, Co, device=dev)
        ops.conv_gemm(conv.conv_s1_fwd(xp, wp, out))
        ref = F.conv2d(x, eff_weight(w, 2), padding=1)
        assert rel(out.permute(0, 3, 1, 2), ref) < 3e-5


@pytest.mark.parametrize("kind", ["up", "s2", "gemm"])
def test_epilogue_column_statistics(dev, kind):
    """cpcsv_gemm_t.stats: the GEMM epilogue adds the per-column sum / sum of squares of what it stores
    (the BatchNorm batch statistics of the conv output, reference model.py:31-32) into an fp64 accumulator"""
    if kind == "up":
        N, H, Ci, Co = 3, 8, 64, 128
        x, xe = split(rnd(N, H, H, Ci, seed=41, dev=dev), 2)
        w = rnd(Co, Ci, 3, 3, seed=42, dev=dev, scale=0.1)
        out = torch.empty(N, 2 * H, 2 * H, Co, device=dev)
        job = conv.upconv_fwd(x, pack_w(w, 2, Co, Ci, 2, dev), out)
    elif kind == "s2":
        N, H, Ci, Co = 5, 16, 64, 64
        x, xe = split(rnd(N, H, H, Ci, seed=43, dev=dev), 2)
        w = rnd(Co, Ci, 4, 4, seed=44, dev=dev, scale=0.1)
        out = torch.empty(N, H // 2, H // 2, Co, device=dev)
        job = conv.conv_s2_fwd(x, pack_w(w, 0, Co, Ci, 2, dev), out, alpha=torch.tensor([0.37], device=dev))
    else:
        M, K, Nn = 90, 128, 512
        a, _ = split(rnd(M, K, seed=45, dev=dev), 2)
        bw, _ = split(rnd(Nn, K, seed=46, dev=dev, scale=0.1), 2)
        out = torch.empty(M, Nn, device=dev)
        job = conv.gemm_nt(a, bw, out)
    job.splits = 1
    C = out.shape[-1]
    stats = torch.zeros(2, C, dtype=torch.float64, device=dev)
    stats[0, 0] = 5.0                      # contributions are ADDED
    job.stats = stats
    ops.conv_gemm(job)
    flat = out.reshape(-1, C).double()
    ref = torch.stack((flat.sum(0), (flat * flat).sum(0)))
    ref[0, 0] += 5.0
    assert float((stats - ref).abs().max() / ref.abs().max()) < 1e-6, kind


@pytest.mark.parametrize("B,T,HW,Ci,Co", [(3, 7, 16, 64, 128), (2, 4, 64, 128, 64), (4, 2, 4, 64, 64), (5, 1, 4, 64, 64)])
def test_temporal_conv_t3(dev, B, T, HW, Ci, Co):
    """Conv3d kernel (3, 1, 1) stride (2, 1, 1) pad (1, 0, 0) (reference model.py:160-189) as even / odd frame
    jobs: forward, data gradient, weight gradient against torch.nn.functional.conv3d, odd and even T, T = 1"""
    side = int(HW ** 0.5)
    x = rnd(B, Ci, T, side, side, seed=3, dev=dev)
    w = rnd(Co - 5, Ci - 2, 3, 1, 1, seed=4, dev=dev, scale=0.05)
    To = (T - 1) // 2 + 1
    xl = x.permute(0, 2, 3, 4, 1).reshape(B, T, HW, Ci).contiguous()          # [B, T, HW, C]
    xp, x_eff = split(xl, 2)
    wp = pack_w(w.view(Co - 5, Ci - 2, 3, 1), 0, Co, Ci, 2, dev)
    out = torch.full((B, To, HW, Co), 7.0, device=dev)
    for job in conv.conv_t3_fwd(xp, wp, out):
        ops.conv_gemm(job)
    xr = x[:, :Ci - 2].double().requires_grad_(True)
    wr = eff_weight(w, 2).double().requires_grad_(True)
    ref = F.conv3d(xr, wr, stride=(2, 1, 1), padding=(1, 0, 0))
    got = out.view(B, To, side, side, Co).permute(0, 4, 1, 2, 3)
    assert rel(got[:, :Co - 5], ref) < 3e-5
    assert float(got[:, Co - 5:].abs().max()) == 0.0
    # backward: single bf16 operands
    dy = rnd(B, Co, To, side, side, seed=5, dev=dev)
    dy[:, Co - 5:] = 0
    dyl = bf16r(dy).permute(0, 2, 3, 4, 1).reshape(B, To, HW, Co).contiguous().to(torch.bfloat16)
    xr2 = bf16r(x[:, :Ci - 2]).double().requires_grad_(True)
    wr2 = bf16r(w).double().requires_grad_(True)
    F.conv3d(xr2, wr2, stride=(2, 1, 1), padding=(1, 0, 0)).backward(bf16r(dy)[:, :Co - 5].double())
    wt = pack_w(w.view(Co - 5, Ci - 2, 3, 1), 1, Ci, Co, 1, dev)[0]
    dx = torch.full((B, T, HW, Ci), 7.0, device=dev)
    for job in conv.conv_t3_dgrad(dyl, wt, dx):
        ops.conv_gemm(job)
    gdx = dx.view(B, T, side, side, Ci).permute(0, 4, 1, 2, 3)
    assert rel(gdx[:, :Ci - 2], xr2.grad) < 1e-5
    assert float(gdx[:, Ci - 2:].abs().max()) == 0.0
    dwt = torch.zeros(3, Co, Ci, device=dev)
    for job in conv.conv_t3_wgrad(dyl, xp[0], dwt):
        ops.conv_gemm(job)
    gw = dwt[:, :Co - 5, :Ci - 2].permute(1, 2, 0)
    assert rel(gw, wr2.grad.view(Co - 5, Ci - 2, 3)) < 1e-5


@pytest.mark.parametrize("geom,N,H,Ci,Co", [("s1", 6, 8, 128, 256), ("s1", 20, 4, 256, 384), ("s2", 5, 16, 128, 512),
                                             ("up", 3, 8, 384, 256), ("s1", 40, 8, 320, 256)])
def test_wgrad_as_cta_pairs(dev, geom, N, H, Ci, Co):
    """weight-gradient jobs with more than one 128-channel M tile and block_n a multiple of 128 run as
    cta_group::2 pairs: even and odd numbers of M tiles, block_n 256 / 128 (and 64: no pair), split-K"""
    x = bf16r(rnd(N, Ci, H, H, seed=31, dev=dev))
    w = bf16r(rnd(Co, Ci, 4 if geom == "s2" else 3, 4 if geom == "s2" else 3, seed=32, dev=dev, scale=0.05))
    Ho = {"s1": H, "s2": H // 2, "up": 2 * H}[geom]
    dy = bf16r(rnd(N, Co, Ho, Ho, seed=33, dev=dev))
    fwd = {"s1": lambda a, b: F.conv2d(a, b, padding=1), "s2": lambda a, b: F.conv2d(a, b, stride=2, padding=1),
           "up": lambda a, b: F.conv2d(F.interpolate(a, scale_factor=2, mode="nearest"), b, padding=1)}[geom]
    _gx, gw = _grad_refs(fwd, x, w, dy)
    dy16, x16 = nhwc(dy).to(torch.bfloat16), nhwc(x).to(torch.bfloat16)
    ntap = {"s1": 9, "s2": 16, "up": 16}[geom]
    dwt = torch.full((ntap, Co, Ci), 7.0, device=dev)
    job = {"s1": conv.conv_s1_wgrad, "s2": conv.conv_s2_wgrad, "up": conv.upconv_wgrad}[geom](dy16, x16, dwt)
    assert job.pair == (job.block_n % 128 == 0)
    ops.conv_gemm(job)
    dw = torch.empty_like(w)
    ops.unpack_conv_wgrad(dwt, Co * Ci, Ci, 2 if geom == "up" else 0, None, dw)
    assert rel(dw, gw) < 1e-5
