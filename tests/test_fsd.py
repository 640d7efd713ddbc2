"""Story-level Frechet distance on the kernel path (cpcsv_b200.fsd; reference fid/vfid_score.py with the
R(2+1)D-18 of fid/residual2p1.py): the tap tables of the new convolution geometries, the whole
``StoryFeatureNet`` against fp64 torchvision ``r2plus1d_18``, the statistics, the Frechet distance against the
scipy-``sqrtm`` formula, ``GANTrainer.calculate_fsd``, and (``-m gpu``) the residual-epilogue kernel
``cpcsv_bn_add_act_pack``.  The CPU cases run the product's host logic on the kernel-contract emulator; the
new entry point's emulation lives here."""
import os
import types

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import emulator
import harness
from cpcsv_b200 import conv, fsd, ops
from oracle import params, presets, synth

torchvision = pytest.importorskip("torchvision")


# ------------------------------------------------------------------------------------------ emulation
def emu_bn_add_act_pack(x, scale, shift, r, rscale, rshift, act, y=None, hi=None, lo=None, dtype=1):
    """include/cpcsv.h cpcsv_bn_add_act_pack: y = act(x*scale + shift + (r*rscale + rshift))"""
    assert x.shape == r.shape and x.shape[1] % 4 == 0 and (rscale is None) == (rshift is None)
    v = torch.addcmul(shift.view(1, -1), x.float(), scale.view(1, -1))
    res = r.float() if rscale is None else torch.addcmul(rshift.view(1, -1), r.float(), rscale.view(1, -1))
    v = emulator._act(v + res, act)
    if y is not None:
        y.copy_(v)
    if hi is not None:
        h, l_ = emulator._split16(v, dtype)
        hi.copy_(h)
        if lo is not None:
            lo.copy_(l_)


def install(monkeypatch):
    emulator.install(monkeypatch)
    monkeypatch.setattr(ops, "bn_add_act_pack", emu_bn_add_act_pack)


def _bf16(t):
    return t.to(torch.bfloat16).double()


def _rel(a, b):
    return float((a.double().cpu() - b.double().cpu()).norm() / b.double().cpu().norm())


# ------------------------------------------------------------------------------------------ tap tables
@pytest.mark.parametrize("T", [4, 5])
def test_temporal_stride1_taps(monkeypatch, T):
    """Conv3d (3, 1, 1) stride 1 pad (1, 0, 0): one three-tap job, zero fill as the temporal padding"""
    install(monkeypatch)
    g = torch.Generator().manual_seed(T)
    B, H, W, Ci, Co = 2, 4, 4, 64, 48
    x = _bf16(torch.randn(B, Ci, T, H, W, generator=g))
    w = _bf16(torch.randn(Co, Ci, 3, 1, 1, generator=g))
    ref = F.conv3d(x, w, padding=(1, 0, 0)).permute(0, 2, 3, 4, 1).reshape(B, T, H * W, Co)
    xp = x.permute(0, 2, 3, 4, 1).reshape(B, T, H * W, Ci).to(torch.bfloat16).contiguous()
    wp = torch.zeros(3, 64, Ci, dtype=torch.bfloat16)
    wp[:, :Co] = w.view(Co, Ci, 3).permute(2, 0, 1).to(torch.bfloat16)
    out = torch.full((B, T, H * W, 64), float("nan"))
    ops.conv_gemm(conv.conv_t3s1_fwd([xp, None], [wp.view(3 * 64, Ci), None], out))
    assert torch.allclose(out[..., :Co].double(), ref, rtol=1e-6, atol=1e-5)
    assert torch.all(out[..., Co:] == 0)


@pytest.mark.parametrize("T", [4, 5])
def test_shortcut_stride2_taps(monkeypatch, T):
    """Conv3d (1, 1, 1) stride (2, 2, 2): one parity-view job per output frame (even frames, rows, columns)"""
    install(monkeypatch)
    g = torch.Generator().manual_seed(10 + T)
    B, H, W, Ci, Co = 3, 8, 8, 128, 64
    x = _bf16(torch.randn(B, Ci, T, H, W, generator=g))
    w = _bf16(torch.randn(Co, Ci, 1, 1, 1, generator=g))
    ref = F.conv3d(x, w, stride=2).permute(0, 2, 3, 4, 1)
    To = (T - 1) // 2 + 1
    assert ref.shape[1] == To
    xp = x.permute(0, 2, 3, 4, 1).to(torch.bfloat16).contiguous()
    out = torch.full((B, To, H // 2, W // 2, Co), float("nan"))
    jobs = conv.conv_p2_fwd([xp, None], [w.view(Co, Ci).to(torch.bfloat16), None], out)
    assert len(jobs) == To
    for job in jobs:
        ops.conv_gemm(job)
    assert torch.allclose(out.double(), ref, rtol=1e-6, atol=1e-5)


# ------------------------------------------------------------------------------------------ references
def preprocess64(stories):
    """what StoryFeatureNet does before the network, in fp64: [-1, 1] -> [0, 1] -> Kinetics mean / std"""
    mean = torch.tensor(fsd.KINETICS_MEAN, dtype=torch.float64, device=stories.device).view(1, 3, 1, 1, 1)
    std = torch.tensor(fsd.KINETICS_STD, dtype=torch.float64, device=stories.device).view(1, 3, 1, 1, 1)
    return ((stories.double() + 1) * 0.5 - mean) / std


def smooth_stories(n, T, generator, side=64):
    """stories in [-1, 1] with structure at several scales (features of white noise barely differ)"""
    x = torch.rand(n, 3, T, side // 8, side // 8, generator=generator) * 2 - 1
    x = F.interpolate(x, size=(T, side, side), mode="trilinear", align_corners=False)
    return (0.8 * x + 0.2 * (torch.rand(n, 3, T, side, side, generator=generator) * 2 - 1)).clamp(-1, 1)


_CALIBRATED = {}


def calibrated_reference(seed=0):
    """torchvision r2plus1d_18 (fc = Identity) with BatchNorm running statistics calibrated by train-mode passes
    (cumulative averages, momentum None) over synthetic stories, then randomised gamma / beta, in eval mode"""
    if seed not in _CALIBRATED:
        torch.manual_seed(seed)
        tv = torchvision.models.video.r2plus1d_18(weights=None)
        tv.fc = torch.nn.Identity()
        g = torch.Generator().manual_seed(seed + 1)
        bns = [m for m in tv.modules() if isinstance(m, torch.nn.BatchNorm3d)]
        for bn in bns:
            bn.momentum = None
            bn.reset_running_stats()
        tv.train()
        with torch.no_grad():
            for _ in range(3):
                tv(preprocess64(smooth_stories(4, 5, g)).float())
            for bn in bns:
                bn.weight.uniform_(0.75, 1.25, generator=g)
                bn.bias.uniform_(-0.1, 0.1, generator=g)
                bn.momentum = 0.1
        _CALIBRATED[seed] = {k: v.clone() for k, v in tv.eval().state_dict().items()}
    tv = torchvision.models.video.r2plus1d_18(weights=None)
    tv.fc = torch.nn.Identity()
    tv.load_state_dict(_CALIBRATED[seed])
    return tv.eval()


def reference_features(tv64, stories, chunk=32):
    with torch.no_grad():
        return torch.cat([tv64(preprocess64(stories[i:i + chunk])) for i in range(0, stories.shape[0], chunk)])


def product_net(dev, seed=0, chunk=256):
    net = fsd.StoryFeatureNet(chunk=chunk)
    net.load_state_dict(calibrated_reference(seed).state_dict())
    return net.to(dev)


# ------------------------------------------------------------------------------------------ feature network
def test_feature_net_emulated_matches_fp64_torchvision(monkeypatch):
    """stem + layer1..4 + pool of the product on the emulated kernels vs fp64 torchvision (2 stories, 3x5x64x64)"""
    install(monkeypatch)
    torch.set_num_threads(min(8, os.cpu_count() or 1))
    g = torch.Generator().manual_seed(3)
    stories = smooth_stories(2, 5, g)
    ref = reference_features(calibrated_reference().double(), stories)
    with torch.no_grad():
        feats = product_net(torch.device("cpu"), chunk=1)(stories)
    assert feats.shape == (2, fsd.FEATURE_DIM) and feats.dtype == torch.float32
    for i in range(2):
        r = _rel(feats[i], ref[i])
        print("story %d relL2 %.2e" % (i, r))
        assert r <= 1e-3, (i, r)


def test_state_dict_names_and_refusals():
    """torchvision's state_dict (fc included) loads strictly, the product's own keys are torchvision's minus fc,
    and train mode / grad-enabled calls raise"""
    tv = torchvision.models.video.r2plus1d_18(weights=None)
    net = fsd.StoryFeatureNet()
    net.load_state_dict(tv.state_dict(), strict=True)
    assert set(net.state_dict()) == {k for k in tv.state_dict() if not k.startswith("fc.")}
    for k, v in net.state_dict().items():
        assert torch.equal(v, tv.state_dict()[k]), k
    assert not net.training
    x = torch.zeros(1, 3, 2, 64, 64)
    with pytest.raises(RuntimeError, match="torch.no_grad"):
        net(x)
    net.train()
    with torch.no_grad(), pytest.raises(RuntimeError, match="eval mode"):
        net(x)
    net.eval()
    with torch.no_grad(), pytest.raises(NotImplementedError, match="powers of two"):
        net(torch.zeros(1, 3, 2, 48, 64))


# ------------------------------------------------------------------------------------------ statistics
def _scipy_fd(mu1, s1, mu2, s2):
    """the Frechet distance as the reference's FID code computes it (scipy.linalg.sqrtm of s1 s2)"""
    from scipy import linalg
    covmean = linalg.sqrtm(s1.dot(s2))
    if isinstance(covmean, tuple):
        covmean = covmean[0]
    if np.iscomplexobj(covmean):
        covmean = covmean.real
    diff = mu1 - mu2
    return float(diff.dot(diff) + np.trace(s1) + np.trace(s2) - 2 * np.trace(covmean))


@pytest.mark.parametrize("n1,n2", [(200, 300), (40, 300)])
def test_frechet_distance_matches_scipy_sqrtm(n1, n2):
    """random SPD covariances; (40, 300): the first one has rank 40 of 64"""
    rng = np.random.default_rng(n1)
    D = 64
    a = rng.standard_normal((D, n1)) * rng.uniform(0.2, 2.0, (D, 1))
    b = rng.standard_normal((D, n2)) + 0.3 * rng.standard_normal((D, D)) @ rng.standard_normal((D, n2)) / 8
    s1, s2 = a @ a.T / n1, b @ b.T / n2
    mu1, mu2 = rng.standard_normal(D), rng.standard_normal(D) * 0.5
    if n1 < D:
        assert np.linalg.matrix_rank(s1) == n1
    ref = _scipy_fd(mu1, s1, mu2, s2)
    got = fsd.frechet_distance(torch.from_numpy(mu1), torch.from_numpy(s1), torch.from_numpy(mu2),
                               torch.from_numpy(s2))
    assert abs(got - ref) <= 1e-8 * abs(ref), (got, ref)
    assert abs(fsd.frechet_distance(torch.from_numpy(mu1), torch.from_numpy(s1), torch.from_numpy(mu1),
                                    torch.from_numpy(s1))) <= 1e-8 * np.trace(s1)


def test_feature_stats_streaming_and_npz_round_trip(tmp_path):
    rng = np.random.default_rng(5)
    feats = rng.standard_normal((301, 16)) @ rng.standard_normal((16, 16)) + rng.standard_normal(16)
    st = fsd.FeatureStats(dim=16)
    for lo, hi in ((0, 7), (7, 128), (128, 129), (129, 301)):
        st.update(torch.from_numpy(feats[lo:hi]).float())
    f32 = feats.astype(np.float32).astype(np.float64)
    assert st.n == 301
    assert np.allclose(st.mu.numpy(), f32.mean(0), rtol=1e-12, atol=1e-12)
    assert np.allclose(st.sigma.numpy(), np.cov(f32, rowvar=False), rtol=1e-10, atol=1e-12)
    path = str(tmp_path / "real_stats.npz")
    st.save(path)
    with np.load(path) as f:
        assert set(f.files) == {"mu", "sigma"} and f["sigma"].shape == (16, 16)
    back = fsd.FeatureStats.load(path)
    assert torch.equal(back.mu, st.mu) and torch.equal(back.sigma, st.sigma)
    assert fsd.frechet_distance(back.mu, back.sigma, st.mu, st.sigma) == pytest.approx(0.0, abs=1e-9)


# ------------------------------------------------------------------------------------------ trainer hook
def _trainer():
    import trainer
    t = trainer.GANTrainer.__new__(trainer.GANTrainer)      # __init__ binds a CUDA device
    logged = []
    t._logger = types.SimpleNamespace(add_scalar=lambda k, v, s: logged.append((k, v, s)))
    return t, logged


def run_calculate_fsd(device):
    """shared with the -m gpu case: tiny-preset generator, two synthetic test batches.  The features are
    reproducible bit for bit; the generator's own GEMMs may split their reductions (fp32 atomics), so on the GPU the
    generated stories -- and the FSD -- repeat up to rounding"""
    p = presets.get("tiny")
    netG = harness.build_product(p, params.init_all(p, 0), device)["G"]
    loader = []
    for seed in (1, 2):
        b = synth.make_batch(p, seed, device=device)
        loader.append({"images": b["st_real"], "description": b["st_desc"], "labels": b["st_labels"]})
    feature_net = product_net(device)
    t, logged = _trainer()
    before = {k: v.clone() for k, v in netG.state_dict().items() if "running" in k or "tracked" in k}
    v1 = t.calculate_fsd(netG, loader, feature_net, epoch=3)
    assert netG.training
    v2 = t.calculate_fsd(netG, loader, feature_net, epoch=4)
    tol = 0.0 if device.type == "cpu" else 1e-4 * abs(v1)
    assert np.isfinite(v1) and v1 > 0 and abs(v1 - v2) <= tol, (v1, v2)
    for k, v in netG.state_dict().items():
        if k in before:
            assert torch.equal(v, before[k]), k
    assert logged == [("Evaluation/fsd", v1, 3), ("Evaluation/fsd", v2, 4)]
    # cached real statistics give the same value without running the real stories again
    real = fsd.story_statistics([b["images"] for b in loader], feature_net)
    v3 = t.calculate_fsd(netG, loader, feature_net, real_stats=real)
    assert abs(v3 - v1) <= tol + 1e-9 * abs(v1), (v3, v1)
    return v1


def test_calculate_fsd_emulated(monkeypatch):
    install(monkeypatch)
    torch.set_num_threads(min(8, os.cpu_count() or 1))
    run_calculate_fsd(torch.device("cpu"))


# ------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("projected", [False, True])
def test_bn_add_act_pack_kernel(projected):
    """cpcsv_bn_add_act_pack against a torch fp64 restatement: strided x / r, padding channels, all outputs"""
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(1 + projected)
    rows, C, Cv = 3001, 192, 150
    x = torch.randn(rows, C + 64, device=dev, generator=g)[:, :C]
    r = torch.randn(rows, C + 32, device=dev, generator=g)[:, 32:]
    x[:, Cv:] = 0
    if not projected:
        r[:, Cv:] = 0

    def affine():
        sc = torch.rand(C, device=dev, generator=g) + 0.5
        sh = torch.randn(C, device=dev, generator=g) * 0.3
        sc[Cv:] = 0
        sh[Cv:] = 0
        return sc, sh
    scale, shift = affine()
    rscale, rshift = affine() if projected else (None, None)
    res = r.double() if not projected else r.double() * rscale.double() + rshift.double()
    ref = torch.relu(x.double() * scale.double() + shift.double() + res)
    y = torch.full((rows, C), float("nan"), device=dev)
    hi = torch.empty(rows, C + 64, device=dev, dtype=torch.bfloat16)[:, :C]
    lo = torch.empty(rows, C + 64, device=dev, dtype=torch.bfloat16)[:, :C]
    ops.bn_add_act_pack(x, scale, shift, r, rscale, rshift, ops.ACT_RELU, y, hi, lo)
    torch.cuda.synchronize()
    assert float((y.double() - ref).abs().max()) <= 1e-6 * float(ref.abs().max())
    assert torch.all(y[:, Cv:] == 0) and torch.all(hi[:, Cv:].float() == 0) and torch.all(lo[:, Cv:].float() == 0)
    assert torch.equal(hi, y.to(torch.bfloat16))
    assert float((hi.double() + lo.double() - y.double()).abs().max()) <= 2 ** -16 * float(y.abs().max())
    # single outputs, identity activation
    y2 = torch.empty(rows, C, device=dev)
    ops.bn_add_act_pack(x, scale, shift, r, rscale, rshift, ops.ACT_NONE, y=y2)
    torch.cuda.synchronize()
    ref2 = x.double() * scale.double() + shift.double() + res
    assert float((y2.double() - ref2).abs().max()) <= 1e-6 * float(ref2.abs().max())


@pytest.mark.gpu
@pytest.mark.timeout(900)
@pytest.mark.parametrize("T", [5, 4])
def test_feature_net_gpu_matches_fp64_torchvision(T):
    dev = torch.device("cuda")
    g = torch.Generator().manual_seed(20 + T)
    stories = smooth_stories(64, T, g).to(dev)
    ref = reference_features(calibrated_reference().double().to(dev), stories)
    with torch.no_grad():
        feats = product_net(dev, chunk=48)(stories)        # two chunks, the second one partial
    errs = [(feats[i].double() - ref[i]).norm().item() / ref[i].norm().item() for i in range(64)]
    print("T=%d per-story relL2 max %.2e median %.2e" % (T, max(errs), sorted(errs)[32]))
    assert max(errs) <= 1e-3


@pytest.mark.gpu
@pytest.mark.timeout(1800)
def test_fsd_gpu_matches_fp64_torchvision_features():
    """FSD between 512 synthetic stories and a perturbation of them, from product features vs fp64 torchvision"""
    dev = torch.device("cuda")
    g = torch.Generator().manual_seed(99)
    a = smooth_stories(512, 5, g)
    b = (0.85 * a + 0.15 * smooth_stories(512, 5, g) + 0.05).clamp(-1, 1)
    tv64 = calibrated_reference().double().to(dev)
    net = product_net(dev)
    vals = {}
    for name, fn in (("product", lambda s: net(s)), ("fp64", lambda s: reference_features(tv64, s, chunk=64))):
        with torch.no_grad():
            sa = fsd.FeatureStats().update(fn(a.to(dev)))
            sb = fsd.FeatureStats().update(fn(b.to(dev)))
        vals[name] = fsd.frechet_distance(sa.mu, sa.sigma, sb.mu, sb.sigma)
    print("FSD product %.6f fp64 %.6f" % (vals["product"], vals["fp64"]))
    assert vals["fp64"] > 0
    assert abs(vals["product"] - vals["fp64"]) <= 1e-3 * vals["fp64"]


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_calculate_fsd_gpu():
    print("FSD tiny %.6f" % run_calculate_fsd(torch.device("cuda")))
