"""Story-level Frechet distance (FSD; the story metric of the paper, reference ``fid/vfid_score.py`` with the
R(2+1)D-18 of ``fid/residual2p1.py``): features of real and generated stories from an R(2+1)D-18 run on the
kernels of libcpcsv.so, their streaming Gaussian statistics, and the Frechet distance between two of them.

The contract is torchvision's ``r2plus1d_18`` forward (stem + layer1..4 + AdaptiveAvgPool3d(1), the 512
features in front of ``fc``) in eval mode, on stories preprocessed as documented in ``StoryFeatureNet``.
Every Conv3d of that network is (1, k, k) or (k, 1, 1); on channels-last activations ``[B * T, H, W, C]``
(frames as batch entries) each is an implicit GEMM the tcgen05 kernel runs with bf16 hi/lo split operands:

* stem (1, 7, 7) stride (1, 2, 2) pad (0, 3, 3) on 3 channels: im2col (K = 147 -> 192) + one GEMM
  (engine.Im2colNode, as the stem of the order-consistency critic);
* (3, 1, 1) stride 1 pad (1, 0, 0): engine.TemporalNode, ``conv.conv_t3s1_fwd`` on ``[B, T, HW, C]`` (one job,
  three frame taps);
* (3, 1, 1) stride (2, 1, 1) pad (1, 0, 0): engine.TemporalNode, ``conv.conv_t3_fwd`` (even / odd frames);
* (1, 3, 3) stride 1 pad (0, 1, 1): engine.ConvNode ``s1`` with frames as batch entries;
* (1, 3, 3) stride (1, 2, 2) pad (0, 1, 1): engine.ConvNode ``s2k3``, the 4x4 / stride-2 parity job with a zero
  4th row / column;
* (1, 1, 1) stride (2, 2, 2) shortcut projection: ``conv.conv_p2_fwd`` (one job per output frame).

Inner BatchNorm + ReLU: engine.BnActNode with the running statistics.  The end of a residual block (its last
BatchNorm, the shortcut's BatchNorm, the add, the ReLU) is one ``cpcsv_bn_add_act_pack`` launch.  Channel
counts are padded to multiples of 64 (stem 45, mid-planes 144 / 230 / 288 / 460 / 576 / 921 / 1152).
Forward only, eval mode only, under ``torch.no_grad()``.  The tape runs with ``split_k=False``, so no job splits
its reduction (split-K partial sums meet in fp32 atomics, in whatever order they arrive): a story's features
are bit-for-bit reproducible and do not depend on the other stories of its chunk, so the FSD of the same
stories is the same number every time.
"""
import numpy as np
import torch
import torch.nn as nn

from . import conv, ops
from .engine import T4, BnActNode, ConvNode, Im2colNode, Tape, TemporalNode, eval_affine, pack_taps, rup, _e
from .nets import _CACHE, _bn_tuple

# torchvision's Kinetics-400 normalisation of the R(2+1)D-18 weights (the reference feeds 64 x 64 frames to
# the network without a resize, SURVEY.md Appendix D)
KINETICS_MEAN = (0.43216, 0.394666, 0.37645)
KINETICS_STD = (0.22803, 0.22145, 0.216989)
FEATURE_DIM = 512


# ------------------------------------------------------------------------------------------ modules
class Conv2Plus1D(nn.Sequential):
    """torchvision.models.video.resnet.Conv2Plus1D: (1, 3, 3) spatial conv, BatchNorm, ReLU, (3, 1, 1) temporal"""

    def __init__(self, in_planes, out_planes, midplanes, stride=1):
        super().__init__(
            nn.Conv3d(in_planes, midplanes, (1, 3, 3), (1, stride, stride), (0, 1, 1), bias=False),
            nn.BatchNorm3d(midplanes), nn.ReLU(inplace=True),
            nn.Conv3d(midplanes, out_planes, (3, 1, 1), (stride, 1, 1), (1, 0, 0), bias=False))


class BasicBlock(nn.Module):
    """torchvision.models.video.resnet.BasicBlock with Conv2Plus1D (parameter names included)"""

    def __init__(self, inplanes, planes, stride=1):
        super().__init__()
        midplanes = (inplanes * planes * 3 * 3 * 3) // (inplanes * 3 * 3 + 3 * planes)
        self.conv1 = nn.Sequential(Conv2Plus1D(inplanes, planes, midplanes, stride), nn.BatchNorm3d(planes),
                                   nn.ReLU(inplace=True))
        self.conv2 = nn.Sequential(Conv2Plus1D(planes, planes, midplanes), nn.BatchNorm3d(planes))
        self.relu = nn.ReLU(inplace=True)
        self.downsample = None
        if stride != 1 or inplanes != planes:
            self.downsample = nn.Sequential(nn.Conv3d(inplanes, planes, 1, stride, bias=False),
                                            nn.BatchNorm3d(planes))
        self.stride = stride


def _stem():
    return nn.Sequential(nn.Conv3d(3, 45, (1, 7, 7), (1, 2, 2), (0, 3, 3), bias=False), nn.BatchNorm3d(45),
                         nn.ReLU(inplace=True),
                         nn.Conv3d(45, 64, (3, 1, 1), (1, 1, 1), (1, 0, 0), bias=False), nn.BatchNorm3d(64),
                         nn.ReLU(inplace=True))


class StoryFeatureNet(nn.Module):
    """R(2+1)D-18 story features on the kernel path: fp32 stories ``[B, 3, T, H, W]`` in ``input_range``
    (the generator's [-1, 1]) -> fp32 ``[B, 512]``.

    Parameter and buffer names are those of ``torchvision.models.video.r2plus1d_18``, so its ``state_dict()``
    (the Kinetics-400 checkpoint included) loads directly; ``fc.*`` entries are ignored.  Preprocessing: map
    ``input_range`` to [0, 1], then ``(x - mean) / std`` per channel; no resize.  Stories go through the
    network ``chunk`` at a time, so memory stays bounded at any batch size.  Eval mode and
    ``torch.no_grad()`` only; the module starts in eval mode."""

    def __init__(self, mean=KINETICS_MEAN, std=KINETICS_STD, input_range=(-1.0, 1.0), chunk=256):
        super().__init__()
        self.mean, self.std = tuple(float(m) for m in mean), tuple(float(s) for s in std)
        self.input_range = (float(input_range[0]), float(input_range[1]))
        assert len(self.mean) == 3 and len(self.std) == 3 and self.input_range[1] > self.input_range[0]
        self.chunk = int(chunk)
        self.stem = _stem()
        cfgs = ((64, 64, 1), (64, 128, 2), (128, 256, 2), (256, 512, 2))
        for i, (cin, cout, stride) in enumerate(cfgs):
            setattr(self, "layer%d" % (i + 1), nn.Sequential(BasicBlock(cin, cout, stride), BasicBlock(cout, cout)))
        self.register_load_state_dict_pre_hook(_drop_fc)
        self.eval()

    def blocks(self):
        return [b for layer in (self.layer1, self.layer2, self.layer3, self.layer4) for b in layer]

    def forward(self, stories):
        if self.training:
            raise RuntimeError("cpcsv_b200: StoryFeatureNet runs in eval mode only (BatchNorm with the running "
                               "statistics of the checkpoint); call .eval() before extracting features")
        if torch.is_grad_enabled():
            raise RuntimeError("cpcsv_b200: StoryFeatureNet is forward-only; call it under torch.no_grad()")
        if stories.dim() != 5 or stories.shape[1] != 3:
            raise ValueError("StoryFeatureNet: expected stories [B, 3, T, H, W], got %s" % (tuple(stories.shape),))
        B, _, T, H, W = stories.shape
        if not (_pow2(H) and _pow2(W) and H >= 32 and W >= 32):
            raise NotImplementedError("StoryFeatureNet: frame sides must be powers of two >= 32, got %dx%d" % (H, W))
        lo, hi = self.input_range
        dev = stories.device
        mean = torch.tensor(self.mean, device=dev, dtype=torch.float32)
        std = torch.tensor(self.std, device=dev, dtype=torch.float32)
        a = 1.0 / ((hi - lo) * std)
        b = (-lo / (hi - lo) - mean) / std
        out = torch.empty(B, FEATURE_DIM, device=dev)
        for s in range(0, B, self.chunk):
            x = stories[s:s + self.chunk].float()
            # [0, 1] and the per-channel normalisation in one elementwise pass that also lays the frames out
            # as batch entries n = b * T + t (NCHW, what the stem's im2col reads)
            frames = torch.addcmul(b.view(1, 1, 3, 1, 1), x.permute(0, 2, 1, 3, 4), a.view(1, 1, 3, 1, 1))
            out[s:s + x.shape[0]] = FeatureRunner(self).run(frames.contiguous().view(-1, 3, H, W), T)
        return out


def _pow2(n):
    return n > 0 and n & (n - 1) == 0


def _drop_fc(module, state_dict, prefix, *args):
    for k in [k for k in state_dict if k.startswith(prefix + "fc.")]:
        del state_dict[k]


# ------------------------------------------------------------------------------------------ tape nodes
class ShortcutNode:
    """Conv3d (1, 1, 1) stride (2, 2, 2), the projected shortcut: [B, T, H, W, Ci] -> [B, To, H/2, W/2, Co]"""

    def __init__(self, tape, x, B, weight, name):
        self.tape, self.x, self.B, self.w, self.name = tape, x, B, weight, name
        self.Co_pad, self.Ci_pad = rup(weight.shape[0], 64), x.C
        assert rup(weight.shape[1], 64) == x.C and x.N % B == 0 and x.H % 2 == 0 and x.W % 2 == 0, name
        self.T = x.N // B
        self.To = (self.T - 1) // 2 + 1
        self.out = T4(B * self.To, x.H // 2, x.W // 2, self.Co_pad)

    def _w4(self):
        w = self.w.detach()
        return w.view(w.shape[0], w.shape[1], 1, 1)

    def forward(self):
        t, x, out = self.tape, self.x, self.out
        wp = pack_taps(t.cache, self.w, self._w4, 0, self.Co_pad, self.Ci_pad, t.planes, t.dtype)
        out.f32 = _e((out.N, out.H, out.W, out.C), x.hi.device)
        xp = [p.view(self.B, self.T, x.H, x.W, x.C) for p in x.planes(t.planes) if p is not None]
        for job in conv.conv_p2_fwd(xp, wp, out.f32.view(self.B, self.To, out.H, out.W, out.C), dtype=t.dtype,
                                    splits=t.splits):
            ops.conv_gemm(job)


class ResidualNode:
    """relu(bn2(z) + shortcut): shortcut = the block input's fp32 values (identity) or bn_d(projection)"""

    def __init__(self, tape, z, r, bn, rbn, name, want_planes=True):
        self.tape, self.z, self.r, self.bn, self.rbn, self.name = tape, z, r, bn, rbn, name
        assert (r.N, r.H, r.W, r.C) == (z.N, z.H, z.W, z.C), name
        self.want_planes = want_planes
        self.out = T4(z.N, z.H, z.W, z.C)

    def forward(self):
        t, z, r, out = self.tape, self.z, self.r, self.out
        dev = z.f32.device
        scale, shift = eval_affine(_bn_tuple(self.bn), z.C, None, self.bn.weight.numel(), self.bn.eps)
        rscale = rshift = None
        if self.rbn is not None:
            rscale, rshift = eval_affine(_bn_tuple(self.rbn), r.C, None, self.rbn.weight.numel(), self.rbn.eps)
        out.f32 = _e((z.N, z.H, z.W, z.C), dev)
        if self.want_planes:
            t16 = ops.TORCH16[t.dtype]
            out.hi = _e((z.N, z.H, z.W, z.C), dev, t16)
            out.lo = _e((z.N, z.H, z.W, z.C), dev, t16) if t.planes == 2 else None
        ops.bn_add_act_pack(z.mat(z.f32), scale, shift, r.mat(r.f32), rscale, rshift, ops.ACT_RELU, z.mat(out.f32),
                            z.mat(out.hi) if out.hi is not None else None,
                            z.mat(out.lo) if out.lo is not None else None, t.dtype)
        z.f32 = r.f32 = None        # nothing reads the conv output or the shortcut again


class FeatureRunner:
    """one chunk of stories through stem + layer1..4 + AdaptiveAvgPool3d(1)"""

    def __init__(self, net):
        self.net = net

    def run(self, frames, T):
        """frames: normalised fp32 [B * T, 3, H, W] (n = b * T + t) -> fp32 [B, 512]"""
        net = self.net
        stem = net.stem
        B = frames.shape[0] // T
        tape = Tape(_CACHE, training=False, need_grad=False, planes=2, dtype=ops.BF16, split_k=False)
        z0 = tape.add(Im2colNode(tape, frames, stem[0].weight, "fsd.stem.0", 2, 3))
        a = tape.add(BnActNode(tape, z0, _bn_tuple(stem[1]), ops.ACT_RELU, "fsd.stem.1"))
        z = tape.add(TemporalNode(tape, a, B, stem[3].weight, "fsd.stem.3", 1))
        # fp32 values too: the identity shortcut of layer1.0
        a = tape.add(BnActNode(tape, z, _bn_tuple(stem[4]), ops.ACT_RELU, "fsd.stem.4", want_f32=True))
        blocks = net.blocks()
        for i, blk in enumerate(blocks):
            a = self._block(tape, a, B, blk, "fsd.block%d" % i, last=i == len(blocks) - 1)
        tape.finish_forward()
        # AdaptiveAvgPool3d(1): mean over the remaining frames and pixels of every story
        return a.f32.view(B, -1, a.C)[:, :, :FEATURE_DIM].mean(1)

    @staticmethod
    def _block(tape, x, B, blk, name, last):
        c1, c2 = blk.conv1[0], blk.conv2[0]
        s = blk.stride
        m = tape.add(ConvNode(tape, "s1" if s == 1 else "s2k3", x, c1[0].weight, name + ".conv1.0.0"))
        m = tape.add(BnActNode(tape, m, _bn_tuple(c1[1]), ops.ACT_RELU, name + ".conv1.0.1"))
        z = tape.add(TemporalNode(tape, m, B, c1[3].weight, name + ".conv1.0.3", s))
        a = tape.add(BnActNode(tape, z, _bn_tuple(blk.conv1[1]), ops.ACT_RELU, name + ".conv1.1"))
        m = tape.add(ConvNode(tape, "s1", a, c2[0].weight, name + ".conv2.0.0"))
        m = tape.add(BnActNode(tape, m, _bn_tuple(c2[1]), ops.ACT_RELU, name + ".conv2.0.1"))
        z = tape.add(TemporalNode(tape, m, B, c2[3].weight, name + ".conv2.0.3", 1))
        r, rbn = x, None
        if blk.downsample is not None:
            r = tape.add(ShortcutNode(tape, x, B, blk.downsample[0].weight, name + ".downsample.0"))
            rbn = blk.downsample[1]
        return tape.add(ResidualNode(tape, z, r, blk.conv2[1], rbn, name + ".out", want_planes=not last))


# ------------------------------------------------------------------------------------------ statistics
class FeatureStats:
    """Streaming mean and covariance of feature rows, in fp64 on the features' device: per ``update`` the sum
    and the sum of outer products.  ``save`` / ``load`` use an ``.npz`` file with keys ``mu`` and ``sigma``
    (the layout of the reference's ``r_cache`` files), so real-data statistics are computed once."""

    def __init__(self, dim=FEATURE_DIM, device=None):
        self.dim, self.device = dim, device
        self.n = 0
        self.s = self.ss = None
        self._mu = self._sigma = None

    def update(self, feats):
        f = feats.detach().to(torch.float64)
        assert f.dim() == 2 and f.shape[1] == self.dim, f.shape
        if self._mu is not None:
            raise RuntimeError("FeatureStats: statistics loaded from a file cannot be extended")
        if self.s is None:
            self.device = f.device
            self.s = torch.zeros(self.dim, dtype=torch.float64, device=f.device)
            self.ss = torch.zeros(self.dim, self.dim, dtype=torch.float64, device=f.device)
        self.s += f.sum(0)
        self.ss.addmm_(f.t(), f)
        self.n += f.shape[0]
        return self

    @property
    def mu(self):
        if self._mu is not None:
            return self._mu
        if self.n < 1:
            raise RuntimeError("FeatureStats: no features yet")
        return self.s / self.n

    @property
    def sigma(self):
        """unbiased covariance (np.cov's default, as the reference's FID code uses)"""
        if self._sigma is not None:
            return self._sigma
        if self.n < 2:
            raise RuntimeError("FeatureStats: a covariance needs at least 2 feature rows")
        mu = self.s / self.n
        sig = (self.ss - self.n * torch.outer(mu, mu)) / (self.n - 1)
        return (sig + sig.t()) * 0.5

    def save(self, path):
        np.savez(path, mu=self.mu.cpu().numpy(), sigma=self.sigma.cpu().numpy())

    @classmethod
    def load(cls, path, device=None):
        with np.load(path) as f:
            mu, sigma = f["mu"], f["sigma"]
        st = cls(dim=mu.shape[0], device=device)
        st._mu = torch.as_tensor(mu, dtype=torch.float64, device=device)
        st._sigma = torch.as_tensor(sigma, dtype=torch.float64, device=device)
        return st


def frechet_distance(mu1, sigma1, mu2, sigma2):
    """|mu1 - mu2|^2 + tr(s1) + tr(s2) - 2 tr((s1 s2)^(1/2)) in fp64 on the statistics' device.

    tr((s1 s2)^(1/2)) = tr((s1^(1/2) s2 s1^(1/2))^(1/2)): the eigenvalues of s1 s2 are those of the symmetric
    positive semi-definite s1^(1/2) s2 s1^(1/2), so two ``eigh`` calls replace the general matrix square root
    (``scipy.linalg.sqrtm`` in the reference's FID code); tiny negative eigenvalues from rounding count as 0."""
    dev = mu1.device if torch.is_tensor(mu1) else None

    def t(v):
        return torch.as_tensor(v, dtype=torch.float64, device=dev)
    mu1, sigma1, mu2, sigma2 = t(mu1), t(sigma1), t(mu2), t(sigma2)
    diff = mu1 - mu2
    s1 = (sigma1 + sigma1.t()) * 0.5
    s2 = (sigma2 + sigma2.t()) * 0.5
    ev1, vec1 = torch.linalg.eigh(s1)
    root1 = (vec1 * ev1.clamp_min(0).sqrt().unsqueeze(0)) @ vec1.t()
    m = root1 @ s2 @ root1
    ev = torch.linalg.eigvalsh((m + m.t()) * 0.5)
    tr_covmean = ev.clamp_min(0).sqrt().sum()
    return float(diff @ diff + torch.trace(s1) + torch.trace(s2) - 2.0 * tr_covmean)


def story_statistics(stories, feature_net, stats=None):
    """add the features of an iterable of story batches ``[B, 3, T, H, W]`` to ``stats`` (a new FeatureStats
    when None) and return it"""
    stats = stats if stats is not None else FeatureStats()
    with torch.no_grad():
        for x in stories:
            stats.update(feature_net(x))
    return stats
