"""Oracle restatement of ``pytorch_ssim._ssim`` (the SSIM of the reference's ``ssim_score.py`` / ``trainer.py``)
for any dtype.  TEST INFRASTRUCTURE: imported by tests and tools only.

The 2-D window is the outer product of the 11-tap Gaussian (sigma 1.5, normalised to sum 1), applied per channel
by ``F.conv2d(padding=5, groups=C)``: border windows see zeros and are not renormalised.
"""
import math

import torch
import torch.nn.functional as F

WINDOW = 11
SIGMA = 1.5
C1 = 0.01 ** 2
C2 = 0.03 ** 2


def gaussian(dtype=torch.float64, device=None):
    g = torch.tensor([math.exp(-(k - WINDOW // 2) ** 2 / (2 * SIGMA ** 2)) for k in range(WINDOW)], dtype=dtype,
                     device=device)
    return g / g.sum()


def ssim_map(x, y):
    """SSIM map [N, C, H, W] of frames x, y [N, C, H, W], computed in their dtype"""
    C = x.shape[1]
    g = gaussian(x.dtype, x.device)
    w = (g[:, None] @ g[None, :]).expand(C, 1, WINDOW, WINDOW).contiguous()

    def conv(t):
        return F.conv2d(t, w, padding=WINDOW // 2, groups=C)

    mu1, mu2 = conv(x), conv(y)
    mu1_sq, mu2_sq, mu1_mu2 = mu1 * mu1, mu2 * mu2, mu1 * mu2
    sigma1_sq = conv(x * x) - mu1_sq
    sigma2_sq = conv(y * y) - mu2_sq
    sigma12 = conv(x * y) - mu1_mu2
    return ((2 * mu1_mu2 + C1) * (2 * sigma12 + C2)) / ((mu1_sq + mu2_sq + C1) * (sigma1_sq + sigma2_sq + C2))


def ssim(x, y, size_average=True):
    """``pytorch_ssim.ssim(x, y, size_average)``: the mean of the map, or per frame [N] (size_average=False)"""
    m = ssim_map(x, y)
    return m.mean() if size_average else m.mean(1).mean(1).mean(1)
