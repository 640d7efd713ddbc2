"""Frame SSIM (the reference's ``ssim_score.py`` / the SSIM loop of its ``trainer.py``, both through
``pytorch_ssim``) on one kernel of libcpcsv.so, ``cpcsv_ssim``.

The contract is ``pytorch_ssim.ssim(x, y, size_average=False)``: an 11-tap Gaussian window (sigma 1.5, normalised to
sum 1) applied per channel with zero padding 5, the moments in fp32, C1 = 0.01^2 and C2 = 0.03^2, and per frame the
mean of the SSIM map over channels and pixels.  The kernel runs one CTA per frame and reduces in a fixed order, so a
frame's score is bit-reproducible and does not depend on the other frames of the call.
"""
import torch

from . import ops


def frame_ssim(x, y, input_range=(0, 1)):
    """Per-frame SSIM of ``x`` against ``y``: fp64 ``[N]`` for frames ``[N, C, H, W]``, fp64 ``[B * T]`` (frame
    ``b * T + t``, the order ``frame_fid.frame_statistics`` flattens stories in) for stories ``[B, C, T, H, W]``.

    ``x`` and ``y`` are fp32 CUDA tensors of the same shape with any strides; they are read in place.
    ``input_range`` is mapped to [0, 1] inside the kernel, the dynamic range C1 and C2 assume: with the default the
    values equal ``pytorch_ssim.ssim(x, y, size_average=False)``, and their mean ``size_average=True``."""
    if x.shape != y.shape:
        raise ValueError("frame_ssim: x %s and y %s differ in shape" % (tuple(x.shape), tuple(y.shape)))
    if x.device != y.device:
        raise ValueError("frame_ssim: x is on %s, y on %s" % (x.device, y.device))
    if x.dim() == 4:
        xv, yv = x.unsqueeze(1), y.unsqueeze(1)
    elif x.dim() == 5:
        xv, yv = x.transpose(1, 2), y.transpose(1, 2)
    else:
        raise ValueError("frame_ssim: expected frames [N, C, H, W] or stories [B, C, T, H, W], got %s"
                         % (tuple(x.shape),))
    lo, hi = float(input_range[0]), float(input_range[1])
    if not hi > lo:
        raise ValueError("frame_ssim: input_range %s is empty" % (tuple(input_range),))
    out = torch.empty(xv.shape[0] * xv.shape[1], dtype=torch.float64, device=x.device)
    ops.ssim(xv, yv, 1.0 / (hi - lo), -lo / (hi - lo), out)
    return out
