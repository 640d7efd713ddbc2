"""Frames / s of per-frame SSIM (cpcsv_b200.ssim.frame_ssim, one kernel) against the pytorch_ssim algorithm
(oracle/ssim.py in fp32: five 11 x 11 depthwise convolutions on cuDNN plus the elementwise map) with TF32 off and
on, on stories of T x 3 x side x side frames in [0, 1] (a near-identical pair: y = clamp(x + 0.05 noise)).

Timing as tools/bench_fsd.py (whose helpers this uses): CUDA events around whole calls after two warm-up calls,
median of ``--reps``.  Both paths score the same contiguous frames [B * T, 3, side, side]; the kernel is also timed on
the story view [B, 3, T, side, side] it takes without a copy.  At 1024 stories each input is 252 MB, twice the L2;
at 256 stories both inputs (126 MB) about fit in it.  Accuracy: per-frame max |d| against the fp64 oracle on the
first 64 frames.  Work from shapes: bytes = both inputs read once plus the fp64 output; FMAs = 5 moments x 11 taps
x 2 passes per pixel and channel for the separable kernel, 5 x 121 for the 2-D window of pytorch_ssim.

Prints one JSON document (and writes it to ``--out`` when given).  Development tool, not the contract benchmark."""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "cpcstoryvisualization-pytorch_b200"))
sys.path.insert(0, ROOT)
from bench_fsd import gpu_info, timed  # noqa: E402
from cpcsv_b200 import ssim  # noqa: E402
from oracle import ssim as ssim_oracle  # noqa: E402

FMA_SEPARABLE = 5 * 11 * 2
FMA_2D = 5 * 11 * 11


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[256, 1024])
    ap.add_argument("--T", type=int, default=5)
    ap.add_argument("--side", type=int, default=64)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_ssim: needs a CUDA device")
    dev = torch.device("cuda")
    torch.backends.cudnn.benchmark = True
    res = {"gpu": gpu_info(), "T": args.T, "side": args.side, "channels": 3, "reps": args.reps,
           "fma_per_pixel_channel": {"kernel_separable": FMA_SEPARABLE, "pytorch_ssim_2d": FMA_2D},
           "hbm_peak_bytes_per_s_datasheet": 7.7e12, "sizes": {}}

    def oracle32(pair):
        return ssim_oracle.ssim(pair[0], pair[1], size_average=False)

    def kernel(pair):
        return ssim.frame_ssim(pair[0], pair[1])

    for B in args.sizes:
        g = torch.Generator(device=dev).manual_seed(B)
        stories_x = torch.rand(B, 3, args.T, args.side, args.side, device=dev, generator=g)
        stories_y = (stories_x + 0.05 * torch.randn(stories_x.shape, device=dev, generator=g)).clamp(0, 1)
        N = B * args.T
        frames = tuple(s.transpose(1, 2).reshape(N, 3, args.side, args.side) for s in (stories_x, stories_y))
        px = N * 3 * args.side * args.side
        bytes_read = 2 * px * 4 + N * 8
        ref = ssim_oracle.ssim(frames[0][:64].double(), frames[1][:64].double(), size_average=False)
        row = {"stories": B, "frames": N, "input_mb_each": px * 4 / 1e6, "bytes": bytes_read,
               "hbm_bound_us": bytes_read / 7.7e12 * 1e6}
        arms = [("kernel_frames", kernel, frames, FMA_SEPARABLE),
                ("kernel_story_view", kernel, (stories_x, stories_y), FMA_SEPARABLE),
                ("cudnn_fp32_strict", oracle32, frames, FMA_2D),
                ("cudnn_fp32_tf32", oracle32, frames, FMA_2D)]
        with torch.no_grad():
            for name, fn, pair, fma in arms:
                torch.backends.cudnn.allow_tf32 = name != "cudnn_fp32_strict"
                med, lo, hi = timed(fn, pair, args.reps)
                s = med * 1e-3
                row[name] = {"ms": med, "ms_min": lo, "ms_max": hi, "frames_per_s": N / s,
                             "bytes_per_s": bytes_read / s, "flop_per_s": 2 * fma * px / s,
                             "max_abs_d_vs_fp64_64_frames": float((fn(pair)[:64] - ref).abs().max())}
            torch.backends.cudnn.allow_tf32 = True
        row["speedup_kernel_vs_cudnn_strict"] = row["cudnn_fp32_strict"]["ms"] / row["kernel_frames"]["ms"]
        row["speedup_kernel_vs_cudnn_tf32"] = row["cudnn_fp32_tf32"]["ms"] / row["kernel_frames"]["ms"]
        res["sizes"][B] = row
        print(json.dumps({B: row}), flush=True)
        del stories_x, stories_y, frames
        torch.cuda.empty_cache()
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt)


if __name__ == "__main__":
    main()
