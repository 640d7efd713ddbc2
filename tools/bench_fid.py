"""Frames / s of InceptionV3 pool3 feature extraction (the frame-FID features, cpcsv_b200.frame_fid) on the B200:
FrameFeatureNet on the project's kernels against the FID InceptionV3 oracle (oracle/fid_inception.py, torchvision
blocks) on cuDNN in fp32 (TF32 allowed, the PyTorch default for convolutions, and TF32 off) and in bf16 autocast,
all with the same weights (BatchNorm statistics calibrated on smooth synthetic frames) and the same
preprocessing (resize to 299 x 299 included), on side x side input frames.

Timing, the per-job GEMM table and the GPU record as tools/bench_fsd.py (whose helpers this uses): CUDA events
around whole calls after two warm-up calls, median of ``--reps``; one profiled call of the kernel path gives every
tcgen05 job's time and its work-over-time rate.  Convolution FLOPs come from shapes: 2 * MACs of the 94 convolutions
at 299 x 299 (11.42 GFLOP per frame).

Prints one JSON document (and writes it to ``--out`` when given).  Development tool, not the contract benchmark."""
import argparse
import json
import os
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "cpcstoryvisualization-pytorch_b200"))
sys.path.insert(0, ROOT)
from bench_fsd import gpu_info, job_table, timed  # noqa: E402
from cpcsv_b200 import frame_fid  # noqa: E402
from oracle.fid_inception import FIDInception  # noqa: E402


def conv_flops_per_frame(ref):
    """2 * MACs of every Conv2d of the network (real channels) for one frame, from the output shapes"""
    total, count = [0], [0]

    def hook(mod, inp, out):
        total[0] += 2 * out.numel() * mod.in_channels * mod.kernel_size[0] * mod.kernel_size[1]
        count[0] += 1

    hs = [m.register_forward_hook(hook) for m in ref.modules() if isinstance(m, torch.nn.Conv2d)]
    with torch.no_grad():
        ref.features(torch.zeros(1, 3, 64, 64, device=next(ref.parameters()).device))
    for h in hs:
        h.remove()
    return total[0], count[0]


def smooth_frames(n, side, dev, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    x = torch.rand(n, 3, side // 8, side // 8, device=dev, generator=g) * 2 - 1
    x = F.interpolate(x, size=(side, side), mode="bilinear", align_corners=False)
    return (0.8 * x + 0.2 * (torch.rand(n, 3, side, side, device=dev, generator=g) * 2 - 1)).clamp(-1, 1)


def calibrated_oracle(dev, side):
    """random weights; BatchNorm running statistics from train-mode passes over synthetic frames (cumulative
    averages), so 94 layers of activations stay O(1)"""
    torch.manual_seed(0)
    ref = FIDInception().to(dev)
    bns = [m for m in ref.modules() if isinstance(m, torch.nn.BatchNorm2d)]
    for bn in bns:
        bn.momentum = None
        bn.reset_running_stats()
    ref.train()
    with torch.no_grad():
        for i in range(4):
            ref.features(smooth_frames(32, side, dev, 100 + i))
    for bn in bns:
        bn.momentum = 0.1
    return ref.eval()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[256, 1024])
    ap.add_argument("--side", type=int, default=64)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_fid: needs a CUDA device")
    dev = torch.device("cuda")
    ref = calibrated_oracle(dev, args.side)
    net = frame_fid.FrameFeatureNet().to(dev)
    net.load_state_dict(ref.state_dict())

    def ref_fp32(x):
        return ref.features(x)

    def ref_bf16(x):
        with torch.autocast("cuda", dtype=torch.bfloat16):
            return ref.features(x).float()

    torch.backends.cudnn.benchmark = True
    flop, nconv = conv_flops_per_frame(ref)
    res = {"gpu": gpu_info(), "side": args.side, "reps": args.reps, "convolutions": nconv,
           "conv_gflop_per_frame": flop / 1e9, "chunk": net.chunk, "sizes": {}}
    for B in args.sizes:
        x = smooth_frames(B, args.side, dev, B)
        row = {}
        with torch.no_grad():
            arms = [("kernels", net), ("cudnn_fp32_tf32", ref_fp32), ("cudnn_fp32_strict", ref_fp32),
                    ("cudnn_bf16_autocast", ref_bf16)]
            feats = {}
            for name, fn in arms:
                torch.backends.cudnn.allow_tf32 = name != "cudnn_fp32_strict"
                med, lo, hi = timed(fn, x, args.reps)
                row[name] = {"ms": med, "ms_min": lo, "ms_max": hi, "frames_per_s": B / (med * 1e-3),
                             "conv_tflops": flop * B / (med * 1e-3) / 1e12}
                feats[name] = fn(x[:64]).double()
            torch.backends.cudnn.allow_tf32 = True
            base = feats["cudnn_fp32_strict"]
            for name in feats:
                row[name]["relL2_vs_fp32_strict_64_frames"] = float((feats[name] - base).norm() / base.norm())
            if B == max(args.sizes):
                try:
                    jobs, summ = job_table(net, x)
                    res["kernel_jobs_at_%d" % B] = jobs
                    res["kernel_summary_at_%d" % B] = summ
                except Exception as e:      # the timings above stand without the per-job table
                    res["kernel_jobs_error"] = repr(e)
        res["sizes"][B] = row
        print(json.dumps({B: row}), flush=True)
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt)


if __name__ == "__main__":
    main()
