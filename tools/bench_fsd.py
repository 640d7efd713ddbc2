"""Stories / s of R(2+1)D-18 story-feature extraction (the FSD features, cpcsv_b200.fsd) on the B200:
StoryFeatureNet on the project's kernels against torchvision ``r2plus1d_18`` on cuDNN in fp32 (TF32 allowed, the
PyTorch default for convolutions, and TF32 off) and in bf16 autocast, all with the same random weights and the
same preprocessing, at T frames of side x side pixels.

Timing: CUDA events around whole calls (preprocessing included) after two warm-up calls, median of ``--reps``;
the inputs of the timed calls are larger than the 126 MB L2 at the default sizes.  ``cudnn.benchmark`` is on for
the cuDNN arms.  A second, profiled call of the kernel path (torch.profiler, after the timed runs) gives the
time of every tcgen05 GEMM job; with the job's executed MMA work (3 MMAs per product with hi/lo split operands,
padded channels included) that is its tensor-core rate and its share of the 2,250 TFLOP/s dense BF16 data-sheet
rate -- an estimate of tensor-pipe activity from work over time, not a hardware counter.

Prints one JSON document (and writes it to ``--out`` when given); the GPU name and power limit are part of it.
Development tool, not the contract benchmark (bench.py)."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "cpcstoryvisualization-pytorch_b200"))
from cpcsv_b200 import fsd, ops  # noqa: E402

PEAK_BF16_TFLOPS = 2250.0


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        info["power_limit, max_sm_clock"] = out[0] if out else None
    except (OSError, subprocess.SubprocessError):
        info["power_limit, max_sm_clock"] = None
    return info


def conv_flops_per_story(T, side):
    """2 * MACs of every Conv3d of r2plus1d_18 (real channels) for one story, from the output shapes"""
    import torchvision
    tv = torchvision.models.video.r2plus1d_18(weights=None).eval()
    total = [0]

    def hook(mod, inp, out):
        k = mod.kernel_size[0] * mod.kernel_size[1] * mod.kernel_size[2]
        total[0] += 2 * out.numel() * mod.in_channels * k

    for m in tv.modules():
        if isinstance(m, torch.nn.Conv3d):
            m.register_forward_hook(hook)
    with torch.no_grad():
        tv(torch.zeros(1, 3, T, side, side))
    return total[0]


def timed(fn, x, reps):
    for _ in range(2):
        fn(x)
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
        e0.record()
        fn(x)
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ts.sort()
    return ts[len(ts) // 2], ts[0], ts[-1]


def job_table(net, x):
    """per tcgen05 GEMM job of one StoryFeatureNet call: shape, executed MMA FLOPs, kernel time"""
    jobs = []
    orig = ops.conv_gemm

    def spy(job):
        rows = job.grid[0] * job.grid[1] * job.grid[2] * job.groups
        K = job.taps_per_group * job.k_blocks * 64
        mmas = 3 if job.planes == 2 else 1
        jobs.append({"rows": rows, "n": job.n_valid, "k": K, "taps": job.taps_per_group, "pair": job.pair,
                     "splits": job.splits, "block_n": job.block_n,
                     "exec_flop": 2.0 * rows * job.n_valid * K * mmas})
        orig(job)

    ops.conv_gemm = spy
    try:
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            net(x)
            torch.cuda.synchronize()
    finally:
        ops.conv_gemm = orig
    kern = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    gemm = [e for e in kern if "conv_gemm_kernel" in e.name]
    assert len(gemm) == len(jobs), (len(gemm), len(jobs))
    for j, e in zip(jobs, gemm):
        us = e.device_time if hasattr(e, "device_time") else e.cuda_time
        j["us"] = us
        j["tflops"] = j["exec_flop"] / (us * 1e-6) / 1e12
        j["share_of_bf16_peak"] = j["tflops"] / PEAK_BF16_TFLOPS
    total_us = sum((e.device_time if hasattr(e, "device_time") else e.cuda_time) for e in kern)
    gemm_us = sum(j["us"] for j in jobs)
    return jobs, {"kernel_us_total": total_us, "gemm_us": gemm_us,
                  "gemm_exec_tflops": sum(j["exec_flop"] for j in jobs) / (gemm_us * 1e-6) / 1e12}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[256, 1024])
    ap.add_argument("--frames", type=int, default=5)
    ap.add_argument("--side", type=int, default=64)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torchvision
    if not torch.cuda.is_available():
        raise SystemExit("bench_fsd: needs a CUDA device")
    dev = torch.device("cuda")
    torch.manual_seed(0)
    tv = torchvision.models.video.r2plus1d_18(weights=None)
    tv.fc = torch.nn.Identity()
    tv = tv.eval().to(dev)
    net = fsd.StoryFeatureNet().to(dev)
    net.load_state_dict(tv.state_dict())
    mean = torch.tensor(fsd.KINETICS_MEAN, device=dev).view(1, 3, 1, 1, 1)
    std = torch.tensor(fsd.KINETICS_STD, device=dev).view(1, 3, 1, 1, 1)

    def tv_fp32(x):
        return tv(((x + 1) * 0.5 - mean) / std)

    def tv_bf16(x):
        with torch.autocast("cuda", dtype=torch.bfloat16):
            return tv(((x + 1) * 0.5 - mean) / std).float()

    torch.backends.cudnn.benchmark = True
    flop = conv_flops_per_story(args.frames, args.side)
    res = {"gpu": gpu_info(), "frames": args.frames, "side": args.side, "reps": args.reps,
           "conv_gflop_per_story": flop / 1e9, "sizes": {}}
    for B in args.sizes:
        g = torch.Generator(device=dev).manual_seed(B)
        x = torch.rand(B, 3, args.frames, args.side, args.side, device=dev, generator=g) * 2 - 1
        row = {}
        with torch.no_grad():
            arms = [("kernels", net), ("cudnn_fp32_tf32", tv_fp32), ("cudnn_fp32_strict", tv_fp32),
                    ("cudnn_bf16_autocast", tv_bf16)]
            feats = {}
            for name, fn in arms:
                torch.backends.cudnn.allow_tf32 = name != "cudnn_fp32_strict"
                med, lo, hi = timed(fn, x, args.reps)
                row[name] = {"ms": med, "ms_min": lo, "ms_max": hi, "stories_per_s": B / (med * 1e-3),
                             "conv_tflops": flop * B / (med * 1e-3) / 1e12}
                feats[name] = fn(x[:64]).double()
            torch.backends.cudnn.allow_tf32 = True
            ref = feats["cudnn_fp32_strict"]
            for name in feats:
                row[name]["relL2_vs_fp32_strict_64_stories"] = float((feats[name] - ref).norm() / ref.norm())
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
