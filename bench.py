#!/usr/bin/env python
"""Contract benchmark: CP-CSV GAN training step (BASELINE.json metric: stories/s).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # reference algorithm on host CPU cores

A "step" is one iteration of the reference's hot loop (trainer.py:290-416) at the
cfg/final.yml batch (18 stories x 5 frames + 90 images, 64x64): no-grad generator passes,
the three discriminator updates and the generator update, including the four Adam steps.
With N > 1 every rank runs that batch on its own GPU (weak scaling, as the reference's
batch x num_gpus) and gradients are averaged with NCCL; ``value`` is the whole-job rate.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

# the step forks into many parallel stream branches; must be set before CUDA initialises
# (see cpcsv_b200/__init__.py)
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "cpcstoryvisualization-pytorch_b200")
for _p in (ROOT, PKG):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

NOMINAL_GFLOP_PER_STEP = 11874.8   # necessary algorithmic work, SURVEY.md section 8(d)
WORKLOAD = ("pororo cfg/final.yml: 18 stories x 5 frames + 90 images, 64x64; G + D_im + D_st + D_se "
            "fwd/bwd + 4 Adam steps")


def preset_dict(st_batch=18, im_batch=90):
    return dict(CUDA=True, USE_SEQ_CONSISTENCY=False, SEGMENT_LEARNING=True, CASCADE_MODEL=False,
                SEGMENT_RATIO=1.0, IMAGE_RATIO=5.0, KL=1.0, DISCRIMINATOR_LR=4e-4, GENERATOR_LR=1e-4,
                VIDEO_LEN=5, TEXT_DIM=356, LABEL_NUM=9, ST_BATCH=st_batch, IM_BATCH=im_batch,
                CONDITION_DIM=124, Z_DIM=100, DF_DIM=124, GF_DIM=256, GF_SEG_DIM=1024, name="pororo")


def apply_cfg(cfg, p):
    cfg.CUDA = p["CUDA"]; cfg.VIDEO_LEN = p["VIDEO_LEN"]; cfg.LABEL_NUM = p["LABEL_NUM"]
    cfg.USE_SEQ_CONSISTENCY = False; cfg.SEGMENT_LEARNING = True; cfg.CASCADE_MODEL = False
    cfg.SEGMENT_RATIO = p["SEGMENT_RATIO"]; cfg.IMAGE_RATIO = p["IMAGE_RATIO"]; cfg.Z_DIM = p["Z_DIM"]
    cfg.TRAIN.IM_BATCH_SIZE = p["IM_BATCH"]; cfg.TRAIN.ST_BATCH_SIZE = p["ST_BATCH"]
    cfg.TRAIN.DISCRIMINATOR_LR = p["DISCRIMINATOR_LR"]; cfg.TRAIN.GENERATOR_LR = p["GENERATOR_LR"]
    cfg.TRAIN.COEFF.KL = p["KL"]
    cfg.GAN.CONDITION_DIM = p["CONDITION_DIM"]; cfg.GAN.Z_DIM = p["Z_DIM"]; cfg.GAN.DF_DIM = p["DF_DIM"]
    cfg.GAN.GF_DIM = p["GF_DIM"]; cfg.GAN.GF_SEG_DIM = p["GF_SEG_DIM"]; cfg.TEXT.DIMENSION = p["TEXT_DIM"]


def synthetic_host_batch(p, seed, pin):
    """the two loader dicts of reference trainer.py:252-274 with synthetic contents (host memory)"""
    g = torch.Generator().manual_seed(seed)
    B, N, V, T, L = p["ST_BATCH"], p["IM_BATCH"], p["VIDEO_LEN"], p["TEXT_DIM"], p["LABEL_NUM"]
    st = {"images": torch.rand(B, 3, V, 64, 64, generator=g) * 2 - 1,
          "description": torch.randn(B, V, T, generator=g),
          "labels": (torch.rand(B, V, L, generator=g) < 0.3).float()}
    im = {"images": torch.rand(N, 3, 64, 64, generator=g) * 2 - 1,
          "description": torch.randn(N, T, generator=g),
          "content": torch.randn(N, V, T, generator=g),
          "labels": (torch.rand(N, L, generator=g) < 0.3).float(),
          "images_seg": torch.rand(N, 1, 64, 64, generator=g) * 2 - 1}
    if pin:
        st = {k: v.pin_memory() for k, v in st.items()}
        im = {k: v.pin_memory() for k, v in im.items()}
    return st, im


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        # median over the samples taken under load (upper half: idle samples sit at the floor clock)
        load = [v for v in sm if mx and v > 0.3 * mx] or sm
        med = load[len(load) // 2] if load else None
        return {"sm_mhz": med, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------- CPU baseline
def cpu_reference_rate(steps, warmup, st_batch=18, im_batch=90, threads=None, prime=True):
    """The reference algorithm (oracle port, fp32, torch CPU ops) on the host cores at the FULL cfg/final.yml
    batch (18 stories + 90 images per step: the same config as the GPU arm).  ``prime``: one step at 2 stories +
    10 images first (thread pool / oneDNN primitive creation, ~1-2 s), not timed.  Returns (stories/s,
    seconds/step, cores)."""
    from oracle import functional as Fn
    from oracle import params, synth
    threads = threads or os.cpu_count() or 1
    torch.set_num_threads(threads)
    if prime:
        q = preset_dict(2, 10)
        q["CUDA"] = False
        Fn.train_step(Fn.OracleModel(params.init_all(q, 0), q, device="cpu"), synth.make_batch(q, 1),
                      synth.NoiseFeed(synth.make_noise(q, 2)))
    p = preset_dict(st_batch, im_batch)
    p["CUDA"] = False
    model = Fn.OracleModel(params.init_all(p, 0), p, device="cpu")
    batch = synth.make_batch(p, 1)
    times = []
    for i in range(warmup + steps):
        feed = synth.NoiseFeed(synth.make_noise(p, 2 + i))
        t0 = time.perf_counter()
        Fn.train_step(model, batch, feed)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    sec = sum(times) / len(times)
    return st_batch / sec, sec, threads


def run_reference_arm(args):
    """``--impl reference``: the reference's own CPU implementation of the step (there is no compiled
    reference: the oracle port of its PyTorch code, all host threads) on THIS arm's config -- the full
    cfg/final.yml batch -- with a bounded number of steps (a CPU step takes ~10-30 s)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = max(1, min(args.steps, 2))
    warm = 1 if args.warmup > 0 else 0
    rate, sec, cores = cpu_reference_rate(steps, warm)
    sample = ("oracle port of the reference step (fp32, torch CPU ops, %d threads); cfg/final.yml model and FULL "
              "batch (18 stories + 90 images per step, same config as the GPU arm); %d warm-up + %d timed steps, "
              "%.1f s/step" % (cores, warm, steps, sec))
    line = {"impl": "reference", "metric": "train stories/s", "value": rate, "unit": "stories/s",
            "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": sec * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": {"workload": WORKLOAD, "sample": sample},
            "cpu_baseline": {"value": rate, "unit": "stories/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": rate, "unit": "stories/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def run_stock_cuda_arm(args, dev=None, p=None):
    """BASELINE.md "second bar" (not part of the driver's contract; run by hand):
    ``bench.py --impl stock-cuda``.  The same oracle port of the reference step, full cfg/final.yml
    batch, on cuda:0 through STOCK PyTorch (cuDNN / cuBLAS / ATen, eager, the reference's own
    execution model), fp32 with TF32 off and on.  Device-timed with CUDA events."""
    import torch.backends.cudnn as cudnn
    from oracle import functional as Fn
    from oracle import params, synth
    dev = dev if dev is not None else torch.device("cuda", 0)
    if p is None:
        p = preset_dict()
        p["CUDA"] = True
    out = {}
    for tf32 in (False, True):
        cudnn.allow_tf32 = tf32
        torch.backends.cuda.matmul.allow_tf32 = tf32
        cudnn.benchmark = True
        model = Fn.OracleModel(params.init_all(p, 0), p, device=dev)
        batch = synth.make_batch(p, 1, device=dev)
        noise = [synth.make_noise(p, 2 + i, device=dev) for i in range(args.warmup + args.steps)]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for i in range(args.warmup + args.steps):
            if i == args.warmup:
                torch.cuda.synchronize()
                e0.record()
            Fn.train_step(model, batch, synth.NoiseFeed(noise[i]))
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / args.steps
        out["tf32_on" if tf32 else "tf32_off"] = {"ms_per_step": ms, "stories_per_s": p["ST_BATCH"] / (ms * 1e-3)}
        del model
        torch.cuda.empty_cache()
    if getattr(args, "return_only", False):
        return out
    line = {"impl": "stock-cuda", "metric": "train stories/s", "unit": "stories/s", "n_gpus": 1,
            "steps": args.steps, "warmup": args.warmup, "value": out["tf32_off"]["stories_per_s"],
            "ms_per_step": out["tf32_off"]["ms_per_step"], "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "execution": "oracle port of the reference step, eager stock PyTorch "
                       "(cuDNN benchmark mode), no per-step host syncs"},
            "tf32_off": out["tf32_off"], "tf32_on": out["tf32_on"]}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- product arm
class StepEngine:
    """Networks, optimisers and a pinned synthetic host batch around the product's own
    ``trainer.GraphedStep`` (the public train_step API on static device buffers, replayed as one
    CUDA graph; three graphs with the NCCL exchanges between them when N > 1)."""

    def __init__(self, p, device, use_graph, grad_sync, segmented=False):
        self.segmented = segmented
        from miscc.config import cfg
        apply_cfg(cfg, p)
        import trainer
        from cpcsv_b200 import nets as knets
        self.trainer, self.knets = trainer, knets
        self.p, self.device = p, device
        torch.manual_seed(1234)             # identical initial weights on every rank (data parallel)
        self.nets = trainer.build_networks(p["VIDEO_LEN"])
        for n in self.nets.values():
            n.to(device).train()
        torch.manual_seed(1234 + int(os.environ.get("RANK", "0")))     # independent noise per rank
        # the product's optimiser: PackedAdam (Adam fused with the weight re-layout), lr in a device tensor
        self.opts = trainer.build_capturable_optimizers(self.nets, device) if use_graph else \
            trainer.build_optimizers(self.nets, fused=True)
        N, B = p["IM_BATCH"], p["ST_BATCH"]
        self.labels = (torch.ones(N, device=device), torch.zeros(N, device=device),
                       torch.ones(B, device=device), torch.zeros(B, device=device))
        st, im = synthetic_host_batch(p, 7, pin=True)
        self.host_st, self.host_im = st, im
        self.dev_st = {k: v.to(device) for k, v in st.items()}
        self.dev_im = {k: v.to(device) for k, v in im.items()}
        self.h2d_bytes = sum(v.numel() * v.element_size() for d in (st, im) for v in d.values())
        self.grad_sync = grad_sync
        self.use_graph = use_graph
        self.gs = trainer.GraphedStep(self.nets, self.opts, self.labels, self.dev_st, self.dev_im,
                                      grad_sync=grad_sync, ratio=1.0, use_graph=use_graph, segmented=segmented)
        self.loss_keys, self.loss_dev, self.loss_host = self.gs.loss_keys, self.gs.loss_dev, self.gs.loss_host

    def _step_body(self):
        self.gs._step_body()

    def capture(self):
        self.gs.capture()

    def step(self):
        self.gs.step()

    overlap_io = False      # --overlap-io: stage the next batch on a copy stream (GraphedStep.load_async)

    def upload(self):
        if self.overlap_io:
            self.gs.load_async(self.host_st, self.host_im)
        else:
            self.gs.load(self.host_st, self.host_im)

    def download(self):
        self.gs.download()


def job_flops(job):
    """executed tensor-core FLOPs of one conv_gemm launch (padded channels and split planes counted)"""
    n, h, w = job.grid
    pix = n * h * w
    if job.mode == 0:
        mmas = 3 if job.planes == 2 else 1
        return 2.0 * pix * job.groups * job.taps_per_group * job.k_blocks * 64 * job.n_valid * mmas
    return 2.0 * pix * job.groups * job.m_valid * job.n_valid


def job_bytes(job):
    """algorithmic HBM bytes of one conv_gemm launch: every operand plane read once (whatever the number of
    filter taps that re-read it through L2 / shared memory), the fp32 output written once"""
    def numel(view):
        n = 1
        for d in view.dims:
            n *= d
        return n
    n, h, w = job.grid
    pix = n * h * w
    a = sum(numel(v) for v in job.a[:job.planes]) * 2
    b = sum(numel(v) for v in job.b[:job.planes]) * 2
    if job.mode == 0:
        out = pix * job.groups * job.n_valid * 4
    else:
        out = job.groups * job.m_valid * job.n_valid * 4
    return a + b + out


def profile_gemm_launches(engine, steps):
    """Average launch duration of the dominant kernel, measured live with CUDA events: the step is
    run eagerly on ONE stream behind a long device-side sleep (so the host stays ahead and each
    event pair brackets its kernel alone; with the step's concurrent branches the second event
    would also wait for kernels of other streams).  The zero fill of split-K outputs is kept
    outside the brackets."""
    from cpcsv_b200 import engine as keng
    from cpcsv_b200 import ops
    orig = ops.conv_gemm
    recs = []

    def timed(job):
        restore = False
        if job.splits > 1 and not job.accumulate:
            job.out.zero_()
            job.accumulate, restore = True, True
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        orig(job)
        e1.record()
        if restore:
            job.accumulate = False
        recs.append((e0, e1, job_flops(job), job_bytes(job)))

    tr = engine.trainer
    flags = (tr.CONCURRENT_D, tr.CONCURRENT_G, tr.EARLY_G, tr.streams.ENABLED, keng.WGRAD_ON_AUX_STREAM)
    tr.CONCURRENT_D = tr.CONCURRENT_G = tr.EARLY_G = tr.streams.ENABLED = keng.WGRAD_ON_AUX_STREAM = False
    try:
        engine._step_body()              # serial warm-up: re-packs weights on this stream
        torch.cuda.synchronize()
        ops.conv_gemm = timed
        for _ in range(steps):
            torch.cuda._sleep(int(0.4 * 1.9e9))
            engine._step_body()
            torch.cuda.synchronize()
    finally:
        ops.conv_gemm = orig
        tr.CONCURRENT_D, tr.CONCURRENT_G, tr.EARLY_G, tr.streams.ENABLED, keng.WGRAD_ON_AUX_STREAM = flags
    ms = sum(r[0].elapsed_time(r[1]) for r in recs)
    fl = sum(r[2] for r in recs)
    return {"launches_per_step": len(recs) / steps, "gemm_ms_per_step": ms / steps,
            "executed_gflop_per_step": fl / steps / 1e9, "achieved_tflops": fl / (ms * 1e-3) / 1e12,
            "avg_launch_us": 1e3 * ms / len(recs), "algorithmic_bytes_per_launch": sum(r[3] for r in recs) / len(recs)}


def run_large_config(args):
    """BASELINE.json configs[3] / configs[4] with the contract's line format (one JSON line per measurement)."""
    torch.cuda.set_device(0)
    device = torch.device("cuda", 0)
    from cpcsv_b200 import _lib
    _lib.load()
    peaks = _recorded("../MEASURED_PEAKS.json") or {}
    peak = peaks.get("bf16_tflops_sustained", 1400.0)
    sampler = ClockSampler(0)
    sampler.start()

    def timed(fn, warm, iters):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0 = _lib.launch_count()
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters, (_lib.launch_count() - c0) / iters

    lines = []
    if args.config == "inference":
        from miscc.config import cfg
        p = preset_dict()
        apply_cfg(cfg, p)
        import trainer
        G = trainer.build_networks(5)["G"].to(device).train()      # inference.py never calls .eval() (SURVEY 3.3)
        for B in (16, 64, 256, 1024):
            motion = torch.randn(B, 5, 365).pin_memory()
            content = torch.randn(B, 5, 356).pin_memory()
            dm, dc = motion.to(device), content.to(device)
            out_host = torch.empty(B, 3, 5, 64, 64).pin_memory()

            def run():
                with torch.no_grad():
                    return G.sample_videos(dm, dc, seg=True)
            run(); run()
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                outs = run()
            ms, launches = timed(g.replay, max(args.warmup, 3), max(3, min(args.steps, 10)))

            def e2e():
                dm.copy_(motion, non_blocking=True)
                dc.copy_(content, non_blocking=True)
                g.replay()
                out_host.copy_(outs[1], non_blocking=True)
            ms_e2e, _ = timed(e2e, 2, max(3, min(args.steps, 10)))
            gf = 66.9 * B          # GFLOP per 5-frame story, SURVEY.md section 8(d)
            lines.append({"metric": "inference stories/s", "value": B / ms * 1e3, "unit": "stories/s", "n_gpus": 1,
                          "steps": max(3, min(args.steps, 10)), "warmup": max(args.warmup, 3), "ms_per_step": ms,
                          "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16",
                          "data": "synthetic",
                          "config": {"workload": "BASELINE configs[3]: sample_videos (generator + segmentation "
                                                 "branch) under no_grad, train-mode BN, %d stories x 5 frames" % B,
                                     "stories": B, "nominal_tflops": gf / ms, "nominal_frac_of_peak": gf / ms / peak,
                                     "precision": "single-pass fp16 forward GEMMs (no-grad path)"},
                          "e2e": {"value": B / ms_e2e * 1e3, "unit": "stories/s",
                                  "h2d_bytes_per_step": (motion.numel() + content.numel()) * 4,
                                  "d2h_bytes_per_step": out_host.numel() * 4, "ms_per_step": ms_e2e},
                          "gpu_launches_per_step": launches})
            del g, outs
    else:
        st_b, im_b = 512, 2560
        eng = StepEngine(preset_dict(st_b, im_b), device, use_graph=False, grad_sync=None)
        if args.job_log:
            # one line per conv_gemm launch, in launch order: joins an ncu launch list (tools/stress_table.py)
            from cpcsv_b200 import ops
            orig, log = ops.conv_gemm, open(args.job_log, "w")

            def logged(job):
                n, h, w = job.grid
                log.write("%s pl=%d grid=%dx%dx%d groups=%d taps=%d kb=%d nv=%d bn=%d mv=%d splits=%d pair=%d\t%.6e\n" % (
                    "fprop/dgrad" if job.mode == 0 else "wgrad", job.planes, n, h, w, job.groups, job.taps_per_group,
                    job.k_blocks, job.n_valid, job.block_n, job.m_valid, job.splits, int(job.pair), job_flops(job)))
                orig(job)
            ops.conv_gemm = logged
        ms, launches = timed(eng.step, max(2, min(args.warmup, 3)), max(2, min(args.steps, 3)))
        if args.job_log:
            ops.conv_gemm = orig
            log.close()
        gf = 659.7 * st_b
        lines.append({"metric": "train stories/s", "value": st_b / ms * 1e3, "unit": "stories/s", "n_gpus": 1,
                      "steps": max(2, min(args.steps, 3)), "warmup": max(2, min(args.warmup, 3)), "ms_per_step": ms,
                      "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
                      "data": "synthetic",
                      "config": {"workload": "BASELINE configs[4]: 512 stories x 5 frames + 2560 images per step, "
                                             "full G + 3 D train step (eager, no CUDA graph)",
                                 "nominal_tflops": gf / ms, "nominal_frac_of_peak": gf / ms / peak,
                                 "max_mem_gb": torch.cuda.max_memory_allocated() / 2 ** 30},
                      "gpu_launches_per_step": launches})
    clocks = sampler.stop()
    for ln in lines:
        ln["clocks"] = clocks
        print(json.dumps(ln), flush=True)


DUMP_SAMPLE = 16384                 # values kept of every larger parameter tensor
DUMP_LIMIT_BYTES = 64 * 2 ** 20


def _state_tensors(nets):
    return [t for n in nets.values() for t in list(n.parameters()) + list(n.buffers())]


def restore_initial_state(eng, initial):
    """Put the training state back where the seeded construction left it: weights and buffers from ``initial``,
    Adam moments and step counters at zero, the optimiser-maintained 16-bit operand planes re-packed from the
    restored weights.  The kernels accumulate with atomics, so two runs of the same build drift apart step by
    step; a step taken from this state sees the same inputs in every run."""
    torch.cuda.synchronize()
    with torch.no_grad():
        for t, s in zip(_state_tensors(eng.nets), initial):
            t.copy_(s)
        for opt in eng.opts.values():
            for st in opt.state.values():
                st["exp_avg"].zero_()
                st["exp_avg_sq"].zero_()
            for st in opt._dev.values():
                st["step"].zero_()
        cache = eng.knets.weight_cache()
        for ent in list(cache.d.values()):
            if ent.spec is not None:
                ent.fill(ent.val)
                cache.refreshed(ent, ent.ref())
    torch.cuda.synchronize()


def dump_outputs(out_dir, nets, losses):
    """What one step of the timed path hands its caller, as .npy files, so that two builds can be compared output
    for output: ``losses.npy`` (float32: the loss vector ``GraphedStep.download`` delivers, in ``trainer.LOSS_KEYS``
    order), ``<net>.params.npy`` (float32: the network's parameters after the step's Adam update, in
    ``named_parameters`` order, of a tensor with more than DUMP_SAMPLE values a fixed seeded sample of DUMP_SAMPLE)
    and ``<net>.buffers.npy`` (float64: every buffer in full -- BatchNorm running statistics and counters,
    spectral-norm vectors)."""
    import numpy as np
    arrays = {"losses": losses.detach().float().cpu().numpy()}
    g = torch.Generator().manual_seed(0)
    for name, net in nets.items():
        parts = []
        for p in net.parameters():
            flat = p.detach().reshape(-1)
            if flat.numel() > DUMP_SAMPLE:
                flat = flat[torch.randint(flat.numel(), (DUMP_SAMPLE,), generator=g).to(flat.device)]
            parts.append(flat.float().cpu())
        arrays[name + ".params"] = torch.cat(parts).numpy()
        arrays[name + ".buffers"] = torch.cat([b.detach().reshape(-1).double().cpu() for b in net.buffers()]).numpy()
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError("--dump-outputs: %d bytes exceed the %d byte limit" % (total, DUMP_LIMIT_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def _recorded(name):
    """a measurement recorded under profiles/ (with its provenance) that the bench line quotes"""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", name)))
    except Exception:
        return None


def _trace(msg):
    if os.environ.get("CPCSV_BENCH_TRACE"):
        print("[bench %.1fs] %s" % (time.perf_counter(), msg), file=sys.stderr, flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="cpcsv_b200")
    ap.add_argument("--no-graph", action="store_true", help="run the step eagerly instead of as one CUDA graph")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--with-stock-cuda", action="store_true",
                    help="also time the oracle step through stock PyTorch / cuDNN on this GPU (TF32 off and on) "
                         "instead of quoting profiles/r02_stock_cuda.json")
    ap.add_argument("--config", default="train", choices=["train", "inference", "stress"],
                    help="train = BASELINE configs[1] (the contract line); inference = configs[3] (no-grad generator "
                         "+ segmentation branch, batch sweep); stress = configs[4] (512 stories + 2560 images / step)")
    ap.add_argument("--job-log", default=None, help="--config stress: write one line per conv_gemm launch (signature, "
                                                    "executed FLOPs) to this file")
    ap.add_argument("--serial-io", action="store_true",
                    help="e2e loop: copy every batch on the step's own stream before the replay (the round-1 path).  "
                         "Default: GraphedStep.load_async, the path GANTrainer.train uses -- the real images of batch "
                         "i+1 are copied straight into the static buffers on a copy stream once step i's graph has "
                         "passed its discriminator stage (measured on one box: 20.41 / 20.68 vs 20.80 / 20.71 ms)")
    ap.add_argument("--overlap-io", action="store_true", help="(default since round 2)")
    ap.add_argument("--whole-graph", action="store_true",
                    help="(default since round 2) N > 1: the NCCL all-reduces are captured inside the ONE step graph")
    ap.add_argument("--segmented", action="store_true",
                    help="three CUDA graphs with the gradient all-reduces issued eagerly between them "
                         "instead of one graph that contains them")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="train config: after the timed loops take one more step of the timed path, untimed, from the "
                         "seeded initial state, and write what it returned (losses, updated parameters -- a seeded "
                         "sample of the large tensors -- and buffers) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl in ("reference", "stock-cuda") or args.config != "train"):
        ap.error("--dump-outputs applies to the train config of this repo's CUDA path")
    if args.impl == "reference":
        run_reference_arm(args)
        return
    if args.impl == "stock-cuda":
        run_stock_cuda_arm(args)
        return
    if args.config != "train":
        run_large_config(args)
        return
    args.warmup = max(args.warmup, 3)
    # N > 1: ONE graph per step with the NCCL all-reduces captured inside (each discriminator's exchange runs
    # under the other discriminators' compute).  Round 1's "hang" of this variant was the process group
    # tear-down at exit, not the replays (see the end of main); --segmented keeps the three-graph variant.

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    from cpcsv_b200 import _lib
    _lib.load()

    p = preset_dict()
    import trainer
    grad_sync = trainer.GradSync() if world > 1 else None
    if args.segmented and world == 1:
        grad_sync = trainer.GradSync(enabled=False)
    eng = StepEngine(p, device, use_graph=not args.no_graph, grad_sync=grad_sync, segmented=args.segmented)
    eng.overlap_io = not args.serial_io and not args.no_graph and not args.segmented
    initial = [t.detach().clone() for t in _state_tensors(eng.nets)] if args.dump_outputs else None

    # warm-up (eager: builds caches, sets kernel attributes), then capture
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(args.warmup):
            eng.step()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    _trace("warm-up done")
    launches0 = _lib.launch_count()
    if not args.no_graph:
        eng.capture()
        torch.cuda.synchronize()
    launches_per_step = _lib.launch_count() - launches0 if not args.no_graph else None
    # Untimed replays until the clocks have settled under the power cap: measured on B200, the first ~20 replays of a
    # fresh process run 0.6 ms / step faster than every later one (sw_power_cap; device-timed loop repeated after the
    # e2e loop: 20.75 vs 20.08 ms first, 20.80 e2e in between).  Both timed loops below see the sustained state.
    settle = int(os.environ.get("CPCSV_BENCH_SETTLE", "40")) if not args.no_graph else 2
    for _ in range(max(2, settle)):
        eng.step()
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_loop(with_io):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        if with_io and eng.overlap_io:
            # the product's pipelined input path (GraphedStep.load_async, as GANTrainer.train uses it): the pinned
            # real images of step i+1 are copied on a copy stream straight into the static buffers once step i's
            # graph has passed its discriminator stage, the small tensors right before replay i+1; all K
            # host-to-device copies and K loss read-backs are inside the timed region
            eng.upload()
            for i in range(args.steps):
                eng.step()
                if i + 1 < args.steps:
                    eng.upload()
                eng.download()
        else:
            for _ in range(args.steps):
                if with_io:
                    eng.upload()
                eng.step()
                if with_io:
                    eng.download()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t)
        return ms

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    _trace("captured, 2 replays done")
    c0 = _lib.launch_count()
    ms_dev = timed_loop(False)
    _trace("device-timed loop done: %.2f ms/step" % (ms_dev / args.steps))
    c1 = _lib.launch_count()
    ms_e2e = timed_loop(True)
    _trace("e2e loop done")
    if os.environ.get("CPCSV_BENCH_REPEAT_DEV"):
        # diagnostic: is the e2e loop slower because of its copies, or because it runs second (power cap)?
        print("[bench] device-timed again after the e2e loop: %.3f ms/step (first %.3f, e2e %.3f)" % (
            timed_loop(False) / args.steps, ms_dev / args.steps, ms_e2e / args.steps), file=sys.stderr, flush=True)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        # one more step through the timed path (same graph, same input upload and loss read-back), untimed, from
        # the seeded initial state; every rank takes it (the graph holds the gradient exchange)
        restore_initial_state(eng, initial)
        eng.upload()
        eng.step()
        eng.download()
        torch.cuda.synchronize()
        if rank == 0:
            dump_outputs(args.dump_outputs, eng.nets, eng.loss_dev)
    if launches_per_step is None:
        launches_per_step = (c1 - c0) / args.steps

    # entries packed while capturing belong to the graph; drop them before running eagerly again
    eng.knets.invalidate_weight_cache()
    prof = profile_gemm_launches(eng, 2)
    _trace("gemm profile done")
    stories = p["ST_BATCH"] * world
    ms_step = ms_dev / args.steps
    ms_step_e2e = ms_e2e / args.steps
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = peaks.get("bf16_tflops_sustained", 1400.0)
    peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained" if peaks else "fallback 1.4 PF sustained (B200_PROFILING.md)"

    traffic = _recorded("r02_gemm_traffic.json") or {}
    line = {
        "metric": "train stories/s", "value": stories / (ms_step * 1e-3), "unit": "stories/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic",
        "config": {"workload": WORKLOAD, "cuda_graph": not args.no_graph,
                   "precision": "fwd convs: bf16 hi/lo split operands (3 MMAs), fp32 accumulate; bwd GEMMs "
                                "single-pass bf16; BN/conditioning/grads fp32",
                   "l2": "per-step working set (activations + 158 M params + Adam state) is ~4 GB >> 126 MB L2; "
                         "no explicit flush",
                   "settle": "%d untimed graph replays after the W warm-up steps, before the timed loops (clocks under "
                             "the power cap)" % max(2, settle),
                   "nominal_gflop_per_step": NOMINAL_GFLOP_PER_STEP,
                   "nominal_tflops": NOMINAL_GFLOP_PER_STEP / ms_step,
                   "nominal_frac_of_peak": NOMINAL_GFLOP_PER_STEP / ms_step / peak},
        "e2e": {"value": stories / (ms_step_e2e * 1e-3), "unit": "stories/s",
                "h2d_bytes_per_step": eng.h2d_bytes, "d2h_bytes_per_step": eng.loss_host.numel() * 4,
                "ms_per_step": ms_step_e2e,
                "io": "GraphedStep.load_async: next batch copied under the running step" if eng.overlap_io
                      else "serial: copy, step, read-back on one stream"},
        "gpu_launches": int(launches_per_step * args.steps),
        "gpu_launches_per_step": launches_per_step,
        "roofline": {"bound": "tensor", "achieved": prof["achieved_tflops"], "peak": peak, "unit": "TFLOP/s",
                     "frac": prof["achieved_tflops"] / peak, "traffic": traffic.get("avg_bytes_per_launch"),
                     "traffic_note": traffic.get("note", "no ncu capture recorded under profiles/"),
                     "algorithmic_bytes_per_launch": prof["algorithmic_bytes_per_launch"],
                     "kernel": "conv_gemm_kernel (tcgen05 implicit GEMM)", "peak_source": peak_src,
                     "executed_gflop_per_step": prof["executed_gflop_per_step"],
                     "gemm_launches_per_step": prof["launches_per_step"],
                     "avg_launch_us": prof["avg_launch_us"],
                     "method": "CUDA events around every conv_gemm launch of 2 eager single-stream steps "
                               "queued behind a device-side sleep; achieved = executed tensor-core FLOPs / "
                               "summed launch durations",
                     "gemm_ms_per_step_serial_events": prof["gemm_ms_per_step"]},
        "clocks": clocks,
    }
    # the "second bar" of BASELINE.md section 4.4: the same step through stock PyTorch / cuDNN on this GPU
    stock = _recorded("r02_stock_cuda.json")
    if rank == 0 and world == 1 and args.with_stock_cuda:
        del eng
        torch.cuda.empty_cache()
        ns = argparse.Namespace(steps=3, warmup=2, return_only=True)
        live = run_stock_cuda_arm(ns, device, dict(preset_dict(), CUDA=True))
        stock = {"tf32_off_ms_per_step": live["tf32_off"]["ms_per_step"], "tf32_on_ms_per_step": live["tf32_on"]["ms_per_step"],
                 "source": "measured in this run (bench.py --with-stock-cuda)"}
    if stock:
        stock = dict(stock)
        stock["speedup_vs_tf32_off"] = stock["tf32_off_ms_per_step"] / ms_step
        stock["speedup_vs_tf32_on"] = stock["tf32_on_ms_per_step"] / ms_step
        line["stock_cuda"] = stock
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        rate, sec, cores = cpu_reference_rate(1, 0)
        line["cpu_baseline"] = {
            "value": rate, "unit": "stories/s", "cores": cores, "kind": "port",
            "sample": "oracle port of the reference step (fp32 torch CPU ops, %d threads) on the cfg/final.yml "
                      "model at the FULL batch (18 stories + 90 images): 1 timed step (%.1f s) after a "
                      "2-story priming step" % (cores, sec)}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        # Leave without tearing the communicator down: destroying a process group whose collectives were
        # captured into CUDA graphs that are still alive blocked at exit on the 2-GPU box
        # (gpurun_out r02_multi2_whole.log).  Every rank is done (barrier), the line is out.
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
