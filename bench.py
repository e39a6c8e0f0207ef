#!/usr/bin/env python
"""bench.py -- enhanced audio-seconds per second of the N-step bridge sampler hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

One "step" = one pass of the whole hot path (fused STFT+compress+pad -> 5-step SB/ode_ei sampler on
the NCSN++ backbone -> fused decompress+iSTFT) over the batch of 256 synthetic 4 s / 16 kHz utterances
of BASELINE.json configs[1] (`infer_folder`: "a batch of 256 ... utterance-sharded over 1/2/4/8").
Utterances are independent units.  With N GPUs the 256 utterances are split into N contiguous shards
(`split_list`, infer_folder.py:149-152), every rank enhances its shard with no data-path collective,
and the enhanced waveforms are gathered onto every rank with ONE NCCL all_gather INSIDE the timed
region (north_star (d)) -- "scaling": "strong".  `--scaling weak` keeps 256 utterances PER GPU instead.

Prints ONE JSON line (see the task contract): value (device-resident inputs), e2e (host buffers,
H2D/D2H inside the timed region), roofline of the dominant kernel (tcgen05 implicit-GEMM convolution,
timed launch by launch with CUDA events through fdbm_plan_profile_forward), cpu_baseline (the CPU
oracle = port of the reference path, on this box's host cores), clocks, gpu_launches.

`--impl reference` times the reference's own CPU path (the oracle port -- the Python reference cannot
travel to the GPU box) with all host threads on a bounded sample of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "rethinking-flow-and-diffusion-bridge-models-for-speech-enhancement_b200")
sys.path.insert(0, PKG)

SR = 16000
UTT_SECONDS = 4.0
N_SAMPLES = int(SR * UTT_SECONDS)
UTTS_PER_GPU = 256
BRIDGE_STEPS = 5
GFLOP_PER_FORWARD = 532.1          # SURVEY.md section 8(d): one ncsnpp_v2 forward on a 4 s utterance (2*MAC)
METRIC = "enhanced audio-sec/sec (5-step SB bridge, ncsnpp_v2)"
UNIT = "audio-s/s"
DUMP_BYTES = 60 * 2 ** 20          # --dump-outputs: stays under 64 MB with room for the .npy headers and row lists


def dump_output(out_dir, name, t, utt_ids=None):
    """--dump-outputs: tensor `t` as out_dir/<name>.npy in float32, so that the outputs of two builds can be compared one for one.
    For per-utterance rows, `utt_ids` names the utterance of each row and goes to out_dir/<name>_rows.npy; more rows than
    DUMP_BYTES holds are cut to a fixed, seeded sample (the same rows for the same ids, whatever the build)."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    a = t.detach().to("cpu", torch.float32).numpy()
    if utt_ids is not None:
        ids = np.asarray(utt_ids, dtype=np.float64)
        if a.nbytes > DUMP_BYTES:                    # one row fits: main() refuses longer utterances
            rows = np.sort(np.random.default_rng(0).choice(a.shape[0], DUMP_BYTES // (a.nbytes // a.shape[0]), replace=False))
            a, ids = a[rows], ids[rows]
        np.save(os.path.join(out_dir, f"{name}_rows.npy"), ids)
    np.save(os.path.join(out_dir, f"{name}.npy"), a)


def set_workload(seconds, steps, predictive):
    """BASELINE.json configs[2] (predictive) and configs[4] (step sweep, 30 s utterances) reuse this script."""
    global UTT_SECONDS, N_SAMPLES, BRIDGE_STEPS, METRIC, GFLOP_PER_FORWARD
    UTT_SECONDS, N_SAMPLES, BRIDGE_STEPS = float(seconds), int(SR * seconds), (1 if predictive else int(steps))
    frames = -(-(1 + N_SAMPLES // 256) // 64) * 64
    GFLOP_PER_FORWARD = (533.0 if predictive else 532.1) * frames / 256.0
    METRIC = ("enhanced audio-sec/sec (predictive ncsnpp_v2_predictive, single pass)" if predictive
              else f"enhanced audio-sec/sec ({BRIDGE_STEPS}-step SB bridge, ncsnpp_v2)")


def synth_batch(n, device, seed=1234):
    """Synthetic noisy utterances (SURVEY.md section 8(d) recipe, vectorised): 8 harmonics of f0~U(100,300) Hz
    with 1/k roll-off and a 3 Hz envelope, plus white noise at SNR~U(0,15) dB.  fp32 [n, N_SAMPLES]."""
    import math
    import torch
    g = torch.Generator(device="cpu").manual_seed(seed)
    f0 = 100 + 200 * torch.rand(n, 1, generator=g)
    phi = 2 * math.pi * torch.rand(n, 8, generator=g)
    phi_e = 2 * math.pi * torch.rand(n, 1, generator=g)
    snr = 15 * torch.rand(n, 1, generator=g)
    t = torch.arange(N_SAMPLES, dtype=torch.float32, device=device)[None] / SR
    f0, phi, phi_e, snr = (v.to(device) for v in (f0, phi, phi_e, snr))
    clean = torch.zeros(n, N_SAMPLES, device=device)
    for k in range(1, 9):
        clean += (1.0 / k) * torch.sin(2 * math.pi * k * f0 * t + phi[:, k - 1:k])
    clean *= 0.3 * 0.5 * (1 + torch.sin(2 * math.pi * 3 * t + phi_e))
    gn = torch.Generator(device=device).manual_seed(seed + 1)
    noise = torch.randn(n, N_SAMPLES, generator=gn, device=device)
    noise *= torch.sqrt(clean.pow(2).mean(1, keepdim=True) / (noise.pow(2).mean(1, keepdim=True) * 10 ** (snr / 10)))
    return (clean + noise).contiguous()


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 100 ms while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.path = index, None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1])); mx.append(float(f[2]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            sm.sort()
            out = {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}
        return out


def cpu_reference_leg(seconds_budget=25.0, steps=1, warmup=0, threads=None, keep_probe=None):
    """The reference's CPU path (oracle port): B=1 utterance loop exactly like infer_folder.py:90-146.
    Returns (audio-s/s, ms per step, description of the sample, cores)."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import fdbm_oracle as O
    cores = threads or os.cpu_count() or 1
    torch.set_num_threads(cores)
    cfg = O.NcsnppConfig()
    sd = O.sensitised_state_dict(cfg, seed=0)
    bridge = O.Bridge("sb", N=BRIDGE_STEPS, sampler_type="ode_ei")
    model = lambda a, b, c: O.ncsnpp_forward(sd, cfg, a, b, c)

    def run(n_samples):
        _, noisy = O.synth_pair(0, n_samples=n_samples)
        t0 = time.perf_counter()
        with torch.no_grad():
            out = O.enhance(noisy[None], model, bridge, O.SpecConfig())
        dt = time.perf_counter() - t0
        if keep_probe is not None and n_samples == SR:        # the 1 s probe doubles as the SI-SDR parity sample
            keep_probe.update(sd=sd, noisy=noisy, ref=out.numpy(), si_sdr=O.si_sdr)
        return dt

    # probe with 1 s of audio, then pick the largest utterance length whose K+W repetitions fit the budget
    probe = run(SR)
    n_runs = max(1, steps + warmup)
    seconds = UTT_SECONDS
    while seconds > 1.0 and probe * seconds * n_runs > seconds_budget * max(1, n_runs) ** 0.5 * 2.5:
        seconds /= 2
    n_samples = int(SR * seconds)
    for _ in range(warmup):
        run(n_samples)
    times = [run(n_samples) for _ in range(max(1, steps))]
    dt = sum(times) / len(times)
    sample = (f"1 of {UTTS_PER_GPU} utterances per step, {seconds:g} s of audio each (B=1 loop like the reference), "
              f"N={BRIDGE_STEPS}, fp32, torch CPU with {cores} threads")
    return seconds / dt, dt * 1e3, sample, cores


def ncu_conv_traffic(micro_batch, n_frames):
    """roofline.traffic: dram__bytes_read.sum + dram__bytes_write.sum of the conv_igemm launches of one forward, per launch,
    from the committed ncu capture of THIS build (profiles/conv_traffic.json, written by tools/ncu_summary.py from an
    `ncu --set full` run; it records the sha256 of csrc/conv_igemm.cu it was taken on).  None when there is no capture for
    this micro-batch / frame count or when the kernel source has changed since the capture."""
    import hashlib
    try:
        rec = json.load(open(os.path.join(ROOT, "profiles", "conv_traffic.json")))
        src = open(os.path.join(PKG, "csrc", "conv_igemm.cu"), "rb").read()
        if rec.get("conv_igemm_sha256") != hashlib.sha256(src).hexdigest():
            return None, "profiles/conv_traffic.json was captured on an older conv_igemm.cu"
        for e in rec.get("captures", []):
            if e["micro_batch"] == micro_batch and e["n_frames"] == n_frames:
                return e["dram_bytes"] / e["launches"], rec.get("source", "profiles/conv_traffic.json")
        return None, "no capture at this micro-batch"
    except Exception as ex:                                          # no capture committed
        return None, f"no capture ({type(ex).__name__})"


def torch_gpu_baseline_leg(dev, n_batch=16, budget_s=20.0):
    """The same-box bar SURVEY.md 8(d) asks for: the reference path in stock PyTorch on THIS GPU (cuFFT STFT, cuDNN
    convolutions, ATen GroupNorm / SiLU / softmax), i.e. the oracle port run on `cuda` instead of `cpu`.  Two precisions:
    fp32 with TF32 convolutions (PyTorch's default, what the reference gets) and bf16 autocast; two batchings: the
    reference's B = 1 file loop (infer_folder.py:93-121) and a batch of `n_batch`.  Baseline only -- not on any product path."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import fdbm_oracle as O
    cfg = O.NcsnppConfig()
    sd = {k: v.to(dev) for k, v in O.sensitised_state_dict(cfg, seed=0).items()}
    table = O.Bridge("sb", N=BRIDGE_STEPS, sampler_type="ode_ei").coefficient_table().tolist()
    times = O.Bridge("sb", N=BRIDGE_STEPS, sampler_type="ode_ei").time_grid()[:-1].tolist()
    win = torch.sqrt(torch.hann_window(512, periodic=True)).to(dev)
    waves = synth_batch(n_batch, dev, seed=777)

    def enhance(y):                                                  # infer_single.py:80-99 / bridge.py:66-87 in torch ops
        norm = y.abs().amax(1, keepdim=True)
        S = torch.stft(y / norm, 512, 256, window=win, center=True, return_complex=True)
        Y = 0.15 * S.abs() ** 0.5 * torch.exp(1j * S.angle())
        T = Y.shape[-1]
        pad = (64 - T % 64) % 64
        if pad:
            idx = torch.arange(T + pad, device=dev)
            Y = Y[..., torch.where(idx < T, idx, 2 * (T - 1) - idx)]
        Y = Y[:, None]
        x = Y.clone()
        for (wx, ws, wy), t in zip(table, times):
            D = O.ncsnpp_forward(sd, cfg, x, Y, torch.full((y.shape[0],), t, device=dev))
            x = wx * x + ws * D + wy * Y
        X = x[:, 0] / 0.15
        X = X.abs() ** 2 * torch.exp(1j * X.angle())
        return torch.istft(X, 512, 256, window=win, center=True, length=y.shape[1]) * norm

    out = {"what": "oracle port (= the reference's torch ops) on cuda: cuFFT + cuDNN + ATen, same weights / sampler; "
                   f"{UTT_SECONDS:g} s utterances, N={BRIDGE_STEPS}"}
    t_start = time.perf_counter()
    for label, autocast in (("fp32_tf32conv", False), ("bf16_autocast", True)):
        for bname, batch in (("B1_loop", waves[:1]), (f"B{n_batch}", waves)):
            if time.perf_counter() - t_start > budget_s:
                break
            try:
                with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
                    enhance(batch); torch.cuda.synchronize()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    reps = 3 if batch.shape[0] == 1 else 1
                    e0.record()
                    for _ in range(reps):
                        enhance(batch)
                    e1.record(); torch.cuda.synchronize()
                ms = e0.elapsed_time(e1) / reps
                out[f"{label}_{bname}"] = {"audio_s_per_s": batch.shape[0] * UTT_SECONDS / (ms * 1e-3), "ms": ms}
            except Exception as ex:                                  # e.g. out of memory at the batched setting
                out[f"{label}_{bname}"] = {"error": f"{type(ex).__name__}: {str(ex)[:120]}"}
            torch.cuda.empty_cache()
    return out


def hbm_kernel_leg(model, waves, dev, reps=20):
    """The HBM-bound kernels of the path timed alone with CUDA events on the whole per-GPU batch (inputs >> L2):
    fused STFT+compress+pad, fused decompress+iSTFT and the bridge update; algorithmic bytes (SURVEY.md 8(d)) / time."""
    import torch
    from fdbm_b200 import _lib
    lib = _lib.load()
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6500.0))
    n, ts = waves.shape
    dm = model.data_module
    y = waves / waves.abs().amax(1, keepdim=True)

    def timeit(fn):
        # `reps` back-to-back launches captured in one CUDA graph: the kernels are tens of microseconds long, so
        # launching them from Python would time the host, not the kernel
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        side = torch.cuda.Stream()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.stream(side):
            with torch.cuda.graph(g, stream=side):
                for _ in range(reps):
                    fn()
        g.replay()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        g.replay()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    Y = dm.stft_compress(y, pad_mode=model.pad_mode)
    frames = Y.shape[-1]
    spec_bytes = Y.numel() * 8
    out = {}
    ms = timeit(lambda: dm.stft_compress(y, pad_mode=model.pad_mode))
    out["stft_compress"] = {"bytes": n * ts * 4 + spec_bytes, "ms": ms}
    ms = timeit(lambda: dm.to_audio(Y[:, 0], ts))
    out["decompress_istft"] = {"bytes": spec_bytes + n * ts * 4, "ms": ms}
    x = Y.clone()
    d = Y.clone()
    coef = torch.tensor([0.8, 0.2, -0.1], device=dev)
    xr, dr, yr = (torch.view_as_real(v) for v in (x, d, Y))

    def step():
        _lib.check(lib.fdbm_bridge_step(xr.data_ptr(), dr.data_ptr(), yr.data_ptr(), coef.data_ptr(), 0, 0, 0,
                                        x.numel(), _lib.current_stream()), "fdbm_bridge_step")
    ms = timeit(step)
    out["bridge_step_ode"] = {"bytes": 4 * spec_bytes, "ms": ms}
    for v in out.values():
        v["GB/s"] = v["bytes"] / (v["ms"] * 1e-3) / 1e9
        v["frac_of_measured_hbm_peak"] = v["GB/s"] / peak
    out["peak_GB/s"] = peak
    out["batch"] = f"{n} utterances x {ts / SR:g} s ({frames} frames)"
    return out


def train_main(args):
    """BASELINE.json configs[3]: the bridge training step (fdbm/model.py:258-275 + hybrid loss + Adam/EMA, train.py:161
    clipping) on `--train-batch` synthetic 65 280-sample crops (exactly 256 frames, data_module.py:58) per GPU, DDP
    gradient all-reduce over NCCL.  One step = sample_prior -> forward -> loss -> backward -> all-reduce -> Adam+EMA."""
    import torch
    import torch.distributed as dist
    from fdbm_b200 import BackboneRegistry, Bridge, SpecsDataModule, _lib, sensitise_
    from fdbm_b200.training import TrainStep
    rank = int(os.environ.get("RANK", "0")); local_rank = int(os.environ.get("LOCAL_RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.check(_lib.load().fdbm_check_device(), "fdbm_check_device")
    B, crop = args.train_batch, 255 * 256
    net = sensitise_(BackboneRegistry.get_by_name("ncsnpp_v2")(), seed=0).to(dev)
    dm = SpecsDataModule(n_fft=512, hop_length=256, num_frames=256, window="sqrthann")
    bridge = Bridge("sb", N=BRIDGE_STEPS, sampler_type="ode_ei")
    ts = TrainStep(net, bridge, dm, batch=B, n_frames=256, loss_scale=1024.0, loss_type=args.loss_type)
    global N_SAMPLES
    N_SAMPLES = crop
    noisy = synth_batch(B, dev, seed=4321 + 1000 * rank)
    clean = synth_batch(B, dev, seed=8765 + 1000 * rank) * 0.5
    noisy = clean + 0.3 * noisy
    norm = noisy.abs().amax(1, keepdim=True)
    X = dm.stft_compress(clean / norm, pad_mode="zero_pad", n_frames_out=256)
    Y = dm.stft_compress(noisy / norm, pad_mode="zero_pad", n_frames_out=256)
    hx = torch.empty(X.shape, dtype=X.dtype, pin_memory=True).copy_(X)
    hy = torch.empty(Y.shape, dtype=Y.dtype, pin_memory=True).copy_(Y)
    hloss = torch.empty(1, pin_memory=True)

    def step_device():
        return ts.training_step(X, Y)

    def step_e2e():
        x = hx.to(dev, non_blocking=True); y = hy.to(dev, non_blocking=True)
        hloss.copy_(ts.training_step(x, y).reshape(1), non_blocking=True)

    def timed(fn, steps):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps - 1):
            fn()
        out = fn()                                   # the last step's result, for --dump-outputs
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), out

    for _ in range(max(args.warmup, 3)):
        step_device()
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    ms, loss = timed(step_device, args.steps)
    if args.dump_outputs and rank == 0:
        dump_output(args.dump_outputs, "loss", loss)
    ms_e2e, _ = timed(step_e2e, args.steps)
    # a few 56 ms steps end before nvidia-smi prints its first line: the sampler covers both timed regions (same step, same load)
    clock_info = clocks.stop() if rank == 0 else None
    # phase split of one step (events around forward / backward / optimiser)
    for _ in range(2):                                  # the second pass is the one reported (the first re-warms allocator paths)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        torch.cuda.synchronize()
        ev[0].record(); t, _, _, x_t = ts.sample_prior(X, Y); D = ts.forward(x_t.contiguous(), Y, t)
        ev[1].record(); ts.loss_and_backward(X, Y)
        ev[2].record(); ts.optimizer_step()
        ev[3].record(); torch.cuda.synchronize()
    lib = _lib.load()
    if rank == 0:
        samples = B * world * args.steps
        value = samples / (ms * 1e-3)
        gflop_step = 3 * 532.1 * B * world
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("bf16_tflops_sustained", 1400.0))
        achieved = gflop_step / world / (ms / args.steps * 1e-3) / 1e3
        print(json.dumps({
            "metric": f"bridge training step throughput (ncsnpp_v2, {args.loss_type} loss, Adam+EMA, DDP)", "value": value, "unit": "crops/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16" if lib.fdbm_operand_is_bf16() else "fp16 (loss-scaled gradients, fp32 master weights)", "data": "synthetic",
            "config": {"workload": f"train: {B} crops of 65 280 samples (256 frames) per GPU, ncsnpp_v2 65.6 M params, "
                                   f"{args.loss_type} loss, Adam lr 1e-4, clip 3.0, EMA 0.999", "global_batch": B * world,
                       "parallelism": f"dp{world}", "l2": "activations kept for backward >> L2"},
            "e2e": {"value": samples / (ms_e2e * 1e-3), "unit": "crops/s", "h2d_bytes_per_step": 2 * X.numel() * 8,
                    "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": (lib.fdbm_plan_num_launches(ts.plan) + lib.fdbm_plan_num_backward_launches(ts.plan)) * args.steps,
            "phase_ms": {"forward": ev[0].elapsed_time(ev[1]), "forward+loss+backward": ev[1].elapsed_time(ev[2]),
                         "allreduce+adam+ema+repack": ev[2].elapsed_time(ev[3])},
            "model_tflops_per_gpu": achieved,
            "roofline": {"bound": "tensor", "kernel": "conv_igemm (fwd, dgrad) + conv_wgrad, whole step", "achieved": achieved, "peak": peak,
                         "unit": "TFLOP/s", "frac": achieved / peak, "traffic": None,
                         "note": "algorithmic 3 x 532.1 GFLOP per crop (fwd + dgrad + wgrad) over the WHOLE step time"},
            "plan_device_GiB": lib.fdbm_plan_device_bytes(ts.plan) / 2 ** 30, "clocks": clock_info}))
    if world > 1:
        dist.destroy_process_group()
    return 0


def tfgridnet_main(args):
    """SURVEY.md 8(f) #1: the backbones config.yaml / config_predictive.yaml actually select.  `--workload tfgridnet`: 5-step SB
    sampler on tfgridnet_5l32c100; `--workload tfgridnet_predictive`: one pass of tfgridnet_5l32c100_predictive.  Same 256 synthetic
    4 s utterances, zero padding to 64 frames (infer_single.py:64-69).  Single process (one GPU)."""
    import torch
    from fdbm_b200 import EnhancementModel, _lib
    from fdbm_b200.model import PredictiveEnhancementModel
    pred = args.workload == "tfgridnet_predictive"
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    _lib.check(_lib.load().fdbm_check_device(), "fdbm_check_device")
    if pred:
        model = PredictiveEnhancementModel("tfgridnet_5l32c100_predictive")
    else:
        model = EnhancementModel("tfgridnet_5l32c100", "sb", bridge_kwargs=dict(N=BRIDGE_STEPS, sampler_type="ode_ei"))
    model = model.to(dev).eval()
    # 36 utterances = 74 tiles of 128 sequences per sweep = 296 CTAs (two directions x two CTAs per tile) = exactly two waves of
    # the 148 SMs; 32 would leave the second wave 78 % full
    mb = min(args.micro_batch, 36)
    waves = synth_batch(args.utts, dev, seed=1234)
    host_in = torch.empty(waves.shape, dtype=torch.float32, pin_memory=True).copy_(waves)
    host_out = torch.empty_like(host_in, pin_memory=True)

    def step_device():
        return model.enhance_many(waves, micro_batch=mb)

    def step_e2e():
        for i in range(0, args.utts, mb):
            chunk = host_in[i:i + mb].to(dev, non_blocking=True)
            n = chunk.shape[0]
            if n < mb:
                chunk = torch.cat([chunk, chunk[-1:].expand(mb - n, -1)], dim=0)
            host_out[i:i + n].copy_(model.enhance_batch(chunk)[:n], non_blocking=True)

    def timed(fn, steps):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps - 1):
            fn()
        out = fn()                                   # the last step's result, for --dump-outputs
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), out

    for _ in range(max(args.warmup, 3)):
        step_device()
    clocks = ClockSampler(0)
    clocks.start()
    ms, enhanced = timed(step_device, args.steps)
    clock_info = clocks.stop()
    if args.dump_outputs:
        dump_output(args.dump_outputs, "enhanced", enhanced, range(args.utts))
    ms_e2e, _ = timed(step_e2e, args.steps)
    n_fwd = 1 if pred else BRIDGE_STEPS
    T, Q = 256, 257
    # algorithmic MACs of the ten BiLSTM sweeps of one forward (input + recurrent projections + ConvTranspose1d), per utterance
    steps_intra, steps_inter = (T + 6) * (Q + 3), (Q + 6) * (T + 3)
    gflop_fwd = 2 * 5 * 2 * (steps_intra + steps_inter) * (128 * 400 + 100 * 400 + 100 * 128) / 1e9
    audio_s = args.utts * UTT_SECONDS
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("bf16_tflops_sustained", 1400.0))
    achieved = gflop_fwd * n_fwd * args.utts * args.steps / (ms * 1e-3) / 1e3
    print(json.dumps({
        "metric": ("enhanced audio-sec/sec (predictive tfgridnet_5l32c100_predictive, single pass)" if pred
                   else f"enhanced audio-sec/sec ({BRIDGE_STEPS}-step SB bridge, tfgridnet_5l32c100)"),
        "value": audio_s * args.steps / (ms * 1e-3), "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp16", "data": "synthetic",
        "config": {"workload": f"{args.workload}: {args.utts} synthetic 4 s 16 kHz utterances, " +
                               ("tfgridnet_5l32c100_predictive (2.11 M params, PyTorch default init), one pass" if pred else
                                f"tfgridnet_5l32c100 (2.16 M params, PyTorch default init), Bridge('sb','bb') ode_ei N={BRIDGE_STEPS}"),
                   "utterances": args.utts, "bridge_steps": n_fwd},
        "run": {"micro_batch": mb, "l2": "ConvTranspose1d partials of one sweep are > 1 GB at micro-batch 32 (>> L2)"},
        "e2e": {"value": audio_s * args.steps / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": args.utts * N_SAMPLES * 4,
                "d2h_bytes_per_step": args.utts * N_SAMPLES * 4, "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": ((args.utts + mb - 1) // mb) * (3 + n_fwd * (4 + 5 * 10 + 1)) * args.steps,
        "roofline": {"bound": "tensor", "kernel": "lstm_sweep_tc_kernel (BiLSTM sweep: tcgen05 UMMA M=128 N=224 per CTA of a 2-CTA cluster, fp16 operands, fp32 TMEM accumulators, hidden state exchanged by cp.async.bulk over DSMEM)",
                     "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak, "traffic": None,
                     "note": f"algorithmic {gflop_fwd:.1f} GFLOP of LSTM + ConvTranspose1d work per forward per utterance over the WHOLE step time; the recurrence is latency-bound (one dependent step every ~2.7 us), see DESIGN.md section 4"},
        "clocks": clock_info}))
    return 0


def files_main(args):
    """SURVEY.md 8(f) #2, the callers' I/O edge of infer_folder.py:91-146: a folder of WAV files of DIFFERENT lengths
    (2-6 s), timed from the file names to the written enhanced files: decode, length bucketing, pinned staging + H2D,
    variable-length STFT, sampler, iSTFT, D2H, 16-bit PCM encode.  Single process (one GPU)."""
    import tempfile
    import numpy as np
    import torch
    from scipy.io import wavfile
    from fdbm_b200 import EnhancementModel, sensitise_, _lib
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    _lib.check(_lib.load().fdbm_check_device(), "fdbm_check_device")
    model = EnhancementModel("ncsnpp_v2", "sb", bridge_kwargs=dict(N=BRIDGE_STEPS, sampler_type="ode_ei"))
    sensitise_(model.dnn, seed=0)
    model = model.to(dev).eval()
    mb = min(args.micro_batch, 64)                # five padded-length buckets of ~50 files each: one micro-batch per bucket
    rng = np.random.default_rng(7)
    tmp = tempfile.mkdtemp(prefix="fdbm_files_")
    paths, outs, total_s = [], [], 0.0
    base = synth_batch(8, torch.device("cpu"), seed=99).numpy()                    # [8, 64000]
    for i in range(args.utts):
        n = int(rng.integers(2 * SR, 6 * SR))
        w = np.tile(base[i % 8], 2)[:n]
        w = w / np.abs(w).max() * 0.7
        p = os.path.join(tmp, "noisy", f"u{i:04d}.wav")
        os.makedirs(os.path.dirname(p), exist_ok=True)
        wavfile.write(p, SR, np.round(w * 32767).astype(np.int16))
        paths.append(p); outs.append(os.path.join(tmp, "enhanced", f"u{i:04d}.wav")); total_s += n / SR
    for _ in range(max(1, min(args.warmup, 2))):                                   # builds one plan + graph per length bucket
        model.enhance_files(paths, outs, micro_batch=mb)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        model.enhance_files(paths, outs, micro_batch=mb)
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / args.steps
    n_bytes = sum(os.path.getsize(p) for p in paths)
    print(json.dumps({
        "metric": f"enhanced audio-sec/sec from WAV files of different lengths ({BRIDGE_STEPS}-step SB bridge, ncsnpp_v2)",
        "value": total_s / dt, "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": max(1, min(args.warmup, 2)),
        "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16" if _lib.load().fdbm_operand_is_bf16() else "fp16", "data": "synthetic",
        "config": {"workload": f"files: {args.utts} synthetic 16 kHz mono 16-bit WAV files of 2-6 s ({total_s:.0f} s of audio), "
                               f"bucketed by padded frame count, micro-batch {mb}, wall clock from file names to written files",
                   "micro_batch": mb, "bridge_steps": BRIDGE_STEPS},
        "e2e": {"value": total_s / dt, "unit": UNIT, "h2d_bytes_per_step": n_bytes * 2, "d2h_bytes_per_step": n_bytes * 2},
        "timing": "host wall clock around enhance_files (includes file decode / encode); not a device-event number"}))
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 3; 20 for --workload train, whose step is 56 ms)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--micro-batch", type=int, default=int(os.environ.get("FDBM_MICRO_BATCH", "128")))
    ap.add_argument("--utts", type=int, default=UTTS_PER_GPU, help="utterances per GPU per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="infer_folder", choices=["infer_folder", "predictive", "train", "files", "tfgridnet", "tfgridnet_predictive"],
                    help="BASELINE.json configs[1] (default, the headline metric), configs[2] or configs[3] (training step)")
    ap.add_argument("--train-batch", type=int, default=16, help="training crops per GPU per step (configs[3]: 8 x 16)")
    ap.add_argument("--loss-type", default="data_prediction_hybrid",
                    choices=["data_prediction_hybrid", "data_prediction", "data_prediction_mel", "data_prediction_melphase"],
                    help="--workload train: BridgeModel's loss head (model.py:162-254); config.yaml trains with the hybrid one")
    ap.add_argument("--bridge-steps", type=int, default=5, help="configs[4]: sampling-step sweep 1/5/10/30")
    ap.add_argument("--seconds", type=float, default=4.0, help="configs[4]: utterance length (30 s long-form)")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="multi-GPU: 'strong' = --utts utterances in TOTAL, sharded (BASELINE configs[1]); 'weak' = --utts per GPU")
    ap.add_argument("--no-gather", action="store_true", help="skip the final NCCL all_gather of the enhanced waveforms")
    ap.add_argument("--no-torch-gpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (enhanced waveforms; the loss for --workload "
                         "train) to DIR/<name>.npy in float32, a seeded sample of the rows where it exceeds 60 MiB; "
                         "DIR/<name>_rows.npy names the utterance of each row")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 20 if args.workload == "train" else 3
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.workload == "files"):
        ap.error("--dump-outputs covers the CUDA path of the in-memory workloads (not --impl reference or --workload files)")
    if args.dump_outputs and args.workload != "train" and int(SR * args.seconds) * 4 > DUMP_BYTES:
        ap.error(f"--dump-outputs: one {args.seconds:g} s utterance is more than the {DUMP_BYTES} bytes a dump may take")
    import torch
    torch.manual_seed(0)             # the Fourier-feature weights are drawn at construction: same arguments, same model and inputs
    predictive = args.workload == "predictive"
    set_workload(args.seconds, args.bridge_steps, predictive)
    if args.workload == "train":
        return train_main(args)
    if args.workload == "files":
        return files_main(args)
    if args.workload.startswith("tfgridnet"):
        return tfgridnet_main(args)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    strong = args.scaling == "strong"
    total_utts = args.utts if strong else args.utts * world
    config = {"workload": (f"{args.workload}: {total_utts} synthetic {UTT_SECONDS:g} s 16 kHz utterances, " +
                           ("ncsnpp_v2_predictive (random init re-sensitised), one backbone pass, "
                            if predictive else
                            f"ncsnpp_v2 (65.6 M params, random init re-sensitised), Bridge('sb','bb') ode_ei N={BRIDGE_STEPS}, ") +
                           "fused STFT/compress/pad and decompress/iSTFT"),
              "utterances": total_utts, "bridge_steps": BRIDGE_STEPS}

    if args.impl == "reference":
        if rank != 0:
            return 0
        v, ms, sample, cores = cpu_reference_leg(steps=args.steps, warmup=args.warmup)
        print(json.dumps({
            "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": args.scaling if args.gpus > 1 else "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
            "note": "ONE CPU process on this box's host cores whatever --gpus says (rank 0 only); a bounded sample, extrapolated",
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}))
        return 0

    import torch
    import torch.distributed as dist
    from fdbm_b200 import EnhancementModel, _lib, gather_waveforms, sensitise_, split_list
    from fdbm_b200.model import PredictiveEnhancementModel
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.check(_lib.load().fdbm_check_device(), "fdbm_check_device")

    # this rank's shard of the utterance list (contiguous chunks, infer_folder.py:149-152)
    if strong:
        shards = split_list(list(range(args.utts)), world)
        my_ids, counts = shards[rank], [len(s) for s in shards]
    else:
        my_ids, counts = list(range(rank * args.utts, (rank + 1) * args.utts)), [args.utts] * world
    n_local = len(my_ids)
    mb = max(1, min(args.micro_batch, n_local))
    do_gather = world > 1 and not args.no_gather
    if predictive:
        model = PredictiveEnhancementModel("ncsnpp_v2_predictive")
    else:
        model = EnhancementModel("ncsnpp_v2", "sb", bridge_kwargs=dict(N=BRIDGE_STEPS, sampler_type="ode_ei"))
    sensitise_(model.dnn, seed=0)
    model = model.to(dev).eval()
    # utterance i is the same signal whatever the GPU count (the generator is keyed by the utterance id, not the rank)
    all_waves = synth_batch(total_utts, dev, seed=1234)
    waves = all_waves[my_ids[0]:my_ids[-1] + 1].contiguous()
    del all_waves
    host_in = torch.empty(waves.shape, dtype=torch.float32, pin_memory=True).copy_(waves)
    n_out = total_utts if do_gather else n_local
    host_out = torch.empty(n_out, waves.shape[1], dtype=torch.float32, pin_memory=True)
    local_out = torch.empty_like(waves)

    def step_device():
        out = model.enhance_many(waves, micro_batch=mb)
        return gather_waveforms(out, counts) if do_gather else out

    def step_e2e():
        for i in range(0, n_local, mb):
            chunk = host_in[i:i + mb].to(dev, non_blocking=True)
            n = chunk.shape[0]
            if n < mb:
                chunk = torch.cat([chunk, chunk[-1:].expand(mb - n, -1)], dim=0)
            local_out[i:i + n] = model.enhance_batch(chunk)[:n]
        host_out.copy_(gather_waveforms(local_out, counts) if do_gather else local_out, non_blocking=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps - 1):
            fn()
        out = fn()                                   # the last step's result, for --dump-outputs
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), out

    for _ in range(max(args.warmup, 3)):
        step_device()
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    ms_total, enhanced = timed(step_device, args.steps)
    clock_info = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_output(args.dump_outputs, "enhanced", enhanced, range(total_utts) if do_gather else my_ids)
    del enhanced
    step_e2e()
    ms_e2e, _ = timed(step_e2e, args.steps)

    audio_s = total_utts * UTT_SECONDS
    value = audio_s * args.steps / (ms_total * 1e-3)
    e2e = audio_s * args.steps / (ms_e2e * 1e-3)

    # roofline of the dominant kernel: every launch of one forward timed with CUDA events
    roofline, shares = None, None
    n_frames = -(-(1 + N_SAMPLES // 256) // 64) * 64
    info = model.dnn.plan_info(mb, n_frames)
    hbm_kernels = None
    if rank == 0:
        Y = model.data_module.stft_compress(waves[:mb] / waves[:mb].abs().amax(1, keepdim=True), pad_mode=model.pad_mode)
        t = torch.full((mb,), 0.5, device=dev)
        prof = [(model.dnn.profile_forward(Y) if predictive else model.dnn.profile_forward(Y, Y, t)) for _ in range(3)][-1]
        hbm_kernels = hbm_kernel_leg(model, waves, dev)
        kind_ms = {}
        for ms, kind, _ in prof:
            kind_ms[kind] = kind_ms.get(kind, 0.0) + ms
        conv_ms = kind_ms.get(0, 0.0)
        conv_flops = sum(f for _, k, f in prof if k == 0)
        n_conv = sum(1 for _, k, _ in prof if k == 0)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("bf16_tflops_sustained", 1400.0))
        achieved = conv_flops / (conv_ms * 1e-3) / 1e12
        roofline = {"bound": "tensor", "kernel": "conv_igemm_kernel (tcgen05 implicit GEMM, 16-bit operands, fp32 accumulate)",
                    "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                    "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)"
                    if peaks else "fallback 1.4 PFLOP/s sustained (B200_PROFILING.md)",
                    "traffic": None if predictive else ncu_conv_traffic(mb, n_frames)[0],
                    "traffic_source": None if predictive else ncu_conv_traffic(mb, n_frames)[1],
                    "traffic_unit": "bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum over the conv launches of one "
                                    "forward at this micro-batch, ncu --set full) / launches",
                    "launches_per_forward": n_conv,
                    "avg_launch_ms": conv_ms / max(1, n_conv),
                    # the same quantity from the TIMED region itself: the convolutions' share of a forward (from the per-launch event
                    # pass) x the device-timed step, i.e. without the event records between the launches of the profile pass
                    "achieved_from_timed_step": None, "frac_from_timed_step": None,
                    "algorithmic_gflop_per_forward_per_utt": conv_flops / mb / 1e9}
        tot = sum(kind_ms.values())
        names = {0: "conv_igemm", 1: "groupnorm_act", 2: "channel_stats", 3: "skinny", 4: "attention", 5: "temb"}
        shares = {names[k]: round(v / tot, 4) for k, v in sorted(kind_ms.items())}
        shares["forward_ms_per_microbatch"] = tot
        if tot > 0 and conv_ms > 0 and n_local % mb == 0:
            n_fwd = (n_local // mb) * (1 if predictive else BRIDGE_STEPS)          # forwards of this rank per step
            hbm_ms = sum(k["ms"] for k in (hbm_kernels or {}).values() if isinstance(k, dict) and "ms" in k) if not predictive else 0.0
            step_ms = ms_total / args.steps
            conv_ms_step = max(step_ms - hbm_ms, 1e-6) * (conv_ms / tot)             # the step is forwards + the three HBM kernels
            roofline["achieved_from_timed_step"] = conv_flops * n_fwd / (conv_ms_step * 1e-3) / 1e12
            roofline["frac_from_timed_step"] = roofline["achieved_from_timed_step"] / peak

    n_micro = (n_local + mb - 1) // mb
    launches_per_step = n_micro * (1 + 1 + BRIDGE_STEPS * (info["launches"] + 1) + 1)
    torch_gpu = None
    if rank == 0 and world == 1 and not args.no_torch_gpu_baseline and not predictive:
        model.dnn.release_plans()                                   # give the stock-PyTorch leg the memory
        torch.cuda.empty_cache()
        torch_gpu = torch_gpu_baseline_leg(dev)

    cpu_baseline = None
    si_sdr_delta = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        probe = {}
        v, ms, sample, cores = cpu_reference_leg(seconds_budget=25.0, keep_probe=probe)
        cpu_baseline = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample, "ms_per_utterance": ms}
        if probe and not predictive:
            # SI-SDR delta (the third part of BASELINE.json's metric): the CUDA path with the oracle's weights on the probe
            # utterance, against a target the reference output scores 15 dB on (the regime of a trained model)
            import numpy as np
            pm = EnhancementModel("ncsnpp_v2", "sb", bridge_kwargs=dict(N=BRIDGE_STEPS, sampler_type="ode_ei"))
            pm.dnn.load_state_dict(probe["sd"])
            pm = pm.to(dev).eval()
            got = pm.enhance(probe["noisy"][None], pad_mode="reflection")
            ref = probe["ref"].reshape(-1).astype(np.float64)
            rng = np.random.default_rng(0)
            nz = rng.standard_normal(ref.shape)
            nz -= ref * (nz @ ref) / (ref @ ref)
            target = ref + nz * np.sqrt((ref @ ref) / (nz @ nz) / 10 ** 1.5)
            si = probe["si_sdr"]
            si_sdr_delta = {"delta_db_on_15dB_target": float(abs(si(target, got) - si(target, ref))),
                            "agreement_db": float(si(ref, got)),
                            "sample": "1 s synthetic utterance, oracle weights, ours (CUDA) vs the reference port (CPU fp32)"}
            pm.dnn.release_plans()
            del pm

    if rank == 0:
        run = {"micro_batch": mb, "parallelism": f"utterance-sharded x{world}", "utterances_per_gpu": counts,
               "final_gather": ("NCCL all_gather of the enhanced waveforms onto every rank, inside the timed region "
                                f"({total_utts * N_SAMPLES * 4 / 1e6:.1f} MB)") if do_gather else "none",
               "l2": f"working set per step >> L2: {info['device_bytes'] / 2**30:.1f} GiB of activations+weights "
                     f"per micro-batch, {n_micro} micro-batches per step per GPU (no explicit flush needed)"}
        print(json.dumps({
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": args.scaling if world > 1 else "weak",
            "vs_baseline": None,
            "dtype": "bf16" if _lib.load().fdbm_operand_is_bf16() else "fp16", "data": "synthetic", "config": config, "run": run,
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": n_local * N_SAMPLES * 4,
                    "d2h_bytes_per_step": n_out * N_SAMPLES * 4, "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": launches_per_step * args.steps,
            "per_backbone_forward_ms_per_utt": ms_total / args.steps / (max(counts) * BRIDGE_STEPS),
            "model_tflops": GFLOP_PER_FORWARD * BRIDGE_STEPS * total_utts * args.steps / (ms_total * 1e-3) / 1e3,
            "roofline": roofline, "kernel_share": shares, "hbm_kernels": hbm_kernels, "cpu_baseline": cpu_baseline,
            "si_sdr": si_sdr_delta, "torch_gpu_baseline": torch_gpu,
            "clocks": clock_info}))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
