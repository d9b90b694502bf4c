#!/usr/bin/env python
"""Benchmark of the vocoder hot path (contract: see the task statement / DESIGN.md "Measurement").

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl cube|reference] [--workload pwn|hifigan] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic mel.  Default workload is
BASELINE.json configs[1]: batch=8 x 10 s utterances, 80-bin synthetic mel, ParallelWaveNet (ClariNet
IAF student) vocoder, per GPU (weak scaling: every rank synthesises its own batch, no data-path
collective).  ``--workload hifigan`` runs configs[2] (batch=64 x 10 s, HiFi-GAN generator).

Prints ONE JSON line (rank 0).  ``value`` is device-timed (CUDA events, inputs resident in HBM);
``e2e`` goes through the host-buffer C-ABI call with H2D/D2H inside the timed region.
``--dump-outputs DIR`` writes what the timed path returned in its last timed step as DIR/<name>.npy (float32); the inputs
are seeded, so two builds of the project can be compared output for output.
``--impl reference`` times the CPU oracle port (the reference ships no runnable CPU code for the
student - weights only - and /root/reference is not on the GPU box) on a bounded sample.
"""
import argparse
import atexit
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# stdout carries exactly ONE JSON line: NCCL's own banner / debug output (it defaults to stdout) goes to stderr
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")

import torch  # noqa: E402

SR = 22050.0
WORKLOADS = {
    # name: (arch, batch per GPU, frames, description)
    "pwn": ("student", 8, 862, "BASELINE configs[1]: batch=8 x 10 s (F=862, T=220672), 80-bin synthetic mel, ParallelWaveNet student"),
    "hifigan": ("hifigan", 64, 919, "BASELINE configs[2]: batch=64 x 10 s (F=919), HiFi-GAN generator (neb-noft rates [3,5,4,4])"),
    # configs[3]: 256 utterances of 2-15 s on rank 0, LPT-sharded over the ranks, NCCL scatter/gather (strong scaling)
    "ragged": ("hifigan", 256, 0, "BASELINE configs[3]: batch=256 variable-length (2-15 s) utterances, HiFi-GAN generator, sharded across the ranks via NCCL p2p scatter/gather"),
    # configs[4]: strings -> PyTorch frontend -> CUDA vocoder, sharded over the ranks
    "e2e": ("hifigan", 128, 0, "BASELINE configs[4]: 128 phoneme strings -> PyTorch frontend (stand-in of the reference's Languasito2 structure, per utterance) -> CUDA HiFi-GAN vocoder -> int16 audio, sharded across the ranks"),
    # the reference API's call shape: ONE utterance per call (cube/api.py:45-66)
    "api1": ("hifigan", 1, 0, "batch-1 latency (TTSCube.__call__ shape): one utterance of 2 s / 10 s, HiFi-GAN and ParallelWaveNet student, host in -> host out"),
    # configs[0]: CPU only (the autoregressive ClariNet teacher), timed on a few steady-state samples and extrapolated
    "teacher_cpu": ("teacher", 1, 173, "BASELINE configs[0]: single 2 s utterance (F=173, T=44288), 80-bin mel, ClariNet teacher (autoregressive) on CPU PyTorch"),
}
# algorithmic work per output sample of the dominant kernel (DESIGN.md "Measurement")
GATE_FLOPS = 2.0 * (2 * 256 * 128 * 3 + 2 * 256 * 80)     # gated dilated conv + conditioning 1x1
GATE_BYTES = 4.0 * (128 + 80 + 256)                        # read h, read c_up, write o (fp32)
BLOCK_FLOPS = GATE_FLOPS + 2.0 * (256 * 256)               # + res/skip 1x1 256 -> 128+128 (fused block kernel)
BLOCK_BYTES = 4.0 * (128 + 80 + 128 + 128 + 128)           # read h, c_up, skip; write h', skip (fp32 equivalents)
HIFI_FLOPS_PER_SAMPLE = 1022.2e3                           # SURVEY 8(d), neb-noft rates
HIFI_BYTES_PER_SAMPLE = 9021.0
FUSED_TRAFFIC = 2.83e9 + 2.21e9                            # dram read + write of one default block-kernel launch (ncu --set full, round 2)
PWN_FLOPS_PER_SAMPLE = 25.63e6
PWN_BYTES_PER_SAMPLE = 103609.0


DUMP_BYTES = 60 << 20            # array data of --dump-outputs: under 64 MB with the .npy headers
DUMP_WORKLOADS = ("pwn", "hifigan", "ragged", "e2e")


def dump_outputs(d, arrays):
    """Write each tensor of `arrays` as d/<name>.npy in float32.  When they exceed 60 MB together, each is replaced by a
    fixed seeded sample of its flattened elements, and the sample's flat indices go to d/<name>_index.npy (float64)."""
    import numpy as np
    os.makedirs(d, exist_ok=True)
    arrays = {k: v.detach().to("cpu", torch.float32).contiguous() for k, v in arrays.items()}
    total = sum(4 * v.numel() for v in arrays.values())
    for name, v in arrays.items():
        if total > DUMP_BYTES:          # 4 bytes of value + 8 bytes of index per kept element
            keep = int(v.numel() * DUMP_BYTES // (3 * total))
            idx = torch.randperm(v.numel(), generator=torch.Generator().manual_seed(0))[:keep].sort().values
            np.save(os.path.join(d, name + "_index.npy"), idx.to(torch.float64).numpy())
            v = v.reshape(-1)[idx]
        np.save(os.path.join(d, name + ".npy"), v.numpy())


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d.get("bf16_tflops_sustained", d["bf16_tflops"]), src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback")


class ClockSampler:
    """nvidia-smi sampling during the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            atexit.register(self.proc.kill)         # a run that fails before stop() must not leave the sampler running
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


HIFIGAN_NEB_CONFIG = {  # data/models/vocoder/neb-noft/config.json: the shipped generator's architecture
    "resblock": "1", "upsample_rates": [3, 5, 4, 4], "upsample_kernel_sizes": [16, 16, 4, 4], "upsample_initial_channel": 512,
    "resblock_kernel_sizes": [3, 7, 11], "resblock_dilation_sizes": [[1, 3, 5], [1, 3, 5], [1, 3, 5]], "num_mels": 80}


def load_weights(arch):
    """Shipped checkpoints when staged under oracle/_ref/weights (binary data copied from the reference tree by
    build()), else seeded random weights of the same architecture (throughput does not depend on the values)."""
    W = os.path.join(ROOT, "oracle", "_ref", "weights")

    def ld(n):
        p = os.path.join(W, n)
        return torch.load(p, map_location="cpu", weights_only=False) if os.path.exists(p) else None

    if arch == "student":
        s, t = ld("pnn_vocoder.network"), ld("nn_vocoder.network")
        if s is not None and t is not None:
            return (s, t), "shipped pnn_vocoder.network + nn_vocoder.network upsampler"
        from oracle import clarinet_ref as C      # fallback only: seeded weights with the shipped key layout
        return (C.random_state_dict("student", 1), C.random_state_dict("teacher", 2)), "seeded random-init weights (shipped checkpoints not staged)"
    g = ld("g_00600000")
    cfg = dict(HIFIGAN_NEB_CONFIG)
    if g is not None:
        return (g["generator"], cfg), "shipped g_00600000"
    from oracle import hifigan_ref as H
    return (H.random_state_dict(cfg, seed=1), cfg), "seeded random-init weights (shipped checkpoint not staged)"


def synthetic_mel01(B, F, seed, num_mels=80):
    """SURVEY 8(d) cfg1/cfg2 input: smooth field in [0, 1] (ClariNet-era min/max normalisation)."""
    g = torch.Generator().manual_seed(seed)
    r = torch.randn(B, num_mels, F + 8, generator=g)
    return torch.sigmoid(torch.nn.functional.avg_pool1d(r, 9, stride=1)[:, :, :F] * 3.0).contiguous()


def synthetic_logmel(B, F, seed, level=0.0, num_mels=80):
    """SURVEY 8(d) cfg3 input: natural-log-mel-like smooth field, loud enough that the shipped generator peaks near 0.9."""
    g = torch.Generator().manual_seed(seed)
    r = 6.0 * torch.randn(B, num_mels, F + 8, generator=g)
    sm = torch.nn.functional.avg_pool1d(r, 9, stride=1)[:, :, :F]
    tilt = torch.linspace(0, 4, num_mels)[None, :, None]
    return torch.clamp(0.5 * sm - tilt + level, -11.5, 2.5).contiguous()


def synth_inputs(arch, B, F, seed):
    if arch == "student":
        z = torch.randn(B, 1, F * 256, generator=torch.Generator().manual_seed(seed + 1))
        return synthetic_mel01(B, F, seed), z
    return synthetic_logmel(B, F, seed), None


def host_cpus():
    """CPUs this process may really use: affinity mask, capped by the cgroup CPU quota (a container whose
    os.cpu_count() says 192 but whose quota is 16 CPUs is throttled to a crawl by 192 busy threads)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(int(txt[0]) / int(txt[1]))))
            else:
                q = int(txt[0])
                per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                if q > 0:
                    n = min(n, max(1, q // per))
        except Exception:
            pass
    return max(1, n)


THREAD_CANDIDATES = (8, 16, 32)     # torch's CPU convs on these tensors stop scaling past a few dozen threads
CPU_CACHE = os.path.join("/tmp", "cube_bench_cpu_threads.json")


def best_cpu_threads(arch, weights):
    """Fastest of {8, 16, 32} threads (clipped to the CPUs this process owns) on a short probe; every probe is
    bounded (a candidate that runs 3x slower than the best so far ends the sweep) and the answer is cached in
    /tmp, so the sweep runs once per box, not once per arm."""
    ncpu = host_cpus()
    try:
        c = json.load(open(CPU_CACHE))
        if c.get("ncpu") == ncpu and arch in c:
            return int(c[arch])
    except Exception:
        c = {}
    cands = sorted({min(t, ncpu) for t in THREAD_CANDIDATES})
    frames = 10 if arch == "student" else 160
    best, best_dt = cands[0], None
    for t in cands:
        _, _, dt = cpu_oracle_rate(arch, weights, frames, t)          # first call at this thread count: warm-up
        _, _, dt = cpu_oracle_rate(arch, weights, frames, t)
        if best_dt is None or dt < best_dt:
            best, best_dt = t, dt
        elif dt > 3.0 * best_dt:
            break
    try:
        c = dict(c) if isinstance(c, dict) else {}
        c.update({"ncpu": ncpu, arch: best})
        json.dump(c, open(CPU_CACHE, "w"))
    except Exception:
        pass
    return best


def cpu_oracle_rate(arch, weights, frames, threads, batch=1):
    """Time the CPU oracle port on `batch` x `frames`; returns (samples/s, samples, seconds)."""
    from oracle import clarinet_ref as C, hifigan_ref as H
    torch.set_num_threads(threads)
    mel, z = synth_inputs(arch, batch, frames, seed=99)
    t0 = time.perf_counter()
    if arch == "student":
        y = C.vocode_student(weights[0], weights[1], mel, z)
    else:
        y = H.generator_forward(weights[0], weights[1], mel)
    dt = time.perf_counter() - t0
    n = int(y.shape[-1]) * batch
    return n / dt, n, dt


def cpu_sample_shape(rate, F, hop, seconds):
    """(batch, frames) of a CPU sample worth about `seconds` at `rate` samples/s: one utterance up to full length,
    then more of them"""
    want = max(8 * hop, rate * seconds)
    frames = int(max(8, min(F, want / hop)))
    batch = int(max(1, min(16, want // (frames * hop))))
    return batch, frames


# CPU sample per step: FIXED shapes, never grown.  The rate of torch's CPU convs depends strongly on the clip length (short
# clips live in cache, long ones stream from DRAM), so sizing a sample from a probe of another length overshoots by multiples
# (round 1 lost its GPU box that way, the first round-2 attempt took 6 min); a fixed shape has a known cost, and the only
# adjustment allowed is to SHRINK it once when the measured time says the run would not fit its wall-clock budget
# (a smaller clip is never slower per sample, so shrinking cannot overshoot).
# (batch, frames).  The student's CPU rate still falls with the clip length at these sizes (16 host threads: ~7 k samples/s at
# 128 frames, 5.7 k at 256, 5.3 k at a full 862-frame utterance, which takes 40 s), so the short per-step sample of the reference
# arm slightly FLATTERS the CPU; the one-off cpu_baseline of the product arm uses a longer clip.
CPU_SAMPLE = {"step": {"student": (1, 128), "hifigan": (2, 919)},          # --impl reference: one of these per step
              "baseline": {"student": (1, 256), "hifigan": (4, 919)}}      # product arm, cpu_baseline leg: measured once


def cpu_fit_sample(arch, weights, threads, F, n_calls, wall_budget_s, kind="step"):
    """(batch, frames) for `n_calls` timed calls within `wall_budget_s`: the fixed shape, shrunk once if one measured call
    says the run would not fit.  The measuring call doubles as a warm-up."""
    cb, frames = CPU_SAMPLE[kind][arch]
    frames = min(frames, F)
    _, n, dt = cpu_oracle_rate(arch, weights, frames, threads, cb)
    if dt * n_calls > wall_budget_s:
        scale = wall_budget_s / (dt * n_calls)
        if cb > 1 and scale * cb >= 1.0:
            cb = max(1, int(cb * scale))
        else:
            frames = max(8, int(frames * cb * scale))
            cb = 1
    return cb, frames


def torch_cuda_baseline(arch, weights, mel, z, steps=2):
    """The reference's own PyTorch ops on the SAME B200 (upstream runs its generator as a cuDNN module on CUDA:
    cube/api.py:60-63, cube/networks/cubegan.py:75-83): the oracle's functional restatement is those very ATen calls,
    run here on cuda:0 in fp32 (TF32 off) on the workload's own batch.  Reported beside the CPU baseline so that
    nobody reads the GPU/CPU ratio as the speed-up over upstream-on-GPU."""
    from oracle import clarinet_ref as C, hifigan_ref as H
    dev = mel.device
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        if arch == "student":
            ws = {k: v.to(dev) for k, v in weights[0].items()}
            wt = {k: v.to(dev) for k, v in weights[1].items() if k.startswith("upsample_conv.")}
            run = lambda: C.vocode_student(ws, wt, mel, z)
        else:
            ws = {k: v.to(dev) for k, v in weights[0].items()}
            run = lambda: H.generator_forward(ws, weights[1], mel)
        y = run()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            y = run()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        n = int(y.shape[0]) * int(y.shape[-1])
        del y
        torch.cuda.empty_cache()
        return {"value": n / (ms / 1e3), "unit": "samples/s", "ms_per_step": ms, "steps": steps,
                "what": "oracle functional restatement (= the reference's torch ops: F.conv1d / conv_transpose1d, cuDNN) on cuda:0, fp32 with TF32 off, "
                        "same batch, device-resident inputs, CUDA events; torch " + torch.__version__}
    except Exception as e:   # e.g. out of memory on a smaller GPU: report, never fail the bench for a side baseline
        torch.cuda.empty_cache()
        return {"value": None, "error": f"{type(e).__name__}: {str(e)[:200]}"}


def run_reference(args, arch, B, F, desc, rank, world):
    """--impl reference: the reference's CPU path (oracle port: the reference ships no runnable CPU code for the
    student, and /root/reference is not on the GPU box) on the host cores, a bounded sample per step; the whole run
    (calibration + warm-up + steps) stays within about two minutes whatever --steps says."""
    if rank != 0:
        return
    t_start = time.perf_counter()
    weights, wdesc = load_weights(arch)
    threads = best_cpu_threads(arch, weights)
    n_calls = max(1, args.steps + args.warmup)
    hop = 256 if arch == "student" else 240
    cb, frames = cpu_fit_sample(arch, weights, threads, F, n_calls, wall_budget_s=100.0)
    for _ in range(args.warmup):
        cpu_oracle_rate(arch, weights, frames, threads, cb)
    tot_s, tot_t = 0, 0.0
    for _ in range(args.steps):
        _, n, dt = cpu_oracle_rate(arch, weights, frames, threads, cb)
        tot_s += n; tot_t += dt
    val = tot_s / tot_t
    sample = (f"B={cb} x {frames} frames ({cb * frames * hop / SR:.2f} s of audio) per step of the same synthetic workload; oracle port "
              f"(torch CPU fp32), {threads} threads = fastest of {list(THREAD_CANDIDATES)} on a host with {host_cpus()} usable CPUs "
              f"(os.cpu_count() = {os.cpu_count()})")
    line = {
        "impl": "reference", "metric": "audio samples/sec", "value": val, "unit": "samples/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / max(1, args.steps),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic; " + wdesc,
        "rtf": val / SR, "config": {"workload": desc},
        "cpu_baseline": {"value": val, "unit": "samples/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": time.perf_counter() - t_start,
    }
    print(json.dumps(line), flush=True)


def run_teacher_cpu(args, desc, rank):
    """BASELINE configs[0]: single 2-s utterance, 80-bin mel -> ClariNet TEACHER on CPU PyTorch (no GPU by definition).
    The teacher is autoregressive: one network evaluation per audio sample.  The reference ships its weights only
    (data/models/nn_vocoder.network), so the CPU path is the oracle port, whose sampler (oracle/clarinet_ref.py:
    teacher_generate) recomputes the causal receptive field for every sample.  Timed: `--steps` steady-state samples
    (full 2 974-sample receptive field each) of the 2-s utterance, extrapolated to its 44 288 samples - stated in `sample`."""
    if rank != 0:
        return
    from oracle import clarinet_ref as C
    W = os.path.join(ROOT, "oracle", "_ref", "weights", "nn_vocoder.network")
    if os.path.exists(W):
        tsd, wdesc = torch.load(W, map_location="cpu", weights_only=False), "shipped nn_vocoder.network"
    else:
        tsd, wdesc = C.random_state_dict("teacher", 2), "seeded random-init teacher (checkpoint not staged)"
    threads = min(host_cpus(), 8)
    torch.set_num_threads(threads)
    F, hop = 173, 256
    T = F * hop
    nb = C.teacher_blocks_of(tsd)
    rf = (C.FRONT_K - 1) + sum((C.KERNEL - 1) * C.dilation_of(i) for i in range(nb)) + 1
    mel = synthetic_mel01(1, F, seed=1234)
    c_up = C.upsample_mel(tsd, mel)
    n = args.steps
    start = rf + 64                                       # steady state: the window is the full receptive field
    g = torch.Generator().manual_seed(7)
    eps = torch.randn(1, start + n + 1, generator=g)
    # prime the history with the first `start` samples of a student-like signal (values do not change the cost)
    x0 = 0.1 * torch.randn(1, 1, start, generator=g)
    w = {k: v.float() for k, v in C.fold_weight_norm(tsd).items()}
    x = torch.zeros(1, 1, start + n + 1)
    x[:, :, :start] = x0
    for _ in range(max(1, args.warmup)):
        C.wavenet_forward(w, "", nb, x[:, :, 1:start], c_up[:, :, 1:start])
    t0 = time.perf_counter()
    for t in range(start - 1, start - 1 + n):
        lo = t + 1 - rf
        ml = C.wavenet_forward(w, "", nb, x[:, :, lo:t + 1], c_up[:, :, lo:t + 1])
        x[:, 0, t + 1] = ml[:, 0, -1] + 0.8 * eps[:, t] * torch.exp(ml[:, 1, -1])      # cube/networks/loss.py:50-52
    dt = time.perf_counter() - t0
    rate = n / dt
    line = {
        "impl": "reference", "metric": "audio samples/sec", "value": rate, "unit": "samples/s", "n_gpus": 0, "steps": n, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / n, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic; " + wdesc, "rtf": rate / SR, "config": {"workload": desc, "frames": F, "samples": T, "receptive_field": rf},
        "cpu_baseline": {"value": rate, "unit": "samples/s", "cores": threads, "kind": "port",
                         "sample": f"{n} consecutive steady-state samples of the 2-s utterance (each = one teacher evaluation over its {rf}-sample "
                                   f"receptive field, naive recompute); the whole utterance extrapolates to {T / rate:.0f} s of CPU"},
        "e2e": {"value": rate, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "utterance_seconds_extrapolated": T / rate, "gpu_launches": 0, "finite": bool(torch.isfinite(x).all()),
    }
    print(json.dumps(line), flush=True)


def run_api1(args, desc, rank, local):
    """Batch-1 latency - the reference API's only call shape (`TTSCube.__call__` synthesises ONE utterance per call,
    cube/api.py:45-66; the frontend is batch-1 by construction, cube/networks/modules.py:945-953): one utterance of 2 s and
    of 10 s through each vocoder, host mel in -> host int16/float audio out (`forward_host`) and device-resident.
    Reports the median latency, the real-time factor and how many tiles each HiFi-GAN stage offers the 148 SMs."""
    if rank != 0:
        return
    import tts_cube_b200 as cube
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    out = {}
    iters = args.steps
    for arch in ("hifigan", "student"):
        weights, wdesc = load_weights(arch)
        if arch == "student":
            voc = cube.ParallelWaveNetVocoder(weights[0], weights[1]).to(dev)
            hop = 256
        else:
            voc = cube.CubeGenerator(weights[1]).to(dev)
            voc.load_state_dict(weights[0])
            hop = 240
        for secs in (2.0, 10.0):
            F = int(round(secs * SR / hop))
            T = voc.out_len(F)
            mel, z = synth_inputs(arch, 1, F, seed=4321)
            mel_d, z_d = mel.to(dev), (z.to(dev) if z is not None else None)
            mel_h, z_h = mel.pin_memory(), (z.pin_memory() if z is not None else None)
            out_h = torch.empty(1, T, dtype=torch.float32).pin_memory()
            call_d = (lambda: voc(mel_d, z_d)) if arch == "student" else (lambda: voc(mel_d))
            call_h = (lambda: voc.forward_host(mel_h, z_h, out=out_h)) if arch == "student" else (lambda: voc.forward_host(mel_h, out=out_h))
            with torch.no_grad():
                for _ in range(max(3, args.warmup)):
                    call_d(); call_h()
                torch.cuda.synchronize()
                dts, hts = [], []
                for _ in range(iters):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(); call_d(); e1.record(); torch.cuda.synchronize()
                    dts.append(e0.elapsed_time(e1))
                    t0 = time.perf_counter(); call_h(); hts.append(1e3 * (time.perf_counter() - t0))
            d_ms, h_ms = statistics.median(dts), statistics.median(hts)
            out[f"{arch}_{int(secs)}s"] = {"frames": F, "samples": T, "device_ms": d_ms, "host_e2e_ms": h_ms,
                                           "rtf_device": (T / SR) / (d_ms / 1e3), "rtf_host_e2e": (T / SR) / (h_ms / 1e3),
                                           "launches": voc._ensure().launches()}
        del voc
        torch.cuda.empty_cache()
    # HiFi-GAN stage occupancy at B=1, 10 s: scheduled tiles per launch vs 148 SMs (neb-noft rates [3,5,4,4])
    L, occ = int(round(10.0 * SR / 240)), {}
    for i, (u, k) in enumerate(zip(HIFIGAN_NEB_CONFIG["upsample_rates"], HIFIGAN_NEB_CONFIG["upsample_kernel_sizes"])):
        L = (L - 1) * u - 2 * ((k - u) // 2) + k
        ch = 512 >> (i + 1)
        rows = {256: 128, 128: 128, 64: 256, 32: 512}[ch]
        occ[f"stage{i}_{ch}ch"] = {"rows": L, "tiles_unfused": (L + rows - 1) // rows,
                                   "tiles_fused_step_k11": (L + rows - 11) // (rows - 10) if ch <= 64 else None}
    ref = out["hifigan_10s"]
    print(json.dumps({
        "metric": "audio samples/sec", "value": ref["samples"] / (ref["device_ms"] / 1e3), "unit": "samples/s", "n_gpus": 1, "steps": iters,
        "warmup": max(3, args.warmup), "ms_per_step": ref["device_ms"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32 in/out; tcgen05 split-fp16", "data": "synthetic; shipped checkpoints when staged", "rtf": ref["rtf_device"],
        "config": {"workload": desc, "headline": "hifigan_10s (value / ms_per_step); every case under `cases`"},
        "e2e": {"value": ref["samples"] / (ref["host_e2e_ms"] / 1e3), "unit": "samples/s", "h2d_bytes_per_step": 80 * ref["frames"] * 4,
                "d2h_bytes_per_step": ref["samples"] * 4, "copies_declared": True},
        "cases": out, "sm_tiles_at_batch1_10s": occ, "gpu_launches": ref["launches"] * iters, "lib": cube.build_info()}), flush=True)


def _standin_frontend(dev, seed=7):
    """A PyTorch stand-in with the SHAPE of the reference frontend (Languasito2: phoneme embedding -> char CNN -> BiLSTM ->
    durations -> frame expansion -> BiLSTM -> 80-d conditioning; cube/networks/modules.py:805-1009).  The reference module
    itself is not on the GPU box and its published weights are download-only, so configs[4] is measured with this
    seeded random-init module of the same structure and size class; it runs per utterance (batch 1), as the reference
    frontend does (modules.py:945-953).  Durations are a seeded function of the phoneme ids (3-12 frames each)."""
    import torch.nn as nn
    torch.manual_seed(seed)

    class Frontend(nn.Module):
        def __init__(self):
            super().__init__()
            self.emb = nn.Embedding(64, 256)
            self.cnn = nn.Sequential(*[m for _ in range(3) for m in (nn.Conv1d(256, 256, 5, padding=2), nn.ReLU())])
            self.rnn_char = nn.LSTM(256, 256, num_layers=2, bidirectional=True, batch_first=True)
            self.rnn_overlay = nn.LSTM(512, 256, num_layers=2, bidirectional=True, batch_first=True)
            self.rnn_cond = nn.LSTM(512, 256, num_layers=1, bidirectional=True, batch_first=True)
            self.out = nn.Linear(512, 80)

        def forward(self, ids):                                   # ids [1, P] -> conditioning [1, F, 80]
            h = self.cnn(self.emb(ids).permute(0, 2, 1)).permute(0, 2, 1)
            h, _ = self.rnn_char(h)
            dur = 3 + (ids[0] * 7 + torch.arange(ids.shape[1], device=ids.device)) % 10
            h = torch.repeat_interleave(h, dur, dim=1)
            h, _ = self.rnn_overlay(h)
            h, _ = self.rnn_cond(h)
            return self.out(h)

    return Frontend().to(dev).eval()


def run_e2e(args, desc, rank, world, local):
    """BASELINE configs[4]: phoneme strings -> PyTorch frontend (per utterance) -> CUDA vocoder -> int16 audio on the host
    of rank 0.  The strings are sharded over the ranks (LPT by length), every rank runs frontend + vocoder on its share,
    the int16 audio is gathered by NCCL point-to-point.  Weak/strong: the 128 strings are fixed (strong scaling)."""
    import torch.distributed as dist
    import tts_cube_b200 as cube
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    weights, wdesc = load_weights("hifigan")
    voc = cube.CubeGenerator(weights[1]).to(dev)
    voc.load_state_dict(weights[0])
    fe = _standin_frontend(dev)
    n_utt = args.batch or 128
    g = torch.Generator().manual_seed(1234 + 5)
    lens = torch.randint(20, 121, (n_utt,), generator=g).tolist()          # 20-120 phonemes per string
    strings = [torch.randint(1, 64, (1, n), generator=g) for n in lens]
    plan = cube.lpt_shard(lens, world)
    mine = plan[rank]

    def step():
        with torch.no_grad():
            conds = [fe(strings[i].to(dev))[0].t() for i in mine]         # [80, F_i]
            # local vocoding (no scatter: the strings were sharded before the frontend), int16 epilogue, gather to rank 0
            from tts_cube_b200.api import _run_local
            wavs = _run_local(lambda m, f: voc(m, f), conds, None, voc.out_len, dev, 64, 64 * 1400)
            a16 = [cube.heads.wav_to_int16(w) for w in wavs]
            n_samples = sum(int(w.numel()) for w in a16)
            if world > 1:
                flat = torch.cat(a16) if a16 else torch.zeros(0, dtype=torch.int16, device=dev)
                sizes = [torch.zeros(1, dtype=torch.int64, device=dev) for _ in range(world)]
                dist.all_gather(sizes, torch.tensor([flat.numel()], dtype=torch.int64, device=dev))
                host = None
                if rank == 0:      # NCCL has no int16: the audio travels as bytes
                    bufs = [torch.empty(2 * int(sz), dtype=torch.uint8, device=dev) for sz in sizes[1:]]
                    ops = [dist.P2POp(dist.irecv, b_, r + 1) for r, b_ in enumerate(bufs) if b_.numel()]
                    for w_ in (dist.batch_isend_irecv(ops) if ops else []):
                        w_.wait()
                    host = [flat.cpu()] + [b_.view(torch.int16).cpu() for b_ in bufs]
                elif flat.numel():
                    for w_ in dist.batch_isend_irecv([dist.P2POp(dist.isend, flat.view(torch.uint8), 0)]):
                        w_.wait()
            else:
                host = [torch.cat(a16).cpu()]
            return n_samples, host

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        n_local, host = step()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        n_local, host = step()
    barrier()
    dt = time.perf_counter() - t0
    t = torch.tensor([dt, float(n_local)], device=dev, dtype=torch.float64)
    if world > 1:
        tm = t.clone(); dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        ts = t.clone(); dist.all_reduce(ts, op=dist.ReduceOp.SUM)
        dt, total = float(tm[0]), float(ts[1])
    else:
        total = float(n_local)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0:
        value = total * args.steps / dt
        if args.dump_outputs:        # rank 0's int16 audio of every string, concatenated in shard order
            dump_outputs(args.dump_outputs, {"audio_int16": torch.cat(host)})
        print(json.dumps({
            "metric": "audio samples/sec", "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32 in/out; tcgen05 split-fp16 x3 (vocoder); f32 cuDNN (frontend)", "data": "synthetic phoneme ids; frontend = seeded stand-in of the reference frontend's structure; " + wdesc,
            "rtf": value / 24000.0, "config": {"workload": desc, "strings": n_utt, "phonemes_min_max": [min(lens), max(lens)],
                                              "seconds_of_audio": total / 24000.0, "parallelism": f"dp{world}: strings sharded by LPT before the frontend; NCCL p2p gather of int16 audio"},
            "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": int(sum(lens) * 8), "d2h_bytes_per_step": int(total * 2), "copies_declared": True,
                    "note": "wall clock, host phoneme ids in -> host int16 audio out, max over ranks"},
            "gpu_launches": voc._ensure().launches() * args.steps, "clocks": clocks, "lib": cube.build_info()}), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_ragged(args, desc, rank, world, local):
    """configs[3]: rank 0 owns 256 variable-length mels; tts_cube_b200.synthesize shards them (LPT), scatters the
    padded mel blocks, every rank vocodes its shard, rank 0 gathers the audio.  Strong scaling: the work is fixed."""
    import torch.distributed as dist
    import tts_cube_b200 as cube
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    weights, wdesc = load_weights("hifigan")
    voc = cube.CubeGenerator(weights[1]).to(dev)
    voc.load_state_dict(weights[0])
    g = torch.Generator().manual_seed(1234 + 3)
    n_utt = args.batch or 256
    secs = torch.empty(n_utt).uniform_(2.0, 15.0, generator=g)
    frames = [int(round(float(s_) * SR / 240)) for s_ in secs]
    mels = None
    if rank == 0:
        big = synthetic_logmel(1, max(frames), seed=77)[0]
        mels = [torch.roll(big, shifts=37 * i, dims=1)[:, :f].contiguous().to(dev) for i, f in enumerate(frames)]
    total = sum(voc.out_len(f) for f in frames)
    emu = args.emulate_world if (world == 1 and args.emulate_world > 1) else 0
    if emu:                                   # one rank's share of an `emu`-GPU run, no communication
        shard = cube.lpt_shard(frames, emu)[0]
        mels = [mels[i] for i in shard]
        frames = [frames[i] for i in shard]
        total = sum(voc.out_len(f) for f in frames)
        n_utt = len(frames)

    stats = {}

    def step():
        with torch.no_grad():
            return cube.synthesize(voc, mels, device=dev, max_batch=64, max_frames=64 * 1400, stats=stats)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        out = step()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches = 0
    barrier()
    ev0.record()
    for _ in range(args.steps):
        out = step()
        launches += voc._ensure().launches()
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t[0])
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0:
        assert all(o.numel() == voc.out_len(f) for o, f in zip(out, frames))
        if args.dump_outputs:        # the waveform of every utterance, concatenated in input order
            dump_outputs(args.dump_outputs, {"wav": torch.cat([o.reshape(-1) for o in out])})
        value = total * args.steps / (ms / 1e3)
        plan = cube.lpt_shard(frames, world)
        loads = [sum(frames[i] for i in p_) for p_ in plan]
        print(json.dumps({
            "metric": "audio samples/sec", "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic; " + wdesc, "rtf": value / SR,
            "config": {"workload": desc + (f" [rank 0's LPT shard of an emulated {emu}-GPU run, on one GPU]" if emu else ""), "utterances": n_utt,
                       "total_seconds_of_audio": total / SR, "frames_min_max": [min(frames), max(frames)], "emulated_world": emu or None,
                       "batches": [len(b_) for b_ in cube.api.make_batches(sorted(range(len(frames)), key=lambda i: -frames[i]), frames, 64, 64 * 1400)],
                       "parallelism": f"dp{world}: LPT shards (max/mean load {max(loads) / (sum(loads) / world):.3f}), NCCL p2p scatter of mel / gather of audio",
                       "l2": "per-step working set >> 126 MB L2"},
            "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                    "note": "device-resident lists in, device-resident lists out (rank 0); includes padding, scatter, gather"},
            "collective": {"kind": "NCCL point-to-point only (batch_isend_irecv): rank 0 -> r padded mel blocks, r -> rank 0 audio blocks",
                           "host_phase_seconds_last_step": {k: v for k, v in stats.items() if k.endswith("_s")},
                           "scatter_bytes": stats.get("scatter_bytes"), "gather_bytes": stats.get("gather_bytes"),
                           "batches_per_rank": stats.get("batches_per_rank")},
            "gpu_launches": launches, "clocks": clocks, "lib": cube.build_info()}))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cube", choices=["cube", "reference"])
    ap.add_argument("--workload", default="pwn", choices=list(WORKLOADS))
    ap.add_argument("--math", default="auto", choices=["auto", "simt", "tc"])
    ap.add_argument("--batch", type=int, default=0, help="override the per-GPU batch (debug)")
    ap.add_argument("--frames", type=int, default=0, help="override frames per utterance (debug)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--emulate-world", type=int, default=0,
                    help="ragged workload on ONE GPU: vocode only rank 0's LPT shard of a world of this size (what one rank of an N-GPU run computes)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path returned in its last timed step as DIR/<name>.npy (float32, at most 64 MB; "
                         "a fixed seeded sample of larger outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "cube" or args.workload not in DUMP_WORKLOADS):
        ap.error(f"--dump-outputs needs --impl cube and one of the workloads {', '.join(DUMP_WORKLOADS)}")
    arch, B, F, desc = WORKLOADS[args.workload]
    B = args.batch or B
    F = args.frames or F
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.workload == "teacher_cpu":
        run_teacher_cpu(args, desc, rank)
        return
    if args.impl == "reference":
        run_reference(args, arch, B, F, desc, rank, world)
        return
    args.warmup = max(args.warmup, 3)
    if args.workload == "ragged":
        run_ragged(args, desc, rank, world, local)
        return
    if args.workload == "api1":
        run_api1(args, desc, rank, local)
        return
    if args.workload == "e2e":
        run_e2e(args, desc, rank, world, local)
        return

    import torch.distributed as dist
    import tts_cube_b200 as cube
    from tts_cube_b200 import _lib
    assert torch.cuda.is_available(), "bench.py --impl cube needs a CUDA device (no CPU fallback)"
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    # auto: tensor cores (split-fp16 x3) for the dense layers of both vocoders
    math = {"auto": _lib.MATH_TC_SPLIT16, "simt": _lib.MATH_FP32_SIMT, "tc": _lib.MATH_TC_SPLIT16}[args.math]
    weights, wdesc = load_weights(arch)
    if arch == "student":
        voc = cube.ParallelWaveNetVocoder(weights[0], weights[1], math=math).to(dev)
    else:
        voc = cube.CubeGenerator(weights[1], math=math).to(dev)
        voc.load_state_dict(weights[0])
    T = voc.out_len(F)
    samples_per_step = B * T
    # two input sets, alternated, resident in HBM; the per-step working set (activations, GBs) is far
    # larger than the 126 MB L2, so nothing survives in L2 from one step to the next
    sets = []
    for k in range(2):
        mel, z = synth_inputs(arch, B, F, seed=1234 + 10 * rank + k)
        sets.append((mel.to(dev), z.to(dev) if z is not None else None, mel.pin_memory(), z.pin_memory() if z is not None else None))
    handle = voc._ensure()

    def step(k):
        mel, z, _, _ = sets[k & 1]
        return voc(mel, z) if arch == "student" else voc(mel)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.no_grad():
        for k in range(args.warmup):
            y = step(k)
        barrier()
        handle.set_profile(True)
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        launches, prof = 0, {}
        barrier()
        ev0.record()
        for k in range(args.steps):
            y = step(k)
            launches += handle.launches()
        ev1.record()
        barrier()
        ms = ev0.elapsed_time(ev1)
        prof = handle.get_profile()       # per-layer-class device time of the LAST timed step
        n_launch_last = handle.launches()
        handle.set_profile(False)
        clocks = sampler.stop() if rank == 0 else None
        # ---- end to end through the host-buffer C-ABI call (H2D + forward + D2H per step) ----
        out_host = torch.empty(B, T, dtype=torch.float32).pin_memory()
        for k in range(2):
            _, _, mh, zh = sets[k & 1]
            voc.forward_host(mh, zh, out=out_host) if arch == "student" else voc.forward_host(mh, out=out_host)
        barrier()
        t0 = time.perf_counter()
        for k in range(args.steps):
            _, _, mh, zh = sets[k & 1]
            voc.forward_host(mh, zh, out=out_host) if arch == "student" else voc.forward_host(mh, out=out_host)
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - t0
    t = torch.tensor([ms, e2e_s * 1e3], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, e2e_ms = float(t[0]), float(t[1])
    assert bool(torch.isfinite(y).all()), "non-finite audio"
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, {"wav": y})
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    pk = peaks()
    total = samples_per_step * world * args.steps
    value = total / (ms / 1e3)
    e2e_val = total / (e2e_ms / 1e3)
    h2d = sets[0][2].numel() * 4 + (sets[0][3].numel() * 4 if sets[0][3] is not None else 0)
    d2h = out_host.numel() * 4
    # ---- roofline of the dominant kernel (device time of its launches inside the last timed step) ----
    if arch == "student":
        fused = prof.get("block_fused", 0.0) > 0.0
        dom = "block_fused" if fused else "gate"
        nlaunch = sum(int(weights[0][k].shape[0] > 0) for k in weights[0] if k.endswith("filter_conv.conv.bias"))
        dom_ms = prof.get(dom, 0.0)
        flops_launch = (BLOCK_FLOPS if fused else GATE_FLOPS) * samples_per_step
        ach = flops_launch * nlaunch / (dom_ms / 1e3) / 1e12 if dom_ms > 0 else None
        roof = {"kernel": "conv_tile_kernel<8,8,8,1> EPI_GATE (gated dilated conv k3 128->2x256 + conditioning 1x1 80->2x256, fp32 FFMA2)" if math == 0
                else ("tc::tc_block_kernel<PAIR, Q8> (whole residual block on a CTA pair: gated dilated conv + conditioning 1x1 -> o kept in smem "
                      "-> res/skip 1x1; tcgen05 cta_group::2 UMMA 256x256, hi*hi in fp16 + two 8-bit correction passes in GEMM1, TMA taps; "
                      "CUBE_TC_PAIR=0 / CUBE_TC_FP8=0 / CUBE_TC_AONCE select the single-CTA / three-fp16-pass / A-once variants)" if fused else
                      "tc::tc_conv_kernel TC_EPI_GATE (same layer on tcgen05: UMMA 128x256x16 f16, split-fp16 x3, TMA taps)"),
                "bound": "tensor", "achieved": ach, "peak": pk["tf_sust"], "unit": "TFLOP/s",
                "frac": (ach / pk["tf_sust"]) if ach else None,
                # dram__bytes_read.sum + dram__bytes_write.sum of one launch of the default kernel (CTA pair + 8-bit correction
                # passes), ncu --set full, round 2; only valid for the default geometry and switches
                "traffic": (FUSED_TRAFFIC if fused else 3.31e9) if (math == 1 and B == 8 and F == 862) else None,
                "traffic_source": ("profiles/r2_ncu_full_tc_block_pair.md (ncu --set full, one launch of the default block kernel: 2.83 GB read + 2.21 GB written)" if fused else
                                   "profiles/r1_ncu_full_tc_conv.md (ncu --set full, gate launch)"),
                "launches_per_step": nlaunch, "avg_launch_ms": dom_ms / max(1, nlaunch),
                "algorithmic_flops_per_launch": flops_launch, "algorithmic_bytes_per_launch": (BLOCK_BYTES if fused else GATE_BYTES) * samples_per_step,
                "share_of_step": dom_ms / (ms / args.steps) if ms > 0 else None,
                "peak_source": pk["src"] + " bf16 sustained (kernel timed inside a long step)",
                "math": "fp32 FFMA (no tensor cores)" if math == 0 else
                        ("tcgen05: fp16 hi*hi + 2 x 8-bit correction passes (GEMM1), split-fp16 x3 (GEMM2)"
                         if fused and os.environ.get("CUBE_TC_FP8", "1") != "0" else "tcgen05 split-fp16 x3")}
        whole = {"flops_per_sample": PWN_FLOPS_PER_SAMPLE, "bytes_per_sample": PWN_BYTES_PER_SAMPLE}
    else:
        dom = "rb"
        fused_ms = prof.get("rb_fused", 0.0)
        dom_ms = prof.get("rb_conv1", 0.0) + prof.get("rb_conv2", 0.0) + fused_ms
        fused_on = fused_ms > 0.0
        # 72 ResBlock convs; on the 32/64-channel stages a launch covers a whole step (conv1 -> lrelu -> conv2 -> + x)
        nlaunch = 36 + 18 if fused_on else 72
        # resblock convs: 95 % of layer-wise bytes, 96 % of FLOPs (SURVEY 8a H3)
        by = 0.95 * HIFI_BYTES_PER_SAMPLE * samples_per_step
        ach = by / (dom_ms / 1e3) / 1e9 if dom_ms > 0 else None
        roof = {"kernel": ("conv_tile_kernel (ResBlock dilated convs, fused lrelu/bias/residual, fp32 FFMA2)" if math == 0 else
                           ("tc::tc_rbstep_kernel<32|64> (one ResBlock step per launch on the narrow stages: conv1 -> lrelu -> conv2 -> + x, a1 kept in "
                            "shared memory) + tc::tc_conv_kernel<256|128> TC_EPI_CONV (wide stages); tcgen05, split-fp16 x3" if fused_on else
                            "tc::tc_conv_kernel<256|128|64|32> TC_EPI_CONV (ResBlock dilated convs on tcgen05, split-fp16 x3)")), "bound": "hbm",
                "achieved": ach, "peak": pk["hbm"], "unit": "GB/s", "frac": (ach / pk["hbm"]) if ach else None, "traffic": None,
                "launches_per_step": nlaunch, "avg_launch_ms": dom_ms / nlaunch, "algorithmic_bytes_per_launch": by / nlaunch,
                "algorithmic_bytes_per_step": by, "fused_step_ms": fused_ms if fused_on else None,
                "share_of_step": dom_ms / (ms / args.steps) if ms > 0 else None, "peak_source": pk["src"] + " copy bandwidth",
                "tensor_frac": 0.96 * HIFI_FLOPS_PER_SAMPLE * samples_per_step / (dom_ms / 1e3) / 1e12 / pk["tf_sust"] if dom_ms > 0 else None}
        whole = {"flops_per_sample": HIFI_FLOPS_PER_SAMPLE, "bytes_per_sample": HIFI_BYTES_PER_SAMPLE}
    whole["hbm_frac_whole_path"] = whole["bytes_per_sample"] * value / world / 1e9 / pk["hbm"]
    whole["tensor_frac_whole_path"] = whole["flops_per_sample"] * value / world / 1e12 / pk["tf_sust"]

    cpu, tgpu = None, None
    if not args.no_cpu_baseline and world == 1:
        with torch.no_grad():
            tgpu = torch_cuda_baseline(arch, weights, sets[0][0], sets[0][1])
    if not args.no_cpu_baseline and world == 1:      # rank 0 at N=1 only (the N>1 lines carry null)
        threads = best_cpu_threads(arch, weights)     # cached in /tmp by the reference arm when that ran first
        hop = 256 if arch == "student" else 240
        cb, frames = cpu_fit_sample(arch, weights, threads, F, n_calls=2, wall_budget_s=40.0, kind="baseline")   # = the warm-up call
        r2, n, dt = cpu_oracle_rate(arch, weights, frames, threads, cb)
        cpu = {"value": r2, "unit": "samples/s", "cores": threads, "kind": "port",
               "sample": f"B={cb} x {frames} frames ({n} samples, {dt:.1f} s of CPU) of the same synthetic workload; oracle port, torch CPU fp32, "
                         f"{threads} threads (fastest of {list(THREAD_CANDIDATES)}; {host_cpus()} usable CPUs)"}

    fp8_on = os.environ.get("CUBE_TC_FP8", "1") != "0" and os.environ.get("CUBE_TC_FUSED", "1") != "0"
    if math == 0:
        math_desc = "f32 (FFMA, no tensor cores)"
    elif arch == "student":
        math_desc = ("f32 in/out; tcgen05: fp16 hi*hi + 2 x fp8 (e4m3/e5m2) correction passes (GEMM1), split-fp16 x3 (GEMM2), f32 accumulate"
                     if fp8_on else "f32 in/out; tcgen05 split-fp16 x3 (hi*hi + hi*lo + lo*hi), f32 accumulate")
    else:
        math_desc = "f32 in/out; tcgen05 split-fp16 x3 (hi*hi + hi*lo + lo*hi), f32 accumulate"
    line = {
        "metric": "audio samples/sec", "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": math_desc, "data": "synthetic; " + wdesc,
        "rtf": value / SR, "rtf_per_gpu": value / SR / world,
        "config": {"workload": desc, "batch_per_gpu": B, "frames": F, "samples_per_utterance": T, "parallelism": f"dp{world} (utterance shards, no data-path collective)",
                   "l2": "per-step activation working set (GBs) >> 126 MB L2; two input sets alternated",
                   "math": math_desc},
        "e2e": {"value": e2e_val, "unit": "samples/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms / args.steps, "copies_declared": True,
                "api": "ParallelWaveNetVocoder.forward_host -> cube_voc_forward_host (pinned host buffers)" if arch == "student" else "CubeGenerator.forward_host -> cube_voc_forward_host"},
        "gpu_launches": launches, "launches_per_step": n_launch_last,
        "roofline": roof, "whole_path": whole, "layer_ms_last_step": prof, "cpu_baseline": cpu, "torch_cuda_baseline": tgpu, "clocks": clocks,
        "workspace_bytes": handle.workspace_bytes(), "lib": cube.build_info(),
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
