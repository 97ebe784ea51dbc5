#!/usr/bin/env python
"""Benchmark of the MFCC + modulation-spectrum hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): per GPU a batch of 1024 x 10 s 16 kHz mono
clips, 25 ms / 10 ms frames, 512-point FFT, 40 mel bands, 13 MFCC + delta +
MFCC-change curve + MFCC modulation spectrum.  One step = one pass of the whole
path over the batch.  ``value`` is audio-seconds per second with the PCM already
resident in HBM; ``e2e`` is the same work through the host-buffer C-ABI call
(pinned host PCM in, host features out, copies inside the timed region).

``--impl reference`` times the reference path's CPU arithmetic (the numpy/scipy
oracle -- librosa itself is not installable here, see DESIGN.md) on all host
cores for the same metric and config, on a bounded sample of the workload.
"""

from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SR = 16000
SECONDS = 10.0
N_SAMPLES = int(SR * SECONDS)
CLIPS = 1024
PARAMS = dict(tStep=0.01, winLen=0.025, n_fft=512, n_mels=40, n_mfcc=13)
METRIC = "audio-seconds/sec (MFCC+modulation spectrum)"
UNIT = "audio-s/s"
WORKLOAD = (
    "BASELINE configs[1]: 1024 x 10 s 16 kHz clips per GPU; win 400 / hop 160 / n_fft 512, 40 mel, "
    "13 MFCC + delta + MFCC-change (zero-phase Butterworth, gradient, norm) + modulation spectrum (1 s windows, 0.5 s hop)"
)


def config_dict(T: int = 1001) -> dict:
    """The workload description printed by BOTH arms (identical keys and values)."""
    return {
        "workload": WORKLOAD,
        "clips_per_gpu_per_step": CLIPS,
        "samples_per_clip": N_SAMPLES,
        "frames_per_clip": T,
        "sample_rate": SR,
        "n_fft": PARAMS["n_fft"],
        "win_length": int(PARAMS["winLen"] * SR),
        "hop_length": int(PARAMS["tStep"] * SR),
        "n_mels": PARAMS["n_mels"],
        "n_mfcc": PARAMS["n_mfcc"],
        "l2": "inputs are 655 MB per step per GPU, larger than the 126 MB L2 (no flush needed)",
    }


# --------------------------------------------------------------------------- CPU arm


def _cpu_init():
    try:
        from threadpoolctl import threadpool_limits

        threadpool_limits(1)
    except Exception:
        pass


_CPU_BATCH = None


def _cpu_one(i):
    import oracle

    f = oracle.mfcc_features(_CPU_BATCH[i], SR, **PARAMS)
    return float(f["totChange"][0])


def cpu_throughput(n_clips: int, repeats: int = 1, warmup: int = 0):
    """audio-s/s of the oracle over ``n_clips`` synthetic clips on all host cores."""
    global _CPU_BATCH
    import multiprocessing as mp

    from modulation_mfcc_b200.synth import synth_batch

    cores = os.cpu_count() or 1
    try:
        cores = len(os.sched_getaffinity(0))
    except Exception:
        pass
    _CPU_BATCH = synth_batch(0, n_clips, N_SAMPLES, SR)
    ctx = mp.get_context("fork")
    times = []
    with ctx.Pool(cores, initializer=_cpu_init) as pool:
        chunk = max(1, n_clips // (cores * 4))
        for r in range(warmup + repeats):
            t0 = time.perf_counter()
            pool.map(_cpu_one, range(n_clips), chunksize=chunk)
            dt = time.perf_counter() - t0
            if r >= warmup:
                times.append(dt)
    _CPU_BATCH = None
    return [n_clips * SECONDS / t for t in times], times, cores


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return None
    cores = os.cpu_count() or 1
    n_clips = CLIPS  # the full batch of one step (about 20 core-seconds of numpy/scipy work per step)
    vals, times, cores = cpu_throughput(n_clips, repeats=args.steps, warmup=args.warmup)
    total = sum(times)
    value = n_clips * SECONDS * len(times) / total
    sample = f"all {n_clips} clips of the workload per step (oracle.mfcc_features per clip, fork pool over all cores, BLAS threads = 1)"
    line = {
        "impl": "reference",
        "metric": METRIC,
        "value": value,
        "unit": UNIT,
        "n_gpus": args.gpus,
        "steps": args.steps,
        "warmup": args.warmup,
        "ms_per_step": 1e3 * total / len(times),
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "f32",
        "data": "synthetic",
        "config": config_dict(),
        "notes": {"arm": "CPU arm: the numpy/scipy restatement of the reference path, pinned bit for bit to the reference's own script/mfcc.py + calc.py (tests/test_reference_pin.py); librosa itself cannot be installed offline (DESIGN.md section 2)"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    return line


# --------------------------------------------------------------------------- clocks


class ClockSampler(threading.Thread):
    """Polls NVML for SM clock and throttle reasons while the timed region runs."""

    def __init__(self, index: int, period: float = 0.002):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self._stop_evt = threading.Event()
        self.armed = False  # the thread records only between arm() and stop(): samples taken while ranks wait at a
        self._names = {}    # barrier would put idle clocks into the median
        self.ok = False
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.nv = None

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4),
            "hw_power_brake": getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80),
        }
        self._names = names
        while not self._stop_evt.is_set():
            if self.armed:
                self.sample()
            time.sleep(self.period)

    def sample(self):
        """One reading of the SM clock and the throttle reasons (any thread)."""
        nv = self.nv
        try:
            self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
            try:
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
            except Exception:
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            for k, bit in self._names.items():
                if r & bit:
                    self.reasons.add(k)
        except Exception:
            pass

    def poll_until(self, event, period: float = 0.002):
        """Sample from the calling thread until the CUDA event has completed: the host enqueues a timed region far
        ahead of the GPU, so this loop runs while the kernels do -- it does not depend on the sampler thread getting
        the GIL (one run of this bench came back with a single sample in a 46 ms region)."""
        if not self.ok:
            return
        while not event.query():
            self.sample()
            time.sleep(period)

    def arm(self):
        self.armed = True

    def stop(self):
        self.armed = False
        self._stop_evt.set()
        self.join(timeout=2)
        med = statistics.median(self.samples) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# --------------------------------------------------------------------------- GPU arm


def _bind_to_gpu_numa_node(index: int):
    """Best effort: run this rank on the CPUs next to its GPU, so that the pinned staging buffers it allocates
    afterwards are NUMA-local to the GPU's PCIe root (first-touch policy)."""
    try:
        import pynvml

        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        n_words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, n_words)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (m >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


class PowerSampler(ClockSampler):
    """ClockSampler that also records board power."""

    def __init__(self, index, period=0.01):
        super().__init__(index, period)
        self.power = []

    def run(self):
        if not self.ok:
            return
        while not self._stop_evt.is_set():
            if self.armed:
                self.sample()
            time.sleep(self.period)

    def sample(self):
        nv = self.nv
        try:
            self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
            self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
        except Exception:
            pass


def run_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    import modulation_mfcc_b200 as mm

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    numa_cpus = _bind_to_gpu_numa_node(local)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return float(x)
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    lib = mm.lib()
    fx = mm.FeatureExtractor(SR, device=local, flags=int(os.environ.get("MMF_FLAGS", "0")), **PARAMS)
    plan, prm = fx.plan, fx.prm
    pcm = mm.synth_batch_device(CLIPS, N_SAMPLES, SR, seed=1234 + rank, device=dev)
    T = plan.num_frames(N_SAMPLES)
    Lw, Hw, nfft, bins = fx.modspec_geometry(T)
    n_win = 1 + (T - Lw) // Hw
    # Per-clip feature gather (north_star: the only cross-GPU traffic).  Every step's MFCC-change curves
    # [1024, T] f64 go to EVERY rank through NVLink peer memory, pushed by the copy engines right after the
    # step while the SMs run the next one (modulation_mfcc_b200.shard.PeerGather); the timed region ends only
    # when all ranks hold all steps' curves.  Rank-major rows: rank r owns [r*R, (r+1)*R), R = n_keep * CLIPS.
    n_keep = max(args.steps, args.warmup, 3)
    gather = None
    if world > 1:
        gather = mm.PeerGather(world * n_keep * CLIPS, (T,), torch.float64, dev,
                               force_collective=bool(int(os.environ.get("MMF_BENCH_NCCL_GATHER", "0"))))
        _GATHER_MODE["mode"] = ("copy-engine pushes over NVLink peer memory after each step, torch symmetric memory"
                                if gather.mode == "peer" else "one in-place NCCL all_gather_into_tensor at the end: " + gather.mode)

    k1_events, k6_events = [], []

    def step(record: bool, slot: int):
        if record:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        lm, cmax = plan.logmel(pcm)  # fused frame/window/rFFT/|X|^2/mel/log kernel (+ clip-max init)
        if record:
            e1.record()
            k1_events.append((e0, e1))
        res = plan.change_from_logmel(lm, cmax, prm, clamp_in_place=False)  # clamp+DCT+delta, IIR, derivative+norm, IIR
        if record:
            e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e2.record()
        mag, band = plan.modspec(res["mfcc"], Lw, Hw, nfft, bins)
        if record:
            e3.record()
            k6_events.append((e2, e3))
        if gather is not None:
            gather.push(res["totChange"], (rank * n_keep + slot % n_keep) * CLIPS)
        return res, mag, band

    for i in range(max(args.warmup, 3)):
        res_w = step(False, i)
    if gather is not None:
        # warm-up at the timed region's size: every slot of every peer's buffer is written once (first touches
        # of a peer mapping are slow), then the same finish() as the timed region
        for i in range(n_keep):
            gather.push(res_w[0]["totChange"], (rank * n_keep + i) * CLIPS)
        gather.finish()
    del res_w
    # the clock sampler (a thread polling NVML / nvidia-smi) is started BEFORE the barrier: starting it between the
    # barrier and the first event skews the ranks by milliseconds, and with a gather that ends on a device-side
    # barrier over all ranks every millisecond of start skew is billed to the ranks that started early (measured at
    # 8 GPUs: 1.08 ms per step in a 30-step region against 0.92 ms in the 2 s sustained loop of the same run)
    sampler = ClockSampler(local)
    sampler.start()
    lib.mmf_launch_count(1)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    barrier()
    sampler.arm()
    ev0.record()
    for i in range(args.steps):
        last = step(True, i)
    gathered = None
    if gather is not None:
        gathered = gather.finish()  # every rank's curves of every step have landed before the clock stops
    ev1.record()
    sampler.poll_until(ev1)
    torch.cuda.synchronize()
    barrier()
    launches = int(lib.mmf_launch_count(0))
    ms_total = max_over_ranks(ev0.elapsed_time(ev1))
    k1_ms = [a.elapsed_time(b) for a, b in k1_events]
    k6_ms = [a.elapsed_time(b) for a, b in k6_events]
    ms_step = ms_total / args.steps
    value = world * CLIPS * SECONDS / (ms_step * 1e-3)
    clocks = sampler.stop()
    # what a caller of the step receives, as the last timed step left it
    dev_res = {"totChange": last[0]["totChange"], "mfcc": last[0]["mfcc"], "delta": last[0]["delta"], "modspec": last[1], "band_energy": last[2]}
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dev_res)
    gather_ok = None
    if gather is not None:
        # the gathered block of this rank's last step must be the curve it computed
        row0 = (rank * n_keep + (args.steps - 1) % n_keep) * CLIPS
        gather_ok = bool(torch.equal(gathered[row0 : row0 + CLIPS], last[0]["totChange"]))
        peer = (rank + 1) % world
        gather_ok = gather_ok and bool(torch.isfinite(gathered[(peer * n_keep) * CLIPS : (peer * n_keep + 1) * CLIPS]).all())

    # ---- sustained: the same step back to back for >= 2 s (clocks and power settle; MEASURED_PEAKS' sustained figure)
    sustained = None
    if not args.no_sustained:
        n_sus = max(200, int(2.2 / (ms_step * 1e-3)))
        ps = PowerSampler(local)
        ps.start()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        barrier()
        ps.arm()
        s0.record()
        for i in range(n_sus):
            step(False, i)
        if gather is not None:
            gather.finish()
        s1.record()
        ps.poll_until(s1, 0.01)
        torch.cuda.synchronize()
        sus_ms = max_over_ranks(s0.elapsed_time(s1))
        pc = ps.stop()
        barrier()
        sustained = {
            "value": world * CLIPS * SECONDS * n_sus / (sus_ms * 1e-3),
            "unit": UNIT,
            "steps": n_sus,
            "seconds": sus_ms * 1e-3,
            "ms_per_step": sus_ms / n_sus,
            "sm_mhz": pc["sm_mhz"],
            "sm_max_mhz": pc["sm_max_mhz"],
            "power_w_median": statistics.median(ps.power) if ps.power else None,
            "power_w_max": max(ps.power) if ps.power else None,
        }

    # ---- end to end through the host-buffer C-ABI call (pinned host PCM in, host features out)
    pcm_host_t = torch.empty((CLIPS, N_SAMPLES), dtype=torch.float32, pin_memory=True)
    pcm_host_t.copy_(pcm)
    torch.cuda.synchronize()
    pcm_host = pcm_host_t.numpy()
    want = ("totChange", "mfcc", "delta", "modspec", "band_energy")
    shapes = {
        "totChange": ((CLIPS, T), torch.float64),
        "mfcc": ((CLIPS, 13, T), torch.float32),
        "delta": ((CLIPS, 13, T), torch.float32),
        "modspec": ((CLIPS, 13, n_win, nfft // 2 + 1), torch.float32),
        "band_energy": ((CLIPS, n_win, len(bins)), torch.float32),
    }
    pinned = {k: torch.empty(s, dtype=d, pin_memory=True) for k, (s, d) in shapes.items()}
    out = {k: v.numpy() for k, v in pinned.items()}
    e2e_steps = max(3, min(args.steps, 10))
    for _ in range(2):
        fx.host_call(pcm_host, want=want, out=out)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        fx.host_call(pcm_host, want=want, out=out)  # synchronous: returns when the results are in host memory
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    barrier()
    e2e_value = world * CLIPS * SECONDS * e2e_steps / e2e_s
    # outside the timed region: what the e2e call (14 chunks over two streams) left in host memory must be
    # bit-identical to the device-resident step
    e2e_verified = all(bool(torch.equal(torch.from_numpy(out[k]), dev_res[k].cpu())) for k in want)
    # raw H2D ceiling of this host for the same pinned buffer, all ranks copying at once
    h2d_buf = torch.empty_like(pcm)
    for _ in range(2):
        h2d_buf.copy_(pcm_host_t, non_blocking=True)
    torch.cuda.synchronize()
    barrier()
    t0 = time.perf_counter()
    for _ in range(5):
        h2d_buf.copy_(pcm_host_t, non_blocking=True)
    torch.cuda.synchronize()
    h2d_s = max_over_ranks(time.perf_counter() - t0)
    barrier()
    h2d_gbs = world * 5 * CLIPS * N_SAMPLES * 4 / h2d_s / 1e9
    del h2d_buf
    # extra (not the contract's `e2e`): the same call fed with 16-bit PCM as it sits in a WAV file --
    # half the H2D bytes, scaled to float32 on the device; inputs are the float batch quantised to int16
    pcm16_t = torch.empty((CLIPS, N_SAMPLES), dtype=torch.int16, pin_memory=True)
    pcm16_t.copy_(torch.clamp(torch.round(pcm * 32768.0), -32768, 32767).to(torch.int16))
    torch.cuda.synchronize()
    pcm16_host = pcm16_t.numpy()
    for _ in range(2):
        fx.host_call(pcm16_host, want=want, out=out)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        fx.host_call(pcm16_host, want=want, out=out)
    e16_s = max_over_ranks(time.perf_counter() - t0)
    barrier()
    e2e16_value = world * CLIPS * SECONDS * e2e_steps / e16_s
    h2d = CLIPS * N_SAMPLES * 4
    d2h = sum(int(np.prod(s)) * (8 if d == torch.float64 else 4) for s, d in shapes.values())
    del pcm_host_t, pcm16_t, pinned, out

    # ---- BASELINE configs[4]: the 100k-clip corpus, block-partitioned over the ranks (CorpusRunner)
    cfg5 = None
    if not args.no_cfg5:
        n_corpus = args.corpus_clips
        lo, hi = mm.shard_range(n_corpus, rank, world)
        free_b, _ = torch.cuda.mem_get_info(dev)
        need = (hi - lo) * N_SAMPLES * 4 + n_corpus * T * 8 + (6 << 30)
        gather = gathered = last = None
        torch.cuda.empty_cache()
        free_b, _ = torch.cuda.mem_get_info(dev)
        ok_mem = max_over_ranks(0.0 if need <= free_b else 1.0) == 0.0
        if ok_mem:
            shard = torch.empty((hi - lo, N_SAMPLES), device=dev, dtype=torch.float32)
            for b0 in range(0, hi - lo, CLIPS):  # stands in for the loader: not timed
                nb = min(CLIPS, hi - lo - b0)
                shard[b0 : b0 + nb] = mm.synth_batch_device(nb, N_SAMPLES, SR, seed=99 + lo + b0, device=dev)
            g5 = mm.PeerGather(n_corpus, (T,), torch.float64, dev) if world > 1 else None
            runner = mm.CorpusRunner(fx, n_corpus, N_SAMPLES, batch=CLIPS, rank=rank, world=world, gather=g5)
            # warm-up pass over the first batches (kernel attributes, allocator pools, peer mappings)
            warm = mm.CorpusRunner(fx, min(n_corpus, 2 * CLIPS * world), N_SAMPLES, batch=CLIPS, rank=rank, world=world)
            warm.run(shard[: warm.hi - warm.lo])
            torch.cuda.synchronize()
            barrier()
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            lib.mmf_launch_count(1)
            c0.record()
            runner.run(shard)
            full = runner.finish()
            c1.record()
            torch.cuda.synchronize()
            c_launch = int(lib.mmf_launch_count(0))
            c_ms = max_over_ranks(c0.elapsed_time(c1))
            barrier()
            # parity sample: one clip of this rank's shard against the single-clip call
            ref1 = fx(shard[:1], want_logmel=False)["totChange"][0]
            row = full[lo] if world > 1 else full[0]
            cfg5 = {
                "workload": f"BASELINE configs[4]: {n_corpus} x 10 s 16 kHz clips, contiguous block partition over {world} GPU(s), batches of {CLIPS}; per-clip MFCC-change curves gathered on every rank, modulation band energies kept per shard",
                "clips": n_corpus,
                "clips_on_rank0": hi - lo,
                "ms": c_ms,
                "value": n_corpus * SECONDS / (c_ms * 1e-3),
                "unit": UNIT,
                "us_per_clip_per_gpu": c_ms * 1e3 / max(1, (n_corpus + world - 1) // world),
                "gather": (g5.mode if g5 is not None else "none"),
                "gathered_shape": list(full.shape),
                "gathered_finite": bool(torch.isfinite(full).all()),
                "sample_matches_single_clip_call": bool(torch.equal(row, ref1)),
                "gpu_launches": c_launch,
                "scaling": "strong (fixed corpus)",
            }
            del shard, full, runner, warm, g5
        else:
            cfg5 = {"skipped": f"needs {need / 2**30:.0f} GiB of HBM on the largest shard, {free_b / 2**30:.0f} GiB free"}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return None

    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    # dominant kernel: fused STFT/mel.  Algorithmic bytes per launch = PCM in + log-mel out.
    alg_bytes = CLIPS * (4 * N_SAMPLES + 4 * PARAMS["n_mels"] * T)
    k1 = statistics.mean(k1_ms)
    achieved = alg_bytes / (k1 * 1e-3) / 1e9
    traffic = traffic_src = None
    try:
        with open(os.path.join(ROOT, "profiles", "stft_mel_traffic.json")) as f:
            tj = json.load(f)
            traffic = tj.get("dram_bytes_per_launch")
            traffic_src = "static: " + tj.get("source", "ncu --set full capture under profiles/ (not measured in this run)")
    except Exception:
        pass
    tc_mel = not (int(os.environ.get("MMF_FLAGS", "0")) & (4096 | 2048 | 16 | 2))
    k1_name = ("stft_mel_tc_kernel<12, 1> (fused frame/window/rFFT/|X|^2 on packed FP32 + mel projection as a tcgen05 bf16x2 "
               "GEMM over 128-frame blocks + log)") if tc_mel else "stft_mel_kernel<512, c2> (fused frame/window/rFFT/|X|^2/mel/log)"
    # the mel GEMM inside K1: per 128-frame block 17 K-slabs x {M128 N96 K16, M128 N48 K16} MMAs (bf16 operand pairs)
    mel_gemm_flops = CLIPS * ((T + 127) // 128) * 17 * (2 * 128 * 96 * 16 + 2 * 128 * 48 * 16) if tc_mel else 0
    # K6 (modulation spectrum): MFCC rows in + magnitudes + band energies out
    k6 = statistics.mean(k6_ms)
    k6_bytes = CLIPS * (4 * 13 * T + 4 * 13 * n_win * (nfft // 2 + 1) + 4 * n_win * len(bins))
    # whole step: compulsory bytes of the fused path (SURVEY section 8d "end-to-end compulsory" + log-mel is
    # NOT an output here): PCM in, MFCC + delta, modulation magnitudes + band energies, totChange f64 out
    step_bytes = CLIPS * (4 * N_SAMPLES + 8 * 13 * T + 4 * 13 * n_win * (nfft // 2 + 1) + 4 * n_win * len(bins) + 8 * T)

    cpu = None
    if world == 1 and not args.no_cpu:
        n_cpu = CLIPS  # the whole batch of one step: ~20 core-seconds of numpy/scipy work
        vals, times, cores = cpu_throughput(n_cpu, repeats=1, warmup=0)
        cpu = {
            "value": vals[0],
            "unit": UNIT,
            "cores": cores,
            "kind": "port",
            "sample": f"{n_cpu} clips of the same workload (oracle.mfcc_features per clip, fork pool over all {cores} cores, BLAS threads = 1), {times[0]:.2f} s wall",
        }

    line = {
        "metric": METRIC,
        "value": value,
        "unit": UNIT,
        "n_gpus": world,
        "steps": args.steps,
        "warmup": max(args.warmup, 3),
        "ms_per_step": ms_step,
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "f32",
        "data": "synthetic",
        "config": config_dict(T),
        "notes": {
            "collective": (f"per-clip MFCC-change curves of every step land on every rank inside the timed region ({gather_mode(world)})" if world > 1 else "none"),
            "gather_verified": gather_ok,
            "fp64_stages": "zero-phase Butterworth and derivative/norm run in f64; the modulation spectrum is a tcgen05 GEMM (fp16 operand pairs, f32 accumulate)",
            "numa_cpus_bound": numa_cpus,
        },
        "clocks": clocks,
        "e2e": {
            "value": e2e_value,
            "unit": UNIT,
            "h2d_bytes_per_step": h2d,
            "d2h_bytes_per_step": d2h,
            "steps": e2e_steps,
            "call": "mmf_features_host (one C-ABI call per step, pinned host buffers)",
            "verified_bit_identical_to_device_path": e2e_verified,
            "h2d_ceiling_gbs_all_ranks": h2d_gbs,
            "h2d_achieved_gbs_all_ranks": world * e2e_steps * h2d / e2e_s / 1e9,
        },
        "e2e_pcm16": {
            "value": e2e16_value,
            "unit": UNIT,
            "h2d_bytes_per_step": CLIPS * N_SAMPLES * 2,
            "d2h_bytes_per_step": d2h,
            "steps": e2e_steps,
            "call": "mmf_features_host_pcm16 (int16 WAV samples in, scaled on the device; extra, not the headline)",
        },
        "gpu_launches": launches,
        "roofline": {
            "kernel": k1_name,
            "bound": "hbm",
            "achieved": achieved,
            "peak": hbm_peak,
            "unit": "GB/s",
            "frac": achieved / hbm_peak,
            "traffic": traffic,
            "traffic_source": traffic_src,
            "peak_source": peak_src,
            "algorithmic_bytes_per_launch": alg_bytes,
            "kernel_ms": k1,
            "kernel_share_of_step": k1 / ms_step,
            "tensor_pipe": {
                "what": "mel projection GEMM issued inside this kernel (tcgen05.mma kind::f16, bf16 operand pairs, fp32 accumulate in TMEM)",
                "flops_per_launch": mel_gemm_flops,
                "achieved_tflops": mel_gemm_flops / (k1 * 1e-3) / 1e12,
                "peak_tflops": float(peaks.get("bf16_tflops", 1680.0)),
                "frac": mel_gemm_flops / (k1 * 1e-3) / 1e12 / float(peaks.get("bf16_tflops", 1680.0)),
                "note": "the GEMM is 4 % of the kernel's work and runs underneath the transform; ncu: tensor pipe 6 % active",
            } if tc_mel else None,
        },
        "roofline_k6": {
            "kernel": "modspec_tc_kernel<128, 7> (modulation spectrum, tcgen05 GEMM)",
            "bound": "hbm",
            "achieved": k6_bytes / (k6 * 1e-3) / 1e9,
            "peak": hbm_peak,
            "unit": "GB/s",
            "frac": k6_bytes / (k6 * 1e-3) / 1e9 / hbm_peak,
            "algorithmic_bytes_per_launch": k6_bytes,
            "kernel_ms": k6,
        },
        "roofline_step": {
            "what": "whole step, compulsory bytes (PCM in; MFCC, delta, modulation magnitudes, band energies, totChange out)",
            "bound": "hbm",
            "achieved": step_bytes / (ms_step * 1e-3) / 1e9,
            "peak": hbm_peak,
            "unit": "GB/s",
            "frac": step_bytes / (ms_step * 1e-3) / 1e9 / hbm_peak,
            "algorithmic_bytes_per_step": step_bytes,
        },
        "sustained": sustained,
        "cfg5": cfg5,
        "cpu_baseline": cpu,
    }
    if world > 1:
        dist.destroy_process_group()
    return line


DUMP_CLIPS = 256  # the whole step's outputs are about 180 MB; this many clips keep a dump near 45 MB


def dump_outputs(out_dir: str, outputs: dict) -> None:
    """Write each output of the step as ``out_dir/<name>.npy`` for the same fixed, seeded sample of clips
    (sorted indices from ``numpy.random.default_rng(0)``), so that two builds can be compared array for array."""
    import numpy as np
    import torch

    os.makedirs(out_dir, exist_ok=True)
    rows = np.sort(np.random.default_rng(0).choice(CLIPS, DUMP_CLIPS, replace=False))
    for name, t in outputs.items():
        sample = t.index_select(0, torch.from_numpy(rows).to(t.device)).cpu().numpy()
        assert sample.dtype in (np.float32, np.float64), (name, sample.dtype)
        np.save(os.path.join(out_dir, name + ".npy"), sample)


_GATHER_MODE = {"mode": "none"}


def gather_mode(world):
    return _GATHER_MODE["mode"]


class _StdoutToStderr:
    """Everything written to fd 1 while the bench runs (NCCL's version banner, library chatter)
    goes to stderr, so that stdout carries exactly one line: the JSON result."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)
        return False


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-sustained", action="store_true", help="skip the >= 2 s sustained-clock leg")
    ap.add_argument("--no-cfg5", action="store_true", help="skip the 100k-clip corpus leg (BASELINE configs[4])")
    ap.add_argument("--corpus-clips", type=int, default=100_000)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help=f"write the last timed step's outputs for {DUMP_CLIPS} fixed clips of rank 0's batch as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the b200 path computed")
    with _StdoutToStderr():
        line = run_reference(args) if args.impl == "reference" else run_b200(args)
    if line is not None:
        print(json.dumps(line), flush=True)
    return 0


if __name__ == "__main__":
    sys.exit(main())
