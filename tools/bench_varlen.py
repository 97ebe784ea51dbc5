#!/usr/bin/env python
"""Clips of different lengths through the MFCC-change path (leg "change") and through the whole feature bundle
(leg "features"), three ways each:

  * varlen: one mmf_mfcc_change_varlen call over the padded batch;
  * loop:   one mmf_mfcc_change call per clip;
  * padded: mmf_mfcc_change over the batch zero-padded to the longest clip (what a caller without the varlen call
            would run; its tails are not the single-clip results).

The features leg runs FeatureExtractor with its defaults (log-mel, MFCC, delta, totChange, and the modulation
spectrum at 1 s / 0.5 s windows: the tcgen05 kernel, the clip kernel for the few window counts it declines): FeatureExtractor.varlen, a loop of one FeatureExtractor call
per clip, and one call over the zero-padded batch (whose windows past a clip's end are spectra of the padding).

The host leg times the host-buffer bundle (every output of FeatureExtractor.host_call) once with float32 and once
with int16 samples, three ways: FeatureExtractor.host_varlen on a pinned packed buffer, host_call on the pinned batch
zero-padded to 20 s, and mfcc_features_many on the list of numpy clips (float32: it takes no int16).  Outputs of the
first two land in pinned arrays.  One pinned host-to-device copy of the packed bytes is timed as the ceiling.  Host
calls end in a synchronise, so a host clock times them.  Each way reports its median ms, audio-s/s and the bytes it
moves each way over PCIe.

The resample leg feeds 1024 int16 clips of 2-20 s at 44.1 kHz (pinned) to FeatureExtractor's defaults at 16 kHz:
one host_varlen(rates=) call, which resamples on the device inside the bundle, against the route before it (each
clip scaled and resampled on the device as the WAV loader does, copied back, then one host_many call).  It also
times the resampler kernels over the same clips with torch.profiler: Plan.resample_poly per clip (whatever kernel
the tree's mmf_resample_poly launches, so the leg can time an older tree too) and, where the tree has it, one
mmf_resample_varlen launch over all of them; and one pinned copy of the packed int16 bytes, against which the
call's own time shows whether resampling and features stay under the copy.

The amplitude leg adds the RMS envelope (FeatureExtractor's amp_* defaults: 0.1 s window, 0.01 s hop, centred) to
host_varlen(want=every output) on the resample leg's corpus (with rates=) and on the host leg's 16 kHz float32 corpus:
the call without it, with the raw envelope and with the 'iir' output filter.  It also times the route without the
bundle, calculate_amplitude_envelope per clip at its native rate, and with torch.profiler the envelope kernels over
the same clips: one mmf_rms_varlen launch, and Plan.rms per clip (whatever kernel the tree's mmf_rms launches).

The hilbert leg times the Hilbert envelope ('Hilb') of the 16 kHz float32 corpus on the device: one
mmf_hilbert_varlen call over the packed clips against Plan.hilbert_envelope per clip (whatever kernels the tree's
mmf_hilbert_envelope launches, so the leg can time an older tree too), as CUDA-event wall time and as kernel time from
torch.profiler.  Where the tree has it, it then times host_varlen(want=every output) on the resample leg's int16
44.1 kHz corpus (with rates=) without the envelope and with amp_method='Hilb', raw and with the 'iir' output filter.

The outfilter leg times the 'fir' (21 taps, 10 Hz) and 'sg' (11 points, order 3) output filters on the 100 Hz curves
and envelopes of the 16 kHz float32 corpus: get_MFCCS_change_many at the bench's frame geometry and
calculate_amplitude_envelope_many (RMS), each also without an output filter, so that the difference is the filter's
cost (a per-clip loop in a tree without mmf_filter_varlen, one ragged call with it).  Where FeatureExtractor takes
outFilter, it then times host_varlen(want=every output) on the resample leg's int16 44.1 kHz corpus (with rates=)
with outFilter None, 'iir' (12 Hz, order 6), 'fir' and 'sg'.

Workload: 1024 clips at 16 kHz with the bench's frame geometry (win 400 / hop 160 / n_fft 512, 40 mel, 13 MFCC,
gradient, Butterworth output filter), lengths uniform in [2 s, 20 s] from a fixed seed.  Prints, per leg, the median
ms of each way and audio-seconds per second as one JSON line, with the GPU's name and power limit.

    python tools/bench_varlen.py [--clips 1024] [--iters 10] [--loop-iters 3]
                                 [--legs change,features,host,resample,amplitude,hilbert,outfilter]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import scipy.signal
import torch

import modulation_mfcc_b200 as mm


def _median_ms(fn, iters):
    times = []
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    return float(np.median(times))


def _median_host_ms(fn, iters):
    times = []
    for _ in range(iters):
        t0 = time.perf_counter()
        fn()
        times.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(times))


def _pinned(shape, dtype):
    t = torch.empty(shape, dtype={np.float32: torch.float32, np.float64: torch.float64, np.int16: torch.int16}[dtype],
                    pin_memory=True)
    return t.numpy()


def _host_leg(fx, pcm, lengths, sr, iters, power_limit, dev):
    """One JSON line per input type; see the module docstring."""
    want = ("totChange", "mfcc", "delta", "modspec", "band_energy")
    B, n_max = pcm.shape
    host = pcm.cpu().numpy()
    clips = [host[i, : lengths[i]] for i in range(B)]
    offsets = np.zeros(B + 1, np.int64)
    np.cumsum(lengths, out=offsets[1:])
    audio_s = sum(lengths) / sr
    for dt in (np.float32, np.int16):
        if dt == np.int16:
            clips_t = [np.clip(np.round(c * 32768.0), -32768, 32767).astype(np.int16) for c in clips]
            floats = [c.astype(np.float32) / 32768.0 for c in clips_t]
        else:
            clips_t = clips
            floats = clips
        packed = _pinned((int(offsets[-1]),), dt)
        padded = _pinned((B, n_max), dt)
        padded[:] = 0
        for i, c in enumerate(clips_t):
            packed[offsets[i] : offsets[i + 1]] = c
            padded[i, : lengths[i]] = c
        # pinned outputs shaped by a first (warm-up) call
        out_v = {k: v for k, v in fx.host_varlen(packed, offsets, want=want).items() if k in want}
        out_v = {k: _pinned(v.shape, v.dtype.type) for k, v in out_v.items()}
        out_p = {k: _pinned(v.shape, v.dtype.type) for k, v in fx.host_call(padded, want=want).items()}
        mm.mfcc_features_many(floats, sr)
        ways = {
            "host_varlen": lambda: fx.host_varlen(packed, offsets, want=want, out=out_v),
            "host_padded": lambda: fx.host_call(padded, want=want, out=out_p),
            "many": lambda: mm.mfcc_features_many(floats, sr),
        }
        dev_out = fx.varlen(torch.zeros((B, n_max), device=dev), lengths)  # what mfcc_features_many copies back
        bytes_io = {
            "host_varlen": (packed.nbytes, sum(v.nbytes for v in out_v.values())),
            "host_padded": (padded.nbytes, sum(v.nbytes for v in out_p.values())),
            "many": (B * n_max * 4, sum(v.numel() * v.element_size() for v in dev_out.values() if hasattr(v, "numel"))),
        }
        src = torch.from_numpy(packed)
        ceiling = lambda: (src.to(dev, non_blocking=True), torch.cuda.synchronize())  # noqa: E731
        ceiling()
        res = {
            "leg": "host",
            "input": np.dtype(dt).name,
            "gpu": torch.cuda.get_device_name(dev),
            "power_limit": power_limit,
            "clips": B,
            "audio_s": audio_s,
            "h2d_ceiling_ms": _median_host_ms(ceiling, iters),
        }
        for k, fn in ways.items():
            fn()
            res[f"{k}_ms"] = _median_host_ms(fn, iters)
            res[f"{k}_audio_s_per_s"] = audio_s / (res[f"{k}_ms"] / 1e3)
            res[f"{k}_h2d_bytes"], res[f"{k}_d2h_bytes"] = bytes_io[k]
        res["h2d_ceiling_audio_s_per_s"] = audio_s / (res["h2d_ceiling_ms"] / 1e3)
        print(json.dumps(res), flush=True)


def _profiled_kernel_ms(fn, match):
    """Device time of the kernels whose name contains `match`, summed over one call of fn (torch.profiler)."""
    from torch.profiler import ProfilerActivity, profile

    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sum(e.device_time_total for e in prof.key_averages() if match in e.key) / 1e3


def _int16_corpus(n_clips, seed, sr_in):
    """The resample leg's corpus: int16 clips of 2-20 s at sr_in, packed in one pinned buffer."""
    rng = np.random.default_rng(seed)
    lengths = [int(n) for n in rng.integers(2 * sr_in, 20 * sr_in + 1, n_clips)]
    offsets = np.zeros(n_clips + 1, np.int64)
    np.cumsum(lengths, out=offsets[1:])
    packed = _pinned((int(offsets[-1]),), np.int16)
    for i in range(n_clips):
        x = mm.synth_clip(seed + i, lengths[i], sr_in)
        packed[offsets[i] : offsets[i + 1]] = np.clip(np.round(x * 32768.0), -32768, 32767).astype(np.int16)
    return packed, offsets, lengths


def _resample_leg(n_clips, iters, seed, power_limit, dev):
    from modulation_mfcc_b200 import _lib

    sr_in, sr = 44100, 16000
    packed, offsets, lengths = _int16_corpus(n_clips, seed, sr_in)
    clips = [packed[offsets[i] : offsets[i + 1]] for i in range(n_clips)]
    audio_s = sum(lengths) / sr_in
    fx = mm.FeatureExtractor(sr, device=0)
    plan = fx.plan
    res = {"leg": "resample", "gpu": torch.cuda.get_device_name(dev), "power_limit": power_limit, "clips": n_clips,
           "sr_in": sr_in, "sr": sr, "audio_s": audio_s, "h2d_bytes": packed.nbytes}
    src = torch.from_numpy(packed)
    copy = lambda: (src.to(dev, non_blocking=True), torch.cuda.synchronize())  # noqa: E731
    copy()
    res["h2d_ms"] = _median_host_ms(copy, iters)
    x_dev = plan.pcm16_to_f32(torch.from_numpy(packed).to(dev))
    rows = [x_dev[offsets[i] : offsets[i + 1]] for i in range(n_clips)]
    # per-clip calls: the filter is designed on the host per call, so only the kernels' device time is counted
    res["resample_poly_per_clip_kernel_ms"] = _profiled_kernel_ms(
        lambda: [plan.resample_poly(r, 160, 441, "hq") for r in rows], "resample")
    if hasattr(_lib.lib(), "mmf_resample_varlen"):
        rs, h = mm.resample_descriptors(lengths, [sr_in] * n_clips, sr)
        y = torch.empty((n_clips, int(rs["n_out"].max())), device=dev)
        st = int(torch.cuda.current_stream(dev).cuda_stream)
        varlen = lambda: _lib.check(_lib.lib().mmf_resample_varlen(  # noqa: E731
            plan._h, x_dev.data_ptr(), n_clips, offsets.ctypes.data, rs.ctypes.data, h.ctypes.data, len(h),
            y.data_ptr(), y.shape[1], st))
        res["resample_varlen_kernel_ms"] = _profiled_kernel_ms(varlen, "resample")
        res["resample_varlen_outputs_per_s"] = float(rs["n_out"].sum()) / (res["resample_varlen_kernel_ms"] / 1e3)

        def before():  # the route without rates=: per clip, the loader's device resample and a copy back
            ys = []
            for c in clips:
                up, down = mm.resample_ratio(sr_in, sr)
                ys.append(plan.resample_poly(plan.pcm16_to_f32(c), up, down, "hq").cpu().numpy())
            return fx.host_many(ys)

        out = {k: v for k, v in fx.host_varlen(packed, offsets, rates=[sr_in] * n_clips).items() if k in
               ("totChange", "mfcc", "delta", "modspec", "band_energy")}
        out = {k: _pinned(v.shape, v.dtype.type) for k, v in out.items()}
        call = lambda: fx.host_varlen(packed, offsets, out=out, rates=[sr_in] * n_clips)  # noqa: E731
        res["host_varlen_rates_ms"] = _median_host_ms(call, iters)
        res["host_varlen_rates_audio_s_per_s"] = audio_s / (res["host_varlen_rates_ms"] / 1e3)
        before()
        res["resample_then_host_many_ms"] = _median_host_ms(before, max(1, iters // 5))
        res["resample_then_host_many_audio_s_per_s"] = audio_s / (res["resample_then_host_many_ms"] / 1e3)
    print(json.dumps(res), flush=True)


def _amplitude_leg(pcm, lengths16, n_clips, iters, seed, power_limit, dev):
    """The RMS envelope inside the host-buffer bundle; see the module docstring."""
    want = ("totChange", "mfcc", "delta", "modspec", "band_energy")
    fxs = {"raw": mm.FeatureExtractor(16000, device=0), "iir": mm.FeatureExtractor(16000, device=0, amp_outFilter="iir")}
    plan = fxs["raw"].plan
    sr_in = 44100
    packed44, offsets44, lengths44 = _int16_corpus(n_clips, seed, sr_in)
    host16 = pcm.cpu().numpy()
    offsets16 = np.zeros(len(lengths16) + 1, np.int64)
    np.cumsum(lengths16, out=offsets16[1:])
    packed16 = _pinned((int(offsets16[-1]),), np.float32)
    for i, n in enumerate(lengths16):
        packed16[offsets16[i] : offsets16[i + 1]] = host16[i, :n]
    corpora = [("int16_44k_rates", packed44, offsets44, [sr_in] * n_clips, sr_in),
               ("float32_16k", packed16, offsets16, None, 16000)]
    for name, packed, offsets, rates, rate in corpora:
        B = len(offsets) - 1
        audio_s = float(offsets[-1] - offsets[0]) / rate
        res = {"leg": "amplitude", "corpus": name, "gpu": torch.cuda.get_device_name(dev), "power_limit": power_limit,
               "clips": B, "audio_s": audio_s, "h2d_bytes": packed.nbytes}
        for k, (fx, w) in {"none": (fxs["raw"], want), "raw": (fxs["raw"], want + ("amplitude",)),
                           "iir": (fxs["iir"], want + ("amplitude",))}.items():
            out = {key: v for key, v in fx.host_varlen(packed, offsets, want=w, rates=rates).items()
                   if key in w}
            out = {key: _pinned(v.shape, v.dtype.type) for key, v in out.items()}
            call = lambda fx=fx, w=w, out=out: fx.host_varlen(packed, offsets, want=w, out=out, rates=rates)  # noqa: E731
            res[f"host_varlen_{k}_ms"] = _median_host_ms(call, iters)
            res[f"host_varlen_{k}_audio_s_per_s"] = audio_s / (res[f"host_varlen_{k}_ms"] / 1e3)
        # the route without the bundle: calculate_amplitude_envelope per clip at its native rate (float32 samples)
        clips = [packed[offsets[i] : offsets[i + 1]] for i in range(B)]
        clips = [c.astype(np.float32) / np.float32(32768.0) if c.dtype == np.int16 else c for c in clips]
        loop = lambda: [mm.calculate_amplitude_envelope(c, rate) for c in clips]  # noqa: E731
        loop()
        res["per_clip_loop_ms"] = _median_host_ms(loop, max(1, iters // 5))
        # kernel time over the same clips: one ragged launch, and mmf_rms per clip (whatever kernel the tree launches)
        x_dev = torch.from_numpy(np.concatenate(clips)).to(dev)
        offs0 = offsets - offsets[0]
        fl, hop = int(0.1 * rate), int(0.01 * rate)
        geom = [(fl, hop)] * B
        rows = [x_dev[offs0[i] : offs0[i + 1]] for i in range(B)]
        res["rms_varlen_kernel_ms"] = _profiled_kernel_ms(lambda: plan.rms_varlen(x_dev, offs0, geom, True), "rms")
        res["rms_per_clip_kernel_ms"] = _profiled_kernel_ms(lambda: [plan.rms(r, fl, hop) for r in rows], "rms")
        res["frames"] = int(mm.plan.amp_sizes(offs0, geom, True)[2][-1])
        print(json.dumps(res), flush=True)


def _hilbert_leg(pcm, lengths16, n_clips, iters, seed, power_limit, dev):
    """The Hilbert envelope; see the module docstring."""
    plan = mm.FeatureExtractor(16000, device=0).plan
    B = len(lengths16)
    offsets = np.zeros(B + 1, np.int64)
    np.cumsum(lengths16, out=offsets[1:])
    x_dev = torch.cat([pcm[i, :n] for i, n in enumerate(lengths16)]).contiguous()
    rows = [x_dev[offsets[i] : offsets[i + 1]] for i in range(B)]
    res = {"leg": "hilbert", "corpus": "float32_16k", "gpu": torch.cuda.get_device_name(dev),
           "power_limit": power_limit, "clips": B, "audio_s": float(offsets[-1]) / 16000}
    loop = lambda: [plan.hilbert_envelope(r) for r in rows]  # noqa: E731
    loop()
    res["per_clip_ms"] = _median_ms(loop, max(1, iters // 5))
    res["per_clip_kernel_ms"] = _profiled_kernel_ms(loop, "")
    if hasattr(plan, "hilbert_varlen"):
        call = lambda: plan.hilbert_varlen(x_dev, offsets)  # noqa: E731
        call()
        res["varlen_ms"] = _median_ms(call, iters)
        res["varlen_kernel_ms"] = _profiled_kernel_ms(call, "")
        from modulation_mfcc_b200 import _lib

        _lib.lib().mmf_launch_count(1)
        call()
        res["varlen_launches"] = _lib.lib().mmf_launch_count(1)
    print(json.dumps(res), flush=True)
    if not hasattr(plan, "hilbert_varlen"):
        return
    # the bundle with and without the envelope: int16 clips at 44.1 kHz resampled to the plan's 16 kHz
    want = ("totChange", "mfcc", "delta", "modspec", "band_energy")
    sr_in = 44100
    packed, offs44, _ = _int16_corpus(n_clips, seed, sr_in)
    rates = [sr_in] * n_clips
    res = {"leg": "hilbert_bundle", "corpus": "int16_44k_rates", "gpu": torch.cuda.get_device_name(dev),
           "power_limit": power_limit, "clips": n_clips, "audio_s": float(offs44[-1]) / sr_in}
    for k, fx, w in (("none", mm.FeatureExtractor(16000, device=0), want),
                     ("hilb_raw", mm.FeatureExtractor(16000, device=0, amp_method="Hilb"), want + ("amplitude",)),
                     ("hilb_iir", mm.FeatureExtractor(16000, device=0, amp_method="Hilb", amp_outFilter="iir"),
                      want + ("amplitude",))):
        out = {key: v for key, v in fx.host_varlen(packed, offs44, want=w, rates=rates).items() if key in w}
        out = {key: _pinned(v.shape, v.dtype.type) for key, v in out.items()}
        call = lambda fx=fx, w=w, out=out: fx.host_varlen(packed, offs44, want=w, out=out, rates=rates)  # noqa: E731
        res[f"host_varlen_{k}_ms"] = _median_host_ms(call, iters)
        res[f"host_varlen_{k}_audio_s_per_s"] = res["audio_s"] / (res[f"host_varlen_{k}_ms"] / 1e3)
    print(json.dumps(res), flush=True)


OUT_FILTERS = {
    "fir": dict(outFilter="fir", outFiltCutOff=[10], outFiltLen=21),
    "sg": dict(outFilter="sg", outFiltCutOff=[12], outFiltLen=11, outFiltPolyOrd=3),
}


def _outfilter_leg(pcm, lengths, n_clips, iters, seed, power_limit, dev):
    """The 'fir' and 'sg' output filters; see the module docstring."""
    sr = 16000
    host = pcm.cpu().numpy()
    clips = [host[i, :n] for i, n in enumerate(lengths)]
    res = {"leg": "outfilter", "corpus": "float32_16k", "gpu": torch.cuda.get_device_name(dev),
           "power_limit": power_limit, "clips": len(clips), "audio_s": sum(lengths) / sr}
    geom = dict(tStep=0.01, winLen=0.025, n_fft=512, n_mels=40, n_mfcc=13, minFreq=0.0, maxFreq=8000.0, device=0)
    for k, kw in (("none", dict(outFilter=None)), *OUT_FILTERS.items()):
        change = lambda kw=kw: mm.get_MFCCS_change_many(clips, sr, **geom, **kw)  # noqa: E731
        env = lambda kw=kw: mm.calculate_amplitude_envelope_many(clips, sr, device=0, **kw)  # noqa: E731
        for name, fn in (("change_many", change), ("envelope_many", env)):
            fn()
            res[f"{name}_{k}_ms"] = _median_host_ms(fn, iters)
    print(json.dumps(res), flush=True)
    try:
        mm.FeatureExtractor(16000, device=0, **OUT_FILTERS["fir"])
    except TypeError:  # a tree whose FeatureExtractor takes no output filter
        return
    want = ("totChange", "mfcc", "delta", "modspec", "band_energy")
    sr_in = 44100
    packed, offs44, _ = _int16_corpus(n_clips, seed, sr_in)
    rates = [sr_in] * n_clips
    res = {"leg": "outfilter_bundle", "corpus": "int16_44k_rates", "gpu": torch.cuda.get_device_name(dev),
           "power_limit": power_limit, "clips": n_clips, "audio_s": float(offs44[-1]) / sr_in}
    settings = {"none": {}, "iir": dict(outFilter="iir", outFiltCutOff=[12], outFiltLen=6), **OUT_FILTERS}
    for k, kw in settings.items():
        fx = mm.FeatureExtractor(16000, device=0, **kw)
        out = {key: _pinned(v.shape, v.dtype.type) for key, v in fx.host_varlen(packed, offs44, want=want,
                                                                               rates=rates).items() if key in want}
        call = lambda fx=fx, out=out: fx.host_varlen(packed, offs44, want=want, out=out, rates=rates)  # noqa: E731
        res[f"host_varlen_{k}_ms"] = _median_host_ms(call, iters)
        res[f"host_varlen_{k}_audio_s_per_s"] = res["audio_s"] / (res[f"host_varlen_{k}_ms"] / 1e3)
    print(json.dumps(res), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--clips", type=int, default=1024)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--loop-iters", type=int, default=3)
    ap.add_argument("--seed", type=int, default=2024)
    ap.add_argument("--legs", default="change,features")
    a = ap.parse_args()
    sr = 16000
    rng = np.random.default_rng(a.seed)
    lengths = [int(n) for n in rng.integers(2 * sr, 20 * sr + 1, a.clips)]
    n_max = 20 * sr
    dev = torch.device("cuda", 0)
    pcm = mm.synth_batch_device(a.clips, n_max, sr, seed=a.seed, device=dev)
    # the varlen call ignores what lies past each length; the padded call needs zeros there
    col = torch.arange(n_max, device=dev)[None, :]
    padded = torch.where(col < torch.tensor(lengths, device=dev)[:, None], pcm, torch.zeros((), device=dev))
    win, hop = mm.frame_sizes(sr, 0.025, 0.01)
    sos = scipy.signal.butter(6, 12.0, "low", fs=sr / hop, output="sos")
    prm = mm.make_change_params(sos, remove_first=1, diff_method=0, out_sos=sos)
    plan = mm.get_plan(mm.MfccConfig(sr, 512, win, hop, 40, 13, 0.0, 8000.0))
    singles = [padded[i : i + 1, : lengths[i]] for i in range(a.clips)]

    fx = mm.FeatureExtractor(sr, device=0)  # the same frame geometry
    ways = {
        "change": (
            lambda: plan.mfcc_change_varlen(pcm, lengths, prm),
            lambda: [plan.mfcc_change(x, prm) for x in singles],
            lambda: plan.mfcc_change(padded, prm),
        ),
        "features": (
            lambda: fx.varlen(pcm, lengths),
            lambda: [fx(x) for x in singles],
            lambda: fx(padded),
        ),
    }
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        power_limit = q.stdout.strip()
    except Exception:
        power_limit = None
    frames = [plan.num_frames(n) for n in lengths]
    for leg in a.legs.split(","):
        if leg == "host":
            _host_leg(fx, pcm, lengths, sr, a.iters, power_limit, dev)
            continue
        if leg == "resample":
            _resample_leg(a.clips, a.iters, a.seed, power_limit, dev)
            continue
        if leg == "amplitude":
            _amplitude_leg(pcm, lengths, a.clips, a.iters, a.seed, power_limit, dev)
            continue
        if leg == "hilbert":
            _hilbert_leg(pcm, lengths, a.clips, a.iters, a.seed, power_limit, dev)
            continue
        if leg == "outfilter":
            _outfilter_leg(pcm, lengths, a.clips, a.iters, a.seed, power_limit, dev)
            continue
        varlen, loop, pad = ways[leg]
        for fn in (varlen, pad, loop):  # warm-up: modules, workspace growth
            fn()
        torch.cuda.synchronize()
        res = {
            "leg": leg,
            "gpu": torch.cuda.get_device_name(dev),
            "power_limit": power_limit,
            "clips": a.clips,
            "audio_s": sum(lengths) / sr,
            "frames_ratio": sum(frames) / (a.clips * max(frames)),  # sum T_i / (n_clips * T_max)
            "varlen_ms": _median_ms(varlen, a.iters),
            "padded_ms": _median_ms(pad, a.iters),
            "loop_ms": _median_ms(loop, a.loop_iters),
        }
        for k in ("varlen", "padded", "loop"):
            res[f"{k}_audio_s_per_s"] = res["audio_s"] / (res[f"{k}_ms"] / 1e3)
        print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
