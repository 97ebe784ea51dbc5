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

Workload: 1024 clips at 16 kHz with the bench's frame geometry (win 400 / hop 160 / n_fft 512, 40 mel, 13 MFCC,
gradient, Butterworth output filter), lengths uniform in [2 s, 20 s] from a fixed seed.  Prints, per leg, the median
ms of each way and audio-seconds per second as one JSON line, with the GPU's name and power limit.

    python tools/bench_varlen.py [--clips 1024] [--iters 10] [--loop-iters 3] [--legs change,features]
"""
import argparse
import json
import os
import subprocess
import sys

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
