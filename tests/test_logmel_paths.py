"""Every STFT + mel-projection (K1/K2: framing, pre-emphasis, Hann window, rFFT, |X|^2, Slaney mel, 10*log10,
per-clip max) kernel path against a float64 reference.

``mmf_plan_create``, ``choose_tile_geometry`` and ``run_stft`` (csrc/c_api.cu) split the shapes ``validate_cfg``
accepts (16 <= n_fft <= 4096, n_mels <= 512) over six kernels:

  path   kernel(s)                                          taken when
  tc     stft_mel_tc_kernel<NBQ, FAST160, VL>               mmf_logmel, n_fft 512, no NO_TC_MEL / MEL_WALK / MMA_MEL /
         (+ mel_empty_bands_kernel when n_act < n_mels)     SPLIT_SMEM / SCALAR_FFT, tc_nb(n_act) <= 112, tile fits;
                                                            NBQ = ceil16(n_act) / 4 (4 .. 28); FAST160 = hop 160, TMA,
                                                            no pre-emphasis; VL = the variable-length change path
  reg    stft_mel_kernel<NFFT, float2 | c2, 256 | 512, MG>  every other power-of-two n_fft in [256, 4096]; c2 (two
                                                            frames on packed FP32) needs n_fft >= 512 and no
                                                            SCALAR_FFT; 512 threads when only one CTA fits an SM and
                                                            n_fft >= 1024; MG = false under MEL_WALK or MMA_MEL (the
                                                            per-bin sparse walk on [bin][frame] rows)
  mma    stft_mel_kernel<.., MG = false>, mel_mma = 1       MMA_MEL where choose_tile_geometry accepts it (it declines
                                                            when the B fragments cost tile width or the second CTA)
  power  stft_mel_kernel writing power                      mmf_stft_power, every NFFT, with and without SPLIT_SMEM
  tcfft  tc_fft512_kernel                                   mmf_stft_power, TC_FFT, n_fft 512, hop <= 512, no
                                                            pre-emphasis
  gen    dft_power_kernel + mel_from_power_kernel           n_fft < 256 or not a power of two

Each GPU case names the kernels it expects; a ``torch.profiler`` probe checks that exactly those K1 kernels ran and
that ``mmf_launch_count`` went up by the expected amount.  Inputs are seeded synthetic audio (tones, a Nyquist
component, DC, noise, a stretch of exact zeros, one all-zero clip per batch) at the case's own shape.

The reference (``_ref_power`` / ``_ref_logmel``) frames the first n samples of each float32 row with n_fft // 2 zeros
of centre padding, applies pre-emphasis y[i] = x[i] - a x[i - 1] (x[-1] = 0) before the padding, multiplies by the
periodic Hann of win samples centred in n_fft and takes |rfft|^2 in float64; the mel projection uses the oracle's
float32 Slaney weights (librosa's) in float64.  Errors are scale-free:
  * power: max_k |P - P_ref| / max_k P_ref per frame; a frame whose reference is all zero must be exactly 0;
  * log-mel, in the linear domain with L = 10^(dB / 10) and R = max(amin, W P_ref): |L - R| / (sum_k W[m, k]
    max_k P_ref[k, t] + R) per cell, floor cells included (the first term is how FFT error, which scales with the
    frame's energy, reaches a band).
Largest values observed on a B200 (1000 W power limit) over the case matrix, the forced geometries and the plan
sweep, and the bounds (BOUND_POWER, BOUND_MEL), each 3 to 5x its maximum:
  power  reg 4.6e-7 (bound 2e-6), tcfft 7.6e-7 (4e-6), gen 2.0e-6 (8e-6)
  mel    reg 1.1e-6 (5e-6), mma 9.9e-7 (3e-6), tc 1.0e-5 (5e-5), gen 1.6e-6 (6e-6)
The tc error is the bf16-pair operands of the tcgen05 GEMM (the product of the two low halves is dropped).
Exact checks: the per-clip max key is the key of the maximum of the clip's own output; floor cells (reference mel
power exactly 0) all hold one value within 1e-5 dB of -100; a clip's bits do not depend on the batch around it, on
the loader (TMA, MMF_FLAG_NO_TMA, an unaligned base, a strided batch with NaN in the gaps), on the tile geometry
(MMF_TF, MMF_SPAN_BUFS, MMF_PT_BUFS, MMF_NO_512) or on the variable-length path; power(2x) == 4 power(x) on the FP32
transforms.  ``test_tolerances_catch_plausible_mistakes`` (CPU) holds the bounds honest: each of ten plausible
mistakes misses the reference by more than 10x the bound of the path that computes each case fixture it can reach.
"""

import os
import re
from typing import NamedTuple

import numpy as np
import pytest

import oracle
import modulation_mfcc_b200 as mm
from modulation_mfcc_b200 import _lib

AMIN = 1e-10
BOUND_POWER = {"reg": 2e-6, "tcfft": 4e-6, "gen": 8e-6}
BOUND_MEL = {"reg": 5e-6, "mma": 3e-6, "tc": 5e-5, "gen": 6e-6}

NO_TMA = _lib.MMF_FLAG_NO_TMA
SPLIT = _lib.MMF_FLAG_SPLIT_SMEM
SCALAR = _lib.MMF_FLAG_SCALAR_FFT
MMA = _lib.MMF_FLAG_MMA_MEL
TCFFT = _lib.MMF_FLAG_TC_FFT
WALK = _lib.MMF_FLAG_MEL_WALK
NO_TC = _lib.MMF_FLAG_NO_TC_MEL
_NO_TC_FLAGS = NO_TC | WALK | MMA | SPLIT | SCALAR


def _torch():
    import torch

    return torch


# ---------------------------------------------------------------------------
# float64 reference
# ---------------------------------------------------------------------------


def _key(maxima):
    """float32 maxima -> the int32 keys the kernels write (bits when the sign bit is clear, else bits ^ 0x7FFFFFFF)."""
    bits = np.ascontiguousarray(maxima, np.float32).view(np.int32)
    return np.where(bits >= 0, bits, bits ^ np.int32(0x7FFFFFFF)).astype(np.int32)


def _window(win, n_fft, mistake=None):
    if mistake == "symmetric_hann":
        n = np.arange(win, dtype=np.float64)
        w = 0.5 - 0.5 * np.cos(2.0 * np.pi * n / max(win - 1, 1)) if win > 1 else np.ones(1)
        out = np.zeros(n_fft)
        lp = (n_fft - win) // 2
        out[lp:lp + win] = w
        return out
    w = oracle.padded_hann(win, n_fft)
    if mistake == "window_left_aligned":
        w = np.roll(w, -((n_fft - win) // 2))
    return w


def _ref_power(x, n, n_fft, win, hop, preemph, *, mistake=None, chunk=2048):
    """|rfft(window * frame)|^2 in float64 of the first ``n`` samples of each float32 row of ``x``: [B, F, T] (or
    [F, T] for one row).  Pre-emphasis y[i] = x[i] - a x[i - 1] with x[-1] = 0 (a = float32(preemph), as the plan
    stores it) comes before the centre padding of n_fft // 2 zeros, so the padding stays exactly zero.  ``mistake``
    (tests of the bounds only) makes one plausible implementation error on purpose."""
    x = np.asarray(x, np.float32)
    one = x.ndim == 1
    x = np.atleast_2d(x)[:, :n].astype(np.float64)
    a = float(np.float32(preemph))
    if a != 0.0 and mistake != "preemph_after_padding":
        y = x.copy()
        y[:, 1:] -= a * x[:, :-1]
        if mistake == "preemph_across_clip_start":
            y[:, 0] -= a * np.roll(x[:, -1], 1)  # the sample before the clip in a packed batch
    else:
        y = x
    pad = n_fft // 2
    T = 1 + (n + 2 * pad - n_fft) // hop
    shift = hop if mistake == "frames_shifted_one_hop" else 0
    yp = np.zeros((x.shape[0], n + 2 * pad + shift + n_fft))
    yp[:, pad:pad + n] = y
    if mistake == "reflect_padding":
        for b in range(x.shape[0]):
            yp[b, :n + 2 * pad] = np.pad(y[b], pad, mode="reflect") if n > pad else np.pad(y[b], pad, mode="wrap")
    if a != 0.0 and mistake == "preemph_after_padding":
        yq = yp.copy()
        yq[:, 1:] -= a * yp[:, :-1]
        yp = yq
    w = _window(win, n_fft, mistake)
    F = n_fft // 2 + 1
    P = np.empty((x.shape[0], F, T))
    for s in range(0, T, chunk):
        t = np.arange(s, min(T, s + chunk))
        frames = yp[:, t[:, None] * hop + shift + np.arange(n_fft)[None, :]]
        X = np.fft.rfft(frames * w, axis=-1)
        p = np.abs(X) if mistake == "magnitude" else X.real ** 2 + X.imag ** 2
        P[:, :, s:s + len(t)] = np.swapaxes(p, -1, -2)
    if mistake == "nyquist_dropped":
        P[:, -1] = 0.0
    return P[0] if one else P


def _mel_weights(sr, n_fft, n_mels, fmin, fmax, mistake=None):
    """The oracle's float32 Slaney filterbank (librosa's weights are the specification) as float64 [n_mels, F]."""
    if mistake == "htk_mel":
        hz2mel = lambda f: 2595.0 * np.log10(1.0 + np.asarray(f, np.float64) / 700.0)  # noqa: E731
        mel2hz = lambda m: 700.0 * (10.0 ** (np.asarray(m) / 2595.0) - 1.0)  # noqa: E731
        fftfreqs = np.fft.rfftfreq(n_fft, 1.0 / sr)
        mel_f = mel2hz(np.linspace(hz2mel(fmin), hz2mel(fmax), n_mels + 2))
        fdiff = np.diff(mel_f)
        ramps = np.subtract.outer(mel_f, fftfreqs)
        W = np.maximum(0, np.minimum(-ramps[:-2] / fdiff[:-1, None], ramps[2:] / fdiff[1:, None]))
        return (W * (2.0 / (mel_f[2:] - mel_f[:-2]))[:, None]).astype(np.float32).astype(np.float64)
    W = oracle.mel_filterbank(sr, n_fft, n_mels, fmin, fmax).astype(np.float64)
    if mistake == "no_slaney_norm":
        mel_f = oracle.mel_to_hz(np.linspace(oracle.hz_to_mel(fmin), oracle.hz_to_mel(fmax), n_mels + 2))
        W = W / (2.0 / (mel_f[2:] - mel_f[:-2]))[:, None]
    return W


def _ref_logmel(P, W, amin=AMIN):
    """10 log10(max(amin, W P)) in float64: [B, n_mels, T]."""
    return 10.0 * np.log10(np.maximum(amin, np.einsum("mk,...kt->...mt", W, P)))


def _power_err(P, Pref):
    """max over frames of max_k |P - P_ref| / max_k P_ref; inf for a non-finite output or a non-zero value in a frame
    whose reference is all zero."""
    P = np.asarray(P, np.float64)
    if not np.all(np.isfinite(P)):
        return float("inf")
    peak = Pref.max(axis=-2)
    d = np.abs(P - Pref).max(axis=-2)
    zero = peak == 0.0
    if np.any(d[zero] != 0.0):
        return float("inf")
    return float(np.max(d[~zero] / peak[~zero], initial=0.0))


def _mel_err(dB, Pref, W, amin=AMIN):
    """max over cells of |L - R| / (sum_k W[m, k] max_k P_ref[k, t] + R) with L = 10^(dB / 10), R = max(amin, W P_ref);
    inf for a non-finite output."""
    dB = np.asarray(dB, np.float64)
    if not np.all(np.isfinite(dB)):
        return float("inf")
    L = 10.0 ** (dB / 10.0)
    R = np.maximum(amin, np.einsum("mk,...kt->...mt", W, Pref))
    scale = W.sum(axis=1)[:, None] * Pref.max(axis=-2)[..., None, :]
    return float(np.max(np.abs(L - R) / (scale + R)))


# ---------------------------------------------------------------------------
# inputs: seeded synthetic audio
# ---------------------------------------------------------------------------


def _audio(B, n, sr, seed, signal="mix"):
    """[B, n] float32.  ``mix``: per clip three tones, a Nyquist component (+-1 alternating), DC and white noise at a
    clip gain between 1e-2 and 1e2 (the second clip 1e-4 quieter still), clicks of 4x the clip's peak on the first and last samples,
    a stretch of exact zeros in the middle of long clips, and a last clip of exact zeros when B > 1.  ``dc``: constant clips.  ``impulse``: unit impulses at the
    first and the last sample.  ``cos``: see test_known_answers."""
    rng = np.random.default_rng(seed)
    i = np.arange(n, dtype=np.float64)
    x = np.zeros((B, n))
    if signal == "dc":
        x[:] = rng.uniform(0.5, 2.0, (B, 1)) * np.where(np.arange(B) % 2, -1.0, 1.0)[:, None]
    elif signal == "impulse":
        x[:, 0] = 1.0
        x[:, -1] = -0.75
    else:
        for b in range(B):
            f = rng.uniform(20.0, 0.45 * sr, 3)
            amp = np.array([0.5, 0.2, 0.05])
            y = (amp[:, None] * np.sin(2 * np.pi * f[:, None] / sr * i + rng.uniform(0, 2 * np.pi, (3, 1)))).sum(0)
            y += 0.1 * np.where(np.arange(n) % 2, -1.0, 1.0) + 0.05 + 0.01 * rng.standard_normal(n)
            y *= 10.0 ** rng.uniform(-2.0, 2.0) * (1e-4 if b == 1 else 1.0)
            if n >= 12000:
                y[n // 2 - 4500:n // 2 + 4500] = 0.0
            y[0], y[-1] = 4 * np.abs(y).max(), -4 * np.abs(y).max()  # clicks at the edges: what lies beyond them shows
            x[b] = y
        if B > 1:
            x[B - 1] = 0.0
    return x.astype(np.float32)


# ---------------------------------------------------------------------------
# the case matrix: expected kernels read off mmf_plan_create, choose_tile_geometry and run_stft
# ---------------------------------------------------------------------------


class Case(NamedTuple):
    id: str
    path: str  # bound key: reg, mma, tc, tcfft, gen
    kind: str  # "logmel" or "power"
    sr: float
    n_fft: int
    win: int
    hop: int
    n_mels: int
    fmin: float
    fmax: float
    n: int
    kernels: tuple  # ((kernel, template arguments), ...) expected, each launched once per 65535-clip chunk if chunked
    preemph: float = 0.0
    flags: int = 0
    B: int = 3
    signal: str = "mix"
    layout: str = "contig"  # contig, strided (NaN gaps), unaligned (NaN before the base)
    env: tuple = ()  # (name, value) tile-geometry overrides read at plan creation
    mma: object = None  # MMA_MEL cases: True = accepted, False = declined

    def cfg(self):
        return mm.MfccConfig(self.sr, self.n_fft, self.win, self.hop, self.n_mels, 1, self.fmin, self.fmax,
                             preemph=self.preemph, flags=self.flags)

    @property
    def T(self):
        return 1 + self.n // self.hop


def _n_act(sr, n_fft, n_mels, fmin, fmax):
    """1 + the last band with a non-zero weight in the plan's own float32 filterbank (stft_mel_tc_active_bands)."""
    _, mel, _ = mm.host_tables(mm.MfccConfig(sr, n_fft, n_fft, 1, n_mels, 1, fmin, fmax))
    nz = np.flatnonzero(mel.any(axis=1))
    return int(nz[-1]) + 1 if nz.size else 1


def _nbq(n_act):
    return (n_act + 15) // 16 * 16 // 4


def _frames_for(T, hop):
    return max(1, (T - 1) * hop)


def TC(id, sr, win, hop, n_mels, fmin, fmax, T, *, pre=0.0, flags=0, layout="contig", **kw):
    n_act = _n_act(sr, 512, n_mels, fmin, fmax)
    fast = hop == 160 and pre == 0.0 and layout != "unaligned" and not flags & NO_TMA  # (a strided batch keeps TMA)
    k = (("stft_mel_tc_kernel", (_nbq(n_act), fast, False)),)
    if n_act < n_mels:
        k += (("mel_empty_bands_kernel", ()),)
    return Case(f"tc_nbq{_nbq(n_act)}_{id}", "tc", "logmel", sr, 512, win, hop, n_mels, fmin, fmax,
                _frames_for(T, hop), k, preemph=pre, flags=flags, layout=layout, **kw)


def _stft(n_fft, flags, threads):
    v = "c2" if n_fft >= 512 and not flags & SCALAR else "float2"
    return ("stft_mel_kernel", (n_fft, v, threads, not flags & (WALK | MMA)))


def R(id, sr, n_fft, win, hop, n_mels, fmin, fmax, T, *, flags=0, threads=256, kind="logmel", mma=None, **kw):
    """register-FFT kernel; at n_fft 512 a log-mel case needs a flag that turns the tcgen05 mel off"""
    path = "mma" if mma else "reg"
    k = _stft(n_fft, flags, threads)
    return Case(f"{'pow' if kind == 'power' else path}_{n_fft}_{k[1][1]}_{threads}_{'mg' if k[1][3] else 'walk'}_{id}",
                path, kind, sr, n_fft, win, hop, n_mels, fmin, fmax, _frames_for(T, hop), (k,), flags=flags, mma=mma,
                **kw)


def G(id, n_fft, win, hop, T, *, kind="logmel", sr=16000.0, n_mels=40, fmin=0.0, fmax=8000.0, **kw):
    k = (("dft_power_kernel", ()),) + ((("mel_from_power_kernel", ()),) if kind == "logmel" else ())
    return Case(f"gen_{kind}_{n_fft}_{id}", "gen", kind, sr, n_fft, win, hop, n_mels, fmin, fmax, _frames_for(T, hop),
                k, **kw)


def TF(id, hop, T, **kw):
    return Case(f"tcfft_{id}", "tcfft", "power", 16000.0, 512, 512, hop, 40, 0.0, 8000.0, _frames_for(T, hop),
                (("tc_fft512_kernel", ()),), flags=TCFFT, **kw)


CASES = [
    # ---- tc: every NBQ, chosen by n_act; T around the 64-frame tile and 128-frame block
    TC("mel16_T129", 16000, 400, 160, 16, 0.0, 8000.0, 129),
    TC("mel16_no_tma_T64", 16000, 400, 160, 16, 0.0, 8000.0, 64, flags=NO_TMA),
    TC("mel32_T65", 16000, 400, 160, 32, 0.0, 8000.0, 65),
    TC("mel64_T128", 16000, 400, 160, 64, 0.0, 8000.0, 128),
    TC("mel80_unaligned_T63", 16000, 400, 160, 80, 0.0, 8000.0, 63, layout="unaligned"),
    TC("mel80_hop128_T65", 16000, 400, 128, 80, 0.0, 8000.0, 65),
    TC("mel96_T64", 16000, 400, 160, 96, 0.0, 8000.0, 64),
    TC("mel26_8k_T65", 8000, 240, 100, 26, 0.0, 4000.0, 65),
    TC("mel40_preemph_T64", 16000, 400, 160, 40, 0.0, 8000.0, 64, pre=0.97),
    TC("mel64_fmin_hop128_T63", 16000, 512, 128, 64, 60.0, 7600.0, 63),
    TC("mel80_T127", 16000, 400, 160, 80, 0.0, 8000.0, 127),
    TC("mel96_hop161_T128", 16000, 320, 161, 96, 0.0, 8000.0, 128),
    TC("gui_default_T200", 10000, 250, 50, 128, 100.0, 10000.0, 200),  # 28 trailing empty bands
    TC("mel112_hop100_T1", 16000, 400, 100, 112, 0.0, 8000.0, 1),
    TC("mel40_T1", 16000, 400, 160, 40, 0.0, 8000.0, 1, B=1),
    # interior empty bands (no bin below n_act): 44.1 kHz, n_fft 512
    TC("44k_mel100_interior_empty", 44100, 512, 100, 100, 0.0, 22050.0, 129),
    TC("44k_mel112_interior_empty", 44100, 441, 100, 112, 0.0, 22050.0, 65, pre=0.97),
    # FAST160 off: no TMA, unaligned base, strided batch; the plain loader with pre-emphasis
    TC("mel40_no_tma_T129", 16000, 400, 160, 40, 0.0, 8000.0, 129, flags=NO_TMA),
    TC("mel40_unaligned_T65", 16000, 400, 160, 40, 0.0, 8000.0, 65, layout="unaligned"),
    TC("mel40_strided_T65", 16000, 400, 160, 40, 0.0, 8000.0, 65, layout="strided"),
    TC("mel40_preemph_unaligned", 16000, 400, 160, 40, 0.0, 8000.0, 100, pre=0.97, layout="unaligned"),
    TC("gui_default_preemph_hop99", 10000, 250, 99, 128, 100.0, 10000.0, 70, pre=0.5),
    TC("mel40_dc", 16000, 400, 160, 40, 0.0, 8000.0, 20, signal="dc"),
    TC("mel40_impulse", 16000, 512, 160, 40, 0.0, 8000.0, 20, signal="impulse"),
    # one long clip: 300 blocks of 128 frames, so every CTA handles several
    TC("mel40_long", 16000, 400, 160, 40, 0.0, 8000.0, 38400, B=1),
    # ---- reg: each NFFT x vector type x mel walk x CTA size that a shape reaches
    R("default", 8000, 256, 200, 80, 32, 0.0, 4000.0, 129),
    R("walk_preemph", 8000, 256, 256, 64, 32, 0.0, 4000.0, 33, flags=WALK, preemph=0.97),
    R("no_tc_mel", 16000, 512, 400, 160, 40, 0.0, 8000.0, 129, flags=NO_TC),
    R("walk", 16000, 512, 400, 160, 40, 0.0, 8000.0, 31, flags=WALK),
    R("scalar_preemph", 16000, 512, 400, 160, 40, 0.0, 8000.0, 32, flags=SCALAR, preemph=0.97),
    R("scalar_walk", 16000, 512, 512, 100, 40, 0.0, 8000.0, 33, flags=SCALAR | WALK),
    R("default", 22050, 1024, 882, 275, 64, 50.0, 11025.0, 100, threads=512),
    R("walk_preemph", 22050, 1024, 1024, 256, 64, 0.0, 11025.0, 33, flags=WALK, preemph=0.97, threads=512),
    R("hop16", 22050, 1024, 1024, 16, 40, 0.0, 11025.0, 40),
    R("hop16_walk", 22050, 1024, 1000, 16, 40, 0.0, 11025.0, 31, flags=WALK),
    R("scalar_mel512", 22050, 1024, 1024, 800, 512, 0.0, 11025.0, 9, flags=SCALAR, threads=512),
    R("scalar_walk_mel128", 22050, 1024, 1024, 1024, 128, 0.0, 11025.0, 9, flags=SCALAR | WALK, threads=512),
    R("scalar", 22050, 1024, 701, 256, 64, 0.0, 11025.0, 17, flags=SCALAR),
    R("scalar_walk", 22050, 1024, 1024, 1024, 64, 0.0, 11025.0, 20, flags=SCALAR | WALK),  # hop = n_fft
    R("default", 44100, 2048, 1102, 441, 128, 0.0, 22050.0, 60, threads=512),
    R("hop16", 44100, 2048, 2048, 16, 40, 0.0, 22050.0, 40),
    R("walk_preemph", 44100, 2048, 2048, 512, 128, 0.0, 22050.0, 9, flags=WALK, preemph=0.97),
    R("scalar", 44100, 2048, 2048, 2048, 128, 0.0, 22050.0, 9, flags=SCALAR, threads=512),  # win = hop = n_fft
    R("scalar_walk", 44100, 2048, 1500, 1500, 128, 0.0, 22050.0, 7, flags=SCALAR | WALK),  # hop = win
    R("default", 48000, 4096, 3840, 960, 96, 20.0, 24000.0, 20),
    R("walk_preemph", 48000, 4096, 4096, 1024, 96, 0.0, 24000.0, 9, flags=WALK, preemph=0.97),
    R("scalar", 48000, 4096, 4096, 1024, 96, 0.0, 24000.0, 8, flags=SCALAR),
    R("scalar_walk", 48000, 4096, 4000, 1024, 96, 0.0, 24000.0, 5, flags=SCALAR | WALK),
    R("scalar_hop16", 48000, 4096, 4096, 16, 40, 0.0, 24000.0, 40, flags=SCALAR, threads=512),
    R("scalar_walk_hop16", 48000, 4096, 4001, 16, 40, 0.0, 24000.0, 33, flags=SCALAR | WALK, threads=512),
    R("hop4096", 48000, 4096, 4096, 4096, 96, 0.0, 24000.0, 4),
    R("hop4096_walk", 48000, 4096, 4096, 4096, 96, 0.0, 24000.0, 3, flags=WALK),
    R("hop4096_scalar", 48000, 4096, 4096, 4096, 96, 0.0, 24000.0, 3, flags=SCALAR),
    R("scalar_walk_mel512", 44100, 2048, 2048, 1500, 512, 0.0, 22050.0, 7, flags=SCALAR | WALK, threads=512),
    # nb 112 at hop 160: the tcgen05 tile does not fit, the plan falls back to the register-FFT kernel
    R("route_tc_nb112_hop160_falls_back", 16000, 512, 400, 160, 112, 0.0, 8000.0, 65),
    R("1024_512thr", 22050, 1024, 1024, 128, 512, 0.0, 11025.0, 40, threads=512),
    # mel projection on mma.sync: accepted, and declined (512 bands of a 2048-point FFT)
    R("mma_40", 16000, 512, 400, 160, 40, 0.0, 8000.0, 129, flags=MMA, mma=True),
    R("mma_preemph", 22050, 1024, 882, 275, 64, 50.0, 11025.0, 33, flags=MMA, mma=True, preemph=0.97),
    R("mma_declined_512", 44100, 2048, 2048, 512, 512, 0.0, 22050.0, 9, flags=MMA, mma=False),
    # hops and windows
    R("hop1", 8000, 256, 256, 1, 32, 0.0, 4000.0, 200),
    R("hop1_walk", 16000, 512, 400, 1, 40, 0.0, 8000.0, 70, flags=WALK),
    R("hop161_odd", 16000, 512, 400, 161, 40, 0.0, 8000.0, 40, flags=NO_TC),
    R("hop_eq_win_301", 8000, 256, 201, 201, 32, 0.0, 4000.0, 30),
    R("hop_2nfft", 8000, 256, 256, 512, 32, 0.0, 4000.0, 12),
    R("win1", 8000, 256, 1, 64, 32, 0.0, 4000.0, 40),
    R("win301_odd", 16000, 512, 301, 160, 40, 0.0, 8000.0, 40, flags=NO_TC),
    # bands
    R("mel1", 16000, 512, 400, 160, 1, 0.0, 8000.0, 40, flags=NO_TC),
    R("mel1_walk", 8000, 256, 200, 80, 1, 300.0, 3000.0, 40, flags=WALK),
    R("mel512", 48000, 4096, 4096, 1024, 512, 0.0, 24000.0, 6),
    R("mel512_walk", 44100, 2048, 2048, 441, 512, 0.0, 22050.0, 9, flags=WALK, threads=512),
    R("fmin300", 16000, 512, 400, 160, 40, 300.0, 8000.0, 40, flags=NO_TC),
    R("fmax_above_nyquist", 10000, 512, 250, 50, 128, 100.0, 10000.0, 60, flags=NO_TC),
    R("fmax_above_nyquist_walk", 10000, 1024, 500, 100, 128, 100.0, 10000.0, 60, flags=WALK),
    R("dc", 22050, 1024, 1024, 256, 64, 0.0, 11025.0, 20, signal="dc", threads=512),
    R("impulse", 16000, 512, 512, 160, 40, 0.0, 8000.0, 12, flags=WALK, signal="impulse"),
    R("strided_preemph", 22050, 1024, 882, 275, 64, 50.0, 11025.0, 17, preemph=0.97, layout="strided", threads=512),
    R("unaligned_preemph", 8000, 256, 200, 80, 32, 0.0, 4000.0, 33, preemph=0.97, layout="unaligned"),
    # ---- power: every NFFT (the register-FFT kernel writing power), SPLIT_SMEM
    R("power", 8000, 256, 200, 80, 32, 0.0, 4000.0, 40, kind="power"),
    R("power", 16000, 512, 400, 160, 40, 0.0, 8000.0, 40, kind="power"),
    R("power_split_smem", 16000, 512, 400, 160, 40, 0.0, 8000.0, 40, kind="power", flags=SPLIT, preemph=0.97),
    R("power_scalar", 16000, 512, 512, 128, 40, 0.0, 8000.0, 33, kind="power", flags=SCALAR),
    R("power", 22050, 1024, 882, 275, 64, 0.0, 11025.0, 20, kind="power", preemph=0.97, threads=512),
    R("power", 44100, 2048, 2048, 441, 128, 0.0, 22050.0, 12, kind="power", threads=512),
    R("power", 48000, 4096, 3840, 960, 96, 0.0, 24000.0, 8, kind="power"),
    R("power_strided", 16000, 512, 400, 160, 40, 0.0, 8000.0, 40, kind="power", layout="strided", preemph=0.97),
    # TC_FFT at hop 513 falls back to the register-FFT kernel
    R("power_tcfft_hop513", 16000, 512, 512, 513, 40, 0.0, 8000.0, 9, kind="power", flags=TCFFT),
    TF("hop1", 1, 300),
    TF("hop160", 160, 129),
    TF("hop512", 512, 40),
    TF("hop160_strided", 160, 65, layout="strided"),
    TF("hop160_unaligned", 160, 65, layout="unaligned"),
    # ---- gen: the FP32 matrix-product DFT, with and without pre-emphasis
    *[G(f"T{T}" + ("_preemph" if pre else ""), nf, win, hop, T, preemph=pre, sr=sr, fmax=sr / 2, n_mels=nm)
      for nf, win, hop, T, sr, nm in [(16, 16, 4, 70, 16000.0, 4), (17, 15, 5, 40, 16000.0, 4),
                                      (32, 25, 8, 66, 16000.0, 8), (64, 64, 16, 65, 16000.0, 16),
                                      (100, 80, 40, 64, 16000.0, 24), (255, 255, 64, 63, 16000.0, 40),
                                      (400, 400, 160, 129, 16000.0, 40), (401, 399, 161, 65, 16000.0, 40),
                                      (4095, 4000, 1024, 12, 48000.0, 96)]
      for pre in (0.0, 0.97)],
    G("power_T65", 400, 400, 160, 65, kind="power"),
    G("power_preemph_T33", 17, 15, 3, 33, kind="power", preemph=0.97),
    G("strided_preemph", 400, 400, 160, 40, layout="strided", preemph=0.97),
    G("unaligned", 100, 80, 40, 40, layout="unaligned"),
    G("fmax_above_nyquist", 400, 400, 100, 40, sr=10000.0, n_mels=128, fmin=100.0, fmax=10000.0),
    G("dc", 255, 255, 64, 20, signal="dc"),
    G("impulse", 401, 401, 100, 20, signal="impulse"),
]

# forced tile geometries: (id, n_fft, flags, env); every one is a register-FFT case on 256 threads whose bits must
# equal the default plan's.  MMF_TF=1 is ignored: the narrowest transform group of a 256-thread CTA holds two frames
# (n_fft 4096 without packing), so a one-frame tile cannot be asked for
GEOMETRIES = [
    ("tf1_ignored", 4096, SCALAR, (("MMF_TF", "1"),)),
    ("tf2", 4096, SCALAR, (("MMF_TF", "2"),)),
    ("tf2_walk", 4096, SCALAR | WALK, (("MMF_TF", "2"),)),
    ("tf4", 4096, 0, (("MMF_TF", "4"),)),
    ("tf4_scalar", 2048, SCALAR, (("MMF_TF", "4"),)),
    ("tf8", 2048, 0, (("MMF_TF", "8"),)),
    ("tf8_walk_preemph", 1024, SCALAR | WALK, (("MMF_TF", "8"),)),
    ("tf16", 1024, 0, (("MMF_TF", "16"),)),
    ("tf16_scalar_walk", 512, SCALAR | WALK, (("MMF_TF", "16"),)),
    ("tf32", 512, NO_TC, (("MMF_TF", "32"),)),
    ("tf32_256", 256, 0, (("MMF_TF", "32"),)),
    ("span_bufs1", 1024, 0, (("MMF_TF", "16"), ("MMF_SPAN_BUFS", "1"))),
    ("span_bufs1_walk", 256, WALK, (("MMF_TF", "32"), ("MMF_SPAN_BUFS", "1"))),
    ("pt_bufs1", 1024, WALK, (("MMF_TF", "16"), ("MMF_PT_BUFS", "1"))),
    ("pt_bufs1_mg", 256, 0, (("MMF_TF", "32"), ("MMF_PT_BUFS", "1"))),
    ("span_pt_bufs1", 2048, SCALAR, (("MMF_TF", "8"), ("MMF_SPAN_BUFS", "1"), ("MMF_PT_BUFS", "1"))),
    ("span_pt_bufs1_mma", 512, MMA, (("MMF_TF", "32"), ("MMF_SPAN_BUFS", "1"), ("MMF_PT_BUFS", "1"))),
    ("no_512", 1024, 0, (("MMF_NO_512", "1"),)),  # the default takes 512 threads at both shapes
    ("no_512_scalar_walk", 4096, SCALAR | WALK, (("MMF_NO_512", "1"),)),
]
_GEO_SHAPE = {256: (8000.0, 256, 64, 32, 4000.0), 512: (16000.0, 400, 160, 40, 8000.0),
              1024: (22050.0, 882, 256, 64, 11025.0), 2048: (44100.0, 2048, 441, 128, 22050.0),
              4096: (48000.0, 4096, 1024, 96, 24000.0)}
_GEO_SHAPE_NO_512 = {1024: (22050.0, 882, 256, 64, 11025.0), 4096: (48000.0, 4096, 16, 40, 24000.0)}

# instantiations the matrix must reach, and the ones no accepted configuration reaches
WANT = ({("stft_mel_tc_kernel", (q, f, v)) for q in range(4, 29, 4) for f in (False, True) for v in (False, True)}
        | {("stft_mel_kernel", (n, v, t, mg)) for n in (256, 512, 1024, 2048, 4096) for v in ("float2", "c2")
           for t in (256, 512) for mg in (False, True) if (v == "float2" or n >= 512) and (t == 256 or n >= 1024)}
        | {(k, ()) for k in ("mel_empty_bands_kernel", "tc_fft512_kernel", "dft_power_kernel", "mel_from_power_kernel")})
# instantiation -> why no configuration the plan accepts launches it
UNREACHABLE = {
    **{("stft_mel_tc_kernel", (28, True, v)): "97-112 non-empty bands at hop 160: four 3072-float span buffers and the "
       "2 x 112-row operand pass 227 KB, so the plan takes stft_mel_kernel (route_tc_nb112_hop160_falls_back)"
       for v in (False, True)},
    **{("stft_mel_kernel", (4096, "c2", 512, mg)): "two frames per thread group make a 512-thread CTA transform 8 frames "
       "at once; at n_fft 4096 no 8-frame tile of 512 threads fits beside its span (every hop 1 .. 8192, 1 .. 512 bands, "
       "with and without MEL_WALK / MMA_MEL)" for mg in (False, True)},
}


def _case_kernels(cases):
    return {k for c in cases for k in c.kernels}


# one geometry per path for the properties that do not need the whole matrix
PATH_GEOMETRY = {
    "tc": TC("prop", 16000, 400, 160, 40, 0.0, 8000.0, 70),
    "tc_empty": TC("prop_empty", 10000, 250, 50, 128, 100.0, 10000.0, 70),
    "reg": R("prop", 22050, 1024, 882, 275, 64, 50.0, 11025.0, 40, threads=512),
    "reg_walk": R("prop", 16000, 512, 400, 160, 40, 0.0, 8000.0, 40, flags=WALK),
    "mma": R("prop", 16000, 512, 400, 160, 40, 0.0, 8000.0, 40, flags=MMA, mma=True),
    "power": R("prop", 44100, 2048, 2048, 441, 128, 0.0, 22050.0, 20, kind="power", threads=512),
    "tcfft": TF("prop", 160, 70),
    "gen": G("prop", 400, 400, 160, 40),
    "gen_power": G("prop", 100, 80, 40, 40, kind="power"),
}


# ---------------------------------------------------------------------------
# the path probe
# ---------------------------------------------------------------------------

_K1 = ("stft_mel_tc_kernel", "stft_mel_kernel", "mel_empty_bands_kernel", "tc_fft512_kernel", "dft_power_kernel",
       "mel_from_power_kernel")
_MANGLED_ARG = re.compile(r"Li(-?\d+)E|Lb([01])E|N(?:S_|3mmf)2(c2)E|6(float2)")


def _demangled_arg(a):
    a = a.strip()
    if a in ("true", "false"):
        return a == "true"
    if re.fullmatch(r"-?\d+", a):
        return int(a)
    return a.split("::")[-1]


def _k1_kernels(names):
    """(kernel, template arguments) of every K1 kernel among profiler kernel names, demangled
    (``void mmf::stft_mel_kernel<512, mmf::c2, 256, true>(...)``) or mangled
    (``_ZN3mmf15stft_mel_kernelILi512ENS_2c2ELi256ELb1EEEv...``).  A name matches whole: stft_mel_kernel is not
    stft_mel_tc_kernel."""
    out = []
    for name in names:
        for k in _K1:
            m = re.search(r"(?<![A-Za-z_])" + k + r"(?=[<(IE]|$)", name)
            if m is None:
                continue
            rest = name[m.end():]
            args = ()
            if rest.startswith("<"):
                args = tuple(_demangled_arg(a) for a in rest[1:rest.index(">")].split(","))
            elif rest.startswith("I"):
                got, i = [], 1
                while (a := _MANGLED_ARG.match(rest, i)) is not None:
                    iv, bv, c2, f2 = a.groups()
                    got.append(int(iv) if iv is not None else bool(int(bv)) if bv is not None else c2 or f2)
                    i = a.end()
                args = tuple(got)
            out.append((k, args))
            break
    return out


def _probe(fn):
    """Run ``fn`` under torch.profiler with CUDA activity: (result, K1 kernels that ran, launch count delta)."""
    torch = _torch()
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    n0 = _lib.lib().mmf_launch_count(0)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    launches = _lib.lib().mmf_launch_count(0) - n0
    names = [e.name for e in prof.events()]
    assert names, "the profiler saw no kernels at all: the path probe cannot tell which K1 kernel ran"
    return res, _k1_kernels(names), launches


def _expect(case, ran, launches, B=None):
    """exactly the case's kernels ran, each once per 65535-clip chunk, and mmf_launch_count counted them (+ the
    clip-max initialisation of a log-mel call)"""
    B = case.B if B is None else B
    chunks = (B + 65534) // 65535
    want = []
    for k in case.kernels:
        per = chunks if k[0] in ("mel_empty_bands_kernel", "dft_power_kernel", "mel_from_power_kernel") else 1
        want += [k] * per
    assert sorted(ran, key=repr) == sorted(want, key=repr), f"{case.id}: expected {want}, K1 kernels that ran: {ran}"
    assert launches == len(want) + (case.kind == "logmel"), (case.id, launches, len(want))


# ---------------------------------------------------------------------------
# running a case
# ---------------------------------------------------------------------------


class _Env:
    """tile-geometry overrides in the environment while a plan is created (restored afterwards)"""

    def __init__(self, env):
        self.env = dict(env)

    def __enter__(self):
        self.old = {k: os.environ.get(k) for k in self.env}
        os.environ.update(self.env)

    def __exit__(self, *exc):
        for k, v in self.old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def _make_plan(case, **over):
    cfg = case.cfg()
    if over:
        cfg = mm.plan.replace(cfg, **over)
    with _Env(case.env):
        return mm.Plan(cfg)


def _device_pcm(x, layout, device):
    """``x`` [B, n] on the device as a contiguous batch, a strided batch whose gap samples are NaN, or an unaligned
    view (base 4 bytes past a 16-byte boundary) whose preceding sample is NaN.  The poisons lie inside the buffer."""
    torch = _torch()
    B, n = x.shape
    if layout == "contig":
        return torch.as_tensor(x).to(device)
    if layout == "strided":
        pitch = (n + 7) // 4 * 4 + 4  # >= 4 gap samples, a 16-byte row pitch (the TMA path stays on)
        buf = torch.full((B, pitch), float("nan"), device=device)
        buf[:, :n] = torch.as_tensor(x).to(device)
        return buf[:, :n]
    assert layout == "unaligned"
    buf = torch.full((B * n + 8,), float("nan"), device=device)
    buf[1:1 + B * n] = torch.as_tensor(x).to(device).reshape(-1)
    v = buf[1:1 + B * n].view(B, n)
    assert v.data_ptr() % 16 == 4
    return v


def _call(plan, kind, pcm):
    if kind == "power":
        return plan.stft_power(pcm), None
    return plan.logmel(pcm)


def _grade(case, out, x, record=None):
    """the case's error against the reference; asserts the bound and the exact checks; returns the errors"""
    Pref = _ref_power(x, case.n, case.n_fft, case.win, case.hop, case.preemph)
    if case.kind == "power":
        e = _power_err(out, Pref)
        if record:
            record(case.id, power=e)
        assert e <= BOUND_POWER[case.path], f"{case.id}: power error {e:.3g} > {BOUND_POWER[case.path]:.3g}"
        return e
    W = _mel_weights(case.sr, case.n_fft, case.n_mels, case.fmin, case.fmax)
    e = _mel_err(out, Pref, W)
    if record:
        record(case.id, mel=e)
    assert e <= BOUND_MEL[case.path], f"{case.id}: mel error {e:.3g} > {BOUND_MEL[case.path]:.3g}"
    # floor cells: reference mel power exactly 0 (an empty band or an all-zero frame) -> one value, ~ -100 dB
    zero = np.einsum("mk,...kt->...mt", W, Pref) == 0.0
    if zero.any():
        fl = out[zero]
        assert np.all(fl == fl[0]) and abs(float(fl[0]) + 100.0) <= 1e-5, (case.id, np.unique(fl)[:4])
    return e


def record(case_id, **errs):
    """one line per case for the observed-maxima table of the docstring (pytest -s)"""
    print("K1ERR", case_id, " ".join(f"{k}={v:.3g}" for k, v in errs.items()))


def _check_keys(case, lm, keys):
    """the clip-max key is the key of the maximum of the clip's own output, bit for bit"""
    want = _key(lm.reshape(lm.shape[0], -1).max(axis=1))
    assert np.array_equal(keys, want), (case.id, keys, want)


# ---------------------------------------------------------------------------
# CPU: the reference, the probe parser, the case table and the bounds
# ---------------------------------------------------------------------------


@pytest.mark.parametrize("sr,n_fft,win,hop,n_mels,fmin,fmax", [
    (16000, 512, 400, 160, 40, 0.0, 8000.0), (10000, 512, 250, 50, 128, 100.0, 10000.0),
    (22050, 1024, 882, 275, 64, 50.0, 11025.0), (16000, 400, 400, 160, 40, 0.0, 8000.0),
    (8000, 17, 15, 5, 4, 0.0, 4000.0)])
def test_reference_agrees_with_the_oracle(sr, n_fft, win, hop, n_mels, fmin, fmax):
    """Without pre-emphasis the reference is the oracle's computation in float64: the oracle's stft_power (complex64
    spectrum, |X|^2 in float32, as librosa stores it) is within 2^-21 of it, relative, in every bin, the mel weights are
    the same numbers, and power_to_db(melspec, top_db=None) of the oracle's float32 projection, graded as if a kernel
    had written it, is within 2e-6 (the float32 accumulation of the oracle's einsum)."""
    x = _audio(2, 3000, sr, 5)[0]
    P = _ref_power(x, len(x), n_fft, win, hop, 0.0)
    Po = oracle.stft_power(x, n_fft, hop, win)
    assert P.shape == Po.shape
    assert np.all(np.abs(Po - P) <= 2.0 ** -21 * P)
    W = _mel_weights(sr, n_fft, n_mels, fmin, fmax)
    Wo = oracle.mel_filterbank(sr, n_fft, n_mels, fmin, fmax)
    assert np.array_equal(W, Wo.astype(np.float64))
    Lo = oracle.power_to_db(np.einsum("ft,mf->mt", Po, Wo, optimize=True), top_db=None)
    assert _mel_err(Lo.astype(np.float32), P, W) <= 2e-6
    # on the oracle's own power the float64 projection and the oracle's log10 agree to float64 rounding
    L = _ref_logmel(Po.astype(np.float64), W)
    assert np.max(np.abs(L - oracle.power_to_db(W @ Po.astype(np.float64), top_db=None))) <= 1e-12


def test_reference_preemphasis_is_the_definition():
    """With pre-emphasis the reference matches a loop that applies the definition sample by sample: y[i] = x[i] -
    a x[i - 1] with x[-1] = 0, then n_fft // 2 zeros each side, the centred periodic Hann, |DFT|^2."""
    n_fft, win, hop, a = 64, 50, 24, 0.97
    x = _audio(2, 301, 8000, 9)
    P = _ref_power(x, 301, n_fft, win, hop, a)
    af = float(np.float32(a))
    w = np.zeros(n_fft)
    lp = (n_fft - win) // 2
    for j in range(win):
        w[lp + j] = 0.5 - 0.5 * np.cos(2 * np.pi * j / win)
    for b in range(2):
        y = [float(x[b, i]) - af * (float(x[b, i - 1]) if i > 0 else 0.0) for i in range(301)]
        yp = [0.0] * (n_fft // 2) + y + [0.0] * (n_fft // 2)
        T = 1 + (len(yp) - n_fft) // hop
        assert P.shape[-1] == T
        for t in (0, 1, T // 2, T - 1):
            fr = np.array([yp[t * hop + j] * w[j] for j in range(n_fft)])
            for k in (0, 1, 7, n_fft // 2):
                X = np.sum(fr * np.exp(-2j * np.pi * k * np.arange(n_fft) / n_fft))
                assert abs(abs(X) ** 2 - P[b, k, t]) <= 1e-9 * max(1.0, P[b, :, t].max())


def test_reference_known_answers():
    """A cosine of amplitude A on bin k0 with win = n_fft: (A n_fft / 4)^2 at k0 and (A n_fft / 8)^2 at k0 +- 1 in
    frames inside the clip; an all-zero clip: exactly 0."""
    n_fft, k0, A = 256, 19, 0.75
    x = (A * np.cos(2 * np.pi * k0 * np.arange(2000) / n_fft)).astype(np.float32)
    P = _ref_power(x, 2000, n_fft, n_fft, 64, 0.0)
    for t in range(2, 1 + (2000 - n_fft) // 64):
        assert abs(P[k0, t] / (A * n_fft / 4) ** 2 - 1) < 1e-6
        assert abs(P[k0 + 1, t] / (A * n_fft / 8) ** 2 - 1) < 1e-6 and abs(P[k0 - 1, t] / (A * n_fft / 8) ** 2 - 1) < 1e-6
    assert np.all(_ref_power(np.zeros(500, np.float32), 500, n_fft, 200, 64, 0.97) == 0.0)


def test_key_encoding_orders():
    v = np.array([-np.inf, -1e30, -100.0, -1.0, -0.0, 0.0, 1.0, 3e38], np.float32)
    k = _key(v)
    assert np.all(np.diff(k[[0, 1, 2, 3, 5, 6, 7]].astype(np.int64)) > 0)


def test_k1_kernel_names_parse():
    """demangled and mangled profiler names, the exact forms the library's kernels carry"""
    names = [
        "void mmf::stft_mel_kernel<512, mmf::c2, 256, true>(CUtensorMap_st, mmf::StftArgs)",
        "void mmf::stft_mel_kernel<4096, float2, 512, false>(CUtensorMap_st, mmf::StftArgs)",
        "void mmf::stft_mel_tc_kernel<20, false, true>(CUtensorMap_st, mmf::StftTcArgs)",
        "_ZN3mmf15stft_mel_kernelILi1024ENS_2c2ELi256ELb0EEEv14CUtensorMap_stNS_8StftArgsE",
        "_ZN3mmf15stft_mel_kernelILi2048E6float2Li512ELb1EEEv14CUtensorMap_stNS_8StftArgsE",
        "_ZN3mmf18stft_mel_tc_kernelILi28ELb1ELb0EEEv14CUtensorMap_stNS_10StftTcArgsE",
        "mmf::mel_empty_bands_kernel(float*, int*, int, int, int const*, int, int, float)",
        "_ZN3mmf22mel_empty_bands_kernelEPfPiiiPKiiif",
        "mmf::tc_fft512_kernel(mmf::TcFftArgs)",
        "mmf::(anonymous namespace)::dft_power_kernel(mmf::(anonymous namespace)::DftArgs)",
        "_ZN3mmf12_GLOBAL__N_121mel_from_power_kernelENS0_10MelPowArgsE",
        "void mmf::mfcc_pk_kernel<4, 16, false>(mmf::PkArgs)", "Memset (Device)",
    ]
    assert _k1_kernels(names) == [
        ("stft_mel_kernel", (512, "c2", 256, True)), ("stft_mel_kernel", (4096, "float2", 512, False)),
        ("stft_mel_tc_kernel", (20, False, True)), ("stft_mel_kernel", (1024, "c2", 256, False)),
        ("stft_mel_kernel", (2048, "float2", 512, True)), ("stft_mel_tc_kernel", (28, True, False)),
        ("mel_empty_bands_kernel", ()), ("mel_empty_bands_kernel", ()), ("tc_fft512_kernel", ()),
        ("dft_power_kernel", ()), ("mel_from_power_kernel", ())]


def test_case_matrix_reaches_every_instantiation():
    """The case table (with the varlen test's two VL instantiations) names every K1 kernel instantiation the build
    compiles, except those listed as unreachable; every case is a configuration validate_cfg accepts, and its
    expected kernels follow the selection rules."""
    got = _case_kernels(CASES) | _case_kernels(c for _, c in VARLEN) | {_stft(n, f, 256) for _, n, f, _ in GEOMETRIES}
    missing = {k for k in WANT if k not in got} - set(UNREACHABLE)
    assert not missing, sorted(missing, key=repr)
    assert {c.path for c in CASES} == {"tc", "reg", "mma", "tcfft", "gen"}
    assert len({c.id for c in CASES}) == len(CASES)
    for c in CASES + [c for _, c in VARLEN] + list(PATH_GEOMETRY.values()):
        assert 16 <= c.n_fft <= 4096 and 1 <= c.win <= c.n_fft and c.hop >= 1 and 1 <= c.n_mels <= 512, c.id
        gen = c.n_fft < 256 or c.n_fft & (c.n_fft - 1)
        names = {k for k, _ in c.kernels}
        if gen:
            assert c.path == "gen" and names <= {"dft_power_kernel", "mel_from_power_kernel"}, c.id
        elif c.path == "tcfft":
            assert c.n_fft == 512 and c.hop <= 512 and c.preemph == 0 and c.flags & TCFFT and c.kind == "power"
        elif c.path == "tc":
            assert c.n_fft == 512 and not c.flags & _NO_TC_FLAGS and c.kind == "logmel", c.id
            n_act = _n_act(c.sr, 512, c.n_mels, c.fmin, c.fmax)
            assert ("mel_empty_bands_kernel" in names) == (n_act < c.n_mels), c.id
        else:
            assert names == {"stft_mel_kernel"}, c.id
            if c.kind == "logmel" and c.n_fft == 512 and "route_" not in c.id:
                assert c.flags & _NO_TC_FLAGS, c.id  # else the tcgen05 mel would take it
            assert c.path == ("mma" if c.mma else "reg"), c.id
    # the tc T edges, the NBQ range, interior empty bands, both FAST160 forms
    tc = [c for c in CASES if c.path == "tc"]
    assert {1, 63, 64, 65, 127, 128, 129} <= {c.T for c in tc} and max(c.T for c in tc) >= 128 * 148 * 2
    assert {k[1][0] for c in tc for k in c.kernels if k[0] == "stft_mel_tc_kernel"} == set(range(4, 29, 4))
    W = _mel_weights(44100, 512, 100, 0.0, 22050.0)
    assert 1 <= int(np.sum(~W.any(axis=1)[:_n_act(44100, 512, 100, 0.0, 22050.0)]))
    # gen n_fft list, pre-emphasis at every NFFT of the register FFT, the MMA declined shape
    assert {16, 17, 32, 64, 100, 255, 400, 401, 4095} <= {c.n_fft for c in CASES if c.path == "gen"}
    assert {256, 512, 1024, 2048, 4096} <= {c.n_fft for c in CASES if c.path in ("reg", "mma") and c.preemph}
    assert {c.mma for c in CASES if c.flags & MMA} == {True, False}
    assert {1, 160, 512} <= {c.hop for c in CASES if c.path == "tcfft"}


_MISTAKES = ["symmetric_hann", "window_left_aligned", "reflect_padding", "frames_shifted_one_hop",
             "preemph_after_padding", "preemph_across_clip_start", "htk_mel", "no_slaney_norm", "magnitude",
             "nyquist_dropped"]


def _mistake_applies(mistake, c):
    """False where the mistake cannot change the case's fixture by a margin its bounds could show"""
    if c.n < c.n_fft or c.win == 1:
        return False  # a clip shorter than one frame samples the window at a few points; win 1: all-zero window
    if mistake == "window_left_aligned":
        return c.win < c.n_fft - 1  # a window that fills n_fft (or all but one sample) has nowhere else to be
    if mistake == "symmetric_hann":
        # the two windows differ by O(1 / win): beyond 1024 samples that is within 10x of the FP32 bounds; one or
        # two wide bands average the window's shape out
        return 2 < c.win <= 1024 and (c.kind == "power" or c.n_mels >= 4)
    if mistake == "reflect_padding":
        return c.signal != "impulse"  # reflection mirrors the zeros next to the edge impulses
    if mistake == "preemph_after_padding":
        # one sample past the clip's end (-a x[n - 1]) is O(1 / n_fft) of the last frame: beyond 2048 samples
        # that is within 10x of the bounds
        return c.preemph != 0.0 and c.signal == "mix" and c.n_fft <= 2048
    if mistake == "preemph_across_clip_start":
        return c.preemph != 0.0 and c.signal == "mix"
    if mistake == "htk_mel":
        return c.kind == "logmel" and c.n_mels >= 4  # fewer, wider triangles average the two scales out
    if mistake == "no_slaney_norm":
        return c.kind == "logmel"
    if mistake == "nyquist_dropped":
        return c.kind == "power" or c.fmax > c.sr / 2  # a band reaches the Nyquist bin only above fmax = sr / 2
    return True


@pytest.mark.parametrize("mistake", _MISTAKES)
def test_tolerances_catch_plausible_mistakes(mistake):
    """Each plausible mistake misses the reference by more than 10x the bound of the path that computes the fixture,
    on the fixtures of every GPU case (float32 output, as the kernels write it) the mistake can reach."""
    worst = {}
    for i, c in enumerate(CASES):
        if not _mistake_applies(mistake, c) or c.n > 200000:
            continue
        x = _audio(c.B, c.n, c.sr, 2000 + i, c.signal)
        ref = _ref_power(x, c.n, c.n_fft, c.win, c.hop, c.preemph)
        bad = _ref_power(x, c.n, c.n_fft, c.win, c.hop, c.preemph, mistake=mistake)
        if c.kind == "power":
            miss = _power_err(bad.astype(np.float32), ref) / BOUND_POWER[c.path]
        else:
            W = _mel_weights(c.sr, c.n_fft, c.n_mels, c.fmin, c.fmax)
            Wb = _mel_weights(c.sr, c.n_fft, c.n_mels, c.fmin, c.fmax, mistake=mistake)
            miss = _mel_err(_ref_logmel(bad, Wb).astype(np.float32), ref, W) / BOUND_MEL[c.path]
        worst[c.id] = miss
    print("K1MISS", mistake, sorted(worst.items(), key=lambda kv: kv[1])[:3])
    assert worst and min(worst.values()) > 10.0, sorted(worst.items(), key=lambda kv: kv[1])[:3]


# ---------------------------------------------------------------------------
# GPU: the case matrix
# ---------------------------------------------------------------------------


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c.id for c in CASES])
def test_k1_path_matches_reference(case, cuda_device):
    x = _audio(case.B, case.n, case.sr, 100 + CASES.index(case), case.signal)
    plan = _make_plan(case)
    try:
        pcm = _device_pcm(x, case.layout, cuda_device)
        (out, keys), ran, launches = _probe(lambda: _call(plan, case.kind, pcm))
        _expect(case, ran, launches)
        out = out.cpu().numpy()
        assert np.all(np.isfinite(out)), case.id
        _grade(case, out, x, record)
        if case.kind == "logmel":
            _check_keys(case, out, keys.cpu().numpy())
        if case.B > 1 and case.signal == "mix" and case.kind == "power":
            assert np.all(out[-1] == 0.0)  # the all-zero clip
        if case.mma is not None:
            # MMA_MEL accepted: not the per-bin walk's bits; declined: exactly the per-bin walk's plan
            walk = _make_plan(case, flags=case.flags & ~MMA | WALK)
            try:
                w, _ = walk.logmel(pcm)
                same = np.array_equal(w.cpu().numpy().view(np.int32), out.view(np.int32))
            finally:
                walk.close()
            assert same != case.mma, (case.id, "mma accepted" if not same else "mma declined")
    finally:
        plan.close()


@pytest.mark.gpu
@pytest.mark.parametrize("geo", GEOMETRIES, ids=[g[0] for g in GEOMETRIES])
def test_forced_tile_geometry_keeps_the_bits(geo, cuda_device, monkeypatch):
    """MMF_TF / MMF_SPAN_BUFS / MMF_PT_BUFS / MMF_NO_512 at plan creation: the kernel runs the forced tile (256
    threads) and gives the default plan's bits, over T = TF - 1, TF, TF + 1 and a longer clip."""
    gid, n_fft, flags, env = geo
    sr, win, hop, n_mels, fmax = (_GEO_SHAPE_NO_512 if gid.startswith("no_512") else _GEO_SHAPE)[n_fft]
    pre = 0.97 if "preemph" in gid else 0.0
    tf = int(dict(env).get("MMF_TF", "0"))
    base = Case(gid, "mma" if flags & MMA else "reg", "logmel", sr, n_fft, win, hop, n_mels, 0.0, fmax, 1,
                (_stft(n_fft, flags, 256),), preemph=pre, flags=flags, B=4, mma=bool(flags & MMA) or None)
    ref = mm.Plan(base.cfg())
    for k, v in env:
        monkeypatch.setenv(k, v)
    forced = mm.Plan(base.cfg())
    try:
        for T in sorted({max(1, tf - 1), max(1, tf), tf + 1, 37}):
            c = base._replace(n=_frames_for(T, hop))
            x = _audio(c.B, c.n, sr, 500 + T)
            pcm = _device_pcm(x, "contig", cuda_device)
            (out, keys), ran, launches = _probe(lambda: forced.logmel(pcm))
            _expect(c, ran, launches)
            a, ka = ref.logmel(pcm)
            out = out.cpu().numpy()
            bad = np.argwhere(out.view(np.int32) != a.cpu().numpy().view(np.int32))
            assert bad.size == 0, (gid, T, bad[:5].tolist())
            assert np.array_equal(keys.cpu().numpy(), ka.cpu().numpy())
            _grade(c, out, x, record)
    finally:
        forced.close()
        ref.close()


# ---------------------------------------------------------------------------
# GPU: properties on one geometry per path
# ---------------------------------------------------------------------------


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(PATH_GEOMETRY))
def test_clip_bits_do_not_depend_on_the_batch(name, cuda_device):
    """A clip gives the same bits (and key) alone, in a batch and in a permuted batch."""
    case = PATH_GEOMETRY[name]._replace(B=5)
    x = _audio(5, case.n, case.sr, 41)
    plan = _make_plan(case)
    try:
        out, keys = _call(plan, case.kind, _device_pcm(x, "contig", cuda_device))
        perm = [3, 0, 4, 2, 1]
        po, pk = _call(plan, case.kind, _device_pcm(x[perm], "contig", cuda_device))
        out = out.cpu().numpy()
        assert np.array_equal(po.cpu().numpy().view(np.int32), out[perm].view(np.int32))
        for b in range(5):
            so, sk = _call(plan, case.kind, _device_pcm(x[b:b + 1], "contig", cuda_device))
            assert np.array_equal(so.cpu().numpy()[0].view(np.int32), out[b].view(np.int32)), (name, b)
            if keys is not None:
                assert int(sk.cpu()[0]) == int(keys.cpu()[b])
        if keys is not None:
            assert np.array_equal(pk.cpu().numpy(), keys.cpu().numpy()[perm])
    finally:
        plan.close()


@pytest.mark.gpu
@pytest.mark.parametrize("preemph", [0.0, 0.97], ids=["plain", "preemph"])
@pytest.mark.parametrize("name", list(PATH_GEOMETRY))
def test_loaders_stay_inside_each_clip(name, preemph, cuda_device):
    """TMA, MMF_FLAG_NO_TMA, an unaligned base whose preceding sample is NaN and a strided batch whose gap samples
    are NaN give identical, finite bits: no loader reads outside a clip's own samples."""
    case = PATH_GEOMETRY[name]
    if preemph and case.path == "tcfft":
        pytest.skip("the tensor-core transform takes no pre-emphasis (the plan falls back to the register FFT)")
    case = case._replace(preemph=preemph)
    x = _audio(case.B, case.n, case.sr, 43)
    plan = _make_plan(case)
    no_tma = _make_plan(case, flags=case.flags | NO_TMA)
    try:
        outs = {}
        for layout in ("contig", "strided", "unaligned"):
            o, k = _call(plan, case.kind, _device_pcm(x, layout, cuda_device))
            outs[layout] = (o.cpu().numpy(), None if k is None else k.cpu().numpy())
        o, k = _call(no_tma, case.kind, _device_pcm(x, "contig", cuda_device))
        outs["no_tma"] = (o.cpu().numpy(), None if k is None else k.cpu().numpy())
        a, ka = outs["contig"]
        assert np.all(np.isfinite(a))
        for layout, (o, k) in outs.items():
            assert np.array_equal(o.view(np.int32), a.view(np.int32)), (name, layout)
            if k is not None:
                assert np.array_equal(k, ka), (name, layout)
        _grade(case, a, x)
    finally:
        no_tma.close()
        plan.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,win,hop,pre,flags", [
    (256, 200, 80, 0.0, 0), (512, 400, 160, 0.97, 0), (512, 512, 128, 0.0, SCALAR), (1024, 882, 275, 0.0, 0),
    (2048, 2048, 441, 0.97, SCALAR), (4096, 3840, 960, 0.0, 0), (100, 80, 40, 0.97, 0), (401, 401, 100, 0.0, 0)])
def test_fp32_transforms_are_linear(n_fft, win, hop, pre, flags, cuda_device):
    """power(2 x) == 4 power(x) bit for bit on the register FFT and the generic DFT: every step is linear in x and
    scaling by 2 is exact away from underflow and overflow."""
    cfg = mm.MfccConfig(16000.0, n_fft, win, hop, 40, 1, 0.0, 8000.0, preemph=pre, flags=flags)
    x = _audio(3, 3000, 16000.0, 47)[:2]
    plan = mm.Plan(cfg)
    try:
        p1 = plan.stft_power(_device_pcm(x, "contig", cuda_device)).cpu().numpy()
        p2 = plan.stft_power(_device_pcm(2 * x, "contig", cuda_device)).cpu().numpy()
    finally:
        plan.close()
    assert np.array_equal(p2.view(np.int32), (4 * p1).view(np.int32))


def _varlen_cases():
    """(id, case) of the variable-length path (mfcc_change_varlen with the log-mel output): the first contiguous tc
    case of every (NBQ, FAST160), with the VL = true instantiation, at 129 frames or more; one register-FFT case."""
    out = {}
    for c in CASES:
        if c.path == "tc" and c.layout != "unaligned":
            k, args = c.kernels[0]
            if args[:2] not in out:
                vc = c._replace(kernels=((k, args[:2] + (True,)),) + c.kernels[1:], n=max(c.n, 128 * c.hop), B=4)
                out[args[:2]] = (f"nbq{args[0]}_{'fast' if args[1] else 'generic'}", vc)
    return list(out.values()) + [("reg", R("varlen", 22050, 1024, 882, 275, 64, 50.0, 11025.0, 60, B=4, threads=512))]


VARLEN = _varlen_cases()


@pytest.mark.gpu
@pytest.mark.parametrize("vid,case", VARLEN, ids=[v[0] for v in VARLEN])
def test_varlen_logmel_equals_solo_calls(vid, case, cuda_device):
    """Clips of different lengths in one call: each clip's log-mel equals its solo call bit for bit; the tc path runs
    its VL = true instantiation, the register-FFT path one stft_mel_kernel launch for the whole batch."""
    lens = [case.n, case.n // 3 + 7, case.n - 3 * case.hop - 1, case.n // 2]
    x = _audio(4, case.n, case.sr, 53)
    plan = _make_plan(case, top_db=None)  # the change path clamps its log-mel output in place unless top_db is off
    try:
        prm = mm.make_change_params(np.array([[1.0, 0, 0, 1.0, 0, 0]]), remove_first=0)
        pcm = _device_pcm(x, "contig", cuda_device)
        res, ran, _ = _probe(lambda: plan.mfcc_change_varlen(pcm, lens, prm, want_logmel=True))
        want = sorted(case.kernels, key=repr)
        assert sorted(ran, key=repr) == want, (vid, ran)
        lm = res["logmel"].cpu().numpy()
        for b, n in enumerate(lens):
            solo, _ = plan.logmel(_device_pcm(x[b:b + 1, :n], "contig", cuda_device))
            solo = solo.cpu().numpy()[0]
            T = solo.shape[-1]
            assert int(res["frames"][b]) == T
            assert np.array_equal(lm[b, :, :T].view(np.int32), solo.view(np.int32)), (vid, b)
            c = case._replace(n=n, B=1)
            _grade(c, solo[None], x[b:b + 1, :n])
    finally:
        plan.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["reg256", "reg512", "reg1024", "reg2048", "reg4096", "gen100", "tcfft"])
def test_known_answers(name, cuda_device):
    """A cosine of amplitude A on bin k0, win = n_fft: (A n_fft / 4)^2 at k0, (A n_fft / 8)^2 at k0 +- 1 and ~0
    elsewhere, in every frame that lies wholly inside the clip."""
    n_fft = int(re.sub(r"\D", "", name) or 512)
    path = "gen" if name.startswith("gen") else name if name == "tcfft" else "reg"
    cfg = mm.MfccConfig(16000.0, n_fft, n_fft, n_fft // 4, 40, 1, 0.0, 8000.0, flags=TCFFT if path == "tcfft" else 0)
    k0, A, n = n_fft // 8 + 3, 0.75, 6 * n_fft
    x = (A * np.cos(2 * np.pi * k0 * np.arange(n) / n_fft)).astype(np.float32)[None]
    plan = mm.Plan(cfg)
    try:
        (P, _), ran, _ = _probe(lambda: _call(plan, "power", _device_pcm(x, "contig", cuda_device)))
    finally:
        plan.close()
    assert {k for k, _ in ran} == {"gen": {"dft_power_kernel"}, "tcfft": {"tc_fft512_kernel"},
                                   "reg": {"stft_mel_kernel"}}[path]
    P = P.cpu().numpy()[0].astype(np.float64)
    peak = (A * n_fft / 4) ** 2
    tol = BOUND_POWER[path] * peak
    inside = [t for t in range(P.shape[1]) if t * cfg.hop_length >= n_fft // 2 and t * cfg.hop_length + n_fft // 2 <= n]
    assert len(inside) >= 3
    for t in inside:
        want = np.zeros(n_fft // 2 + 1)
        want[k0] = peak
        want[k0 - 1] = want[k0 + 1] = (A * n_fft / 8) ** 2
        assert np.max(np.abs(P[:, t] - want)) <= tol, (name, t, np.max(np.abs(P[:, t] - want)) / peak)


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["tc", "gen", "gen_power"])
def test_clip_chunks_of_65535(path, cuda_device):
    """65 537 tiny clips: the tc path's mel_empty_bands_kernel (trailing empty bands) and both generic kernels are
    launched for clips [0, 65535) and [65535, 65537); clips on both sides of the boundary match the reference."""
    base = {"tc": PATH_GEOMETRY["tc_empty"], "gen": G("chunks", 16, 16, 4, 2, n_mels=4),
            "gen_power": G("chunks", 16, 16, 4, 2, kind="power")}[path]
    B = 65537
    case = base._replace(B=B, n=5 if path != "tc" else 60, preemph=0.97 if path == "gen" else 0.0)
    if path == "tc":
        case = case._replace(kernels=(("stft_mel_tc_kernel", (28, False, False)), ("mel_empty_bands_kernel", ())))
    rng = np.random.default_rng(59)
    x = (rng.standard_normal((B, case.n)) * rng.uniform(0.01, 10.0, (B, 1))).astype(np.float32)
    x[65534:65536] *= 100.0
    plan = _make_plan(case)
    try:
        (out, keys), ran, launches = _probe(lambda: _call(plan, case.kind, _device_pcm(x, "contig", cuda_device)))
    finally:
        plan.close()
    _expect(case, ran, launches)
    out = out.cpu().numpy()
    sel = np.r_[0:3, 65530:65537]
    _grade(case._replace(B=len(sel)), out[sel], x[sel])
    if keys is not None:
        _check_keys(case, out, keys.cpu().numpy())


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft", [256, 1024])
def test_largest_accepted_hop(n_fft, cuda_device):
    """The largest hop a plan accepts (found by bisection; a refusal is MMF_ERR_UNSUPPORTED for shared memory) runs
    within its bound."""
    def make(hop):
        try:
            return mm.Plan(mm.MfccConfig(16000.0, n_fft, n_fft, hop, 40, 1, 0.0, 8000.0))
        except mm.MmfError as e:
            assert e.code == _lib.MMF_ERR_UNSUPPORTED and "shared memory" in e.msg, e
            return None

    lo, hi = n_fft, 1 << 20
    p = make(hi)
    assert p is None
    while hi - lo > 1:
        mid = (lo + hi) // 2
        p = make(mid)
        if p is None:
            hi = mid
        else:
            p.close()
            lo = mid
    case = R("largest_hop", 16000.0, n_fft, n_fft, lo, 40, 0.0, 8000.0, 3)
    x = _audio(2, case.n + 5, 16000.0, 61)
    case = case._replace(n=x.shape[1], B=2, kernels=())
    plan = make(lo)
    try:
        out, keys = plan.logmel(_device_pcm(x, "contig", cuda_device))
    finally:
        plan.close()
    record(case.id + f"_hop{lo}")
    _grade(case, out.cpu().numpy(), x, record)


_SWEEP = [(nf, nm, hop, fl) for nf in (16, 256, 512, 1024, 2048, 4096) for nm in (1, 128, 512)
          for hop in (1, max(1, nf // 4), nf, 2 * nf) for fl in (0, SCALAR, WALK, MMA, NO_TC)]


@pytest.mark.gpu
def test_plan_acceptance_sweep(cuda_device):
    """Every plan over n_fft x n_mels x hop x flags is refused at creation (MMF_ERR_UNSUPPORTED, shared memory) or
    runs mmf_logmel within the bound of the path that ran; no launch fails."""
    x = _audio(2, 700, 16000.0, 67)[:1]
    pcm = _device_pcm(x, "contig", cuda_device)
    refused, worst = [], {}
    for nf, nm, hop, fl in _SWEEP:
        cfg = mm.MfccConfig(16000.0, nf, nf, hop, nm, 1, 0.0, 8000.0, flags=fl)
        try:
            plan = mm.Plan(cfg)
        except mm.MmfError as e:
            assert e.code == _lib.MMF_ERR_UNSUPPORTED and "shared memory" in e.msg, (nf, nm, hop, fl, e)
            refused.append((nf, nm, hop, fl))
            continue
        try:
            (out, keys), ran, _ = _probe(lambda: plan.logmel(pcm))
        finally:
            plan.close()
        names = {k for k, _ in ran}
        path = ("tc" if "stft_mel_tc_kernel" in names else "gen" if "dft_power_kernel" in names
                else "mma" if fl & MMA else "reg")
        case = Case(f"sweep_{nf}_{nm}_{hop}_{fl}", path, "logmel", 16000.0, nf, nf, hop, nm, 0.0, 8000.0, 700, ())
        out = out.cpu().numpy()
        worst[case.id] = _grade(case._replace(B=1), out, x)
        _check_keys(case, out, keys.cpu().numpy())
        print("K1SWEEP", case.id, sorted(ran, key=repr))
    print("K1SWEEP refused", refused)
    record("sweep_max", mel=max(worst.values()))
