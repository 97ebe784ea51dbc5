"""Plans: a frozen frame/spectrum configuration bound to one CUDA device.

A :class:`Plan` owns the device-side constant tables (Hann window, FFT twiddles,
sparse Slaney mel bank, padded DCT rows) and exposes one method per C-ABI entry
point, taking and returning ``torch`` CUDA tensors (torch is used for device
memory and streams only; all arithmetic happens in ``libmmf_b200.so``).
"""

from __future__ import annotations

import ctypes as C
import math
from collections import OrderedDict
from dataclasses import dataclass, replace

import numpy as np

from . import _lib
from ._lib import (
    MmfError,
    check,
    mmf_amp_params,
    mmf_change_params,
    mmf_config,
    mmf_env_params,
    mmf_modspec_params,
    mmf_out_filter,
)


@dataclass(frozen=True)
class MfccConfig:
    """Arguments librosa.feature.mfcc sees at script/mfcc.py:387 (+ librosa defaults)."""

    sample_rate: float
    n_fft: int = 512
    win_length: int = 400
    hop_length: int = 160
    n_mels: int = 128
    n_mfcc: int = 13
    fmin: float = 0.0
    fmax: float | None = None
    amin: float = 1e-10
    top_db: float | None = 80.0
    preemph: float = 0.0
    device: int = 0
    flags: int = 0

    def to_c(self) -> mmf_config:
        return mmf_config(
            float(self.sample_rate),
            int(self.n_fft),
            int(self.win_length),
            int(self.hop_length),
            int(self.n_mels),
            int(self.n_mfcc),
            float(self.fmin),
            float(self.sample_rate / 2 if self.fmax is None else self.fmax),
            float(self.amin),
            float(-1.0 if self.top_db is None else self.top_db),
            float(self.preemph),
            int(self.device),
            int(self.flags),
        )

    @property
    def n_bins(self) -> int:
        return self.n_fft // 2 + 1


def frame_sizes(sigSr: float, winLen: float, tStep: float) -> tuple[int, int]:
    """``int(winLen*sigSr)``, ``int(tStep*sigSr)`` -- Python truncation, script/mfcc.py:382-384."""
    return int(winLen * sigSr), int(tStep * sigSr)


def num_frames(n_samples: int, n_fft: int, hop_length: int) -> int:
    return int(_lib.lib().mmf_num_frames(int(n_samples), int(n_fft), int(hop_length)))


def host_tables(cfg: MfccConfig):
    """(window[n_fft], mel[n_mels, F], dct[n_mfcc, n_mels]) exactly as a plan uploads them (no GPU needed)."""
    c = cfg.to_c()
    w = np.zeros(cfg.n_fft, np.float32)
    m = np.zeros((cfg.n_mels, cfg.n_bins), np.float32)
    d = np.zeros((cfg.n_mfcc, cfg.n_mels), np.float32)
    check(_lib.lib().mmf_host_tables(C.byref(c), w.ctypes.data, m.ctypes.data, d.ctypes.data))
    return w, m, d


def sos_zi(sos: np.ndarray):
    """(zi[n_sections, 2], padlen) as scipy.signal.sosfilt_zi / sosfiltfilt compute them."""
    sos = np.ascontiguousarray(sos, dtype=np.float64)
    zi = np.zeros((sos.shape[0], 2), np.float64)
    padlen = C.c_int32(0)
    check(_lib.lib().mmf_sos_zi(sos.ctypes.data, sos.shape[0], zi.ctypes.data, C.byref(padlen)))
    return zi, int(padlen.value)


def make_change_params(
    sos: np.ndarray, *, remove_first: int = 1, diff_method: int = 0, out_sos: np.ndarray | None = None
) -> mmf_change_params:
    """Pack the post-MFCC parameters of get_MFCCS_change (script/mfcc.py:393-425)."""
    prm = mmf_change_params()
    sos = np.ascontiguousarray(sos, dtype=np.float64)
    if sos.ndim != 2 or sos.shape[1] != 6 or sos.shape[0] > 16:
        raise ValueError("sos must be [n_sections <= 16, 6]")
    prm.remove_first = int(bool(remove_first))
    prm.diff_method = int(diff_method)
    prm.n_sections = sos.shape[0]
    for i, v in enumerate(sos.ravel()):
        prm.sos[i] = v
    if out_sos is None:
        prm.out_kind = 1
        prm.out_n_sections = 0
    else:
        out_sos = np.ascontiguousarray(out_sos, dtype=np.float64)
        if out_sos.ndim != 2 or out_sos.shape[1] != 6 or out_sos.shape[0] > 16:
            raise ValueError("out_sos must be [n_sections <= 16, 6]")
        prm.out_kind = 0
        prm.out_n_sections = out_sos.shape[0]
        for i, v in enumerate(out_sos.ravel()):
            prm.out_sos[i] = v
    return prm


def _torch():
    import torch

    return torch


def _stream_ptr(device) -> int:
    return int(_torch().cuda.current_stream(device).cuda_stream)


def design_resample_filter(n_in: int, up: int, down: int, quality: str = "scipy"):
    """Taps (float32, zero-padded for the polyphase bookkeeping), samples to drop at the front of the full
    convolution, and output length, for ``y = upfirdn(h, x, up, down)[n_pre_remove : n_pre_remove + n_out]``.

    ``"scipy"`` restates scipy/signal/_signaltools.py resample_poly (filter design and edge bookkeeping) -- the
    output is bit-compatible with it up to float32 rounding.  ``"hq"`` keeps the bookkeeping and swaps the filter:
    Kaiser-windowed sinc with the transition band 0.913 .. 1.0 of the lower Nyquist at 120 dB (beta 12.27,
    90 taps per phase side), i.e. libsoxr HQ's band limits -- what ``librosa.load`` applies at script/mfcc.py:373.
    Content below 0.9 of the lower Nyquist comes through within 1e-5 of the ideal band-limited resampling
    (tests/test_host.py::test_hq_resampler_is_transparent_below_the_band_edge); libsoxr's own output cannot be
    compared here (not installed, no network)."""
    import scipy.signal

    half_len, n_pre_pad, n_post_pad, n_pre_remove, n_out = _resample_geometry(n_in, up, down, quality)
    max_rate = max(up, down)
    if quality == "scipy":
        h = scipy.signal.firwin(2 * half_len + 1, 1.0 / max_rate, window=("kaiser", 5.0))
    else:
        h = scipy.signal.firwin(2 * half_len + 1, 0.9565 / max_rate, window=("kaiser", 12.27))
    h = h.astype(np.float32) * up
    h = np.concatenate((np.zeros(n_pre_pad, dtype=h.dtype), h, np.zeros(n_post_pad, dtype=h.dtype)))
    return np.ascontiguousarray(h, dtype=np.float32), n_pre_remove, n_out


def _resample_geometry(n_in: int, up: int, down: int, quality: str):
    """The edge bookkeeping of :func:`design_resample_filter` without the filter design: (half_len, n_pre_pad,
    n_post_pad, n_pre_remove, n_out).  The taps are ``n_pre_pad`` zeros, the ``2 * half_len + 1`` designed taps and
    ``n_post_pad`` zeros; only the padding depends on ``n_in``."""
    from scipy.signal._upfirdn import _output_len

    n_out = n_in * up
    n_out = n_out // down + bool(n_out % down)
    if quality not in ("scipy", "hq"):
        raise ValueError("quality must be 'scipy' or 'hq'")
    half_len = (10 if quality == "scipy" else 90) * max(up, down)
    n_pre_pad = down - half_len % down
    n_post_pad = 0
    n_pre_remove = (half_len + n_pre_pad) // down
    while _output_len(2 * half_len + 1 + n_pre_pad + n_post_pad, n_in, up, down) < n_out + n_pre_remove:
        n_post_pad += 1
    return half_len, n_pre_pad, n_post_pad, n_pre_remove, n_out


def resample_ratio(sr_in: float, sr: float):
    """``(up, down)`` that brings audio at ``sr_in`` to ``sr``: ``Fraction(sr / sr_in).limit_denominator(1000)``,
    reduced by the gcd as :meth:`Plan.resample_poly` reduces it; ``(1, 1)`` when the rates are equal.  The WAV loader
    and the packed resampling bundle share it, so a clip gets the same ratio on either route."""
    from fractions import Fraction

    if float(sr_in) == float(sr):
        return 1, 1
    fr = Fraction(float(sr) / float(sr_in)).limit_denominator(1000)
    g = math.gcd(fr.numerator, fr.denominator)
    return fr.numerator // g, fr.denominator // g


# mmf_resample_clip as a numpy record (C layout; mmf_abi_sizeof(3) checks it)
RESAMPLE_CLIP = np.dtype(
    [("up", np.int32), ("down", np.int32), ("tap0", np.int64), ("len_h", np.int32), ("n_pre_remove", np.int64),
     ("n_out", np.int64)],
    align=True,
)


def resample_descriptors(lengths, rates, sr: float):
    """The tap table and the ``mmf_resample_clip`` descriptors that bring clips of ``lengths`` samples at ``rates``
    to ``sr`` with the ``"hq"`` filter (the loader's).  One table entry per distinct ratio, designed for the longest
    clip of that ratio and zero-padded to the longest ``len_h`` of any of them (the designs of one ratio differ only in
    trailing zeros); each clip's ``len_h``, ``n_pre_remove`` and ``n_out`` are ``design_resample_filter``'s for its own
    length.  Plan-rate clips get ``up = down = 1``.  Returns ``(rs, h)``: a ``RESAMPLE_CLIP`` array and float32 taps."""
    lengths = np.asarray(lengths, dtype=np.int64).reshape(-1)
    rates = list(np.asarray(rates, dtype=np.float64).reshape(-1))
    if len(rates) != len(lengths):
        raise ValueError(f"rates has {len(rates)} entries for {len(lengths)} clips")
    rs = np.zeros(len(lengths), RESAMPLE_CLIP)
    ratio = [resample_ratio(r, sr) for r in rates]
    groups = {}
    for i, (up, down) in enumerate(ratio):
        n = int(lengths[i])
        rs[i]["up"], rs[i]["down"] = up, down
        if (up, down) == (1, 1):
            rs[i]["n_out"] = n
            continue
        half_len, n_pre_pad, n_post_pad, n_pre_remove, n_out = _resample_geometry(n, up, down, "hq")
        rs[i]["len_h"] = n_pre_pad + 2 * half_len + 1 + n_post_pad
        rs[i]["n_pre_remove"], rs[i]["n_out"] = n_pre_remove, n_out
        groups.setdefault((up, down), []).append(i)
    tables, tap0 = [], 0
    for (up, down), idx in groups.items():
        longest = max(idx, key=lambda i: int(lengths[i]))
        h, _, _ = design_resample_filter(int(lengths[longest]), up, down, "hq")
        h = np.concatenate([h, np.zeros(max(int(rs[i]["len_h"]) for i in idx) - len(h), np.float32)])
        rs["tap0"][idx] = tap0
        tables.append(h)
        tap0 += len(h)
    h = np.concatenate(tables) if tables else np.zeros(0, np.float32)
    return rs, np.ascontiguousarray(h, dtype=np.float32)


class Plan:
    """Device-resident plan (``mmf_plan``).  Not thread-safe: one plan per host thread."""

    def __init__(self, cfg: MfccConfig):
        torch = _torch()
        if not torch.cuda.is_available():
            raise MmfError(_lib.MMF_ERR_CUDA, "no CUDA device available (this package has no CPU fallback)")
        self.cfg = cfg
        self.device = torch.device("cuda", cfg.device)
        self._h = C.c_void_p()
        c = cfg.to_c()
        check(_lib.lib().mmf_plan_create(C.byref(self._h), C.byref(c)))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            _lib.lib().mmf_plan_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- helpers -----------------------------------------------------------
    def _pcm(self, pcm):
        torch = _torch()
        if not isinstance(pcm, torch.Tensor):
            pcm = torch.as_tensor(np.ascontiguousarray(pcm, dtype=np.float32)).to(self.device, non_blocking=True)
        if pcm.device != self.device:
            pcm = pcm.to(self.device)
        if pcm.dtype != torch.float32:
            pcm = pcm.to(torch.float32)
        if pcm.dim() == 1:
            pcm = pcm[None, :]
        if pcm.dim() != 2:
            raise ValueError("pcm must be [n_clips, n_samples]")
        if pcm.stride(1) != 1:
            pcm = pcm.contiguous()
        return pcm

    def num_frames(self, n_samples: int) -> int:
        return num_frames(n_samples, self.cfg.n_fft, self.cfg.hop_length)

    # -- kernels -----------------------------------------------------------
    def stft_power(self, pcm):
        """|STFT|^2 -> float32 [B, F, T]."""
        torch = _torch()
        pcm = self._pcm(pcm)
        B, N = pcm.shape
        T = self.num_frames(N)
        out = torch.empty((B, self.cfg.n_bins, T), device=self.device, dtype=torch.float32)
        check(
            _lib.lib().mmf_stft_power(
                self._h, pcm.data_ptr(), B, N, pcm.stride(0) if B > 1 else N, out.data_ptr(), _stream_ptr(self.device)
            )
        )
        return out

    def logmel(self, pcm):
        """Unclamped log-mel [B, n_mels, T] float32 and the per-clip max keys [B] int32."""
        torch = _torch()
        pcm = self._pcm(pcm)
        B, N = pcm.shape
        T = self.num_frames(N)
        out = torch.empty((B, self.cfg.n_mels, T), device=self.device, dtype=torch.float32)
        cmax = torch.empty((B,), device=self.device, dtype=torch.int32)
        check(
            _lib.lib().mmf_logmel(
                self._h,
                pcm.data_ptr(),
                B,
                N,
                pcm.stride(0) if B > 1 else N,
                out.data_ptr(),
                cmax.data_ptr(),
                _stream_ptr(self.device),
            )
        )
        return out, cmax

    def mfcc(self, logmel, clipmax, *, delta: bool = False, clamp_in_place: bool = True):
        """top_db clamp + DCT-II: MFCC [B, n_mfcc, T] (and np.gradient delta)."""
        torch = _torch()
        B, _, T = logmel.shape
        out = torch.empty((B, self.cfg.n_mfcc, T), device=self.device, dtype=torch.float32)
        d = torch.empty_like(out) if delta else None
        check(
            _lib.lib().mmf_mfcc(
                self._h,
                logmel.data_ptr(),
                clipmax.data_ptr(),
                B,
                T,
                out.data_ptr(),
                d.data_ptr() if delta else None,
                1 if clamp_in_place else 0,
                _stream_ptr(self.device),
            )
        )
        return (out, d) if delta else out

    def sosfiltfilt(self, x, sos):
        """scipy.signal.sosfiltfilt(sos, x) along the last axis -> float64."""
        torch = _torch()
        sos = np.ascontiguousarray(sos, dtype=np.float64)
        if x.dtype not in (torch.float32, torch.float64):
            x = x.to(torch.float64)
        x = x.contiguous()
        T = x.shape[-1]
        rows = x.numel() // T
        y = torch.empty(x.shape, device=self.device, dtype=torch.float64)
        check(
            _lib.lib().mmf_sosfiltfilt(
                self._h,
                x.data_ptr(),
                1 if x.dtype == torch.float32 else 0,
                rows,
                T,
                T,
                sos.ctypes.data,
                sos.shape[0],
                y.data_ptr(),
                T,
                _stream_ptr(self.device),
            )
        )
        return y

    def delta_norm(self, x, method: int = 0):
        """x float64 [B, rows, T] -> sqrt(sum_rows d^2)/rows, float64 [B, T]."""
        torch = _torch()
        x = x.contiguous()
        B, R, T = x.shape
        out = torch.empty((B, T), device=self.device, dtype=torch.float64)
        check(_lib.lib().mmf_delta_norm(self._h, x.data_ptr(), B, R, T, method, out.data_ptr(), _stream_ptr(self.device)))
        return out

    def fir_filtfilt(self, x, b):
        """scipy.signal.filtfilt(b, 1, x) along the last axis, float64."""
        torch = _torch()
        b = np.ascontiguousarray(b, dtype=np.float64)
        x = x.to(torch.float64).contiguous()
        T = x.shape[-1]
        rows = x.numel() // T
        y = torch.empty_like(x)
        work = torch.empty((rows, T + 6 * len(b)), device=self.device, dtype=torch.float64)
        check(
            _lib.lib().mmf_fir_filtfilt(
                self._h, x.data_ptr(), rows, T, b.ctypes.data, len(b), y.data_ptr(), work.data_ptr(), _stream_ptr(self.device)
            )
        )
        return y

    def stencil(self, x, coef, edge_l, edge_r):
        """Banded stencil with dense boundary rows along the last axis, float64."""
        torch = _torch()
        coef = np.ascontiguousarray(coef, dtype=np.float64)
        edge_l = np.ascontiguousarray(edge_l, dtype=np.float64)
        edge_r = np.ascontiguousarray(edge_r, dtype=np.float64)
        half = (len(coef) - 1) // 2
        n_edge, n_edge_in = edge_l.shape if edge_l.size else (0, 0)
        x = x.to(torch.float64).contiguous()
        T = x.shape[-1]
        rows = x.numel() // T
        y = torch.empty_like(x)
        check(
            _lib.lib().mmf_stencil(
                self._h,
                x.data_ptr(),
                rows,
                T,
                coef.ctypes.data,
                half,
                edge_l.ctypes.data if n_edge else None,
                edge_r.ctypes.data if n_edge else None,
                n_edge,
                n_edge_in,
                y.data_ptr(),
                _stream_ptr(self.device),
            )
        )
        return y

    def filter_varlen(self, x, offsets_or_lengths, filt: "OutFilter"):
        """The output filter ``filt`` (:func:`fir_filter` / :func:`stencil_filter`) over rows of any lengths, in a
        fixed number of launches (``mmf_filter_varlen``).  ``x`` is a float64 or float32 device tensor: 1-D packed,
        row ``i`` being ``x[offsets[i]:offsets[i + 1]]`` (``offsets_or_lengths`` holds ``B + 1`` offsets), or 2-D
        ``[B, T_max]`` padded, row ``i`` being ``x[i, :lengths[i]]`` (``B`` lengths).  Returns float64 in the same
        layout (the padding is 0); each row equals :meth:`fir_filtfilt` / :meth:`stencil` on that row
        alone, bit for bit."""
        torch = _torch()
        if x.dtype not in (torch.float32, torch.float64):
            x = x.to(torch.float64)
        x = x.contiguous()
        v = np.ascontiguousarray(np.asarray(offsets_or_lengths, dtype=np.int64).reshape(-1))
        if x.dim() == 1:
            if v.shape[0] < 2:
                raise ValueError("offsets needs at least two entries")
            x_off, T = np.ascontiguousarray(v[:-1]), np.ascontiguousarray(np.diff(v))
            if v[-1] > x.shape[0] or v[0] < 0 or np.any(T < 0):
                raise ValueError("offsets must be non-decreasing and within the buffer")
        elif x.dim() == 2:
            if v.shape[0] != x.shape[0]:
                raise ValueError(f"{v.shape[0]} lengths for {x.shape[0]} rows")
            if np.any(v > x.shape[1]):
                raise ValueError(f"a length exceeds the row length {x.shape[1]}")
            x_off, T = np.arange(x.shape[0], dtype=np.int64) * x.shape[1], v
        else:
            raise ValueError("filter_varlen takes a 1-D packed or a 2-D padded tensor")
        y = torch.zeros(x.shape, device=self.device, dtype=torch.float64)
        check(
            _lib.lib().mmf_filter_varlen(
                self._h, C.byref(filt.c), x.data_ptr(), 1 if x.dtype == torch.float32 else 0, T.shape[0],
                x_off.ctypes.data, T.ctypes.data, y.data_ptr(), x_off.ctypes.data, _stream_ptr(self.device),
            )
        )
        return y

    def modspec(self, mfcc, win: int, hop: int, nfft: int, band_bins=None, *, want_mag: bool = True):
        """Modulation spectrum of [B, C, T] float32 trajectories.

        Returns (mag [B, C, n_win, nfft/2+1] or None, band [B, n_win, n_bands] or None)."""
        torch = _torch()
        mfcc = mfcc.contiguous()
        B, Cc, T = mfcc.shape
        n_win = 1 + (T - win) // hop if T >= win and hop >= 1 else 0
        nb = nfft // 2 + 1
        mag = torch.empty((B, Cc, n_win, nb), device=self.device, dtype=torch.float32) if want_mag else None
        band = None
        lo = hi = None
        n_bands = 0
        if band_bins is not None and len(band_bins):
            n_bands = len(band_bins)
            lo = np.ascontiguousarray([b[0] for b in band_bins], dtype=np.int32)
            hi = np.ascontiguousarray([b[1] for b in band_bins], dtype=np.int32)
            band = torch.empty((B, n_win, n_bands), device=self.device, dtype=torch.float32)
        # called for n_win == 0 too: the library validates the geometry (and launches nothing)
        check(
            _lib.lib().mmf_modspec(
                self._h,
                mfcc.data_ptr(),
                B,
                Cc,
                T,
                win,
                hop,
                nfft,
                mag.data_ptr() if want_mag and n_win > 0 else None,
                band.data_ptr() if band is not None and n_win > 0 else None,
                lo.ctypes.data if lo is not None else None,
                hi.ctypes.data if hi is not None else None,
                n_bands,
                _stream_ptr(self.device),
            )
        )
        return mag, band

    def modspec_varlen(self, mfcc, frames, win: int, hop: int, nfft: int, band_bins=None, *, want_mag: bool = True):
        """:meth:`modspec` for clips of different lengths: ``mfcc [B, C, T_max]`` holds clip ``i`` in its first
        ``frames[i]`` frames (as :meth:`mfcc_change_varlen` returns it; whatever follows is ignored).  Outputs are
        padded to the most windows of any clip; windows ``[0, windows[i])`` of clip ``i`` equal :meth:`modspec` on
        that clip alone, bit for bit, and the rest is 0.  Returns ``(mag [B, C, W, nfft/2+1] or None,
        band [B, W, n_bands] or None, windows)``, ``windows`` a numpy int64 ``[B]``."""
        torch = _torch()
        mfcc = mfcc.contiguous()
        B, Cc, P = mfcc.shape
        T = np.ascontiguousarray(np.asarray(frames, dtype=np.int64).reshape(-1))
        if T.shape[0] != B:
            raise ValueError(f"frames has {T.shape[0]} entries for {B} clips")
        windows = np.where(T >= win, 1 + (T - win) // max(hop, 1), 0) if hop >= 1 else np.zeros(B, np.int64)
        W = int(windows.max()) if B else 0
        nb = nfft // 2 + 1
        mag = torch.empty((B, Cc, W, nb), device=self.device, dtype=torch.float32) if want_mag else None
        band = None
        lo = hi = None
        n_bands = 0
        if band_bins is not None and len(band_bins):
            n_bands = len(band_bins)
            lo = np.ascontiguousarray([b[0] for b in band_bins], dtype=np.int32)
            hi = np.ascontiguousarray([b[1] for b in band_bins], dtype=np.int32)
            band = torch.empty((B, W, n_bands), device=self.device, dtype=torch.float32)
        # called for W == 0 too: the library validates the lengths and the geometry (and launches nothing)
        check(
            _lib.lib().mmf_modspec_varlen(
                self._h,
                mfcc.data_ptr(),
                B,
                Cc,
                T.ctypes.data,
                P,
                win,
                hop,
                nfft,
                mag.data_ptr() if want_mag and W > 0 else None,
                band.data_ptr() if band is not None and W > 0 else None,
                lo.ctypes.data if lo is not None else None,
                hi.ctypes.data if hi is not None else None,
                n_bands,
                _stream_ptr(self.device),
            )
        )
        return mag, band, windows

    def rms(self, pcm, frame_length: int, hop_length: int, center: bool = True):
        """librosa.feature.rms -> float32 [B, T_rms]."""
        torch = _torch()
        pcm = self._pcm(pcm)
        B, N = pcm.shape
        pad = frame_length // 2 if center else 0
        if N + 2 * pad < frame_length:
            raise ValueError(f"Input is too short (n={N}) for frame_length={frame_length}")
        T = 1 + (N + 2 * pad - frame_length) // hop_length
        out = torch.empty((B, T), device=self.device, dtype=torch.float32)
        check(
            _lib.lib().mmf_rms(
                self._h,
                pcm.data_ptr(),
                B,
                N,
                pcm.stride(0) if B > 1 else N,
                frame_length,
                hop_length,
                1 if center else 0,
                out.data_ptr(),
                _stream_ptr(self.device),
            )
        )
        return out

    def rms_varlen(self, x, offsets, geom, center: bool = True):
        """:meth:`rms` for clips of different lengths and frame geometries packed back to back, in one launch.

        ``x`` is a 1-D float32 device tensor (or host array); clip ``i`` is ``x[offsets[i]:offsets[i + 1]]`` with
        ``geom[i] = (frame_length_i, hop_i)``.  Returns ``(amp, amp_offsets)``: the float32 envelopes packed clip after
        clip, clip ``i``'s at ``amp[amp_offsets[i]:amp_offsets[i + 1]]``, each equal to :meth:`rms` on that clip alone,
        bit for bit."""
        torch = _torch()
        x = x if isinstance(x, torch.Tensor) else torch.as_tensor(np.ascontiguousarray(x, dtype=np.float32))
        x = x.to(device=self.device, dtype=torch.float32).contiguous()
        if x.dim() != 1:
            raise ValueError("rms_varlen takes a 1-D packed buffer")
        offs, geom, amp_off = amp_sizes(offsets, geom, center)
        if offs[-1] > x.shape[0]:
            raise ValueError(f"offsets[{len(offs) - 1}] = {offs[-1]} is past the end of the {x.shape[0]}-sample buffer")
        amp = torch.empty((int(amp_off[-1]),), device=self.device, dtype=torch.float32)
        check(
            _lib.lib().mmf_rms_varlen(
                self._h, x.data_ptr(), len(offs) - 1, offs.ctypes.data, geom.ctypes.data, 1 if center else 0,
                amp.data_ptr(), _stream_ptr(self.device),
            )
        )
        return amp, amp_off

    def hilbert_varlen(self, x, offsets):
        """:meth:`hilbert_envelope` for clips of different lengths packed back to back (``mmf_hilbert_varlen``).

        ``x`` is a 1-D float32 device tensor (or host array); clip ``i`` is ``x[offsets[i]:offsets[i + 1]]``.  Returns
        ``(amp, amp_offsets)``: the float32 envelopes packed clip after clip, clip ``i``'s at
        ``amp[amp_offsets[i]:amp_offsets[i + 1]]`` (``amp_offsets = offsets - offsets[0]``), each equal to
        :meth:`hilbert_envelope` on that clip alone, bit for bit."""
        torch = _torch()
        x = x if isinstance(x, torch.Tensor) else torch.as_tensor(np.ascontiguousarray(x, dtype=np.float32))
        x = x.to(device=self.device, dtype=torch.float32).contiguous()
        if x.dim() != 1:
            raise ValueError("hilbert_varlen takes a 1-D packed buffer")
        offs = np.ascontiguousarray(np.asarray(offsets, dtype=np.int64).reshape(-1))
        amp_off = env_sizes(offs, make_env_params("Hilb"))
        if offs[-1] > x.shape[0]:
            raise ValueError(f"offsets[{len(offs) - 1}] = {offs[-1]} is past the end of the {x.shape[0]}-sample buffer")
        amp = torch.empty((int(amp_off[-1]),), device=self.device, dtype=torch.float32)
        check(
            _lib.lib().mmf_hilbert_varlen(
                self._h, x.data_ptr(), len(offs) - 1, offs.ctypes.data, amp.data_ptr(), _stream_ptr(self.device)
            )
        )
        return amp, amp_off

    def hilbert_envelope(self, x):
        """``np.abs(scipy.signal.hilbert(x))`` along the last axis, float32 on the device."""
        torch = _torch()
        x = x if isinstance(x, torch.Tensor) else torch.as_tensor(np.ascontiguousarray(x, dtype=np.float32))
        x = x.to(device=torch.device("cuda", self.cfg.device), dtype=torch.float32)
        squeeze = x.ndim == 1
        if squeeze:
            x = x[None, :]
        x = x.contiguous()
        amp = torch.empty_like(x)
        check(
            _lib.lib().mmf_hilbert_envelope(
                self._h, x.data_ptr(), x.shape[0], x.shape[1], x.stride(0), amp.data_ptr(), amp.stride(0), _stream_ptr(x.device)
            )
        )
        return amp[0] if squeeze else amp

    def find_peaks(self, x, *, minima: bool = False, max_peaks: int | None = None):
        """``scipy.signal.find_peaks(x)`` (default arguments) for every float64 row of ``x`` on the
        device.  Returns ``(idx [rows, max_peaks] int32, count [rows] int32)``; row ``r`` holds its
        ``min(count[r], max_peaks)`` peak indices in ascending order."""
        torch = _torch()
        x = x if isinstance(x, torch.Tensor) else torch.as_tensor(np.ascontiguousarray(x, dtype=np.float64))
        x = x.to(device=torch.device("cuda", self.cfg.device), dtype=torch.float64)
        if x.ndim == 1:
            x = x[None, :]
        x = x.contiguous()
        rows, T = x.shape
        if max_peaks is None:
            max_peaks = max(1, (T - 1) // 2)  # peaks need a lower sample between them
        idx = torch.full((rows, max_peaks), -1, device=x.device, dtype=torch.int32)
        cnt = torch.empty((rows,), device=x.device, dtype=torch.int32)
        check(
            _lib.lib().mmf_find_peaks(
                self._h, x.data_ptr(), rows, T, x.stride(0), 1 if minima else 0, max_peaks, idx.data_ptr(), cnt.data_ptr(),
                _stream_ptr(x.device),
            )
        )
        return idx, cnt

    def pcm16_to_f32(self, pcm16):
        """int16 PCM (CUDA tensor or numpy) -> float32 in [-1, 1) on the device (x / 32768)."""
        torch = _torch()
        x = pcm16 if isinstance(pcm16, torch.Tensor) else torch.as_tensor(np.ascontiguousarray(pcm16))
        x = x.to(device=torch.device("cuda", self.cfg.device), dtype=torch.int16).contiguous()
        y = torch.empty(x.shape, device=x.device, dtype=torch.float32)
        check(_lib.lib().mmf_pcm16_to_f32(self._h, x.data_ptr(), x.numel(), y.data_ptr(), _stream_ptr(x.device)))
        return y

    def resample_poly(self, x, up: int, down: int, quality: str = "scipy"):
        """Rational-rate conversion of float32 rows on the device (polyphase FIR, float64 accumulation).

        ``quality="scipy"``: exactly ``scipy.signal.resample_poly(x, up, down, axis=-1)`` (Kaiser-5 FIR, 10 taps per
        phase side, constant padding).  ``quality="hq"``: the band limits of libsoxr's HQ recipe that
        ``librosa.load(sr=...)`` uses at script/mfcc.py:373 (pass band to 0.913 of the lower Nyquist, stop band from
        the Nyquist, 120 dB).  The filter is designed on the host (:func:`design_resample_filter`)."""
        torch = _torch()
        import math

        x = x if isinstance(x, torch.Tensor) else torch.as_tensor(np.ascontiguousarray(x, dtype=np.float32))
        x = x.to(device=torch.device("cuda", self.cfg.device), dtype=torch.float32)
        squeeze = x.ndim == 1
        if squeeze:
            x = x[None, :]
        x = x.contiguous()
        g = math.gcd(int(up), int(down))
        up, down = int(up) // g, int(down) // g
        n_in = x.shape[-1]
        if up == 1 and down == 1:
            return x[0] if squeeze else x
        h, n_pre_remove, n_out = design_resample_filter(n_in, up, down, quality)
        y = torch.empty((x.shape[0], n_out), device=x.device, dtype=torch.float32)
        for c0 in range(0, x.shape[0], 65535):
            xs = x[c0 : c0 + 65535]
            ys = y[c0 : c0 + 65535]
            check(
                _lib.lib().mmf_resample_poly(
                    self._h, xs.data_ptr(), xs.shape[0], n_in, xs.stride(0), h.ctypes.data, len(h), up, down,
                    n_pre_remove, n_out, ys.data_ptr(), ys.stride(0), _stream_ptr(x.device),
                )
            )
        return y[0] if squeeze else y

    def mfcc_change(self, pcm, prm: mmf_change_params, *, want_logmel=False, want_mfcc=False, want_delta=False):
        """Whole get_MFCCS_change on device-resident PCM -> dict of CUDA tensors."""
        torch = _torch()
        pcm = self._pcm(pcm)
        B, N = pcm.shape
        T = self.num_frames(N)
        tot = torch.empty((B, T), device=self.device, dtype=torch.float64)
        logmel = torch.empty((B, self.cfg.n_mels, T), device=self.device, dtype=torch.float32) if want_logmel else None
        mfcc = (
            torch.empty((B, self.cfg.n_mfcc, T), device=self.device, dtype=torch.float32)
            if (want_mfcc or want_delta)
            else None
        )
        delta = torch.empty((B, self.cfg.n_mfcc, T), device=self.device, dtype=torch.float32) if want_delta else None
        check(
            _lib.lib().mmf_mfcc_change(
                self._h,
                pcm.data_ptr(),
                B,
                N,
                pcm.stride(0) if B > 1 else N,
                C.byref(prm),
                tot.data_ptr(),
                logmel.data_ptr() if logmel is not None else None,
                mfcc.data_ptr() if mfcc is not None else None,
                delta.data_ptr() if delta is not None else None,
                _stream_ptr(self.device),
            )
        )
        return {"totChange": tot, "logmel": logmel, "mfcc": mfcc, "delta": delta}

    def mfcc_change_varlen(self, pcm, lengths, prm: mmf_change_params, *, want_logmel=False, want_mfcc=False,
                           want_delta=False):
        """:meth:`mfcc_change` for clips of different lengths: row ``i`` of ``pcm`` ``[B, N_max]`` holds clip ``i`` in
        its first ``lengths[i]`` samples (whatever follows is ignored).  Outputs are padded to the longest clip's
        frame count; frames ``[0, frames[i])`` of clip ``i`` equal :meth:`mfcc_change` on that clip alone, bit for
        bit, and the rest is 0.  Returns the dict of :meth:`mfcc_change` plus ``frames`` (numpy int64 ``[B]``)."""
        torch = _torch()
        pcm = self._pcm(pcm)
        B, N = pcm.shape
        lens = np.ascontiguousarray(np.asarray(lengths, dtype=np.int64).reshape(-1))
        if lens.shape[0] != B:
            raise ValueError(f"lengths has {lens.shape[0]} entries for {B} clips")
        # mmf_num_frames for every clip at once (a ctypes call per clip costs ~1 us each)
        padded = lens + 2 * (self.cfg.n_fft // 2)
        frames = np.where(padded < self.cfg.n_fft, 0, 1 + np.maximum(padded - self.cfg.n_fft, 0) // self.cfg.hop_length)
        T = int(frames.max()) if B else 0
        tot = torch.empty((B, T), device=self.device, dtype=torch.float64)
        logmel = torch.empty((B, self.cfg.n_mels, T), device=self.device, dtype=torch.float32) if want_logmel else None
        mfcc = (
            torch.empty((B, self.cfg.n_mfcc, T), device=self.device, dtype=torch.float32)
            if (want_mfcc or want_delta)
            else None
        )
        delta = torch.empty((B, self.cfg.n_mfcc, T), device=self.device, dtype=torch.float32) if want_delta else None
        check(
            _lib.lib().mmf_mfcc_change_varlen(
                self._h,
                pcm.data_ptr(),
                B,
                lens.ctypes.data,
                pcm.stride(0) if B > 1 else N,
                C.byref(prm),
                tot.data_ptr(),
                logmel.data_ptr() if logmel is not None else None,
                mfcc.data_ptr() if mfcc is not None else None,
                delta.data_ptr() if delta is not None else None,
                _stream_ptr(self.device),
            )
        )
        return {"totChange": tot, "logmel": logmel, "mfcc": mfcc, "delta": delta, "frames": frames}

    def change_from_logmel(self, logmel, clipmax, prm: mmf_change_params, *, want_delta=True, clamp_in_place=True):
        """Second half of :meth:`mfcc_change` for a log-mel already on the device."""
        torch = _torch()
        B, _, T = logmel.shape
        tot = torch.empty((B, T), device=self.device, dtype=torch.float64)
        mfcc = torch.empty((B, self.cfg.n_mfcc, T), device=self.device, dtype=torch.float32)
        delta = torch.empty_like(mfcc) if want_delta else None
        check(
            _lib.lib().mmf_change_from_logmel(
                self._h,
                logmel.data_ptr(),
                clipmax.data_ptr(),
                B,
                T,
                C.byref(prm),
                tot.data_ptr(),
                mfcc.data_ptr(),
                delta.data_ptr() if delta is not None else None,
                1 if clamp_in_place else 0,
                _stream_ptr(self.device),
            )
        )
        return {"totChange": tot, "mfcc": mfcc, "delta": delta}

    def features_host(self, pcm_host: np.ndarray, prm: mmf_change_params, mod=None, *, want=("totChange",), out=None):
        """The whole bundle through ONE C-ABI call with host buffers (H2D/D2H inside).

        ``mod`` = (win, hop, nfft, band_bins) or None; ``want`` subset of
        totChange/mfcc/delta/modspec/band_energy; ``out`` may hold preallocated
        (ideally pinned) numpy arrays to receive the results."""
        pcm_host = np.asarray(pcm_host)
        pcm16 = pcm_host.dtype == np.int16  # raw WAV samples: scaled by 1/32768 on the device
        if not pcm16 and pcm_host.dtype != np.float32:
            pcm_host = pcm_host.astype(np.float32)
        if pcm_host.ndim == 1:
            pcm_host = pcm_host[None, :]
        isz = pcm_host.dtype.itemsize
        if pcm_host.strides[1] != isz:
            pcm_host = np.ascontiguousarray(pcm_host)
        B, N = pcm_host.shape
        T = self.num_frames(N)
        nm = self.cfg.n_mfcc
        out = {} if out is None else out
        mp = _modspec_params(mod)
        n_win = nb = n_bands = 0
        if mod is not None:
            win, hop, nfft, bins = mod
            n_win = 1 + (T - win) // hop if T >= win else 0
            nb, n_bands = nfft // 2 + 1, len(bins)
        shapes = {
            "totChange": ((B, T), np.float64),
            "mfcc": ((B, nm, T), np.float32),
            "delta": ((B, nm, T), np.float32),
            "modspec": ((B, nm, n_win, nb), np.float32),
            "band_energy": ((B, n_win, n_bands), np.float32),
        }
        ptr = {k: _out_array(out, k, *sd).ctypes.data if k in want or k == "totChange" else None
               for k, sd in shapes.items()}
        fn = _lib.lib().mmf_features_host_pcm16 if pcm16 else _lib.lib().mmf_features_host
        check(
            fn(
                self._h,
                pcm_host.ctypes.data,
                B,
                N,
                pcm_host.strides[0] // isz if B > 1 else N,
                C.byref(prm),
                C.byref(mp) if mp is not None else None,
                ptr["totChange"],
                ptr["mfcc"],
                ptr["delta"],
                ptr["modspec"],
                ptr["band_energy"],
            )
        )
        return out

    def features_host_varlen(self, pcm_host: np.ndarray, offsets, prm: mmf_change_params, mod=None, *,
                             want=("totChange",), out=None, rates=None, amp=None, amp_method="RMS",
                             change_out=None):
        """:meth:`features_host` for clips of different lengths packed back to back in one host buffer.

        ``pcm_host`` is 1-D float32 or int16 (raw WAV samples, scaled by 1/32768 on the device); clip ``i`` is
        ``pcm_host[offsets[i]:offsets[i + 1]]``, ``offsets`` int64 ``[B + 1]``.  Returns the keys of
        :meth:`features_host` as flat packed arrays, clip after clip with no padding (clip ``i``'s ``[n_mfcc, T_i]``
        MFCC block starts at ``n_mfcc * frame_offsets[i]``, its ``[n_mfcc, n_win_i, nfft/2+1]`` modulation block at
        ``n_mfcc * (nfft/2+1) * window_offsets[i]``), plus ``frames``, ``windows`` (int64 ``[B]``), ``frame_offsets``
        and ``window_offsets`` (int64 ``[B + 1]``).  Each clip's blocks equal :meth:`features_host` on that clip
        alone, bit for bit.  Pinned buffers (``pcm_host`` and the arrays in ``out``) make the copies asynchronous.

        ``rates``: one source sample rate per clip.  Each clip then crosses PCIe at its own rate and is resampled on
        the device to the plan's rate with the loader's filter (:func:`resample_descriptors`), straight into the rows
        the ragged path reads; its blocks equal :meth:`features_host` on ``resample_poly(x, up, down, "hq")`` of that
        clip alone (after ``pcm16_to_f32`` for int16), bit for bit, and ``frames`` count frames at the plan's rate.

        ``amp = (geom, center, out_sos or None)`` adds each clip's RMS envelope, taken from its native samples (int16
        scaled by 1/32768) with ``geom[i] = (frame_length_i, hop_i)``: ``amplitude``, float32, or float64 through the
        zero-phase ``out_sos`` when one is given, packed at ``amp_offsets`` (int64 ``[B + 1]``).  Clip ``i``'s block
        equals :meth:`rms` (then :meth:`sosfiltfilt`) on that clip alone, bit for bit.  ``amp_method="Hilb"``: the
        Hilbert envelope instead, one value per native sample (``geom`` and ``center`` are not read), equal to
        :meth:`hilbert_envelope` (then :meth:`sosfiltfilt`) on that clip alone, bit for bit.

        ``change_out``: an :class:`OutFilter` run over each raw change curve (``prm`` must ask for the raw curve,
        ``out_sos=None``); clip ``i``'s ``totChange`` then equals :meth:`filter_varlen` on its raw curve alone."""
        pcm_host = np.asarray(pcm_host)
        pcm16 = pcm_host.dtype == np.int16
        if not pcm16 and pcm_host.dtype != np.float32:
            pcm_host = pcm_host.astype(np.float32)
        if pcm_host.ndim != 1:
            raise ValueError("features_host_varlen takes a 1-D packed buffer")
        pcm_host = np.ascontiguousarray(pcm_host)
        offs = np.ascontiguousarray(np.asarray(offsets, dtype=np.int64).reshape(-1))
        B = offs.shape[0] - 1
        if B < 1:
            raise ValueError("offsets needs at least two entries")
        if offs[-1] > pcm_host.shape[0]:
            raise ValueError(f"offsets[{B}] = {offs[-1]} is past the end of the {pcm_host.shape[0]}-sample buffer")
        mp = _modspec_params(mod)
        frame_off = np.empty(B + 1, np.int64)
        win_off = np.empty(B + 1, np.int64)
        # the library owns the size formulas (and checks the offsets, naming a bad clip)
        sizes = lambda o: check(  # noqa: E731
            _lib.lib().mmf_features_varlen_sizes(
                C.byref(self.cfg.to_c()), C.byref(mp) if mp is not None else None, B, o.ctypes.data,
                frame_off.ctypes.data, win_off.ctypes.data,
            )
        )
        sizes(offs)
        if rates is not None:
            # the blocks follow the lengths at the plan's rate: sizes of the prefix sums of n_out
            rs, h = resample_descriptors(np.diff(offs), rates, self.cfg.sample_rate)
            out_offs = np.zeros(B + 1, np.int64)
            np.cumsum(rs["n_out"], out=out_offs[1:])
            sizes(out_offs)
        nm = self.cfg.n_mfcc
        F, Wt = int(frame_off[-1]), int(win_off[-1])
        nb = n_bands = 0
        if mod is not None:
            nb, n_bands = int(mod[2]) // 2 + 1, len(mod[3])
        shapes = {
            "totChange": ((F,), np.float64),
            "mfcc": ((nm * F,), np.float32),
            "delta": ((nm * F,), np.float32),
            "modspec": ((nm * Wt * nb,), np.float32),
            "band_energy": ((Wt * n_bands,), np.float32),
        }
        out = {} if out is None else out
        ptr = {}
        for k, sd in shapes.items():
            a = _out_array(out, k, *sd) if k in want or k == "totChange" else None
            # (size 0: no modulation window in any clip, nothing to write)
            ptr[k] = a.ctypes.data if a is not None and a.size else None
        if ("modspec" in want or "band_energy" in want) and mp is None:
            raise ValueError("modspec / band_energy requested without modulation parameters")
        # one entry point for every variant: rs = NULL means every clip at the plan's rate, amp = NULL no envelope
        rs_p = h_p = None
        n_h = 0
        if rates is not None:
            rs_p, h_p, n_h = rs.ctypes.data, h.ctypes.data if len(h) else None, len(h)
        amp_p = geom_p = a_p = af_p = None
        if amp is not None:
            geom, center, out_sos = amp
            env = make_env_params(amp_method, center, out_sos)
            if amp_method == "RMS":
                _, geom, amp_off = amp_sizes(offs, geom, center)
                geom_p = geom.ctypes.data
            else:
                amp_off = env_sizes(offs, env)
            a = _out_array(out, "amplitude", (int(amp_off[-1]),), np.float64 if out_sos is not None else np.float32)
            amp_p = C.byref(env)
            a_p, af_p = (None, a.ctypes.data) if out_sos is not None else (a.ctypes.data, None)
        check(
            _lib.lib().mmf_features_host_varlen_out(
                self._h, pcm_host.ctypes.data, 1 if pcm16 else 0, B, offs.ctypes.data, rs_p, h_p, n_h,
                C.byref(prm), C.byref(mp) if mp is not None else None, amp_p, geom_p,
                C.byref(change_out.c) if change_out is not None else None,
                ptr["totChange"], ptr["mfcc"], ptr["delta"], ptr["modspec"], ptr["band_energy"], a_p, af_p,
            )
        )
        out["frames"] = np.diff(frame_off)
        out["windows"] = np.diff(win_off)
        out["frame_offsets"] = frame_off
        out["window_offsets"] = win_off
        if amp is not None:
            out["amp_offsets"] = amp_off
        return out

    def mfcc_change_host(self, pcm_host: np.ndarray, prm: mmf_change_params, *, want_mfcc: bool = False):
        """Host buffers in and out through the single C-ABI call (H2D/D2H inside).

        float32 samples go through ``mmf_mfcc_change_host``; int16 samples (raw WAV PCM) through
        ``mmf_features_host_pcm16``, which scales them by 1/32768 on the device."""
        pcm_host = np.asarray(pcm_host)
        pcm16 = pcm_host.dtype == np.int16
        if not pcm16 and pcm_host.dtype != np.float32:
            pcm_host = pcm_host.astype(np.float32)
        if pcm_host.ndim == 1:
            pcm_host = pcm_host[None, :]
        isz = pcm_host.dtype.itemsize
        if pcm_host.strides[1] != isz or pcm_host.strides[0] % isz:
            pcm_host = np.ascontiguousarray(pcm_host)
        B, N = pcm_host.shape
        T = self.num_frames(N)
        tot = np.empty((B, T), np.float64)
        mf = np.empty((B, self.cfg.n_mfcc, T), np.float32) if want_mfcc else None
        stride = pcm_host.strides[0] // isz if B > 1 else N
        if pcm16:
            check(
                _lib.lib().mmf_features_host_pcm16(
                    self._h, pcm_host.ctypes.data, B, N, stride, C.byref(prm), None, tot.ctypes.data,
                    mf.ctypes.data if want_mfcc else None, None, None, None,
                )
            )
        else:
            check(
                _lib.lib().mmf_mfcc_change_host(
                    self._h, pcm_host.ctypes.data, B, N, stride, C.byref(prm), tot.ctypes.data,
                    mf.ctypes.data if want_mfcc else None,
                )
            )
        return (tot, mf) if want_mfcc else tot


def _out_array(out: dict, key: str, shape, dtype) -> np.ndarray:
    """``out[key]`` when it is a C-contiguous array of this shape and dtype, else a new one, stored there."""
    a = out.get(key)
    if a is None or a.shape != shape or a.dtype != dtype or not a.flags.c_contiguous:
        a = np.empty(shape, dtype)
        out[key] = a
    return a


def amp_sizes(offsets, geom, center: bool):
    """``(offsets, geom, amp_offsets)`` of a packed batch's RMS envelopes (``mmf_amp_varlen_sizes``, no device
    needed): ``offsets`` as int64 ``[B + 1]``, ``geom`` as int32 ``[B, 2]`` rows ``(frame_length_i, hop_i)``, and the
    prefix sums of ``T_amp_i = 1 + (len_i + 2 pad_i - frame_length_i) // hop_i``.  A bad clip raises
    :class:`MmfError` naming it."""
    offs = np.ascontiguousarray(np.asarray(offsets, dtype=np.int64).reshape(-1))
    B = offs.shape[0] - 1
    geom = np.ascontiguousarray(np.asarray(geom, dtype=np.int32).reshape(-1, 2))
    if geom.shape[0] != B:
        raise ValueError(f"geom has {geom.shape[0]} rows for {B} clips")
    amp_off = np.zeros(B + 1, np.int64)
    check(_lib.lib().mmf_amp_varlen_sizes(B, offs.ctypes.data, geom.ctypes.data, 1 if center else 0,
                                          amp_off.ctypes.data))
    return offs, geom, amp_off


def make_amp_params(center: bool, out_sos=None) -> mmf_amp_params:
    """Pack the envelope parameters of the host-buffer bundle: ``center`` and the optional zero-phase output filter."""
    ap = mmf_amp_params()
    ap.center = 1 if center else 0
    if out_sos is not None:
        out_sos = np.ascontiguousarray(out_sos, dtype=np.float64)
        if out_sos.ndim != 2 or out_sos.shape[1] != 6 or out_sos.shape[0] > 16:
            raise ValueError("out_sos must be [n_sections <= 16, 6]")
        ap.out_n_sections = out_sos.shape[0]
        for i, v in enumerate(out_sos.ravel()):
            ap.out_sos[i] = v
    return ap


AMP_METHODS = {"RMS": _lib.MMF_ENV_RMS, "Hilb": _lib.MMF_ENV_HILBERT}


class OutFilter:
    """A 'fir' or 'sg' output filter as the library takes it (``mmf_out_filter``), holding its host coefficients.
    Build one with :func:`fir_filter` or :func:`stencil_filter`."""

    def __init__(self, kind: int, arrays):
        self.kind, self.arrays = kind, arrays  # the arrays stay alive as long as the struct that points at them
        self.c = mmf_out_filter()
        self.c.kind = kind

    def check(self, lengths) -> None:
        """The library's checks for rows of ``lengths`` samples, without a device (``mmf_filter_varlen_check``)."""
        T = np.ascontiguousarray(np.asarray(lengths, dtype=np.int64).reshape(-1))
        check(_lib.lib().mmf_filter_varlen_check(C.byref(self.c), T.shape[0], T.ctypes.data))


def fir_filter(b) -> OutFilter:
    """scipy.signal.filtfilt(b, 1, x) (applyFilter's 'fir', script/mfcc.py:126)."""
    b = np.ascontiguousarray(b, dtype=np.float64).reshape(-1)
    f = OutFilter(_lib.MMF_FILT_FIR, (b,))
    f.c.n_taps, f.c.taps = b.shape[0], b.ctypes.data
    return f


def stencil_filter(coef, edge_l, edge_r) -> OutFilter:
    """A banded stencil with dense edge rows, as :meth:`Plan.stencil` takes it (applyFilter's 'sg', np.gradient,
    findiff)."""
    coef = np.ascontiguousarray(coef, dtype=np.float64).reshape(-1)
    edge_l = np.ascontiguousarray(edge_l, dtype=np.float64)
    edge_r = np.ascontiguousarray(edge_r, dtype=np.float64)
    f = OutFilter(_lib.MMF_FILT_SG, (coef, edge_l, edge_r))
    n_edge, n_edge_in = edge_l.shape if edge_l.size else (0, 0)
    f.c.half, f.c.coef = (coef.shape[0] - 1) // 2, coef.ctypes.data
    f.c.n_edge, f.c.n_edge_in = n_edge, n_edge_in
    f.c.edge_l = edge_l.ctypes.data if n_edge else None
    f.c.edge_r = edge_r.ctypes.data if n_edge else None
    return f


def make_env_params(method: str = "RMS", center: bool = True, out_sos=None) -> mmf_env_params:
    """:func:`make_amp_params` with the envelope method: ``'RMS'`` or ``'Hilb'``."""
    if method not in AMP_METHODS:
        raise ValueError(f"amplitude method must be 'RMS' or 'Hilb', not {method!r}")
    ap = make_amp_params(center, out_sos)
    ep = mmf_env_params()
    ep.method, ep.center, ep.out_n_sections = AMP_METHODS[method], ap.center, ap.out_n_sections
    ep.out_sos[:] = list(ap.out_sos)
    return ep


def env_sizes(offsets, env: mmf_env_params, geom=None):
    """``amp_offsets`` of a packed batch's envelopes (``mmf_env_varlen_sizes``, no device needed); ``geom`` (RMS only)
    as in :func:`amp_sizes`.  A bad clip raises :class:`MmfError` naming it."""
    offs = np.ascontiguousarray(np.asarray(offsets, dtype=np.int64).reshape(-1))
    g = None if geom is None else np.ascontiguousarray(np.asarray(geom, dtype=np.int32).reshape(-1, 2))
    amp_off = np.zeros(offs.shape[0], np.int64)
    check(_lib.lib().mmf_env_varlen_sizes(offs.shape[0] - 1, offs.ctypes.data, C.byref(env),
                                          g.ctypes.data if g is not None else None, amp_off.ctypes.data))
    return amp_off


def _modspec_params(mod):
    """``mod`` = (win, hop, nfft, band_bins) or None -> mmf_modspec_params or None."""
    if mod is None:
        return None
    win, hop, nfft, bins = mod
    mp = mmf_modspec_params()
    mp.win, mp.hop, mp.nfft, mp.n_bands = int(win), int(hop), int(nfft), len(bins)
    for i, (lo, hi) in enumerate(bins):
        mp.band_lo[i], mp.band_hi[i] = int(lo), int(hi)
    return mp


_PLANS: "OrderedDict[MfccConfig, Plan]" = OrderedDict()
_MAX_PLANS = 16


def get_plan(cfg: MfccConfig) -> Plan:
    """Keyed least-recently-used cache of plans (window, mel bank, DCT, twiddles stay on the device).

    An evicted plan is only dropped from the cache: objects that still hold it (a ``FeatureExtractor``, a
    caller's local) keep a live handle, and ``Plan.__del__`` frees the device memory with the last reference."""
    p = _PLANS.get(cfg)
    if p is None:
        while len(_PLANS) >= _MAX_PLANS:
            _PLANS.popitem(last=False)
        p = Plan(cfg)
        _PLANS[cfg] = p
    else:
        _PLANS.move_to_end(cfg)
    return p


def clear_plans() -> None:
    for p in _PLANS.values():
        p.close()
    _PLANS.clear()


__all__ = [
    "amp_sizes",
    "make_amp_params",
    "design_resample_filter",
    "resample_descriptors",
    "resample_ratio",
    "MfccConfig",
    "Plan",
    "get_plan",
    "clear_plans",
    "frame_sizes",
    "num_frames",
    "host_tables",
    "sos_zi",
    "make_change_params",
    "replace",
]
