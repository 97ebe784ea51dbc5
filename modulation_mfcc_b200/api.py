"""Host-side mirror of the reference's feature functions, backed by the CUDA library.

Same names, positional/keyword structure, return types and error behaviour as
``script/mfcc.py`` / ``script/calc.py`` of aaron-randreth/modulation-mfcc:

* ``get_MFCCS_change``      script/mfcc.py:291-427
* ``applyFilter``           script/mfcc.py:29-135  == script/calc.py:23-129
* ``get_amplitude`` / ``calculate_amplitude_envelope``
                            script/mfcc.py:137-259 == script/calc.py:221-343
* ``load_channel``          script/mfcc.py:262-289
* ``get_velocity``          script/calc.py:593-650

plus batch entry points that keep everything on the device
(``get_MFCCS_change_batch``, ``mfcc_features_batch``).  Filter *design* (Butterworth
sections, Kaiser FIR taps, Savitzky-Golay / finite-difference stencils) happens on
the host at plan time with scipy, exactly as the reference designs its filters;
every operation that touches signal data runs in ``libmmf_b200.so`` on the GPU.
There is no CPU fallback.
"""

from __future__ import annotations

import math
from functools import lru_cache

import numpy as np
import scipy.signal

from . import _lib
from ._lib import MmfError
from .plan import MfccConfig, Plan, frame_sizes, get_plan, make_change_params, resample_ratio

MODULATION_BANDS_HZ = ((0.5, 2.0), (2.0, 4.0), (4.0, 8.0), (8.0, 16.0), (16.0, 32.0))


class ParameterError(Exception):
    """Stands in for ``librosa.util.exceptions.ParameterError`` (what ``librosa.feature.mfcc`` raises for
    invalid audio at script/mfcc.py:387)."""


def _require_float_audio(a):
    """``librosa.util.valid_audio``: integer PCM is rejected, not silently rescaled.  (The corpus path for raw
    16-bit samples is ``FeatureExtractor.host_call`` / ``mmf_features_host_pcm16``, which documents its 1/32768
    scale.)"""
    dt = getattr(a, "dtype", None)
    is_float = dt is not None and (dt.is_floating_point if hasattr(dt, "is_floating_point") else np.issubdtype(dt, np.floating))
    if not is_float:
        raise ParameterError("Audio data must be floating-point")


@lru_cache(maxsize=64)
def _butter_sos_cached(order, wn, btype):
    return scipy.signal.butter(order, wn if not isinstance(wn, tuple) else list(wn), btype=btype, output="sos")


def _butter_sos(order, wn, btype):
    """``scipy.signal.butter(order, wn, btype, output='sos')`` with the design cached: the GUI calls the
    path with the same filter over and over, and the design costs as much as the whole GPU pass."""
    try:
        key = tuple(float(v) for v in wn) if np.ndim(wn) else float(wn)
        return _butter_sos_cached(int(order), key, str(btype)).copy()
    except TypeError:  # unhashable / odd arguments: let scipy validate them
        return scipy.signal.butter(order, wn, btype=btype, output="sos")


def _torch():
    import torch

    return torch


def _raise_from(e: MmfError):
    """Map C-ABI error codes onto the exception types the reference's callers see."""
    if e.code == _lib.MMF_ERR_TOO_SHORT:
        raise ValueError(e.msg) from None  # scipy's sosfiltfilt/filtfilt raise ValueError
    if e.code == _lib.MMF_ERR_INVALID:
        raise ValueError(e.msg) from None
    raise e


def _any_plan(device=None) -> Plan:
    """A plan just to reach the filter kernels (they do not depend on the STFT config)."""
    return get_plan(MfccConfig(sample_rate=16000.0, device=_device_index(device)))


def _device_index(device) -> int:
    if device is None:
        torch = _torch()
        return torch.cuda.current_device() if torch.cuda.is_available() else 0
    if isinstance(device, int):
        return device
    torch = _torch()
    d = torch.device(device)
    return d.index if d.index is not None else torch.cuda.current_device()


def _to_dev(x, dtype, device_index: int):
    torch = _torch()
    if isinstance(x, torch.Tensor):
        return x.to(device=torch.device("cuda", device_index), dtype=dtype)
    return torch.as_tensor(np.ascontiguousarray(x)).to(device=torch.device("cuda", device_index), dtype=dtype)


# ---------------------------------------------------------------------------
# linear-operator probing: turn a (linear, shift-invariant in the interior)
# scipy filter into interior stencil + dense boundary rows for mmf_stencil
# ---------------------------------------------------------------------------


def _stencil_from_operator(fn, support: int):
    """Probe ``fn`` (linear map along axis 0) with unit impulses.

    Returns (coef[2*half+1], edge_l[n_edge, n_in], edge_r[n_edge, n_in]) such that
    y[t] = sum_o coef[o+half]*x[t+o] in the interior and the first/last n_edge
    outputs are edge_l/edge_r applied to the first/last n_in inputs.
    """
    L = 4 * support + 5
    M = np.asarray(fn(np.eye(L)), dtype=np.float64)  # M[t, j] = response at t to an impulse at j
    mid = L // 2
    half = support
    coef = M[mid, mid - half : mid + half + 1].copy()
    nz = np.nonzero(coef)[0]
    if len(nz):
        h = max(half - nz[0], nz[-1] - half)
    else:
        h = 0
    coef = coef[half - h : half + h + 1]
    half = h

    def interior_row(t):
        r = np.zeros(L)
        lo, hi = t - half, t + half + 1
        if lo < 0 or hi > L:
            return None
        r[lo:hi] = coef
        return r

    n_edge = 0
    for t in range(mid):
        r = interior_row(t)
        if r is None or not np.allclose(M[t], r, rtol=0, atol=1e-13 * max(1.0, np.abs(coef).max())):
            n_edge = t + 1
    n_edge = max(n_edge, half)
    if n_edge == 0:
        return coef, np.zeros((0, 0)), np.zeros((0, 0))
    rows_l = M[:n_edge]
    n_in = int(np.max(np.nonzero(np.abs(rows_l).sum(axis=0))[0])) + 1 if np.any(rows_l) else 1
    rows_r = M[L - n_edge :]
    first = int(np.min(np.nonzero(np.abs(rows_r).sum(axis=0))[0])) if np.any(rows_r) else L - 1
    n_in = max(n_in, L - first, 1)
    return coef, rows_l[:, :n_in].copy(), rows_r[:, L - n_in :].copy()


@lru_cache(maxsize=64)
def _savgol_stencil(window: int, polyorder: int, deriv: int):
    return _stencil_from_operator(
        lambda e: scipy.signal.savgol_filter(e, window, polyorder, deriv=deriv, axis=0, mode="interp"), window
    )


def _fd_weights(offsets, deriv):
    offsets = np.asarray(offsets, dtype=np.float64)
    n = len(offsets)
    A = np.vander(offsets, n, increasing=True).T
    rhs = np.zeros(n)
    rhs[deriv] = math.factorial(deriv)
    return np.linalg.solve(A, rhs)


@lru_cache(maxsize=64)
def _findiff_stencil(deriv: int, acc: int):
    """findiff.FinDiff(0, h, deriv, acc=acc) for unit spacing: central stencil of
    half-width p = (deriv+1)//2 - 1 + acc//2, equal-accuracy one-sided stencils on
    the first/last p points (script/calc.py:635-637)."""
    p = (deriv + 1) // 2 - 1 + acc // 2
    c_off = np.arange(-p, p + 1)
    coef = _fd_weights(c_off, deriv)
    num = 2 * p + 1 + (1 if deriv % 2 == 0 else 0)
    f_off = np.arange(0, num)
    f_w = _fd_weights(f_off, deriv)
    b_w = _fd_weights(-f_off[::-1], deriv)
    n_in = num + p - 1
    el = np.zeros((p, n_in))
    er = np.zeros((p, n_in))
    for t in range(p):
        el[t, t : t + num] = f_w
        # output index T-p+t uses inputs (T-p+t) - (num-1) .. (T-p+t); edge window covers T-n_in .. T-1
        end = n_in - p + t
        er[t, end - num + 1 : end + 1] = b_w
    return coef, el, er


# ---------------------------------------------------------------------------
# applyFilter
# ---------------------------------------------------------------------------


def _apply_filter_dev(plan: Plan, x_dev, sr, *, filt, cutOff, filtLen, filtType, polyOrd, coeffs=None):
    """Validation (same order and messages as script/mfcc.py:82-96) + GPU filtering
    of a float64 device tensor along its last axis."""
    if (filt is None) | (cutOff is None) | (cutOff is None):
        if cutOff is None:
            raise Exception("Cannot apply filter without specifying a cut Off freq. (CutOff is None).")
        else:
            raise Exception(
                "Cannot apply filter without specifying a filter method among iir, fir and  sg (filt is None)."
            )
    filtTypes = np.array(["bandpass", "lowpass", "highpass"])
    try:
        filtType = filtTypes[np.argwhere([t.startswith(filtType) for t in filtTypes]).flatten()][0]
    except Exception:
        raise Exception("filtType must be one among: lowpass, highpass, bandpass. Partial matches allowed.")
    if any((sr / 2) <= np.array(cutOff)):
        raise Exception(
            "Cut off frequencies must be smaller than the half of the sampling freq. of the signal submitted to the filter"
        )
    if (len(cutOff) > 0) & (any(np.diff(cutOff) <= 0)):
        raise Exception("If two cut off freqs are provided: cutOff[0]<cutOff[1]")
    cutOff = np.array(cutOff)
    ok = ((len(cutOff) == 1) and ((filtType == "lowpass") | (filtType == "highpass"))) | (
        (len(cutOff) == 2) and (filtType == "bandpass")
    )
    y = None
    try:
        if filt == "iir":
            if coeffs is None:
                w = cutOff / (sr / 2)
                if ok:
                    sos = _butter_sos(filtLen, w, filtType)
                else:
                    raise Exception(
                        "only one or two cut off frequencies allowed. If two freqs are provided, filtType must be bandpass"
                    )
            else:
                # reference quirk (script/mfcc.py:100-111): `sos` is never bound when coeffs is given
                raise NameError("name 'sos' is not defined")
            y = plan.sosfiltfilt(x_dev, sos)
        if filt == "fir":
            if coeffs is None:
                w = cutOff / (sr / 2)
                if ok:
                    bFil = scipy.signal.firwin(filtLen, w, window=("kaiser", 7.4), pass_zero=filtType)
                else:
                    raise Exception(
                        "only one or two cut off frequencies allowed. If two freqs are provided, filtType must be bandpass"
                    )
            else:
                raise NameError("name 'bFil' is not defined")
            y = plan.fir_filtfilt(x_dev, bFil)
        if filt == "sg":
            if len(cutOff) == 1:
                if x_dev.shape[-1] < filtLen:
                    raise ValueError("If mode is 'interp', window_length must be less than or equal to the size of x.")
                coef, el, er = _savgol_stencil(int(filtLen), int(polyOrd), 0)
                y = plan.stencil(x_dev, coef, el, er)
            else:
                raise Exception("sg (savitsky Golay) filters can only be lowpass (one cutOff freq allowed)")
    except MmfError as e:
        _raise_from(e)
    return y


def applyFilter(x, sr, /, *, filt="iir", cutOff=[None], filtLen=6, filtType="low", polyOrd=3, coeffs=None, device=None):
    """Drop-in for ``applyFilter`` (script/mfcc.py:29-135, script/calc.py:23-129).

    Filters along the last axis (scipy's default); returns float64 ndarray, or
    ``None`` when ``filt`` names no known method (as the reference does)."""
    di = _device_index(device)
    plan = _any_plan(di)
    torch = _torch()
    # validation that does not need the data happens inside _apply_filter_dev before any GPU work
    x_dev = _to_dev(np.asarray(x), torch.float64, di) if not isinstance(x, torch.Tensor) else x.to(torch.float64)
    y = _apply_filter_dev(plan, x_dev, sr, filt=filt, cutOff=cutOff, filtLen=filtLen, filtType=filtType, polyOrd=polyOrd, coeffs=coeffs)
    if y is None:
        return None
    return y.cpu().numpy() if not isinstance(x, torch.Tensor) else y


# ---------------------------------------------------------------------------
# get_MFCCS_change
# ---------------------------------------------------------------------------


def _parse_wav(path: str):
    """Host half of the WAV loader: ``(file_sr, samples)``, shaped [channels, n] or [n] (one channel).  16-bit PCM
    stays int16 (scaled by 1/32768 on the device); 32-bit and 8-bit PCM and float files become float32 in [-1, 1]
    here.  Anything but RIFF/WAVE raises ``ValueError`` naming the path."""
    from scipy.io import wavfile

    try:
        file_sr, data = wavfile.read(path)
    except ValueError as e:
        # librosa.load goes through soundfile/audioread and also decodes FLAC, OGG, MP3 ...; here the
        # container is parsed on the host and only RIFF/WAVE (PCM 8/16/32-bit, float32/64) is supported
        raise ValueError(f"{path}: only RIFF/WAVE files can be decoded by the B200 loader ({e})") from None
    if data.ndim == 2:
        data = data.T
        if data.shape[0] == 1:
            data = data[0]
    data = np.ascontiguousarray(data)
    if data.dtype == np.int16:
        return file_sr, data
    if data.dtype == np.int32:
        return file_sr, (data.astype(np.float64) / 2147483648.0).astype(np.float32)
    if data.dtype == np.uint8:
        return file_sr, (data.astype(np.float32) - 128.0) / 128.0
    return file_sr, data.astype(np.float32)


def _read_audio(path: str, sr: float, device=None, *, to_host: bool = True):
    """Decode a WAV file to float32 in [-1, 1] shaped [channels, n] or [n] and bring
    it to ``sr`` (librosa.load(path, sr=sr, mono=False) at script/mfcc.py:373).

    Decode/resample sits *before* the measured path (SURVEY.md section 8f rank 2).
    The file is parsed on the host (scipy's WAV reader); 16-bit PCM is scaled on the
    device (``mmf_pcm16_to_f32``) and the rate conversion is a polyphase resampler on
    the device (``mmf_resample_poly``: polyphase FIR with libsoxr HQ's band limits -- pass band to 0.913
    of the lower Nyquist, 120 dB -- which is what librosa.load applies; within 1e-5 of the ideal band-limited
    resampling below the band edge, not bit-identical to libsoxr: DESIGN.md section 6b).  A corpus of files goes
    through :meth:`FeatureExtractor.host_files` instead, in one call."""
    torch = _torch()
    file_sr, data = _parse_wav(path)
    plan = _any_plan(_device_index(device))
    try:
        if data.dtype == np.int16:
            y = plan.pcm16_to_f32(data)
        else:
            y = _to_dev(data, torch.float32, plan.cfg.device)
        if sr is not None and float(file_sr) != float(sr):
            up, down = resample_ratio(file_sr, sr)
            y = plan.resample_poly(y, up, down, quality="hq")
    except MmfError as e:
        _raise_from(e)
    return np.ascontiguousarray(y.cpu().numpy()) if to_host else y


def load_channel(file_path: str, signal_sample_rate: float = 10_000, channel_nb: int = 0):
    """Drop-in for ``load_channel`` (script/mfcc.py:262-289): all channels at the
    requested rate (the reference's channel selection is commented out)."""
    return _read_audio(file_path, signal_sample_rate)


def _change_setup(sigSr, tStep, winLen, n_mfcc, n_fft, minFreq, maxFreq, n_mels, preemph, device, flags=0):
    win_length, hop_length = frame_sizes(sigSr, winLen, tStep)  # script/mfcc.py:382-384
    cfg = MfccConfig(
        sample_rate=float(sigSr),
        n_fft=int(n_fft),
        win_length=win_length,
        hop_length=hop_length,
        n_mels=int(n_mels),
        n_mfcc=int(n_mfcc),
        fmin=float(minFreq),
        fmax=float(maxFreq),
        preemph=float(preemph),
        device=_device_index(device),
        flags=flags,
    )
    try:
        return get_plan(cfg)
    except MmfError as e:
        _raise_from(e)


def _time_anchors(T: int, tStep: float, winLen: float) -> np.ndarray:
    return np.round(np.multiply(np.arange(1, T + 1), tStep) + winLen / 2, 4)  # script/mfcc.py:390


def get_MFCCS_change_batch(
    audio,
    sigSr,
    /,
    *,
    tStep=0.001,
    winLen=0.025,
    n_mfcc=13,
    n_fft=512,
    minFreq=100,
    maxFreq=10000,
    removeFirst=1,
    filtCutoff=12,
    filtOrd=6,
    diffMethod="grad",
    outFilter="iir",
    outFiltType="low",
    outFiltCutOff=[None],
    outFiltLen=6,
    outFiltPolyOrd=3,
    n_mels=128,
    preemph=0.0,
    return_features=False,
    device=None,
    flags=0,
):
    """``get_MFCCS_change`` for a batch ``[B, N]`` of equal-length clips.

    ``audio`` may be a numpy array (host) or a CUDA tensor (stays on the device and
    the result is returned as CUDA tensors).  Returns ``(totChange [B, T], T [T])``
    and, with ``return_features``, a dict with ``logmel``, ``mfcc``, ``delta``."""
    torch = _torch()
    if not isinstance(audio, torch.Tensor):
        audio = np.asarray(audio)
    _require_float_audio(audio)
    plan, prm, post = _change_request(
        sigSr, tStep, winLen, n_mfcc, n_fft, minFreq, maxFreq, removeFirst, filtCutoff, filtOrd, diffMethod, outFilter,
        outFiltType, outFiltCutOff, outFiltLen, outFiltPolyOrd, n_mels, preemph, device, flags,
    )
    on_device = isinstance(audio, torch.Tensor) and audio.is_cuda
    try:
        if not on_device and not return_features and post is None:
            a = np.asarray(audio)
            tot = plan.mfcc_change_host(a if a.ndim == 2 else a[None, :], prm)
            T = _time_anchors(tot.shape[-1], tStep, winLen)
            return tot, T
        pcm = audio if on_device else _to_dev(np.asarray(audio), torch.float32, plan.cfg.device)
        res = plan.mfcc_change(pcm, prm, want_logmel=return_features, want_mfcc=return_features, want_delta=return_features)
        tot = res["totChange"]
        if post is not None:
            tot = _apply_filter_dev(plan, tot, 1 / tStep, **post)
            if tot is None:  # unknown filter name: the reference returns None from applyFilter
                T = _time_anchors(res["totChange"].shape[-1], tStep, winLen)
                return (None, T, res) if return_features else (None, T)
    except MmfError as e:
        _raise_from(e)
    T = _time_anchors(tot.shape[-1], tStep, winLen)
    if not on_device:
        tot = tot.cpu().numpy()
        if return_features:
            res = {k: (v.cpu().numpy() if v is not None else None) for k, v in res.items()}
    if return_features:
        res["totChange"] = tot
        return tot, T, res
    return tot, T


def _change_request(sigSr, tStep, winLen, n_mfcc, n_fft, minFreq, maxFreq, removeFirst, filtCutoff, filtOrd, diffMethod,
                    outFilter, outFiltType, outFiltCutOff, outFiltLen, outFiltPolyOrd, n_mels, preemph, device, flags):
    """Plan, packed change parameters and the deferred 'fir'/'sg' output filter of one get_MFCCS_change request."""
    plan = _change_setup(sigSr, tStep, winLen, n_mfcc, n_fft, minFreq, maxFreq, n_mels, preemph, device, flags)
    cutOffNorm = filtCutoff / ((1 / tStep) / 2)  # script/mfcc.py:398
    sos = _butter_sos(filtOrd, cutOffNorm, "low")  # script/mfcc.py:400
    method = 0 if diffMethod == "grad" else 1

    # output filter: None -> Goldstein's low-pass with the same sos (mfcc.py:417-421);
    # 'iir' -> fused second sosfiltfilt; 'fir'/'sg' -> raw change, then the generic kernels
    out_sos = None
    post = None
    if outFilter is None:
        out_sos = sos
    else:
        # run the reference's validation up front (same exceptions, same order)
        if outFilter == "iir":
            out_sos = _design_iir(1 / tStep, outFiltCutOff, outFiltLen, outFiltType)
        else:
            post = dict(filt=outFilter, cutOff=outFiltCutOff, filtLen=outFiltLen, filtType=outFiltType, polyOrd=outFiltPolyOrd)
    return plan, make_change_params(sos, remove_first=removeFirst, diff_method=method, out_sos=out_sos), post


def get_MFCCS_change_many(
    clips,
    sigSr,
    /,
    *,
    tStep=0.001,
    winLen=0.025,
    n_mfcc=13,
    n_fft=512,
    minFreq=100,
    maxFreq=10000,
    removeFirst=1,
    filtCutoff=12,
    filtOrd=6,
    diffMethod="grad",
    outFilter="iir",
    outFiltType="low",
    outFiltCutOff=[None],
    outFiltLen=6,
    outFiltPolyOrd=3,
    n_mels=128,
    preemph=0.0,
    return_features=False,
    device=None,
    flags=0,
):
    """``get_MFCCS_change`` for a list of 1-D clips of any lengths, in one batched call.

    ``clips`` holds numpy arrays and/or CUDA tensors.  Returns one ``(totChange, T)`` per clip -- or
    ``(totChange, T, feats)`` with ``return_features`` -- equal to what ``get_MFCCS_change`` returns for that clip:
    numpy for a numpy clip, CUDA tensors for a CUDA clip.  A clip too short for the filters raises the
    single-clip call's exception, its message naming the clip's index."""
    torch = _torch()
    clips = [c if isinstance(c, torch.Tensor) else np.asarray(c) for c in clips]
    for c in clips:
        _require_float_audio(c)
        if c.ndim != 1:
            raise ValueError("get_MFCCS_change_many takes 1-D clips")
    if not clips:
        return []
    plan, prm, post = _change_request(
        sigSr, tStep, winLen, n_mfcc, n_fft, minFreq, maxFreq, removeFirst, filtCutoff, filtOrd, diffMethod, outFilter,
        outFiltType, outFiltCutOff, outFiltLen, outFiltPolyOrd, n_mels, preemph, device, flags,
    )
    lengths = [int(c.shape[0]) for c in clips]
    n_max = max(max(lengths), 1)
    dev = plan.device
    if all(not isinstance(c, torch.Tensor) for c in clips):  # one host->device copy of the padded batch
        host = np.zeros((len(clips), n_max), np.float32)
        for i, c in enumerate(clips):
            host[i, : lengths[i]] = c
        pcm = torch.as_tensor(host).to(dev)
    else:
        pcm = torch.zeros((len(clips), n_max), device=dev, dtype=torch.float32)
        for i, c in enumerate(clips):
            pcm[i, : lengths[i]] = c.to(dev) if isinstance(c, torch.Tensor) else torch.as_tensor(np.asarray(c, np.float32))
    try:
        res = plan.mfcc_change_varlen(
            pcm, lengths, prm, want_logmel=return_features, want_mfcc=return_features, want_delta=return_features
        )
        frames = res.pop("frames")
        tots = [res["totChange"][i, : frames[i]] for i in range(len(clips))]
        if post is not None:
            filtered = []
            for i, t in enumerate(tots):
                try:
                    filtered.append(_apply_filter_dev(plan, t, 1 / tStep, **post))
                except ValueError as e:  # a curve too short for the output filter: name the clip
                    raise ValueError(f"clip {i}: {e}") from None
            tots = filtered
    except MmfError as e:
        _raise_from(e)
    out = []
    for i, c in enumerate(clips):
        on_device = isinstance(c, torch.Tensor) and c.is_cuda
        conv = (lambda v: v) if on_device else (lambda v: v.cpu().numpy())
        tot = tots[i]
        T = _time_anchors(int(frames[i]), tStep, winLen)
        tot = conv(tot) if tot is not None else None
        if return_features:
            feats = {k: (conv(v[i, ..., : frames[i]]) if v is not None else None) for k, v in res.items() if k != "totChange"}
            feats["totChange"] = tot
            out.append((tot, T, feats))
        else:
            out.append((tot, T))
    return out


def _design_iir(sr, cutOff, filtLen, filtType):
    """The validation + butter() of applyFilter's 'iir' branch (script/mfcc.py:82-106)."""
    if cutOff is None:
        raise Exception("Cannot apply filter without specifying a cut Off freq. (CutOff is None).")
    filtTypes = np.array(["bandpass", "lowpass", "highpass"])
    try:
        filtType = filtTypes[np.argwhere([t.startswith(filtType) for t in filtTypes]).flatten()][0]
    except Exception:
        raise Exception("filtType must be one among: lowpass, highpass, bandpass. Partial matches allowed.")
    if any((sr / 2) <= np.array(cutOff)):
        raise Exception(
            "Cut off frequencies must be smaller than the half of the sampling freq. of the signal submitted to the filter"
        )
    if (len(cutOff) > 0) & (any(np.diff(cutOff) <= 0)):
        raise Exception("If two cut off freqs are provided: cutOff[0]<cutOff[1]")
    cutOff = np.array(cutOff)
    w = cutOff / (sr / 2)
    if ((len(cutOff) == 1) and ((filtType == "lowpass") | (filtType == "highpass"))) | (
        (len(cutOff) == 2) and (filtType == "bandpass")
    ):
        return _butter_sos(filtLen, w, filtType)
    raise Exception("only one or two cut off frequencies allowed. If two freqs are provided, filtType must be bandpass")


def get_MFCCS_change(
    audioIn,
    sigSr,
    /,
    *,
    channelN=0,
    tStep=0.001,
    winLen=0.025,
    n_mfcc=13,
    n_fft=512,
    minFreq=100,
    maxFreq=10000,
    removeFirst=1,
    filtCutoff=12,
    filtOrd=6,
    diffMethod="grad",
    outFilter="iir",
    outFiltType="low",
    outFiltCutOff=[None],
    outFiltLen=6,
    outFiltPolyOrd=3,
    n_mels=128,
    preemph=0.0,
    return_features=False,
    device=None,
):
    """Drop-in for ``get_MFCCS_change`` (script/mfcc.py:291-427).

    Additive keywords (all default to the reference's behaviour): ``n_mels`` (the
    reference never passes it, so librosa's 128), ``preemph`` (0 = none),
    ``return_features``, ``device``.  Returns ``(totChange, T)`` as float64 arrays."""
    from_file = type(audioIn) == str
    if from_file:  # script/mfcc.py:372-373; the decoded, resampled audio stays on the device
        myAudio = _read_audio(audioIn, sigSr, device, to_host=False)
    else:
        myAudio = audioIn
    if len(np.shape(myAudio)) > 1:  # script/mfcc.py:377-380
        y = myAudio[channelN, :]
    else:
        y = myAudio
    out = get_MFCCS_change_batch(
        y[None, :] if from_file else np.asarray(y)[None, :],
        sigSr,
        tStep=tStep,
        winLen=winLen,
        n_mfcc=n_mfcc,
        n_fft=n_fft,
        minFreq=minFreq,
        maxFreq=maxFreq,
        removeFirst=removeFirst,
        filtCutoff=filtCutoff,
        filtOrd=filtOrd,
        diffMethod=diffMethod,
        outFilter=outFilter,
        outFiltType=outFiltType,
        outFiltCutOff=outFiltCutOff,
        outFiltLen=outFiltLen,
        outFiltPolyOrd=outFiltPolyOrd,
        n_mels=n_mels,
        preemph=preemph,
        return_features=return_features,
        device=device,
    )
    host = (lambda v: v.cpu().numpy()) if from_file else (lambda v: v)
    if return_features:
        tot, T, feats = out
        feats = {k: (host(v[0]) if v is not None else None) for k, v in feats.items()}
        return (host(tot[0]) if tot is not None else None), T, feats
    tot, T = out
    return (host(tot[0]) if tot is not None else None), T


# ---------------------------------------------------------------------------
# get_velocity
# ---------------------------------------------------------------------------


def get_velocity(x, sr, difference=1, method="gradient", width=3, accOrder=2, polyOrder=2, device=None):
    """Drop-in for ``get_velocity`` (script/calc.py:593-650).

    Like the reference, the derivative runs along axis 0 of ``x`` (``savgol_filter(axis=0)`` at calc.py:639,
    ``FinDiff(0, ...)`` at :636); ``'gradient'`` on N-D input makes ``np.gradient`` return one array per axis,
    which the reference then feeds back into ``np.gradient`` -- reproduced only for 1-D input, N-D raises."""
    if method not in ("finDiff", "sg", "gradient"):
        raise ValueError("Méthode inconnue. Utilisez 'gradient', 'sg' ou 'finDiff'.")
    torch = _torch()
    is_tensor = isinstance(x, torch.Tensor)
    xa = x if is_tensor else np.asarray(x)
    if xa.ndim == 0:
        raise ValueError("get_velocity: x must have at least one dimension")
    if xa.ndim > 1 and method == "gradient":
        raise ValueError("get_velocity (B200): method='gradient' is supported for 1-D trajectories only")
    di = _device_index(device)
    plan = _any_plan(di)
    xd = _to_dev(xa, torch.float64, di)
    nd = xd.dim()
    if nd > 1:  # the kernels run along the last axis: bring axis 0 there
        xd = xd.movedim(0, -1).contiguous()
    try:
        if method == "finDiff":
            coef, el, er = _findiff_stencil(int(difference), int(accOrder))
            y = plan.stencil(xd, coef, el, er) * (float(sr) ** int(difference))
        elif method == "sg":
            if xd.shape[-1] < width:
                raise ValueError("If mode is 'interp', window_length must be less than or equal to the size of x.")
            coef, el, er = _savgol_stencil(int(width), int(polyOrder), int(difference))
            y = plan.stencil(xd, coef, el, er)
        else:
            h = 1 / sr
            grad = (np.array([-0.5, 0.0, 0.5]) / h, np.array([[-1.0, 1.0]]) / h, np.array([[-1.0, 1.0]]) / h)
            y = xd
            for _ in range(difference):
                if y.shape[-1] < 2:
                    raise ValueError(
                        "Shape of array too small to calculate a numerical gradient, at least (edge_order + 1) elements are required."
                    )
                y = plan.stencil(y, *grad)
    except MmfError as e:
        _raise_from(e)
    if nd > 1:
        y = y.movedim(-1, 0).contiguous()
    return y if is_tensor else y.cpu().numpy()


# ---------------------------------------------------------------------------
# amplitude envelope
# ---------------------------------------------------------------------------


def calculate_amplitude_envelope(
    x,
    sr,
    /,
    *,
    method="RMS",
    winLen=0.1,
    hopLen=0.01,
    center=True,
    outFilter=None,
    outFiltType="low",
    outFiltCutOff=[12],
    outFiltLen=6,
    outFiltPolyOrd=3,
    device=None,
):
    """Drop-in for ``calculate_amplitude_envelope`` / ``get_amplitude``
    (script/calc.py:221-343, script/mfcc.py:137-259), method ``'RMS'``.

    ``'Hilb'`` is the full-length Hilbert envelope (``mmf_hilbert_envelope``); like the reference
    (lower-case typo at script/calc.py:333) its time axis comes out on the hop grid.  ``'RMSpraat'``
    (Praat) raises NotImplementedError -- there is no CPU fallback."""
    torch = _torch()
    if method == "RMS":
        frLen = int(hopLen * sr)
        winLenS = int(winLen * sr)
        di = _device_index(device)
        plan = _any_plan(di)
        xa = np.asarray(x)
        if xa.ndim != 1:
            raise ValueError("calculate_amplitude_envelope (B200): only mono signals are supported")
        try:
            amp_dev = plan.rms(_to_dev(xa, torch.float32, di), winLenS, frLen, bool(center))[0]
        except MmfError as e:
            _raise_from(e)
    elif method == "Hilb":
        di = _device_index(device)
        plan = _any_plan(di)
        xa = np.asarray(x)
        if xa.ndim != 1:
            raise ValueError("calculate_amplitude_envelope (B200): only mono signals are supported")
        try:
            amp_dev = plan.hilbert_envelope(_to_dev(xa, torch.float32, di))
        except MmfError as e:
            _raise_from(e)
    elif method == "RMSpraat":
        raise NotImplementedError("amplitude method 'RMSpraat' calls Praat and is outside the B200 hot path (no CPU fallback)")
    else:
        # the reference falls through with `amp` unbound -> UnboundLocalError (script/calc.py:333)
        raise UnboundLocalError("cannot access local variable 'amp' where it is not associated with a value")
    ampT = np.arange(amp_dev.shape[0]) * hopLen  # script/calc.py:333-337
    ampSr = 1 / hopLen
    if outFilter is not None:
        y = _apply_filter_dev(
            plan, amp_dev, ampSr, filt=outFilter, filtType=outFiltType, cutOff=outFiltCutOff, filtLen=outFiltLen, polyOrd=outFiltPolyOrd
        )
        return (y.cpu().numpy() if y is not None else None), ampT
    return amp_dev.cpu().numpy(), ampT


get_amplitude = calculate_amplitude_envelope


def calculate_amplitude_envelope_many(
    clips,
    sr,
    /,
    *,
    method="RMS",
    winLen=0.1,
    hopLen=0.01,
    center=True,
    outFilter=None,
    outFiltType="low",
    outFiltCutOff=[12],
    outFiltLen=6,
    outFiltPolyOrd=3,
    device=None,
):
    """:func:`calculate_amplitude_envelope` (method ``'RMS'``) for a list of 1-D clips of any lengths: one packed
    upload and one ``mmf_rms_varlen`` launch for all of them.  ``sr`` is one rate for every clip or one rate per clip;
    each clip's frame geometry is ``int(winLen * sr_i)``, ``int(hopLen * sr_i)``.  The output filter, if any, runs per
    clip as the single call runs it.  Returns one ``(amp, ampT)`` per clip, equal to
    ``calculate_amplitude_envelope(clip, sr_i, ...)`` bit for bit; an error names the clip's index."""
    if method != "RMS":
        raise ValueError(f"calculate_amplitude_envelope_many takes method 'RMS' only, not {method!r}")
    clips = [np.asarray(c) for c in clips]
    if any(c.ndim != 1 for c in clips):
        raise ValueError("calculate_amplitude_envelope_many takes 1-D clips")
    if not clips:
        return []
    rates = [float(r) for r in (sr if np.ndim(sr) else [sr] * len(clips))]
    if len(rates) != len(clips):
        raise ValueError(f"sr has {len(rates)} rates for {len(clips)} clips")
    di = _device_index(device)
    plan = _any_plan(di)
    offsets = np.zeros(len(clips) + 1, np.int64)
    np.cumsum([c.shape[0] for c in clips], out=offsets[1:])
    geom = [(int(winLen * r), int(hopLen * r)) for r in rates]
    try:
        packed = np.concatenate([c.astype(np.float32, copy=False) for c in clips])
        amp, amp_off = plan.rms_varlen(packed, offsets, geom, bool(center))
        out = []
        host = amp.cpu().numpy() if outFilter is None else None
        for i in range(len(clips)):
            a0, a1 = int(amp_off[i]), int(amp_off[i + 1])
            ampT = np.arange(a1 - a0) * hopLen  # script/calc.py:333-337
            if outFilter is None:
                out.append((host[a0:a1], ampT))
                continue
            try:
                y = _apply_filter_dev(plan, amp[a0:a1], 1 / hopLen, filt=outFilter, filtType=outFiltType,
                                      cutOff=outFiltCutOff, filtLen=outFiltLen, polyOrd=outFiltPolyOrd)
            except ValueError as e:  # an envelope too short for the output filter: name the clip
                raise ValueError(f"clip {i}: {e}") from None
            out.append((y.cpu().numpy() if y is not None else None, ampT))
    except MmfError as e:
        _raise_from(e)
    return out


# ---------------------------------------------------------------------------
# batch feature bundle (log-mel, MFCC, delta, MFCC change, modulation spectrum)
# ---------------------------------------------------------------------------


def modspec_sizes(T: int, frame_rate: float, mod_win_s: float = 1.0, mod_hop_s: float = 0.5):
    Lw = int(round(mod_win_s * frame_rate))
    Hw = max(1, int(round(mod_hop_s * frame_rate)))
    nfft = 1 << max(1, (Lw - 1).bit_length())
    n_win = 1 + (T - Lw) // Hw if T >= Lw else 0
    return Lw, Hw, nfft, n_win


def band_bins(nfft: int, frame_rate: float, bands_hz=MODULATION_BANDS_HZ):
    """[lo, hi) bin ranges of the modulation bands on the k*frame_rate/nfft axis."""
    freqs = np.arange(nfft // 2 + 1) * frame_rate / nfft
    out = []
    for lo, hi in bands_hz:
        sel = np.nonzero((freqs >= lo) & (freqs < hi))[0]
        out.append((int(sel[0]), int(sel[-1]) + 1) if len(sel) else (0, 0))
    return out


class FeatureExtractor:
    """Reusable batch pipeline: PCM ``[B, N]`` on the device -> log-mel, MFCC, delta,
    MFCC-change curve and MFCC modulation spectrum, all left on the device."""

    def __init__(
        self,
        sr: float,
        *,
        tStep: float = 0.01,
        winLen: float = 0.025,
        n_fft: int = 512,
        n_mels: int = 40,
        n_mfcc: int = 13,
        fmin: float = 0.0,
        fmax: float | None = None,
        removeFirst: int = 1,
        filtCutoff: float = 12,
        filtOrd: int = 6,
        mod_win_s: float = 1.0,
        mod_hop_s: float = 0.5,
        bands_hz=MODULATION_BANDS_HZ,
        preemph: float = 0.0,
        device=None,
        flags: int = 0,
        amp_winLen: float = 0.1,
        amp_hopLen: float = 0.01,
        amp_center: bool = True,
        amp_outFilter=None,
        amp_outFiltType="low",
        amp_outFiltCutOff=[12],
        amp_outFiltLen=6,
    ):
        # the envelope's output filter is validated before any device work, with applyFilter's exceptions
        if amp_outFilter is None:
            self.amp_sos = None
        elif amp_outFilter == "iir":
            self.amp_sos = _design_iir(1 / amp_hopLen, amp_outFiltCutOff, amp_outFiltLen, amp_outFiltType)
        else:
            raise ValueError(f"the feature bundle takes amp_outFilter None or 'iir', not {amp_outFilter!r} (use "
                             "calculate_amplitude_envelope_many for 'fir' and 'sg')")
        self.amp_winLen, self.amp_hopLen, self.amp_center = float(amp_winLen), float(amp_hopLen), bool(amp_center)
        self.sr, self.tStep, self.winLen = float(sr), float(tStep), float(winLen)
        self.plan = _change_setup(sr, tStep, winLen, n_mfcc, n_fft, fmin, sr / 2 if fmax is None else fmax, n_mels, preemph, device, flags)
        sos = _butter_sos(filtOrd, filtCutoff / ((1 / tStep) / 2), "low")
        self.prm = make_change_params(sos, remove_first=removeFirst, diff_method=0, out_sos=sos)
        self.mod_win_s, self.mod_hop_s, self.bands_hz = mod_win_s, mod_hop_s, bands_hz
        self.frame_rate = 1.0 / tStep

    def modspec_geometry(self, T: int):
        Lw, Hw, nfft, _ = modspec_sizes(T, self.frame_rate, self.mod_win_s, self.mod_hop_s)
        return Lw, Hw, nfft, band_bins(nfft, self.frame_rate, self.bands_hz)

    def _amp(self, want, n_clips, rates):
        """The ``amp`` argument of :meth:`Plan.features_host_varlen` when ``want`` holds ``"amplitude"``: each clip's
        frame geometry at its own rate (``rates``, else the extractor's), as calc.py:326-331 computes it."""
        if "amplitude" not in want:
            return None
        rates = [self.sr] * n_clips if rates is None else [float(r) for r in rates]
        geom = [(int(self.amp_winLen * r), int(self.amp_hopLen * r)) for r in rates]
        return geom, self.amp_center, self.amp_sos

    def host_call(self, pcm_host, *, want=("totChange", "mfcc", "delta", "modspec", "band_energy"), out=None):
        """Host buffers in, host buffers out, through the single C-ABI bundle call."""
        pcm_host = np.asarray(pcm_host)
        T = self.plan.num_frames(pcm_host.shape[-1])
        mod = self.modspec_geometry(T) if ("modspec" in want or "band_energy" in want) else None
        try:
            return self.plan.features_host(pcm_host, self.prm, mod, want=want, out=out)
        except MmfError as e:
            _raise_from(e)

    def host_varlen(self, pcm_host, offsets, *, want=("totChange", "mfcc", "delta", "modspec", "band_energy"),
                    out=None, rates=None):
        """:meth:`host_call` for clips of different lengths packed back to back in one 1-D host buffer (float32, or
        int16 WAV samples): clip ``i`` is ``pcm_host[offsets[i]:offsets[i + 1]]``.  Returns the packed arrays of
        :meth:`Plan.features_host_varlen` with this extractor's modulation geometry; each clip's blocks equal
        :meth:`host_call` on that clip alone, bit for bit.  ``rates``: each clip's sample rate; clips are then
        resampled to the extractor's rate on the device as the WAV loader resamples them, and each clip's blocks
        equal :meth:`host_call` on the loader's resampled clip.

        ``"amplitude"`` in ``want`` adds each clip's RMS envelope with this extractor's ``amp_*`` settings, taken at
        the clip's own rate (``rates``, else the extractor's) from its native samples (int16 scaled by 1/32768):
        ``amplitude`` packed at ``amp_offsets``; clip ``i``'s block equals :func:`calculate_amplitude_envelope` on that
        clip as float32, bit for bit."""
        mod = self.modspec_geometry(0) if ("modspec" in want or "band_energy" in want) else None
        try:
            amp = self._amp(want, len(offsets) - 1, rates)
            return self.plan.features_host_varlen(pcm_host, offsets, self.prm, mod, want=want, out=out, rates=rates,
                                                  amp=amp)
        except MmfError as e:
            _raise_from(e)

    def host_many(self, clips, *, want=("totChange", "mfcc", "delta", "modspec", "band_energy"), rates=None):
        """:meth:`host_varlen` for a list of 1-D numpy clips of any lengths (all int16, or anything else as float32).
        Concatenates them once and returns one dict per clip of zero-copy views into the packed arrays, shaped as
        :func:`mfcc_features_batch` returns one clip without its batch axis (``totChange [T]``, ``mfcc`` /
        ``delta [n_mfcc, T]``, ``modspec [n_mfcc, W, nfft/2+1]``, ``band_energy [W, n_bands]``), plus ``T``, the
        frame times (at the extractor's rate when ``rates`` are given).  With ``"amplitude"`` in ``want``, each dict
        also holds ``amplitude`` and ``ampT``, what :func:`calculate_amplitude_envelope` returns for the clip.  A corpus
        already held in one buffer should call :meth:`host_varlen` with its offsets instead, which saves the
        concatenation."""
        clips = [np.asarray(c) for c in clips]
        if not clips:
            return []
        if any(c.ndim != 1 for c in clips):
            raise ValueError("host_many takes 1-D clips")
        dt = np.int16 if all(c.dtype == np.int16 for c in clips) else np.float32
        offsets = np.zeros(len(clips) + 1, np.int64)
        np.cumsum([c.shape[0] for c in clips], out=offsets[1:])
        res = self.host_varlen(np.concatenate(clips).astype(dt, copy=False), offsets, want=want, rates=rates)
        nm = self.plan.cfg.n_mfcc
        _, _, nfft, bins = self.modspec_geometry(0)
        nb, n_bands = nfft // 2 + 1, len(bins)
        fo, wo = res["frame_offsets"], res["window_offsets"]
        out = []
        for i in range(len(clips)):
            f0, f1, w0, w1 = int(fo[i]), int(fo[i + 1]), int(wo[i]), int(wo[i + 1])
            T, W = f1 - f0, w1 - w0
            d = {"totChange": res["totChange"][f0:f1]}
            for k in ("mfcc", "delta"):
                if k in res:
                    d[k] = res[k][nm * f0 : nm * f1].reshape(nm, T)
            if "modspec" in res:
                d["modspec"] = res["modspec"][nm * nb * w0 : nm * nb * w1].reshape(nm, W, nb)
            if "band_energy" in res:
                d["band_energy"] = res["band_energy"][n_bands * w0 : n_bands * w1].reshape(W, n_bands)
            d["T"] = _time_anchors(T, self.tStep, self.winLen)
            if "amplitude" in res:
                a0, a1 = int(res["amp_offsets"][i]), int(res["amp_offsets"][i + 1])
                d["amplitude"] = res["amplitude"][a0:a1]
                d["ampT"] = np.arange(a1 - a0) * self.amp_hopLen  # script/calc.py:333-337
            out.append(d)
        return out

    def host_files(self, paths, *, channel: int = 0, want=("totChange", "mfcc", "delta", "modspec", "band_energy")):
        """A corpus of WAV files at any sample rates through one :meth:`host_many` call.  Each file is parsed on the
        host, channel ``channel`` of a multi-channel file is kept, and its native samples cross PCIe once (as int16
        when every file is 16-bit PCM, else as float32) to be resampled on the device to the extractor's rate.
        Returns one dict per file, as :meth:`host_many` does; each file's blocks equal :meth:`host_call` on
        ``_read_audio(path, sr)[channel]``, bit for bit (rows are resampled independently, so selecting the channel
        first changes nothing).  A file that is not RIFF/WAVE raises ``ValueError`` naming its path.  ``amplitude`` is
        taken at the file's own rate on samples in [-1, 1]: for a 16-bit file, times 32768 it equals
        :func:`calculate_amplitude_envelope` of the raw samples, as the GUI computes it (``main.py:843-849``)."""
        rates, clips = [], []
        for p in paths:
            file_sr, data = _parse_wav(p)
            rates.append(float(file_sr))
            clips.append(data[channel] if data.ndim > 1 else data)
        if clips and not all(c.dtype == np.int16 for c in clips):
            # (float)x * 2^-15, as the device scales int16
            clips = [c.astype(np.float32) / np.float32(32768.0) if c.dtype == np.int16 else c for c in clips]
        return self.host_many(clips, want=want, rates=rates)

    def __call__(self, pcm, *, want_logmel: bool = True, want_modspec: bool = True):
        res = self.plan.mfcc_change(pcm, self.prm, want_logmel=want_logmel, want_mfcc=True, want_delta=True)
        if want_modspec:
            T = res["mfcc"].shape[-1]
            Lw, Hw, nfft, _ = modspec_sizes(T, self.frame_rate, self.mod_win_s, self.mod_hop_s)
            mag, band = self.plan.modspec(res["mfcc"], Lw, Hw, nfft, band_bins(nfft, self.frame_rate, self.bands_hz))
            res["modspec"], res["band_energy"] = mag, band
        return res

    def varlen(self, pcm, lengths, *, want_logmel: bool = True, want_modspec: bool = True):
        """:meth:`__call__` for clips of different lengths: row ``i`` of ``pcm [B, N_max]`` holds clip ``i`` in its
        first ``lengths[i]`` samples (whatever follows is ignored).  Returns the dict of :meth:`__call__`, padded
        to the longest clip (frames) and to the most modulation windows of any clip, plus ``frames`` and
        ``windows`` (numpy int64 ``[B]``); clip ``i``'s first ``frames[i]`` frames and ``windows[i]`` windows equal
        :meth:`__call__` on that clip alone, bit for bit, and the padding is 0."""
        res = self.plan.mfcc_change_varlen(pcm, lengths, self.prm, want_logmel=want_logmel, want_mfcc=True,
                                           want_delta=True)
        frames = res["frames"]
        # the modulation geometry does not depend on T, only each clip's window count does
        Lw, Hw, nfft, _ = modspec_sizes(0, self.frame_rate, self.mod_win_s, self.mod_hop_s)
        if want_modspec:
            mag, band, windows = self.plan.modspec_varlen(res["mfcc"], frames, Lw, Hw, nfft,
                                                          band_bins(nfft, self.frame_rate, self.bands_hz))
            res["modspec"], res["band_energy"] = mag, band
        else:
            windows = np.where(frames >= Lw, 1 + (frames - Lw) // Hw, 0)
        res["windows"] = windows
        return res


def mfcc_features_batch(audio, sr, *, device=None, **kw):
    """One-shot :class:`FeatureExtractor` call; numpy in -> numpy out, CUDA in -> CUDA out."""
    torch = _torch()
    fx = FeatureExtractor(sr, device=device, **kw)
    on_device = isinstance(audio, torch.Tensor) and audio.is_cuda
    try:
        res = fx(audio if on_device else _to_dev(np.asarray(audio), torch.float32, fx.plan.cfg.device))
    except MmfError as e:
        _raise_from(e)
    T = res["totChange"].shape[-1]
    res["T"] = _time_anchors(T, fx.tStep, fx.winLen)
    if not on_device:
        res = {k: (v.cpu().numpy() if hasattr(v, "cpu") else v) for k, v in res.items()}
    return res


def mfcc_features_many(clips, sr, *, device=None, **kw):
    """:func:`mfcc_features_batch` for a list of 1-D clips of any lengths, in one batched call
    (:meth:`FeatureExtractor.varlen`).

    ``clips`` holds numpy arrays and/or CUDA tensors.  Returns one dict per clip, equal bit for bit to
    ``mfcc_features_batch(clip[None], sr, **kw)`` with the batch axis dropped: numpy for a numpy clip, CUDA tensors
    for a CUDA clip.  A clip too short for the filters raises the single-clip call's ``ValueError``, its message
    naming the clip's index."""
    torch = _torch()
    clips = [c if isinstance(c, torch.Tensor) else np.asarray(c) for c in clips]
    for c in clips:
        _require_float_audio(c)
        if c.ndim != 1:
            raise ValueError("mfcc_features_many takes 1-D clips")
    if not clips:
        return []
    fx = FeatureExtractor(sr, device=device, **kw)
    lengths = [int(c.shape[0]) for c in clips]
    n_max = max(max(lengths), 1)
    dev = fx.plan.device
    if all(not isinstance(c, torch.Tensor) for c in clips):  # one host->device copy of the padded batch
        host = np.zeros((len(clips), n_max), np.float32)
        for i, c in enumerate(clips):
            host[i, : lengths[i]] = c
        pcm = torch.as_tensor(host).to(dev)
    else:
        pcm = torch.zeros((len(clips), n_max), device=dev, dtype=torch.float32)
        for i, c in enumerate(clips):
            pcm[i, : lengths[i]] = c.to(dev) if isinstance(c, torch.Tensor) else torch.as_tensor(np.asarray(c, np.float32))
    try:
        res = fx.varlen(pcm, lengths)
    except MmfError as e:
        _raise_from(e)
    frames, windows = res.pop("frames"), res.pop("windows")
    on_dev = [isinstance(c, torch.Tensor) and c.is_cuda for c in clips]
    host = {k: v.cpu().numpy() for k, v in res.items() if v is not None} if not all(on_dev) else {}
    out = []
    for i in range(len(clips)):
        src = res if on_dev[i] else host
        T, W = int(frames[i]), int(windows[i])
        d = {
            "totChange": src["totChange"][i, :T],
            "logmel": src["logmel"][i, :, :T],
            "mfcc": src["mfcc"][i, :, :T],
            "delta": src["delta"][i, :, :T],
            "modspec": src["modspec"][i, :, :W],
            "band_energy": src["band_energy"][i, :W],
        }
        if not on_dev[i]:
            d = {k: np.ascontiguousarray(v) for k, v in d.items()}
        d["T"] = _time_anchors(T, fx.tStep, fx.winLen)
        out.append(d)
    return out
