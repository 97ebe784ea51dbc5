"""Every zero-phase IIR (K4) and MFCC-change (K5, fused per-clip) kernel path against a long-double reference.

The float64 half of get_MFCCS_change -- zero-phase Butterworth of the kept MFCC rows, derivative + norm over rows,
output filter of the curve -- runs on these kernels (csrc/change_fused.cu, csrc/sos_par.cuh, csrc/post_kernels.cu),
chosen by ``sosfiltfilt_any``, ``change_route``, ``change_fused_supported`` / ``change_fused_lm_supported`` and
``change_split_out`` (csrc/c_api.cu):

  path     kernels                                             taken when
  par      sosfiltfilt_par_kernel<float|double, 1..4, false>   L = T + 2 padlen <= 32 * 191 = 6112, <= 4 sections
  long     sos_long_kernel x4 + sos_long_carry_kernel x2       L > 6112, <= 4 sections, rows * L * 8 <= 1 GiB
  seq      sosfiltfilt_kernel<float|double, 1..8 | 0>          > 4 sections (0: 9 .. 16), or the 1 GiB fallback
  fused    change_fused_kernel<NS, NS, false, false>           a delta output wanted, or MMF_FLAG_SEPARATE_MFCC
  folded   change_fused_kernel<NS, NS, true, false>            the default without a delta output; MMF_FLAG_FOLD_MFCC
                                                               with one
  split    fused or folded, then sosfiltfilt_par_kernel        an 'iir' output filter and >= 32 clips
           <double, NS_out, false> over the curves
  unfused  K4 + delta_norm_kernel + K4                         MMF_FLAG_UNFUSED_CHANGE, T > 12 * 32 * 9 = 3456, the
                                                               220 KB shared-memory limit, or unequal section counts
                                                               without the split

The boundaries are computed from Python restatements of ``sos_par_chunk``, ``sosfiltfilt_any`` and
``fused_row_doubles`` / ``change_route``, which ``test_case_matrix_reaches_every_instantiation`` checks against each
case's intended path.  Each GPU case names its kernels, and a ``torch.profiler`` probe asserts that exactly those
K4 / K5 kernels ran (mangled or demangled names).  The probes run once per module in a child process (``probed``
says why); each test then runs its own call with the launch count checked and grades it.

The reference (``_ref_sosfiltfilt``, ``_ref_change``) is scipy's sosfiltfilt restated in long double: the odd
extension is built in the input's dtype (as scipy and the kernels build it), then widened; the change stage starts
from the kernel's own float32 MFCC output, so K1 - K3 error never enters the grade.

Bounds:
  * filter error: max |y - ref| over a row / max |x| of that row;
  * curve error: max |curve - ref| over a clip / max |filtered row| of that clip;
one bound per path and conditioning class, the class being the smallest normalised cutoff wn of the cascade:
w (wn >= 0.1), m (>= 0.02), i (>= 0.003), x (>= 0.001), u (< 0.001; the long path only).
Largest values observed on a B200 (1000 W power limit) over the case matrix; every bound (BOUND_FILT, BOUND_CURVE)
is 1.5x .. 7x the largest value observed in its class (long u: 6e-8, a float32 row's own resolution):
  filter  par   w 1.1e-15, m 1.4e-13, i 5.3e-11, x 5.4e-10
          long  w 1.2e-15, m 1.3e-13, i 4.4e-11, x 4.1e-10, u 4.0e-8 (order 8, wn 0.00015, T 20 000)
          seq   w 2.3e-14, m 1.9e-13, i 1.3e-12
  curve   folded w 2.5e-16, m 3.9e-16; fused w 2.8e-17, m 1.5e-15; split w 3.5e-17; unfused w 3.8e-17, m 4.0e-17
The scan's error grows as the cutoff falls (scipy's own float64 sosfiltfilt is at 1.9e-12 for the par x case and
2.1e-11 for the long u case); at every accepted configuration measured it stays under a float32 row's own
resolution, 6e-8.  The curve is graded on the scale of the filtered rows, which it is far below.
``test_tolerances_catch_plausible_*_mistakes`` (CPU) hold the bounds honest: every listed mistake misses the reference
by more than 10x every bound it applies to, on the fixtures of the GPU cases.
"""

import json
import os
import re
import subprocess
import sys
from functools import partial
from typing import NamedTuple

import numpy as np
import pytest
import scipy.signal

import modulation_mfcc_b200 as mm
from modulation_mfcc_b200 import _lib

LD = np.longdouble

# constants of csrc/change_fused.cu and csrc/mmf_internal.h the routes depend on
PAR_MAX_CHUNK = 191  # kSosParMaxChunk
PAR_MAX_SECTIONS = 4  # kParMaxSections
LONG_CL = 33  # kLongCL
FUSED_MAX_T = 12 * 32 * 9  # kFusedMaxWarps * 32 * kFusedPerThread
FUSED_SMEM = 220 * 1024
FUSED_NC = 16  # kFusedNC
SEQ_FALLBACK_BYTES = 1 << 30

UNFUSED = _lib.MMF_FLAG_UNFUSED_CHANGE
SEPARATE = _lib.MMF_FLAG_SEPARATE_MFCC
FOLD = _lib.MMF_FLAG_FOLD_MFCC
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

BOUND_FILT = {
    ("par", "w"): 5e-15, ("par", "m"): 5e-13, ("par", "i"): 2e-10, ("par", "x"): 2e-9,
    ("long", "w"): 5e-15, ("long", "m"): 5e-13, ("long", "i"): 2e-10, ("long", "x"): 2e-9, ("long", "u"): 6e-8,
    ("seq", "w"): 1e-13, ("seq", "m"): 1e-12, ("seq", "i"): 5e-12,
}
BOUND_CURVE = {
    ("folded", "w"): 1e-15, ("folded", "m"): 2e-15, ("fused", "w"): 2e-16, ("fused", "m"): 5e-15,
    ("split", "w"): 2e-16, ("unfused", "w"): 2e-16, ("unfused", "m"): 2e-16,
}

TOP_DB = 80.0


def _torch():
    import torch

    return torch


# ---------------------------------------------------------------------------
# long-double reference
# ---------------------------------------------------------------------------


def _padlen(sos, adjust=True):
    """scipy.signal.sosfiltfilt's default padlen: 3 * (2n + 1 - min(#b2 == 0, #a2 == 0))."""
    n = sos.shape[0]
    k = min(int(np.sum(sos[:, 2] == 0)), int(np.sum(sos[:, 5] == 0))) if adjust else 0
    return 3 * (2 * n + 1 - k)


def _ref_sosfiltfilt(sos, x, mistake=None):
    """scipy.signal.sosfiltfilt(sos, x) along the last axis of ``x [rows, T]`` in long double.

    The odd extension is computed in x's dtype, then widened (scipy extends a float32 row in float32); the passes
    start from sosfilt_zi * the first sample of their input.  ``mistake`` (tests of the bounds only) makes one
    plausible implementation error on purpose."""
    x = np.asarray(x)
    p = _padlen(sos, adjust=mistake != "padlen_unadjusted")
    xe = x.astype(np.float64) if mistake == "ext_in_float64" else x
    two = xe.dtype.type(2)
    left = two * xe[..., :1] - xe[..., p:0:-1]
    right = two * xe[..., -1:] - xe[..., -2:-p - 2:-1]
    ext = np.concatenate([left, xe, right], axis=-1).astype(LD)
    s = np.asarray(sos, np.float64).astype(LD)
    zi = scipy.signal.sosfilt_zi(s)[:, None, :]
    first = ext[..., 1:2] if mistake == "zi_second_sample" else ext[..., :1]
    f, _ = scipy.signal.sosfilt(s, ext, axis=-1, zi=zi * first[None])
    r = f[..., ::-1]
    zb = np.zeros_like(zi * r[None, ..., :1]) if mistake == "bwd_zero_state" else zi * r[None, ..., :1]
    b, _ = scipy.signal.sosfilt(s, r, axis=-1, zi=zb)
    return b[..., ::-1][..., p:p + x.shape[-1]]


def _ref_diff(f, method, mistake=None):
    """d/dt along the last axis: np.gradient (method 0) or savgol_filter(3, 2, deriv=1, mode='interp') (method 1).

    Both share the interior (f[t+1] - f[t-1]) / 2; method 1's edges are the second-order one-sided differences.
    For T < 3 (method 1) the kernels fall back to the first-order edges of np.gradient, where savgol_filter
    raises; T = 1 gives 0."""
    T = f.shape[-1]
    d = np.zeros_like(f)
    if T == 1:
        return d
    half = 1 if mistake == "gradient_without_half" else 2
    d[..., 1:-1] = (f[..., 2:] - f[..., :-2]) / half
    if method == 0 or T < 3 or mistake == "sg_first_order_edges":
        d[..., 0] = f[..., 1] - f[..., 0]
        d[..., -1] = f[..., -1] - f[..., -2]
    else:
        d[..., 0] = (-3 * f[..., 0] + 4 * f[..., 1] - f[..., 2]) / 2
        d[..., -1] = (3 * f[..., -1] - 4 * f[..., -2] + f[..., -3]) / 2
    return d


def _ref_change(mfcc, first, sos, method, out_sos, mistake=None):
    """(curve [B, T], scale [B]) of get_MFCCS_change after the MFCC, from the kernel's float32 ``mfcc [B, n, T]``:
    row filter, derivative, sqrt(sum d^2) / rows, output cascade (``out_sos`` None: the raw curve).  scale is
    max |filtered row| of each clip."""
    m = np.asarray(mfcc, np.float32)
    keep = m if mistake == "norm_keeps_c0" else m[:, first:]
    B, R, T = keep.shape
    f = _ref_sosfiltfilt(sos, keep.reshape(B * R, T), mistake=mistake).reshape(B, R, T)
    d = _ref_diff(f, method, mistake)
    raw = np.sqrt(np.sum(d * d, axis=1)) / R
    scale = np.abs(f[:, (first if mistake == "norm_keeps_c0" else 0):]).reshape(B, -1).max(axis=1)
    if out_sos is None:
        return raw, scale
    o = sos if mistake == "out_filter_is_row_filter" else out_sos
    return _ref_sosfiltfilt(o, raw, mistake=mistake if mistake in ("zi_second_sample", "bwd_zero_state") else None), scale


def _filt_err(y, ref, x):
    """max over rows of max |y - ref| / max |x row|; inf for a non-finite output."""
    y = np.asarray(y, np.float64)
    if not np.all(np.isfinite(y)):
        return float("inf")
    scale = np.abs(np.asarray(x, np.float64)).max(axis=-1)
    return float(np.max(np.abs(y.astype(LD) - ref).max(axis=-1) / scale))


def _curve_err(tot, ref, scale):
    tot = np.asarray(tot, np.float64)
    if not np.all(np.isfinite(tot)):
        return float("inf")
    return float(np.max(np.abs(tot.astype(LD) - ref).max(axis=-1) / scale))


def _cls(wn):
    w = float(np.min(np.atleast_1d(wn)))
    return "w" if w >= 0.1 else "m" if w >= 0.02 else "i" if w >= 0.003 else "x" if w >= 0.001 else "u"


def _design(kind, order, wn):
    if kind == "band":
        return scipy.signal.butter(order, [wn, 2 * wn], btype="bandpass", output="sos")
    return scipy.signal.butter(order, wn, btype="highpass" if kind == "high" else "lowpass", output="sos")


def _rows(rows, T, seed, dtype):
    """Random walks over an offset, in the input dtype."""
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((rows, T)).cumsum(axis=-1) * (4.0 / np.sqrt(T)) + rng.uniform(-3, 3, (rows, 1)) + 1.5
    # sample-to-sample noise across binades: the float32 odd extension 2 x[0] - x[k] rounds
    x += rng.standard_normal((rows, T)) * 0.4
    return x.astype(dtype)


# ---------------------------------------------------------------------------
# routes: Python restatements of the C++ decisions
# ---------------------------------------------------------------------------


def _par_chunk(p, T):
    """sos_par_chunk: the chunk length of a row of T samples, -1 when the row does not fit shared memory."""
    L = T + 2 * p
    return -1 if L > 32 * PAR_MAX_CHUNK else ((L + 31) // 32) | 1


def _k4_path(ns, p, rows, T):
    """sosfiltfilt_any."""
    if ns <= PAR_MAX_SECTIONS and _par_chunk(p, T) > 0:
        return "par"
    L = T + 2 * p
    n_sb = (L + 32 * LONG_CL - 1) // (32 * LONG_CL)
    if ns <= PAR_MAX_SECTIONS and L > 32 * LONG_CL and rows * n_sb < 0x7FFFFFFF * 4 and rows * L * 8 <= SEQ_FALLBACK_BYTES:
        return "long"
    return "seq"


def _k4_kernels(path, dt, ns):
    if path == "par":
        return [("sosfiltfilt_par_kernel", (dt, ns, False))]
    if path == "long":
        return ([("sos_long_kernel", (dt, ns, b, a)) for b in (False, True) for a in (False, True)]
                + [("sos_long_carry_kernel", (dt, ns, b)) for b in (False, True)])
    return [("sosfiltfilt_kernel", (dt, ns if ns <= 8 else 0))]


def _fused_row_doubles(cl1, cl2, rows):
    d = rows * 32 * cl1
    return max(d, 32 * cl2) if cl2 is not None else d


def _change_route(n_mels, n_mfcc, first, sos, out_sos, n_clips, T, want_delta, flags):
    """change_route -> (path, kernels); path 'split' when the fused or folded kernel leaves the output filter to its
    own launch."""
    rows = n_mfcc - first
    ns1, p1 = sos.shape[0], _padlen(sos)
    out_iir = out_sos is not None
    cl1 = _par_chunk(p1, T) if ns1 <= PAR_MAX_SECTIONS else -1
    cl2 = (_par_chunk(_padlen(out_sos), T) if out_sos.shape[0] <= PAR_MAX_SECTIONS else -1) if out_iir else None
    split = out_iir and n_clips >= 32

    def supported(extra):
        if rows < 1 or T > FUSED_MAX_T or (out_iir and not split and out_sos.shape[0] != ns1):
            return False
        smem = _fused_row_doubles(cl1, cl2 if out_iir else None, rows) * 8
        return smem <= FUSED_SMEM and smem + extra <= FUSED_SMEM

    path = "unfused"
    if not (flags & UNFUSED or cl1 < 0 or (out_iir and cl2 < 0)):
        folds = (flags & FOLD or not want_delta) and not flags & (SEPARATE | _lib.MMF_FLAG_MMA_DCT) and n_mfcc <= FUSED_NC
        if folds and supported(n_mels * FUSED_NC * 4):
            path = "folded"
        elif supported(0):
            path = "fused"
    if path != "unfused":
        ks = [("change_fused_kernel", (ns1, ns1, path == "folded", False))]
        if split:
            ks += [("sosfiltfilt_par_kernel", ("double", out_sos.shape[0], False))]
            path = "split"
        return path, ks
    ks = _k4_kernels(_k4_path(ns1, p1, n_clips * rows, T), "float", ns1) + [("delta_norm_kernel", ())]
    if out_iir:
        ks += _k4_kernels(_k4_path(out_sos.shape[0], _padlen(out_sos), n_clips, T), "double", out_sos.shape[0])
    return path, ks


def _last(pred, lo, hi):
    """largest T in [lo, hi] with pred(T), pred true at lo and monotone."""
    assert pred(lo)
    while lo < hi:
        mid = (lo + hi + 1) // 2
        lo, hi = (mid, hi) if pred(mid) else (lo, mid - 1)
    return lo


# ---------------------------------------------------------------------------
# kernel probe
# ---------------------------------------------------------------------------

_NAMES = ("sosfiltfilt_par_kernel", "sos_long_carry_kernel", "sos_long_kernel", "sosfiltfilt_kernel",
          "change_fused_kernel", "delta_norm_kernel")


def _arg(a, mangled):
    if mangled:
        if a in ("f", "d"):
            return "float" if a == "f" else "double"
        v = int(a[2:-1])
        return bool(v) if a[1] == "b" else v
    a = a.strip()
    if a in ("float", "double"):
        return a
    if a in ("true", "false"):
        return a == "true"
    return int(re.sub(r"[^\d-]", "", a))


def _k45_kernels(names):
    """(kernel, template arguments) of every K4 / K5 kernel among profiler kernel names, demangled or mangled."""
    out = []
    for name in names:
        for k in _NAMES:
            m = re.search(r"(?<![\w])" + k + r"<([^>]*)>", name)
            if m:
                out.append((k, tuple(_arg(a, False) for a in m.group(1).split(","))))
                break
            m = re.search(r"(?<=\d)" + k + r"I((?:[fd]|L[ib]-?\d+E)+)E", name)
            if m:
                out.append((k, tuple(_arg(a, True) for a in re.findall(r"[fd]|L[ib]-?\d+E", m.group(1)))))
                break
            if re.search(r"(?<![\w])" + k + r"(?:\(|$)", name) or re.search(r"(?<=\d)" + k + r"E", name):
                out.append((k, ()))
                break
    return out


def _probe(fn):
    """Run ``fn`` under torch.profiler with CUDA activity; return (result, K4 / K5 kernels that ran)."""
    torch = _torch()
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events()]
    assert names, "the profiler saw no kernels at all: the path probe cannot tell which kernel ran"
    return res, _k45_kernels(names)


def _expect(ran, want):
    assert sorted(ran, key=repr) == sorted(want, key=repr), f"expected {want}, K4 / K5 kernels that ran: {ran}"


def _run(fn, want, k3=0):
    """``fn()`` with its launch count checked: one per kernel of ``want``, plus ``k3`` MFCC-stage launches.  Which
    kernels ran is the probe's to say (``probed``)."""
    torch = _torch()
    torch.cuda.synchronize()
    n0 = _lib.lib().mmf_launch_count(0)
    res = fn()
    torch.cuda.synchronize()
    assert _lib.lib().mmf_launch_count(0) - n0 == len(want) + k3, want
    return res


# ---------------------------------------------------------------------------
# the case matrix
# ---------------------------------------------------------------------------


class K4Case(NamedTuple):
    id: str
    kind: str  # low, high, band
    order: int
    wn: float
    dt: str  # float or double
    T: int
    rows: int
    path: str  # the intended path


def _sos(case):
    return _design(case.kind, case.order, case.wn)


def K4(kind, order, wn, dt, T, rows, path):
    sos = _design(kind, order, wn)
    if T == "min":
        T = _padlen(sos) + 1
    elif T == "last_par":
        T = _last(lambda t: _par_chunk(_padlen(sos), t) > 0, _padlen(sos) + 1, 1 << 20)
    elif T == "first_long":
        T = _last(lambda t: _par_chunk(_padlen(sos), t) > 0, _padlen(sos) + 1, 1 << 20) + 1
    elif isinstance(T, str):  # "L<n>": the odd-extended row is n samples long
        T = int(T[1:]) - 2 * _padlen(sos)
    return K4Case(f"{path}_{dt[0]}{sos.shape[0]}_{kind}{order}_wn{wn}_T{T}_r{rows}", kind, order, wn, dt, T, rows, path)


F, D = "float", "double"
K4_CASES = [
    # par: every instantiation, T at padlen + 1 and at the last T of the chunk-parallel kernel, odd orders
    *[K4("low", 2 * ns, 0.3, dt, 1001, 5, "par") for dt in (F, D) for ns in (1, 2, 3, 4)],
    K4("low", 6, 0.3, F, "min", 7, "par"), K4("low", 1, 0.3, D, "min", 3, "par"),
    K4("low", 8, 0.024, F, "last_par", 7, "par"), K4("low", 3, 0.3, D, "last_par", 5, "par"),
    *[K4("low", o, 0.024, F, 1001, 7, "par") for o in (1, 3, 5, 7)],
    K4("low", 6, 0.024, F, 3456, 7, "par"), K4("low", 8, 0.003, D, 3456, 5, "par"),
    K4("low", 8, 0.0015, F, 5000, 5, "par"), K4("low", 5, 0.003, F, 2001, 6, "par"),
    K4("high", 4, 0.3, D, 500, 5, "par"), K4("band", 2, 0.1, F, 777, 7, "par"),
    K4("band", 4, 0.024, D, 3000, 5, "par"),
    # long: every instantiation at the first T past the chunk-parallel kernel; ill-conditioned cascades
    *[K4("low", 2 * ns, 0.3, dt, "first_long", 3, "long") for dt in (F, D) for ns in (1, 2, 3, 4)],
    K4("low", 8, 0.024, F, "first_long", 7, "long"), K4("low", 5, 0.024, D, 9000, 3, "long"),
    K4("low", 6, 0.0015, F, 20000, 3, "long"), K4("low", 8, 0.0015, D, 20000, 3, "long"),
    K4("low", 8, 0.003, F, 12000, 3, "long"), K4("high", 3, 0.024, F, 7001, 3, "long"),
    K4("low", 8, 0.00015, F, 20000, 2, "long"), K4("low", 8, 0.00015, D, 20000, 2, "long"),
    # seq: 5 .. 8 sections and the generic 9 .. 16, both input types; rows across two warps
    *[K4("low", 2 * ns, 0.3, dt, 1001, 37, "seq") for dt in (F, D) for ns in (5, 6, 7, 8)],
    K4("low", 9, 0.024, D, "min", 33, "seq"), K4("low", 11, 0.024, F, "L1024", 7, "seq"),
    K4("low", 13, 0.024, F, "L1025", 5, "seq"), K4("low", 15, 0.003, D, 2001, 5, "seq"),
    K4("low", 18, 0.3, F, 1001, 37, "seq"), K4("low", 24, 0.024, D, 1001, 7, "seq"),
    K4("low", 32, 0.3, F, "min", 3, "seq"), K4("low", 31, 0.3, D, 6001, 1, "seq"),
    K4("low", 17, 0.024, F, 7000, 7, "seq"), K4("low", 12, 0.003, F, 4000, 5, "seq"),
    K4("high", 12, 0.3, F, 999, 7, "seq"), K4("band", 10, 0.1, D, 1500, 5, "seq"),
    K4("band", 5, 0.024, F, 2500, 6, "seq"), K4("low", 10, 0.024, F, "last_par", 3, "seq"),
    K4("low", 10, 0.024, D, "first_long", 3, "seq"),
]

# the 1 GiB fallback: rows * L * 8 > 1 GiB sends rows of <= 4 sections to the sequential kernel.  Every
# instantiation at the first row count past the limit, and two at the last row count the super-block scan takes.
FALLBACK_T = 11000


def _gib_rows(ns):
    """the most rows of FALLBACK_T samples the super-block scan takes for an order-2ns low-pass"""
    p = _padlen(scipy.signal.butter(2 * ns, 0.024, output="sos"))
    return _last(lambda r: _k4_path(ns, p, r, FALLBACK_T) == "long", 1, 1 << 20)


FALLBACK = [(dt, ns, "seq") for dt in (F, D) for ns in (1, 2, 3, 4)] + [(F, 1, "long"), (D, 4, "long")]


class ChangeCase(NamedTuple):
    id: str
    n_mels: int
    n_mfcc: int
    first: int
    method: int
    order: int
    wn: float
    out: str  # raw, same, oddpad (same section count, other padlen), unequal (other section count)
    n_clips: int
    T: int
    want_delta: bool
    flags: int
    path: str  # the intended path


def _change_sos(case):
    sos = scipy.signal.butter(case.order, case.wn, output="sos")
    if case.out == "raw":
        return sos, None
    if case.out == "same":
        return sos, sos
    if case.out == "oddpad":
        out = scipy.signal.butter(case.order - 1, 0.1, output="sos")
        assert out.shape[0] == sos.shape[0] and _padlen(out) != _padlen(sos)
        return sos, out
    return sos, scipy.signal.butter(2 if sos.shape[0] > 1 else 4, 0.1, output="sos")


def _route_of(case, T=None):
    sos, out = _change_sos(case)
    return _change_route(case.n_mels, case.n_mfcc, case.first, sos, out, case.n_clips, case.T if T is None else T,
                         case.want_delta, case.flags)


def CH(n_mels, n_mfcc, first, method, order, out, n_clips, T, path, *, wn=0.24, delta=False, flags=0, edge=None):
    c = ChangeCase("", n_mels, n_mfcc, first, method, order, wn, out, n_clips, 0, delta, flags, path)
    p = _padlen(scipy.signal.butter(order, wn, output="sos"))
    if T == "min":
        T = p + 1
    elif T == "edge":  # the last T on the case's fused form
        T = _last(lambda t: _route_of(c, t)[0] == edge, p + 1, FUSED_MAX_T)
    elif T == "edge+1":
        T = _last(lambda t: _route_of(c, t)[0] == edge, p + 1, FUSED_MAX_T) + 1
    rows = n_mfcc - first
    cid = (f"{path}_ns{(order + 1) // 2}_mels{n_mels}_rows{rows}_m{method}_rf{first}_{out}_clips{n_clips}_T{T}"
           + ("_delta" if delta else "") + ("_unfusedflag" if flags & UNFUSED else "")
           + ("_separate" if flags & SEPARATE else "") + ("_fold" if flags & FOLD else "") + ("_wn" + str(wn) if wn != 0.24 else ""))
    return c._replace(id=cid, T=T)


CHANGE_CASES = [
    # folded: NS 1 .. 4, rows 1 / 7 / 12 / 15, both methods, removeFirst 0 / 1, every output kind
    CH(40, 13, 1, 0, 2, "raw", 1, 1001, "folded"),
    CH(40, 8, 1, 1, 4, "same", 31, 1001, "folded"),
    CH(40, 15, 0, 0, 6, "oddpad", 3, 1001, "folded"),
    CH(40, 13, 1, 1, 8, "same", 2, 1001, "folded", wn=0.024),
    CH(40, 2, 1, 0, 6, "same", 1, "min", "folded"),
    CH(40, 1, 0, 1, 3, "raw", 2, "min", "folded"),
    CH(40, 8, 1, 0, 6, "same", 1, 3456, "folded"),
    CH(40, 16, 1, 1, 6, "same", 2, "edge", "folded", edge="folded"),
    CH(512, 16, 1, 0, 4, "raw", 2, "edge", "folded", edge="folded"),
    CH(40, 13, 1, 1, 6, "same", 2, 1001, "folded", delta=True, flags=FOLD),
    # fused (the MFCC kernel first): NS 1 .. 4; the folded form's shared-memory edge at n_mels 512
    CH(40, 13, 1, 0, 2, "same", 1, 1001, "fused", delta=True),
    CH(40, 8, 0, 1, 4, "oddpad", 3, 1001, "fused", delta=True),
    CH(40, 13, 1, 1, 6, "raw", 31, 1001, "fused", delta=True, wn=0.024),
    CH(40, 16, 1, 0, 8, "same", 2, 777, "fused", flags=SEPARATE),
    CH(512, 8, 1, 0, 6, "same", 1, 3456, "fused"),
    CH(512, 16, 1, 0, 4, "raw", 2, "edge+1", "fused", edge="folded"),
    CH(40, 16, 1, 1, 6, "same", 2, "edge", "fused", delta=True, edge="fused"),
    # split: 32 clips with an 'iir' output filter, equal and unequal section counts
    CH(40, 13, 1, 0, 6, "same", 32, 1001, "split"),
    CH(40, 13, 1, 1, 6, "unequal", 32, 1001, "split", delta=True),
    CH(40, 13, 0, 0, 4, "oddpad", 33, 500, "split"),
    # unfused: the flag, T past the fused kernel, the shared-memory limit, unequal sections without the split,
    # sequential row warps that straddle clips (5 clips x 12 rows), long rows
    CH(40, 13, 1, 0, 6, "same", 5, 1001, "unfused", flags=UNFUSED),
    CH(40, 13, 1, 1, 10, "same", 5, 1001, "unfused", flags=UNFUSED),
    CH(40, 13, 1, 0, 10, "raw", 5, 700, "unfused"),
    CH(40, 8, 1, 0, 6, "same", 1, 3457, "unfused"),
    CH(40, 16, 1, 0, 6, "same", 2, "edge+1", "unfused", edge="folded"),
    CH(40, 13, 1, 1, 6, "unequal", 31, 1001, "unfused"),
    CH(40, 12, 0, 0, 4, "same", 2, 7000, "unfused", wn=0.024),
    CH(40, 13, 1, 0, 6, "unequal", 32, 4000, "unfused", delta=True),
]


# ---------------------------------------------------------------------------
# CPU: the reference, the matrix and the bounds
# ---------------------------------------------------------------------------


@pytest.mark.parametrize("kind,order,wn,dt", [("low", 6, 0.24, np.float64), ("low", 5, 0.024, np.float64),
                                              ("band", 4, 0.1, np.float64), ("low", 8, 0.003, np.float32),
                                              ("high", 3, 0.3, np.float32)])
def test_reference_agrees_with_scipy(kind, order, wn, dt):
    """On float64 rows the reference is scipy.signal.sosfiltfilt to its own float64 rounding; on float32 rows too
    (scipy extends them in float32, as the reference does), but not with the extension done in long double."""
    sos = _design(kind, order, wn)
    x = _rows(3, 777, 5, dt)
    ref = _ref_sosfiltfilt(sos, x)
    assert _filt_err(scipy.signal.sosfiltfilt(sos, x), ref, x) < 1e-12
    if dt == np.float32:
        wrong = scipy.signal.sosfiltfilt(sos.astype(LD), x.astype(LD))
        assert _filt_err(wrong.astype(np.float64), ref, x) > 1e-11


def test_reference_diff_matches_numpy_and_savgol():
    f = _rows(4, 50, 9, np.float64)
    assert np.allclose(_ref_diff(f, 0), np.gradient(f, axis=-1), rtol=0, atol=1e-14)
    sg = scipy.signal.savgol_filter(f, 3, 2, deriv=1, axis=-1, mode="interp")
    assert np.allclose(_ref_diff(f, 1), sg, rtol=0, atol=1e-12)
    # T < 3: first-order edges for both methods (savgol_filter cannot take a 3-sample window there)
    assert np.array_equal(_ref_diff(f[:, :2], 1), np.gradient(f[:, :2], axis=-1))
    assert np.all(_ref_diff(f[:, :1], 1) == 0)


def test_reference_known_answers():
    """A constant row stays that constant through a low-pass, a high-pass takes it to ~0; the curve of rows c_r * t is
    sqrt(sum c_r^2) / rows away from the edges."""
    sos = scipy.signal.butter(6, 0.024, output="sos")
    x = np.full((2, 500), 3.25)
    # exactly c * g^2, g the DC gain of the float64 coefficients (1 - g ~ 1e-14 from their rounding)
    s = sos.astype(LD)
    g = np.prod(s[:, :3].sum(axis=1) / s[:, 3:].sum(axis=1))
    assert abs(g - 1) < 1e-12
    assert np.max(np.abs(_ref_sosfiltfilt(sos, x) - LD(3.25) * g * g)) < 1e-15
    hp = scipy.signal.butter(4, 0.1, btype="highpass", output="sos")
    assert np.max(np.abs(_ref_sosfiltfilt(hp, x))) < 1e-15
    m = np.zeros((1, 4, 300), np.float32)
    m[0, 1:] = np.array([1.0, -2.0, 0.5], np.float32)[:, None] * np.arange(300, dtype=np.float32)[None] / 128
    raw, scale = _ref_change(m, 1, scipy.signal.butter(2, 0.3, output="sos"), 1, None)
    want = np.sqrt(1.0 + 4.0 + 0.25) / 128 / 3
    assert np.max(np.abs(raw[0, 50:-50] - LD(want))) < 1e-12 * want  # away from the edge transients


def test_case_matrix_reaches_every_instantiation():
    """Each case's intended path is the restated route's, and together the cases (with the 1 GiB fallback) target
    every kernel instantiation of the table: par and long <float|double, 1..4>, seq <float|double, 1..8 | 0>,
    change_fused_kernel <NS, NS, FROM_LM> for NS 1..4, the split and delta_norm_kernel."""
    targets = []
    for c in K4_CASES:
        sos = _sos(c)
        assert c.T > _padlen(sos), c.id
        assert _k4_path(sos.shape[0], _padlen(sos), c.rows, c.T) == c.path, c.id
        assert c.rows % 4 and c.rows % 32, c.id
        targets += _k4_kernels(c.path, c.dt, sos.shape[0])
    for dt, ns, path in FALLBACK:
        sos = scipy.signal.butter(2 * ns, 0.024, output="sos")
        rows = _gib_rows(ns) + (path == "seq")
        assert _k4_path(ns, _padlen(sos), rows, FALLBACK_T) == path
        assert (rows * (FALLBACK_T + 2 * _padlen(sos)) * 8 > SEQ_FALLBACK_BYTES) == (path == "seq")
        targets += _k4_kernels(path, dt, ns)
    assert {p for _, _, p in FALLBACK} == {"seq", "long"}
    for c in CHANGE_CASES:
        path, ks = _route_of(c)
        assert path == c.path, (c.id, path)
        targets += ks
    want = {("sosfiltfilt_par_kernel", (dt, ns, False)) for dt in (F, D) for ns in range(1, 5)}
    want |= {k for dt in (F, D) for ns in range(1, 5) for k in _k4_kernels("long", dt, ns)}
    want |= {("sosfiltfilt_kernel", (dt, ns)) for dt in (F, D) for ns in range(0, 9)}
    want |= {("change_fused_kernel", (ns, ns, lm, False)) for ns in range(1, 5) for lm in (False, True)}
    want |= {("delta_norm_kernel", ())}
    assert want <= set(targets), want - set(targets)
    assert {c.path for c in CHANGE_CASES} == {"folded", "fused", "split", "unfused"}
    # the switches, each from both sides
    last_par = {c.id: _last(lambda t: _par_chunk(_padlen(_sos(c)), t) > 0, _padlen(_sos(c)) + 1, 1 << 20)
                for c in K4_CASES}
    for path, dT in [("par", 0), ("long", 1), ("seq", 0), ("seq", 1)]:
        assert any(c.path == path and c.T == last_par[c.id] + dT for c in K4_CASES), (path, dT)
    for path in ("par", "seq"):
        assert any(c.path == path and c.T == _padlen(_sos(c)) + 1 for c in K4_CASES), path
    assert {1, 7, 12, 15} <= {c.n_mfcc - c.first for c in CHANGE_CASES}
    assert {1, 31, 32} <= {c.n_clips for c in CHANGE_CASES}
    assert {FUSED_MAX_T, FUSED_MAX_T + 1, 1001} <= {c.T for c in CHANGE_CASES}
    assert {"raw", "same", "oddpad", "unequal"} == {c.out for c in CHANGE_CASES}
    # the shared-memory edges: the last T of the folded form and the first past it, at n_mels 40 and 512
    for n_mels in (40, 512):
        edge = [c for c in CHANGE_CASES if c.n_mels == n_mels and c.path != "unfused" and
                _route_of(c, c.T + 1)[0] not in (c.path, "split")]
        assert any(c.path == "folded" for c in edge), n_mels
        assert any(_route_of(c, c.T - 1)[0] == "folded" and c.path != "folded" for c in CHANGE_CASES
                   if c.n_mels == n_mels), n_mels


def test_probe_reads_mangled_and_demangled_names():
    """_k45_kernels on the library's own kernel symbols (mangled and demangled) and on names it must ignore."""
    names = [
        "_ZN3mmf22sosfiltfilt_par_kernelIfLi1ELb0EEEvPKT_lililNS_6SosParEPdlNS_11FusedVarlenEi",
        "void mmf::sosfiltfilt_par_kernel<double, 4, false>(double const*, long, int, long, int, long, mmf::SosPar, "
        "double*, long, mmf::FusedVarlen, int)",
        "_ZN3mmf15sos_long_kernelIdLi2ELb1ELb1EEEvPKT_lilPKdlllNS_6SosParES5_PdS7_S7_l",
        "void mmf::sos_long_kernel<double, 4, true, false>(double const*, long, int, long, double const*, long, long, "
        "long, mmf::SosPar, double const*, double*, double*, double*, long)",
        "_ZN3mmf21sos_long_carry_kernelIfLi2ELb0EEEvPKT_lilPKdlllNS_6SosParES5_Pd",
        "void mmf::sos_long_carry_kernel<double, 2, true>(double const*, long, int, long, double const*, long, long, "
        "long, mmf::SosPar, double const*, double*)",
        "_ZN3mmf18sosfiltfilt_kernelIfLi7EEEvPKT_lllilNS_7SosArgsEPdl",
        "void mmf::sosfiltfilt_kernel<float, 0>(float const*, long, long, long, int, long, mmf::SosArgs, double*, long)",
        "_ZN3mmf19change_fused_kernelILi2ELi2ELb0ELb1EEEvPKfiiiiiNS_6SosParES3_iPdNS_13FusedMfccArgsEiNS_11FusedVarlenE",
        "void mmf::change_fused_kernel<4, 4, true, false>(float const*, int, int, int, int, int, mmf::SosPar, "
        "mmf::SosPar, int, double*, mmf::FusedMfccArgs, int, mmf::FusedVarlen)",
        "_ZN3mmf17delta_norm_kernelEPKdiliPd",
        "mmf::delta_norm_kernel(double const*, int, long, int, double*)",
        "void mmf::mfcc_pk_kernel<7, 16, false>(float*, int const*, int, int, int, float, float*, float*, int)",
        "_ZN3mmf14mfcc_pk_kernelILi7ELi16ELb0EEEvPfPKiiiifS1_S1_i",
        "cudaLaunchKernel",
        "void at::native::vectorized_elementwise_kernel<4, at::native::FillFunctor<double>, std::array<char*, 1ul> >"
        "(int, at::native::FillFunctor<double>, std::array<char*, 1ul>)",
    ]
    assert _k45_kernels(names) == [
        ("sosfiltfilt_par_kernel", ("float", 1, False)), ("sosfiltfilt_par_kernel", ("double", 4, False)),
        ("sos_long_kernel", ("double", 2, True, True)), ("sos_long_kernel", ("double", 4, True, False)),
        ("sos_long_carry_kernel", ("float", 2, False)), ("sos_long_carry_kernel", ("double", 2, True)),
        ("sosfiltfilt_kernel", ("float", 7)), ("sosfiltfilt_kernel", ("float", 0)),
        ("change_fused_kernel", (2, 2, False, True)), ("change_fused_kernel", (4, 4, True, False)),
        ("delta_norm_kernel", ()), ("delta_norm_kernel", ()),
    ]


def test_every_gpu_case_has_a_probe_job():
    """Each GPU test's cases map onto JOBS one to one, so the probe process sees every case the suite grades."""
    keys = (["k4:" + c.id for c in K4_CASES] + [_key_of("gib", p) for p in FALLBACK]
            + [_key_of("strided", p) for p in _STRIDED] + [_key_of("constant", p) for p in _CONSTANT]
            + ["change:" + c.id for c in CHANGE_CASES] + [_key_of("delta", p) for p in _DELTA])
    assert len(keys) == len(set(keys)) and set(keys) == set(JOBS)


_K4_MISTAKES = ["ext_in_float64", "zi_second_sample", "bwd_zero_state", "padlen_unadjusted"]
_CHANGE_MISTAKES = ["gradient_without_half", "sg_first_order_edges", "norm_keeps_c0", "out_filter_is_row_filter"]


def _applies(mistake, sos, dt, wn):
    if mistake == "ext_in_float64":
        # the extension's float32 rounding moves a filtered row by 1e-12 .. 2e-8 of its scale on these fixtures, least
        # at low cutoffs: visible under the bounds of the classes w and m only (the scan's own rounding is larger below)
        return dt == F and _cls(wn) in ("w", "m")
    if mistake == "padlen_unadjusted":
        return _padlen(sos) != _padlen(sos, adjust=False)
    return True


@pytest.mark.parametrize("mistake", _K4_MISTAKES)
def test_tolerances_catch_plausible_filter_mistakes(mistake):
    """Each plausible K4 mistake misses the reference by more than 10x the bound of every case it applies to, on
    two rows of that case's fixture (float64 output, as the kernels write it)."""
    worst = {}
    for i, c in enumerate(K4_CASES):
        sos = _sos(c)
        if not _applies(mistake, sos, c.dt, c.wn):
            continue
        x = _rows(2, c.T, 1000 + i, np.float32 if c.dt == F else np.float64)
        ref = _ref_sosfiltfilt(sos, x)
        wrong = _ref_sosfiltfilt(sos, x, mistake=mistake).astype(np.float64)
        worst[c.id] = _filt_err(wrong, ref, x) / BOUND_FILT[(c.path, _cls(c.wn))]
    assert worst and min(worst.values()) > 10.0, min(worst.items(), key=lambda kv: kv[1])


@pytest.mark.parametrize("mistake", _CHANGE_MISTAKES + _K4_MISTAKES[:3])
def test_tolerances_catch_plausible_change_mistakes(mistake):
    """Each plausible mistake of the change stage misses the reference curve by more than 10x the bound of every
    case it applies to, on synthetic float32 MFCC rows of the case's shape (two clips)."""
    worst = {}
    for i, c in enumerate(CHANGE_CASES):
        sos, out = _change_sos(c)
        if mistake == "sg_first_order_edges" and c.method != 1:
            continue
        if mistake == "norm_keeps_c0" and c.first != 1:
            continue
        if mistake == "out_filter_is_row_filter" and (out is None or out is sos):
            continue
        rng = np.random.default_rng(2000 + i)
        m = (rng.standard_normal((2, c.n_mfcc, c.T)).cumsum(axis=-1) * (30.0 / np.sqrt(c.T))
             + rng.uniform(-40, 40, (2, c.n_mfcc, 1))).astype(np.float32)
        ref, scale = _ref_change(m, c.first, sos, c.method, out)
        wrong, _ = _ref_change(m, c.first, sos, c.method, out, mistake=mistake)
        worst[c.id] = _curve_err(wrong.astype(np.float64), ref, scale) / BOUND_CURVE[(c.path, _cls(c.wn))]
    assert worst and min(worst.values()) > 10.0, min(worst.items(), key=lambda kv: kv[1])


# ---------------------------------------------------------------------------
# GPU jobs: each builds one call on seeded inputs and names the kernels it must run
# ---------------------------------------------------------------------------

_PLAN_CFG = mm.MfccConfig(16000, 512, 400, 160, 40, 13, 0.0, 8000.0)
_CHANGE_GEOS = {40: (16000, 512, 400, 160, 0.0, 8000.0), 512: (48000, 4096, 3840, 960, 4000.0, 24000.0)}


class Job(NamedTuple):
    fn: object  # the call
    want: list  # the K4 / K5 kernels it must launch
    k3: int  # MFCC-stage launches besides them
    ctx: dict  # inputs the grade needs


def _k4_job(case, dev):
    torch = _torch()
    plan = mm.get_plan(_PLAN_CFG)
    sos = _sos(case)
    x = _rows(case.rows, case.T, 300 + case.order * 17 + case.T, np.float32 if case.dt == F else np.float64)
    xd = torch.as_tensor(x).to(dev)
    return Job(lambda: plan.sosfiltfilt(xd, sos), _k4_kernels(case.path, case.dt, sos.shape[0]), 0,
               dict(x=x, sos=sos))


def _gib_job(dt, ns, path, dev):
    torch = _torch()
    plan = mm.get_plan(_PLAN_CFG)
    sos = scipy.signal.butter(2 * ns, 0.024, output="sos")
    rows = _gib_rows(ns) + (path == "seq")
    g = torch.Generator(device=dev).manual_seed(11 + ns)
    x = torch.randn((rows, FALLBACK_T), generator=g, device=dev, dtype=torch.float64)
    x = x.cumsum_(dim=1).mul_(4.0 / FALLBACK_T ** 0.5).add_(1.5).to(torch.float32 if dt == F else torch.float64)
    return Job(lambda: plan.sosfiltfilt(x, sos), _k4_kernels(path, dt, ns), 0, dict(x=x, sos=sos, rows=rows))


_STRIDED = [("par", 6, 1001, F), ("par", 4, 333, D), ("long", 6, 7000, F), ("long", 3, 6500, D), ("seq", 12, 1001, F),
            ("seq", 20, 900, D)]
_POISON = np.array([0x7FF8DEADBEEF0001], np.int64).view(np.float64)[0]


def _strided_job(path, order, T, dt, dev):
    """mmf_sosfiltfilt on 7 rows with x_row_stride = T + 5 (NaN in the gaps) and y_row_stride = T + 3 (a NaN payload
    in the gaps)."""
    torch = _torch()
    plan = mm.get_plan(_PLAN_CFG)
    sos = np.ascontiguousarray(scipy.signal.butter(order, 0.024, output="sos"))
    rows = 7
    npdt = np.float32 if dt == F else np.float64
    x = _rows(rows, T, 40 + order, npdt)
    xb = np.full((rows, T + 5), np.nan, npdt)
    xb[:, :T] = x
    yb = np.full((rows, T + 3), _POISON)
    xd, yd = torch.as_tensor(xb).to(dev), torch.as_tensor(yb).to(dev)

    def call():
        _lib.check(_lib.lib().mmf_sosfiltfilt(plan._h, xd.data_ptr(), 1 if dt == F else 0, rows, T, T + 5,
                                              sos.ctypes.data, sos.shape[0], yd.data_ptr(), T + 3,
                                              int(torch.cuda.current_stream(dev).cuda_stream)))
        return yd

    return Job(call, _k4_kernels(path, dt, sos.shape[0]), 0, dict(x=x, sos=sos, yb=yb))


_CONSTANT = [(p, o, T, kind) for p, o, T in [("par", 6, 1001), ("long", 8, 8000), ("seq", 12, 1001)]
             for kind in ("low", "high")]


def _constant_job(path, order, T, kind, dev):
    torch = _torch()
    plan = mm.get_plan(_PLAN_CFG)
    sos = _design(kind, order, 0.024)
    xd = torch.full((5, T), -7.5, device=dev, dtype=torch.float32)
    return Job(lambda: plan.sosfiltfilt(xd, sos), _k4_kernels(path, F, sos.shape[0]), 0, dict(sos=sos))


def _key(maxima):
    """float32 maxima -> the int32 keys the kernels decode (key_to_float's inverse)."""
    bits = np.ascontiguousarray(maxima, np.float32).view(np.int32)
    return np.where(bits >= 0, bits, bits ^ np.int32(0x7FFFFFFF)).astype(np.int32)


def _logmel(B, n_mels, T, seed):
    """[B, n_mels, T] float32 random walks in dB over a per-mel offset, and the clips' maxima."""
    rng = np.random.default_rng(seed)
    off = np.linspace(22.0, -58.0, n_mels)[None, :, None] + rng.uniform(-6, 6, (1, n_mels, 1))
    walk = rng.standard_normal((B, n_mels, T)).cumsum(axis=-1) * (6.0 / np.sqrt(T))
    x = (off + walk + 2.0 * rng.standard_normal((B, n_mels, T))).astype(np.float32)
    return x, x.reshape(B, -1).max(axis=1)


def _change_job(case, dev):
    torch = _torch()
    sr, n_fft, win, hop, fmin, fmax = _CHANGE_GEOS[case.n_mels]
    plan = mm.get_plan(mm.MfccConfig(sr, n_fft, win, hop, case.n_mels, case.n_mfcc, fmin, fmax, top_db=TOP_DB,
                                     flags=case.flags))
    sos, out = _change_sos(case)
    x, cmax = _logmel(case.n_clips, case.n_mels, case.T, 500 + case.T + case.n_mfcc)
    lm, km = torch.as_tensor(x).to(dev), torch.as_tensor(_key(cmax)).to(dev)
    prm = mm.make_change_params(sos, remove_first=case.first, diff_method=case.method, out_sos=out)
    want = _route_of(case)[1]
    folded = any(k == "change_fused_kernel" and a[2] for k, a in want)  # no separate MFCC launch
    return Job(lambda: plan.change_from_logmel(lm, km, prm, want_delta=case.want_delta, clamp_in_place=False), want,
               0 if folded else 1, dict(sos=sos, out=out))


_DELTA = [(3, 5, 1, 0), (3, 5, 1, 1), (3, 5, 2, 0), (3, 5, 2, 1), (2, 4, 3, 1), (2, 12, 1001, 0), (2, 12, 1001, 1),
          (65537, 3, 7, 1)]


def _delta_job(B, R, T, method, dev):
    torch = _torch()
    plan = mm.get_plan(_PLAN_CFG)
    x = _rows(B * R, T, 70 + T, np.float64).reshape(B, R, T)
    xd = torch.as_tensor(x).to(dev)
    return Job(lambda: plan.delta_norm(xd, method), [("delta_norm_kernel", ())] * ((B + 65534) // 65535), 0, dict(x=x))


def _key_of(kind, params):
    return kind + ":" + "_".join(str(p) for p in params)


# every GPU case: key -> job builder (device -> Job)
JOBS = {}
for _c in K4_CASES:
    JOBS["k4:" + _c.id] = partial(_k4_job, _c)
for _p in FALLBACK:
    JOBS[_key_of("gib", _p)] = partial(_gib_job, *_p)
for _p in _STRIDED:
    JOBS[_key_of("strided", _p)] = partial(_strided_job, *_p)
for _p in _CONSTANT:
    JOBS[_key_of("constant", _p)] = partial(_constant_job, *_p)
for _c in CHANGE_CASES:
    JOBS["change:" + _c.id] = partial(_change_job, _c)
for _p in _DELTA:
    JOBS[_key_of("delta", _p)] = partial(_delta_job, *_p)


def _probe_all(out_path):
    """Run every job once under torch.profiler and write {key: [[kernel, template arguments], ...]} to out_path."""
    torch = _torch()
    dev = torch.device("cuda", 0)
    ran = {}
    for key, build in JOBS.items():
        job = build(dev)
        _, ran[key] = _probe(job.fn)
        del job
        if key.startswith("gib:"):
            torch.cuda.empty_cache()
    with open(out_path, "w") as f:
        json.dump({k: [[n, list(a)] for n, a in v] for k, v in ran.items()}, f)


@pytest.fixture(scope="module")
def probed(cuda_device, tmp_path_factory):
    """The K4 / K5 kernels each job launches, seen by torch.profiler in a child process.

    The probes run in their own process: this module's GPU cases would otherwise be the first torch.profiler
    sessions of a whole-suite run, and then later modules' probes (test_logmel_paths, test_mfcc_paths, ...) saw
    none of this library's kernels.  The child builds every job from the same seeds and shapes as the test that
    grades it, and the dispatch depends on shapes and cascades alone."""
    out = tmp_path_factory.mktemp("probe") / "kernels.json"
    env = dict(os.environ)
    env["PYTHONPATH"] = ROOT + os.pathsep + env.get("PYTHONPATH", "")
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.abspath(__file__), str(out)]
    r = subprocess.run(cmd, env=env, cwd=ROOT, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, f"the probe process failed:\n{r.stdout[-2000:]}\n{r.stderr[-4000:]}"
    with open(out) as f:
        data = json.load(f)
    assert set(data) == set(JOBS)
    return {k: [(n, tuple(a)) for n, a in v] for k, v in data.items()}


def _graded(probed, key, dev):
    """Build job ``key``, check that the probe saw exactly its kernels, run it with its launch count checked."""
    job = JOBS[key](dev)
    _expect(probed[key], job.want)
    return _run(job.fn, job.want, job.k3), job.ctx


# ---------------------------------------------------------------------------
# GPU: K4 through Plan.sosfiltfilt and the C ABI
# ---------------------------------------------------------------------------


@pytest.mark.gpu
@pytest.mark.parametrize("case", K4_CASES, ids=[c.id for c in K4_CASES])
def test_sosfiltfilt_path_matches_reference(case, probed, cuda_device, record_property):
    y, ctx = _graded(probed, "k4:" + case.id, cuda_device)
    err = _filt_err(y.cpu().numpy(), _ref_sosfiltfilt(ctx["sos"], ctx["x"]), ctx["x"])
    record_property("filt_err", err)
    record_property("cls", f"{case.path}/{_cls(case.wn)}")
    assert err <= BOUND_FILT[(case.path, _cls(case.wn))], err


@pytest.mark.gpu
@pytest.mark.parametrize("dt,ns,path", FALLBACK, ids=[_key_of("", p)[1:] for p in FALLBACK])
def test_one_gib_switch(dt, ns, path, probed, cuda_device, record_property):
    """Rows of 11 000 samples of a <= 4-section cascade: at the last row count with rows * L * 8 <= 1 GiB the
    super-block scan, one row more the sequential kernel.  Every row is finite; the first, the last and rows around
    warp boundaries match the reference."""
    torch = _torch()
    y, ctx = _graded(probed, _key_of("gib", (dt, ns, path)), cuda_device)
    x, rows = ctx["x"], ctx["rows"]
    assert bool(torch.isfinite(y).all())
    sample = [0, 1, 30, 31, 32, 33, 4095, 4096, 6143, 6144, rows - 33, rows - 32, rows - 1]
    xs = x[sample].cpu().numpy()
    err = _filt_err(y[sample].cpu().numpy(), _ref_sosfiltfilt(ctx["sos"], xs), xs)
    record_property("filt_err", err)
    record_property("cls", f"{path}/m")
    assert err <= BOUND_FILT[(path, "m")], err
    del x, y, ctx
    torch.cuda.empty_cache()


@pytest.mark.gpu
@pytest.mark.parametrize("path,order,T,dt", _STRIDED)
def test_strided_rows_through_the_c_abi(path, order, T, dt, probed, cuda_device):
    """x_row_stride = T + 5 and y_row_stride = T + 3: the gaps of x hold NaN (never read), the gaps of y hold a NaN
    payload that must stay bit for bit."""
    yd, ctx = _graded(probed, _key_of("strided", (path, order, T, dt)), cuda_device)
    y = yd.cpu().numpy()
    assert np.array_equal(y[:, T:].view(np.int64), ctx["yb"][:, T:].view(np.int64)), "the gaps of y were written"
    assert _filt_err(y[:, :T], _ref_sosfiltfilt(ctx["sos"], ctx["x"]), ctx["x"]) <= BOUND_FILT[(path, "m")]


@pytest.mark.gpu
@pytest.mark.parametrize("path,order,T,kind", _CONSTANT)
def test_constant_rows_known_answers(path, order, T, kind, probed, cuda_device):
    """A constant row stays that constant through a low-pass; a high-pass of it is ~0."""
    y, _ = _graded(probed, _key_of("constant", (path, order, T, kind)), cuda_device)
    want = -7.5 if kind == "low" else 0.0
    assert np.max(np.abs(y.cpu().numpy() - want)) <= 7.5 * BOUND_FILT[(path, "m")]


# ---------------------------------------------------------------------------
# GPU: the change stage through change_from_logmel
# ---------------------------------------------------------------------------


@pytest.mark.gpu
@pytest.mark.parametrize("case", CHANGE_CASES, ids=[c.id for c in CHANGE_CASES])
def test_change_path_matches_reference(case, probed, cuda_device, record_property):
    r, ctx = _graded(probed, "change:" + case.id, cuda_device)
    ref, scale = _ref_change(r["mfcc"].cpu().numpy(), case.first, ctx["sos"], case.method, ctx["out"])
    err = _curve_err(r["totChange"].cpu().numpy(), ref, scale)
    record_property("curve_err", err)
    record_property("cls", f"{case.path}/{_cls(case.wn)}")
    assert err <= BOUND_CURVE[(case.path, _cls(case.wn))], err


# ---------------------------------------------------------------------------
# GPU: delta_norm_kernel known answers and limits
# ---------------------------------------------------------------------------


def _ref_delta_norm(x, method):
    d = _ref_diff(np.asarray(x, np.float64).astype(LD), method)
    return np.sqrt(np.sum(d * d, axis=1)) / x.shape[1]


@pytest.mark.gpu
@pytest.mark.parametrize("B,R,T,method", _DELTA)
def test_delta_norm_known_answers(B, R, T, method, probed, cuda_device):
    """T = 1 gives 0.  For T = 2 both methods give the first-order difference at both frames: np.gradient does, and
    savgol_filter(3, 2, deriv=1) cannot fit a 3-sample window to 2 frames, so the kernels take np.gradient's
    edges there rather than fail.  More than 65 535 clips run in launches of 65 535."""
    tot, ctx = _graded(probed, _key_of("delta", (B, R, T, method)), cuda_device)
    x = ctx["x"]
    tot = tot.cpu().numpy()
    if T == 1:
        assert np.all(tot == 0.0)
        return
    ref = _ref_delta_norm(x, method)
    if T == 2:
        want = np.sqrt(np.sum((x[:, :, 1] - x[:, :, 0]).astype(LD) ** 2, axis=1)) / R
        assert np.max(np.abs(ref - want[:, None])) < 1e-16 * want.max()
    scale = np.abs(x).reshape(B, -1).max(axis=1)
    assert _curve_err(tot, ref, scale) <= 1e-15


if __name__ == "__main__":
    _probe_all(sys.argv[1])
