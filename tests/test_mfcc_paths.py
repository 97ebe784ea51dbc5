"""Every MFCC-stage (K3: top_db clamp + DCT-II + np.gradient delta) kernel path against a float64 reference.

``mmf_mfcc`` / ``mfcc_launch`` (csrc/c_api.cu, csrc/post_kernels.cu) and ``run_post`` split the shapes
``validate_cfg`` accepts (n_mels <= 512, n_mfcc <= min(128, n_mels)) over five kernels:

  path   kernel                                  taken when
  pk     mfcc_pk_kernel<NP, PITCH, false>        default; n_mfcc <= 32, n_mels % 8 == 0, T < 2^27;
                                                 NP = 4 for n_mfcc <= 8 else ceil(n_mfcc / 2), PITCH = 16 / 32
  fp32   mfcc_kernel<NC, false>                  n_mels % 8 != 0, n_mfcc > 32 or T >= 2^27; NC = 16 / 32 / 64 / 128
  mma    mfcc_mma_kernel<NT>                     MMF_FLAG_MMA_DCT, n_mfcc <= 32; NT = ceil(n_mfcc / 8)
  tc     mfcc_tc_kernel<KS>                      MMF_FLAG_TC_DCT without MMA_DCT, power-of-two n_fft,
                                                 n_mfcc <= 16, n_mels <= 96; KS = ceil(n_mels / 16)
  fused  change_fused_kernel<.., true, false>    change_from_logmel without a delta output (or MMF_FLAG_FOLD_MFCC
                                                 with one), n_mfcc <= 16 (FROM_LM = true)

Each GPU case names the path and instantiation it is meant to reach, and a ``torch.profiler`` probe checks that
exactly that K3 kernel ran.  The inputs are seeded synthetic log-mel in dB uploaded directly (not produced by
K1), so any shape is reachable.

Checks, against ``_ref_mfcc`` on the same float32 input:
  * MFCC: max |d| / ||clamped frame||_2 per frame <= BOUND[path] (the DCT is orthonormal, so the frame's norm
    bounds every coefficient);
  * delta: bit-identical to the float32 np.gradient of the kernel's own MFCC output (this pins the one-frame
    halo exactly, whatever the DCT error), and within 2 * BOUND[path] of the float64 gradient of the reference,
    graded on the largest norm of the three frames involved;
  * clamp: with clamp_in_place = 1 the log-mel written back is bit-identical to the reference clamp; with 0 the
    input is unchanged byte for byte.
Largest values observed on a B200 (1000 W power limit) over the case matrix; every bound is at most about 10x
(the delta's 2x bound follows from the MFCC bound, so its margin is wider):
  mfcc   pk 2.8e-6, fp32 3.1e-6, mma 1.3e-6, tc 2.2e-7, fused 2.7e-6  (pk, fp32 and fused at n_mels 512)
  delta  pk 4.6e-7, fp32 4.0e-7, mma 2.5e-7, tc 9.2e-8, fused 1.4e-7
``test_tolerances_catch_plausible_mistakes`` (CPU) holds these bounds honest: each of six plausible mistakes
misses the reference by more than 10x every path's bound on the case fixtures.
"""

import re
from typing import NamedTuple

import numpy as np
import pytest
import scipy.fft
import scipy.signal

import oracle
import modulation_mfcc_b200 as mm
from modulation_mfcc_b200 import _lib
from modulation_mfcc_b200.synth import synth_batch

# pk, fp32 and fused accumulate the n_mels products of each coefficient in float32, one FMA after the other: the
# error grows with n_mels and peaks at n_mels 512 (the reference's float64 sum of the same inputs differs by that)
BOUND = {"pk": 1e-5, "fp32": 1e-5, "mma": 5e-6, "tc": 1e-6, "fused": 1e-5}

TOP_DB = 80.0
MMA = _lib.MMF_FLAG_MMA_DCT
TC = _lib.MMF_FLAG_TC_DCT
FOLD = _lib.MMF_FLAG_FOLD_MFCC


def _torch():
    import torch

    return torch


# ---------------------------------------------------------------------------
# float64 reference
# ---------------------------------------------------------------------------


def _key(maxima):
    """float32 maxima -> the int32 keys the kernels decode (inverse of key_to_float / float_key): the bits when the
    sign bit is clear, else bits ^ 0x7FFFFFFF, so that signed integer order is float order."""
    bits = np.ascontiguousarray(maxima, np.float32).view(np.int32)
    return np.where(bits >= 0, bits, bits ^ np.int32(0x7FFFFFFF)).astype(np.int32)


def _unkey(keys):
    k = np.asarray(keys, np.int32)
    return np.where(k >= 0, k, k ^ np.int32(0x7FFFFFFF)).astype(np.int32).view(np.float32)


def _ref_mfcc(logmel, clipmax_f32, top_db, n_mfcc, delta, *, mistake=None):
    """(clamped float32 log-mel, float64 MFCC [B, n_mfcc, T], float64 delta or None) of ``logmel [B, n_mels, T]``.

    The clamp is the kernels' float32 arithmetic: thr = float32(max) - float32(top_db), then max(x, thr); no clamp
    when top_db < 0.  The MFCCs are scipy's orthonormal DCT-II in float64 of the clamped float32 values, the delta
    np.gradient along time (edge_order 1; 0 when T = 1).  ``mistake`` (tests of the bounds only) makes one
    plausible implementation error on purpose."""
    x = np.asarray(logmel, np.float32)
    B, n_mels, T = x.shape
    cmax = np.asarray(clipmax_f32, np.float32).reshape(B)
    if mistake == "wrong_clip_threshold":
        cmax = np.roll(cmax, 1)
    if top_db >= 0:
        thr = (cmax - np.float32(top_db)).astype(np.float32)[:, None, None]
        clamped = x if mistake == "clamp_after_dct" else np.maximum(x, thr)
    else:
        clamped = x.copy()
    dct_type = 3 if mistake == "dct_iii" else 2
    mfcc = scipy.fft.dct(clamped.astype(np.float64), type=dct_type, norm="ortho", axis=-2)[:, :n_mfcc]
    if mistake == "clamp_after_dct" and top_db >= 0:
        mfcc = np.maximum(mfcc, thr)
        clamped = np.maximum(x, thr)
    if mistake == "c0_without_sqrt_half":
        mfcc[:, 0] *= np.sqrt(2.0)
    if not delta:
        return clamped, mfcc, None
    if T == 1:
        d = np.zeros_like(mfcc)
    else:
        d = np.gradient(mfcc, axis=-1)
        if mistake == "delta_without_half" and T > 2:
            d[..., 1:-1] *= 2.0
        if mistake == "halo_shifted":
            d[..., :-1] = d[..., 1:].copy()
    return clamped, mfcc, d


def _frame_norm(clamped):
    """||clamped frame||_2 per (clip, frame): [B, T]."""
    return np.sqrt(np.sum(np.asarray(clamped, np.float64) ** 2, axis=-2))


def _mfcc_err(mfcc, ref, norm):
    """max over frames of max |d| / ||clamped frame||; inf for a non-finite output."""
    mfcc = np.asarray(mfcc, np.float64)
    if not np.all(np.isfinite(mfcc)):
        return float("inf")
    d = np.abs(mfcc - ref).max(axis=-2)
    return float(np.max(d / np.maximum(norm, 1e-30), initial=0.0))


def _nbr_norm(norm):
    """largest frame norm among t - 1, t, t + 1: the frames a delta value depends on."""
    n = norm.copy()
    n[..., 1:] = np.maximum(n[..., 1:], norm[..., :-1])
    n[..., :-1] = np.maximum(n[..., :-1], norm[..., 1:])
    return n


def _delta_f32(c):
    """np.gradient along time in float32 arithmetic, as every K3 kernel computes it from its own MFCCs."""
    c = np.asarray(c, np.float32)
    d = np.zeros_like(c)
    T = c.shape[-1]
    if T == 1:
        return d
    d[..., 0] = c[..., 1] - c[..., 0]
    d[..., -1] = c[..., -1] - c[..., -2]
    if T > 2:
        d[..., 1:-1] = (c[..., 2:] - c[..., :-2]) / np.float32(2.0)
    return d


# ---------------------------------------------------------------------------
# inputs: seeded synthetic log-mel in dB
# ---------------------------------------------------------------------------


def _logmel(B, n_mels, T, seed, top_db=TOP_DB):
    """[B, n_mels, T] float32 random walks along time over a per-mel offset (about -100 .. +40 dB) and the clips'
    float32 maxima [B].

    Every clip has a different maximum, the last one a negative maximum; a few cells sit exactly at the
    threshold and one ulp either side of it."""
    rng = np.random.default_rng(seed)
    off = np.linspace(22.0, -58.0, n_mels)[None, :, None] + rng.uniform(-6, 6, (1, n_mels, 1))
    walk = rng.standard_normal((B, n_mels, T)).cumsum(axis=-1) * (2.0 / np.sqrt(max(T, 1) / 64.0))
    x = off + walk + 3.0 * rng.standard_normal((B, n_mels, T))
    x = np.clip(x, -100.0, 40.0)
    for b in range(B):
        x[b] += 12.0 - 7.25 * b - (x[b].max() - 28.0)  # clip maxima 40, 32.75, 25.5, ...
    if B > 1:
        x[B - 1] -= x[B - 1].max() + 3.5  # a clip whose maximum is negative
    x = x.astype(np.float32)
    cmax = x.reshape(B, -1).max(axis=1)
    if top_db >= 0:
        for b in range(B):
            thr = np.float32(cmax[b] - np.float32(top_db))
            cells = rng.integers(0, n_mels * T, size=min(6, n_mels * T))
            for i, v in zip(cells, [thr, np.nextafter(thr, np.float32(np.inf)), np.nextafter(thr, np.float32(-np.inf))] * 2):
                m, t = divmod(int(i), T)
                if x[b, m, t] != cmax[b]:
                    x[b, m, t] = v
        cmax = x.reshape(B, -1).max(axis=1)
    return x, cmax


# ---------------------------------------------------------------------------
# the case matrix: expected path and instantiation read off mfcc_launch, mmf_mfcc and run_post
# ---------------------------------------------------------------------------


class Case(NamedTuple):
    id: str
    n_mels: int
    n_mfcc: int
    T: int
    delta: bool
    path: str
    inst: object  # (NP, PITCH) for pk, NC for fp32, NT for mma, KS for tc, FROM_LM for fused
    flags: int = 0
    call: str = "mfcc"  # "mfcc" (Plan.mfcc) or "change" (Plan.change_from_logmel)
    geo: str = "auto"  # "auto" or "generic" (a non-power-of-two n_fft)
    remove_first: int = 1
    B: int = 3


def _pk(n_mfcc):
    np_ = 4 if n_mfcc <= 8 else (n_mfcc + 1) // 2
    return (np_, 16 if np_ <= 8 else 32)


def _nc(n_mfcc):
    return 16 if n_mfcc <= 16 else 32 if n_mfcc <= 32 else 64 if n_mfcc <= 64 else 128


def P(n_mels, n_mfcc, T, delta, **kw):
    return Case(f"pk_np{_pk(n_mfcc)[0]}_mels{n_mels}_mfcc{n_mfcc}_T{T}" + ("_delta" if delta else ""),
                n_mels, n_mfcc, T, delta, "pk", _pk(n_mfcc), **kw)


def F(n_mels, n_mfcc, T, delta, **kw):
    return Case(f"fp32_nc{_nc(n_mfcc)}_mels{n_mels}_mfcc{n_mfcc}_T{T}" + ("_delta" if delta else ""),
                n_mels, n_mfcc, T, delta, "fp32", _nc(n_mfcc), **kw)


def M(n_mels, n_mfcc, T, delta, **kw):
    return Case(f"mma_nt{(n_mfcc + 7) // 8}_mels{n_mels}_mfcc{n_mfcc}_T{T}" + ("_delta" if delta else ""),
                n_mels, n_mfcc, T, delta, "mma", (n_mfcc + 7) // 8, flags=MMA, **kw)


def K(n_mels, n_mfcc, T, delta, **kw):
    return Case(f"tc_ks{(n_mels + 15) // 16}_mels{n_mels}_mfcc{n_mfcc}_T{T}" + ("_delta" if delta else ""),
                n_mels, n_mfcc, T, delta, "tc", (n_mels + 15) // 16, flags=TC, **kw)


def U(n_mels, n_mfcc, T, delta=False, flags=0, remove_first=1):
    return Case(f"fused_mels{n_mels}_mfcc{n_mfcc}_T{T}" + ("_rf" if remove_first else "") + ("_fold_delta" if delta else ""),
                n_mels, n_mfcc, T, delta, "fused", True, flags=flags | (FOLD if delta else 0), call="change",
                remove_first=remove_first)


CASES = [
    # pk: every NP from 4 to 16; T around the 128-frame block (126 owned with the delta), 1, 2 and ~1000
    P(8, 1, 1, True), P(8, 1, 126, True), P(16, 8, 2, True), P(40, 9, 125, True), P(48, 12, 126, True),
    P(40, 13, 127, True), P(64, 16, 128, False), P(128, 17, 129, True), P(256, 20, 127, False),
    P(512, 21, 129, True), P(96, 24, 1000, True), P(200, 25, 300, False), P(120, 28, 2, False),
    P(72, 29, 1, False), P(32, 31, 129, False), P(512, 32, 1000, True), P(24, 13, 128, False),
    # fp32: n_mels % 8 != 0, n_mfcc > 32; NC 128 at n_mels 272 and 512 stages the DCT rows in two chunks
    F(1, 1, 1, True), F(13, 13, 127, True), F(13, 13, 128, False), F(41, 20, 126, True), F(41, 32, 129, False),
    F(64, 33, 300, True), F(200, 40, 2, False), F(512, 64, 129, True), F(128, 128, 128, True),
    F(271, 100, 1000, True), F(272, 128, 127, True), F(512, 128, 300, True), F(512, 65, 1, False),
    F(300, 80, 129, False),
    # mma: 4 warps of 30 owned frames with the delta (120 per block), 32 without (128); n_mels 13 = a partial k-step
    M(13, 8, 119, True), M(40, 1, 1, True), M(40, 13, 120, True), M(128, 16, 128, False), M(64, 20, 121, True),
    M(13, 13, 2, True), M(512, 32, 127, False), M(512, 25, 1000, True), M(48, 24, 129, False),
    # tc: KS 1 .. 6; n_mels 1, 17 and 81 leave a partial K slab
    K(1, 1, 1, True), K(16, 13, 126, True), K(17, 16, 127, True), K(32, 16, 128, False), K(40, 13, 129, False),
    K(48, 13, 127, False), K(64, 13, 1000, True), K(80, 9, 125, True), K(81, 16, 2, False), K(96, 16, 127, True), K(72, 7, 128, True),
    # fused: 32-frame warp tiles (30 owned with a delta output)
    U(40, 2, 31), U(40, 13, 32, remove_first=0), U(64, 16, 33), U(512, 16, 300), U(40, 13, 31, delta=True),
    # routing: one line each
    Case("route_tc_mels128_lands_on_pk", 128, 13, 129, True, "pk", _pk(13), flags=TC),
    Case("route_mma_with_tc_lands_on_mma", 40, 13, 129, True, "mma", 2, flags=MMA | TC),
    Case("route_mma_mfcc33_lands_on_fp32", 64, 33, 129, True, "fp32", 64, flags=MMA),
    Case("route_tc_generic_nfft_lands_on_pk", 40, 13, 129, True, "pk", _pk(13), flags=TC, geo="generic"),
    # run_post does not exclude TC_DCT from folding: without a delta output the fused kernel takes the DCT
    Case("route_tc_change_without_delta_lands_on_fused", 40, 13, 129, False, "fused", True, flags=TC, call="change"),
]

# instantiations the matrix must reach
WANT = ({("pk", _pk(n)) for n in (1, 9, 11, 13, 15, 17, 19, 21, 23, 25, 27, 29, 31)}
        | {("fp32", nc) for nc in (16, 32, 64, 128)} | {("mma", nt) for nt in (1, 2, 3, 4)}
        | {("tc", ks) for ks in range(1, 7)} | {("fused", True)})

# one geometry per path for the properties that do not need the whole matrix
PATH_GEOMETRY = {
    "pk": P(40, 13, 300, True),
    "fp32": F(41, 20, 300, True),
    "mma": M(40, 13, 300, True),
    "tc": K(40, 13, 300, True),
    "fused": U(40, 13, 300),
}

_KERNELS = {"mfcc_pk_kernel": "pk", "mfcc_kernel": "fp32", "mfcc_mma_kernel": "mma", "mfcc_tc_kernel": "tc",
            "change_fused_kernel": "fused"}


def _targs(text, mangled):
    if mangled:  # Li16E / Lb0E
        return tuple(int(v) if k == "i" else bool(int(v)) for k, v in re.findall(r"L([ib])(\d+)E", text))
    out = []
    for a in text.split(","):
        a = a.strip()
        out.append(True if a == "true" else False if a == "false" else int(re.sub(r"[^\d-]", "", a)))
    return tuple(out)


def _k3_kernels(names):
    """(path, instantiation) of every K3 kernel among profiler kernel names, demangled or mangled.  Names match on
    word boundaries: mfcc_kernel is not mfcc_pk_kernel, mfcc_tc_kernel or mfcc_mma_kernel."""
    out = []
    for name in names:
        for tok, path in _KERNELS.items():
            m = re.search(r"(?<![\w])" + tok + r"<([^>]*)>", name)
            mangled = False
            if m is None:
                m = re.search(r"(?<=\d)" + tok + r"I((?:L[ib]\d+E)+)E", name)
                mangled = True
            if m is None:
                continue
            a = _targs(m.group(1), mangled)
            if path == "pk":
                out.append((path, (a[0], a[1]) if not a[2] else ("VL", a)))
            elif path == "fp32":
                out.append((path, a[0] if not a[1] else ("VL", a)))
            elif path == "fused":
                out.append((path, a[2] if not a[3] else ("VL", a)))
            else:
                out.append((path, a[0]))
    return out


def _probe(fn):
    """Run ``fn`` under torch.profiler with CUDA activity; return (result, K3 kernels that ran, launch count delta)."""
    torch = _torch()
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    n0 = _lib.lib().mmf_launch_count(0)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    launches = _lib.lib().mmf_launch_count(0) - n0
    names = [e.name for e in prof.events()]
    assert names, "the profiler saw no kernels at all: the path probe cannot tell which K3 kernel ran"
    return res, _k3_kernels(names), launches


def _expect_path(ran, path, inst, launches, n_launches=1):
    want = (path, inst)
    assert ran and all(k == want for k in ran), f"expected only {want}, K3 kernels that ran: {ran}"
    assert len(ran) == n_launches and launches == n_launches, (ran, launches)


# plan geometries (sample_rate, n_fft, win_length, hop_length, fmin, fmax): K3 does not depend on them, but the
# plan must create; many mels want a long FFT and a high fmin so that no Slaney filter is empty
_GEOS = [(16000, 512, 400, 160, 0.0, 8000.0), (48000, 4096, 3840, 960, 4000.0, 24000.0),
         (48000, 4096, 4096, 1024, 0.0, 24000.0), (44100, 2048, 2048, 512, 0.0, 22050.0)]
_GENERIC = [(16000, 400, 400, 160, 0.0, 8000.0)]


def _plan(n_mels, n_mfcc, flags, geo="auto", top_db=TOP_DB):
    geos = _GENERIC if geo == "generic" else (_GEOS if n_mels <= 64 else _GEOS[1:] + _GEOS[:1])
    errors = []
    for sr, n_fft, win, hop, fmin, fmax in geos:
        cfg = mm.MfccConfig(sr, n_fft, win, hop, n_mels, n_mfcc, fmin, fmax, top_db=top_db, flags=flags)
        try:
            return mm.get_plan(cfg)
        except mm.MmfError as e:
            errors.append(f"{sr}/{n_fft}: {e}")
    raise AssertionError(f"no plan geometry creates n_mels={n_mels} n_mfcc={n_mfcc}: {errors}")


def _prm(remove_first):
    return mm.make_change_params(scipy.signal.butter(2, 0.2, output="sos"), remove_first=remove_first)


def _run(plan, case, lm, km, clamp):
    """One K3 call of the case's kind on device tensors: (mfcc, delta or None)."""
    if case.call == "change":
        r = plan.change_from_logmel(lm, km, _prm(case.remove_first), want_delta=case.delta, clamp_in_place=clamp)
        return r["mfcc"], r["delta"]
    r = plan.mfcc(lm, km, delta=case.delta, clamp_in_place=clamp)
    return r if case.delta else (r, None)


def _check(mfcc, delta, x, cmax, top_db, n_mfcc, path, record=None, frames=slice(None)):
    """Grade the kernel's outputs on frames ``frames`` of the reference computed from ``x``."""
    clamped, rm, rd = _ref_mfcc(x, cmax, top_db, n_mfcc, delta is not None)
    norm = _frame_norm(clamped)
    em = _mfcc_err(mfcc, rm[..., frames], norm[..., frames])
    if record is not None:
        record("mfcc_err", em)
    assert em <= BOUND[path], f"MFCC error {em:.3g} > {BOUND[path]:.3g}"
    if delta is None:
        return clamped
    want = _delta_f32(mfcc) if frames == slice(None) else None
    if want is not None:
        bad = np.argwhere(delta.view(np.int32) != want.view(np.int32))
        assert bad.size == 0, f"delta is not the float32 gradient of the kernel's own MFCC at {bad[:5].tolist()}"
    ed = _mfcc_err(delta, rd[..., frames], _nbr_norm(norm)[..., frames])
    if record is not None:
        record("delta_err", ed)
    assert ed <= 2 * BOUND[path], f"delta error {ed:.3g} > {2 * BOUND[path]:.3g}"
    return clamped


# ---------------------------------------------------------------------------
# CPU: the reference, the fixtures and the bounds
# ---------------------------------------------------------------------------


def test_key_encoding_round_trips_and_orders():
    v = np.array([-np.inf, -1e30, -80.5, -1.0, -1e-40, -0.0, 0.0, 1e-40, 1.0, 40.25, 3e38, np.inf], np.float32)
    k = _key(v)
    assert np.array_equal(_unkey(k).view(np.int32), v.view(np.int32))
    assert np.all(np.diff(k[[0, 1, 2, 3, 4, 6, 7, 8, 9, 10, 11]].astype(np.int64)) > 0)


@pytest.mark.parametrize("n_mels,n_mfcc,top_db", [(40, 13, 80.0), (128, 20, 80.0), (40, 13, None)])
def test_reference_agrees_with_oracle(n_mels, n_mfcc, top_db, monkeypatch):
    """On the oracle's own log-mel (rounded to float32, the kernels' input type) ``_ref_mfcc`` gives exactly the
    oracle's float32-cast clamp, MFCC (scipy.fftpack's DCT-II) and np.gradient delta."""
    sr = 16000
    y = synth_batch(5, 1, sr, sr)[0]
    seen = {}
    orig = oracle.mfcc_oracle.power_to_db

    def power_to_db_f32(S, amin=1e-10, top_db=80.0):
        L = orig(S, amin=amin, top_db=None).astype(np.float32).astype(np.float64)
        seen["L"] = L
        return np.maximum(L, L.max() - top_db) if top_db is not None else L

    monkeypatch.setattr(oracle.mfcc_oracle, "power_to_db", power_to_db_f32)
    M, inter = oracle.mfcc(y, sr, n_mfcc=n_mfcc, win_length=400, hop_length=160, n_fft=512, n_mels=n_mels,
                           top_db=top_db, return_intermediates=True)
    L = seen["L"].astype(np.float32)[None]
    clamped, rm, rd = _ref_mfcc(L, L.max(axis=(1, 2)), -1.0 if top_db is None else top_db, n_mfcc, True)
    assert np.array_equal(clamped[0], inter["logmel"].astype(np.float32))
    assert np.array_equal(rm[0].astype(np.float32), M.astype(np.float32))
    assert np.array_equal(rd[0].astype(np.float32), np.gradient(M, axis=1).astype(np.float32))
    # the reference's DCT is independent of the plan's float32 table and agrees with the oracle's matrix form
    D = oracle.dct_ortho_matrix(n_mfcc, n_mels)
    assert np.array_equal(rm[0].astype(np.float32), (D @ clamped[0].astype(np.float64)).astype(np.float32))


def test_reference_known_answers():
    """A constant frame has only c0 = c * sqrt(n_mels); a frame equal to DCT row k0 has only coefficient k0 = 1;
    T = 1 gives a zero delta and T = 2 the one-sided difference at both ends."""
    n_mels, k0 = 40, 5
    D = oracle.dct_ortho_matrix(16, n_mels)
    x = np.stack([np.full(n_mels, -17.25), D[k0]], axis=1)[None].astype(np.float32)
    _, m, d = _ref_mfcc(x, x.max(axis=(1, 2)), -1.0, 16, True)
    assert abs(m[0, 0, 0] - (-17.25) * np.sqrt(n_mels)) < 1e-12 and np.all(np.abs(m[0, 1:, 0]) < 1e-12)
    e = np.zeros(16)
    e[k0] = 1.0
    assert np.all(np.abs(m[0, :, 1] - e) < 1e-6)
    assert np.array_equal(d[0, :, 0], m[0, :, 1] - m[0, :, 0]) and np.array_equal(d[0, :, 1], d[0, :, 0])
    _, _, d1 = _ref_mfcc(x[..., :1], x.max(axis=(1, 2)), -1.0, 16, True)
    assert np.all(d1 == 0.0)


def test_fixtures_reach_the_clamp_edges():
    """Every clip of a fixture has its own maximum, the last one negative; 10 .. 30 % of the cells sit below the
    threshold, and some sit exactly at it and one ulp either side."""
    for n_mels, T in [(40, 300), (512, 129), (8, 1000), (13, 2)]:
        x, cmax = _logmel(3, n_mels, T, 7)
        assert len(set(cmax.tolist())) == 3 and cmax[2] < 0
        assert np.array_equal(cmax, x.reshape(3, -1).max(axis=1))
        thr = (cmax - np.float32(TOP_DB)).astype(np.float32)[:, None, None]
        below = float(np.mean(x < thr))
        if n_mels * T >= 300:
            assert 0.10 <= below <= 0.30, below
        for b in range(3):
            t = thr[b, 0, 0]
            for v in (t, np.nextafter(t, np.float32(np.inf)), np.nextafter(t, np.float32(-np.inf))):
                assert np.any(x[b] == v)


def test_case_matrix_reaches_every_instantiation():
    """The case table names every K3 kernel and instantiation: pk NP 4 .. 16, fp32 NC 16 / 32 / 64 / 128, mma
    NT 1 .. 4, tc KS 1 .. 6 and the fused kernel from log-mel; the T edges of each kernel's block; the routing
    lines.  Each GPU case then proves with the probe that it ran there."""
    got = {(c.path, c.inst) for c in CASES}
    assert WANT <= got, WANT - got
    assert {np_ for p, (np_, _) in ((c.path, c.inst) for c in CASES if c.path == "pk")} == set(range(4, 17))
    for c in CASES:
        assert 1 <= c.n_mfcc <= min(128, c.n_mels) and c.n_mels <= 512  # validate_cfg accepts every case
        mma = c.flags & MMA and c.n_mfcc <= 32
        tc = c.flags & TC and not c.flags & MMA and c.geo != "generic" and c.n_mfcc <= 16 and c.n_mels <= 96
        fused = c.call == "change" and c.n_mfcc <= 16 and not c.flags & MMA and (not c.delta or c.flags & FOLD)
        pk = c.n_mfcc <= 32 and c.n_mels % 8 == 0
        want = "fused" if fused else "mma" if mma else "tc" if tc else "pk" if pk else "fp32"
        assert c.path == want, (c.id, want)
        inst = {"pk": _pk(c.n_mfcc), "fp32": _nc(c.n_mfcc), "mma": (c.n_mfcc + 7) // 8, "tc": (c.n_mels + 15) // 16,
                "fused": True}[want]
        assert c.inst == inst, c.id
    Ts = {c.path: set() for c in CASES}
    for c in CASES:
        Ts[c.path].add((c.T, c.delta))
    for path, edges in [("pk", [(125, 1), (126, 1), (127, 1), (127, 0), (128, 0), (129, 0), (129, 1)]),
                        ("fp32", [(126, 1), (127, 1), (128, 0), (129, 0), (127, 1), (128, 1)]),
                        ("mma", [(119, 1), (120, 1), (121, 1), (127, 0), (128, 0), (129, 0)]),
                        ("tc", [(125, 1), (126, 1), (127, 1), (127, 0), (128, 0), (129, 0)]),
                        ("fused", [(31, 0), (32, 0), (33, 0), (31, 1)])]:
        assert {(t, bool(d)) for t, d in edges} <= Ts[path], path
    for path in ("pk", "fp32", "mma", "tc"):
        assert {1, 2} <= {t for t, _ in Ts[path]} and max(t for t, _ in Ts[path]) >= 1000
    assert any(c.n_mels >= 272 and c.n_mfcc > 64 for c in CASES)  # the chunked DCT table


_MISTAKES = ["c0_without_sqrt_half", "dct_iii", "wrong_clip_threshold", "clamp_after_dct", "delta_without_half",
             "halo_shifted"]


@pytest.mark.parametrize("mistake", _MISTAKES)
def test_tolerances_catch_plausible_mistakes(mistake):
    """Each plausible implementation mistake misses the reference by more than 10x the bound of every path, on
    the fixtures of the GPU cases (float32 output, as the kernels write it)."""
    delta_mistake = mistake in ("delta_without_half", "halo_shifted")
    worst = {}
    for i, c in enumerate(CASES):
        if delta_mistake and c.T < 3:
            continue  # no central difference, no halo to shift
        if mistake in ("dct_iii", "clamp_after_dct") and c.n_mels == 1:
            continue  # a one-point DCT is the identity: neither mistake changes anything
        x, cmax = _logmel(c.B, c.n_mels, min(max(c.T, 64), 300), 1000 + i)
        clamped, rm, rd = _ref_mfcc(x, cmax, TOP_DB, c.n_mfcc, True)
        wc, wm, wd = _ref_mfcc(x, cmax, TOP_DB, c.n_mfcc, True, mistake=mistake)
        if mistake == "wrong_clip_threshold" and np.array_equal(wc, clamped):
            continue  # the fixture has no cell between the two clips' thresholds
        if mistake == "clamp_after_dct" and np.array_equal(x, clamped):
            continue  # nor any cell below the threshold
        norm = _frame_norm(clamped)
        if delta_mistake:
            miss = _mfcc_err(wd.astype(np.float32), rd, _nbr_norm(norm)) / (2 * max(BOUND.values()))
        else:
            miss = _mfcc_err(wm.astype(np.float32), rm, norm) / max(BOUND.values())
        worst[c.id] = miss
    assert worst and min(worst.values()) > 10.0, min(worst.items(), key=lambda kv: kv[1])


# ---------------------------------------------------------------------------
# GPU: the case matrix
# ---------------------------------------------------------------------------


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c.id for c in CASES])
def test_mfcc_path_matches_reference(case, cuda_device, record_property):
    torch = _torch()
    plan = _plan(case.n_mels, case.n_mfcc, case.flags, case.geo)
    x, cmax = _logmel(case.B, case.n_mels, case.T, 100 + case.n_mels * 7 + case.n_mfcc)
    lm = torch.as_tensor(x).to(cuda_device)
    km = torch.as_tensor(_key(cmax)).to(cuda_device)
    # clamp_in_place = 0: the input stays byte for byte as it was
    (mfcc, delta), ran, launches = _probe(lambda: _run(plan, case, lm, km, False))
    _expect_path(ran, case.path, case.inst, launches)
    assert torch.equal(lm.cpu().view(torch.int32), torch.as_tensor(x).view(torch.int32)), "clamp_in_place=0 wrote"
    mfcc = mfcc.cpu().numpy()
    delta = delta.cpu().numpy() if delta is not None else None
    clamped = _check(mfcc, delta, x, cmax, TOP_DB, case.n_mfcc, case.path, record_property)
    # clamp_in_place = 1: the same outputs, and the log-mel written back is the reference clamp bit for bit
    (m1, d1), ran, launches = _probe(lambda: _run(plan, case, lm, km, True))
    _expect_path(ran, case.path, case.inst, launches)
    assert np.array_equal(m1.cpu().numpy().view(np.int32), mfcc.view(np.int32))
    if delta is not None:
        assert np.array_equal(d1.cpu().numpy().view(np.int32), delta.view(np.int32))
    assert np.array_equal(lm.cpu().numpy().view(np.int32), clamped.view(np.int32)), "written-back clamp differs"


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["pk", "tc"])
def test_clip_chunks_of_65535(path, cuda_device):
    """65 537 clips: mmf_mfcc launches clips [0, 65535) and [65535, 65537) separately; clips on both sides of the
    boundary match the reference with their own thresholds."""
    torch = _torch()
    n_mels, n_mfcc, flags = (8, 4, 0) if path == "pk" else (16, 13, TC)
    B, T = 65537, 5
    inst = _pk(n_mfcc) if path == "pk" else 1
    plan = _plan(n_mels, n_mfcc, flags)
    rng = np.random.default_rng(3)
    x = (rng.standard_normal((B, n_mels, T)) * 30.0 - 20.0).astype(np.float32)
    cmax = x.reshape(B, -1).max(axis=1) + rng.uniform(0.0, 60.0, B).astype(np.float32)  # thresholds differ per clip
    lm = torch.as_tensor(x).to(cuda_device)
    km = torch.as_tensor(_key(cmax)).to(cuda_device)
    (mfcc, delta), ran, launches = _probe(lambda: plan.mfcc(lm, km, delta=True, clamp_in_place=True))
    _expect_path(ran, path, inst, launches, n_launches=2)
    clamped = _check(mfcc.cpu().numpy(), delta.cpu().numpy(), x, cmax, TOP_DB, n_mfcc, path)
    assert np.array_equal(lm.cpu().numpy().view(np.int32), clamped.view(np.int32))


@pytest.mark.gpu
@pytest.mark.parametrize("path,T", [("pk", (1 << 27) - 1), ("fp32", 1 << 27)], ids=["pk_T2e27m1", "fp32_T2e27"])
def test_long_clip_row_arithmetic(path, T, cuda_device):
    """One clip of 2^27 - 1 frames (the last the pk kernel takes, with its 32-bit row arithmetic) and of 2^27
    (the first the fp32 kernel takes), n_mels 8, n_mfcc 1, with the delta; checked on sampled frame ranges."""
    torch = _torch()
    n_mels = 8
    plan = _plan(n_mels, 1, 0)
    t = torch.arange(T, device=cuda_device, dtype=torch.float32).mul_(0.00137)
    off = torch.linspace(30.0, -90.0, n_mels, device=cuda_device)
    lm = torch.sin(t)[None, None, :] * 25.0 + off[None, :, None]
    del t
    cmax = np.array([lm.max().item()], np.float32)
    km = torch.as_tensor(_key(cmax)).to(cuda_device)
    (mfcc, delta), ran, launches = _probe(lambda: plan.mfcc(lm, km, delta=True, clamp_in_place=False))
    _expect_path(ran, path, _pk(1) if path == "pk" else 16, launches)
    for a, b in [(0, 300), (126 * 1000 - 5, 126 * 1000 + 260), (1 << 26, (1 << 26) + 300),
                 ((1 << 27) - 2000, (1 << 27) - 1700), (T - 300, T)]:
        lo, hi = max(a - 1, 0), min(b + 1, T)
        x = lm[:, :, lo:hi].cpu().numpy()
        sel = slice(a - lo, a - lo + (b - a))
        clamped, rm, rd = _ref_mfcc(x, cmax, TOP_DB, 1, True)  # one-sided only where the clip ends
        norm = _frame_norm(clamped)
        m = mfcc[:, :, a:b].cpu().numpy()
        d = delta[:, :, a:b].cpu().numpy()
        assert _mfcc_err(m, rm[..., sel], norm[..., sel]) <= BOUND[path], (a, b)
        assert _mfcc_err(d, rd[..., sel], _nbr_norm(norm)[..., sel]) <= 2 * BOUND[path], (a, b)
        # the delta from the kernel's own MFCCs in float32 (the frames either side of the range included)
        want = _delta_f32(mfcc[:, :, lo:hi].cpu().numpy())
        assert np.array_equal(d.view(np.int32), want[..., sel].view(np.int32)), (a, b)
    del lm, mfcc, delta
    torch.cuda.empty_cache()


# ---------------------------------------------------------------------------
# GPU: known answers, top_db 0 and top_db disabled
# ---------------------------------------------------------------------------


@pytest.mark.gpu
@pytest.mark.parametrize("path", list(PATH_GEOMETRY))
def test_known_answers_with_top_db_disabled(path, cuda_device):
    """No clamp (top_db < 0): a constant frame gives c0 = c * sqrt(n_mels) and ~0 elsewhere, a frame equal to DCT
    row k0 gives ~1 at k0 and ~0 elsewhere, the rest matches the unclamped reference, and clamp_in_place leaves
    the log-mel as it was."""
    torch = _torch()
    case = PATH_GEOMETRY[path]
    plan = _plan(case.n_mels, case.n_mfcc, case.flags, top_db=None)
    x, cmax = _logmel(case.B, case.n_mels, case.T, 11, top_db=-1.0)
    x[:, :, :4] -= 300.0  # far below any threshold: only an unclamped kernel keeps them
    k0 = case.n_mfcc - 1
    D = oracle.dct_ortho_matrix(case.n_mfcc, case.n_mels).astype(np.float32)
    x[0, :, 10] = -17.25
    x[0, :, 20] = 30.0 * D[k0]
    cmax = x.reshape(case.B, -1).max(axis=1)
    lm = torch.as_tensor(x).to(cuda_device)
    km = torch.as_tensor(_key(cmax)).to(cuda_device)
    (mfcc, delta), ran, launches = _probe(lambda: _run(plan, case, lm, km, True))
    _expect_path(ran, case.path, case.inst, launches)
    mfcc = mfcc.cpu().numpy()
    _check(mfcc, delta.cpu().numpy() if delta is not None else None, x, cmax, -1.0, case.n_mfcc, case.path)
    assert np.array_equal(lm.cpu().numpy().view(np.int32), x.view(np.int32))
    tol = BOUND[case.path]
    c = mfcc[0, :, 10].astype(np.float64)
    assert abs(c[0] + 17.25 * np.sqrt(case.n_mels)) <= tol * 17.25 * np.sqrt(case.n_mels)
    assert np.all(np.abs(c[1:]) <= tol * 17.25 * np.sqrt(case.n_mels))
    c = mfcc[0, :, 20].astype(np.float64)
    e = np.zeros(case.n_mfcc)
    e[k0] = 30.0
    assert np.all(np.abs(c - e) <= 30.0 * (tol + 1e-6))  # the float32 row itself is ~6e-8 relative


@pytest.mark.gpu
@pytest.mark.parametrize("path", list(PATH_GEOMETRY))
def test_known_answers_with_top_db_zero(path, cuda_device):
    """top_db = 0 clamps every cell to its clip's maximum: the written-back log-mel is exactly that maximum, and
    every frame has only c0 = max * sqrt(n_mels)."""
    torch = _torch()
    case = PATH_GEOMETRY[path]
    plan = _plan(case.n_mels, case.n_mfcc, case.flags, top_db=0.0)
    x, cmax = _logmel(case.B, case.n_mels, case.T, 12, top_db=0.0)
    lm = torch.as_tensor(x).to(cuda_device)
    km = torch.as_tensor(_key(cmax)).to(cuda_device)
    (mfcc, delta), ran, launches = _probe(lambda: _run(plan, case, lm, km, True))
    _expect_path(ran, case.path, case.inst, launches)
    assert np.array_equal(lm.cpu().numpy(), np.broadcast_to(cmax[:, None, None], x.shape))
    mfcc = mfcc.cpu().numpy().astype(np.float64)
    scale = np.abs(cmax.astype(np.float64))[:, None] * np.sqrt(case.n_mels)
    tol = BOUND[case.path] * scale
    assert np.all(np.abs(mfcc[:, 0] - cmax[:, None].astype(np.float64) * np.sqrt(case.n_mels)) <= tol)
    assert np.all(np.abs(mfcc[:, 1:]) <= tol[:, None])
    if delta is not None:
        assert np.all(np.abs(delta.cpu().numpy()) <= 2 * tol[:, None])
