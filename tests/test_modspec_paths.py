"""Every modulation-spectrum (K6, ``mmf_modspec``) kernel path against a float64 reference in geometry units.

``run_modspec`` (csrc/c_api.cu) splits the range the C ABI accepts over four kernels:

  path     kernel                          taken when
  tc       modspec_tc_kernel<128, KS>      nfft == 128, 2 <= win <= 128 and fits() holds; KS = ceil(win / 16)
  clip     modspec_clip_kernel<NFFT, V>    nfft 32 .. 1024 and the chunk's rows fit 110 KB
  fast     modspec_fast_kernel<NFFT>       nfft 32 .. 1024 when the clip kernel declines (n_coef * win * 4 too large)
  generic  modspec_kernel                  nfft 2048 and 4096 (fp64 radix-2)

Each GPU case names the path and the instantiation it is meant to reach, and a ``torch.profiler`` probe checks
that exactly that K6 kernel ran, so that a change to ``fits()`` or ``need()`` cannot quietly move the cases
onto one kernel.

Bounds, against ``_ref_modspec`` on the same float32 input:
  * magnitudes: max |d| per row (one (clip, coefficient, window) spectrum) <= RTOL_MAG[path] * max of the
    reference row; a row whose reference is all zero must be exactly zero;
  * band energies: |d| <= RTOL_BAND[path] * (E + BAND_FLOOR * E_win), E_win = the window's energy over all
    coefficients and bins.  Kernel errors scale with the spectrum's peak, not with the band, so a band that holds
    almost nothing is graded on the window's scale; bands with real energy are graded relative to themselves.
Largest values observed on a B200 (1000 W power limit) over the case matrix; every bound is at most about 10x:
  mag   tc 3.1e-6, clip 3.5e-6, fast 1.4e-6, generic 5.1e-8
  band  tc 1.2e-6, clip 8.9e-7, fast 4.0e-7, generic 4.6e-8
``test_tolerances_catch_plausible_mistakes`` (CPU) holds these bounds honest: each of five plausible mistakes
misses the reference by more than 10x its bound on the same fixtures.
"""

import re
from typing import NamedTuple

import numpy as np
import pytest

import oracle
import modulation_mfcc_b200 as mm
from modulation_mfcc_b200 import _lib
from modulation_mfcc_b200.synth import synth_batch

RTOL_MAG = {"tc": 2e-5, "clip": 2e-5, "fast": 1.4e-5, "generic": 5e-7}
RTOL_BAND = {"tc": 2e-6, "clip": 2e-6, "fast": 2e-6, "generic": 5e-7}
BAND_FLOOR = 1e-3
ABS_TOL = 1e-3  # north_star: modulation magnitudes of MFCC-scale trajectories, 1e-3 absolute

FR = 100.0  # frames per second of the trajectories (tStep 10 ms)


def _torch():
    import torch

    return torch


# ---------------------------------------------------------------------------
# float64 reference in geometry units (win, hop, nfft, [lo, hi) bins)
# ---------------------------------------------------------------------------


def _ref_modspec(M, win, hop, nfft, bins, *, mistake=None):
    """|rfft(n=nfft)| of mean-removed, periodic-Hann windows of ``M [..., C, T]`` in float64.

    Returns (mag [..., C, n_win, nfft/2+1], band [..., n_win, n_bands], e_win [..., n_win]) where
    band[b] = sum over coefficients and bins [lo, hi) of |X|^2 and e_win the same over all bins.
    ``mistake`` (tests of the bounds only) makes one plausible implementation error on purpose."""
    M = np.asarray(M, dtype=np.float32).astype(np.float64)
    T = M.shape[-1]
    n_win = 1 + (T - win) // hop
    start = 1 if mistake == "late_window" else 0
    idx = start + (np.arange(n_win) * hop)[:, None] + np.arange(win)[None, :]
    seg = M[..., np.minimum(idx, T - 1)]  # [..., C, n_win, win]
    if mistake != "no_mean":
        seg = seg - seg.mean(axis=-1, keepdims=True)
    n = np.arange(win)
    period = win - 1 if (mistake == "symmetric_hann" and win > 1) else win
    w = 0.5 - 0.5 * np.cos(2.0 * np.pi * n / period)
    mag = np.abs(np.fft.rfft(seg * w, n=nfft, axis=-1))
    p = mag**2
    if mistake == "shifted_bin":
        mag = np.roll(mag, 1, axis=-1)
    hi_extra = 1 if mistake == "band_hi_included" else 0
    band = np.stack([p[..., lo : hi + hi_extra if hi > lo else hi].sum(axis=(-3, -1)) for lo, hi in bins], axis=-1) \
        if len(bins) else np.zeros(p.shape[:-3] + (n_win, 0))
    return mag, band, p.sum(axis=(-3, -1))


def _mag_err(mag, ref):
    """max over rows of max |d| / max |ref row|; inf when a row whose reference is all zero is not exactly zero."""
    mag = np.asarray(mag, np.float64)
    d = np.abs(mag - ref).max(axis=-1)
    scale = ref.max(axis=-1)
    if np.any(d[scale == 0] != 0):
        return float("inf")
    return float(np.max(np.where(scale > 0, d / np.where(scale > 0, scale, 1.0), 0.0), initial=0.0))


def _band_err(band, ref, e_win):
    """max |d| / (ref + BAND_FLOOR * E_win) over windows and bands; an all-zero reference window must be exactly zero."""
    band = np.asarray(band, np.float64)
    d = np.abs(band - ref)
    scale = ref + BAND_FLOOR * e_win[..., None]
    if np.any(d[scale == 0] != 0):
        return float("inf")
    return float(np.max(np.where(scale > 0, d / np.where(scale > 0, scale, 1.0), 0.0), initial=0.0))


def _edge_bands(nfft):
    """16 bands: DC alone, Nyquist alone, an empty one, the full range, overlapping ones and small ones."""
    H = nfft // 2
    return [(0, 1), (H, H + 1), (5, 5), (0, H + 1), (2, 9), (6, 12), (1, 2), (1, 3),
            (3, 7), (H - 1, H + 1), (H - 3, H), (4, H // 2), (H // 2, H), (7, 8), (0, 2), (10, 11)]


def _bands(kind, nfft):
    if kind == "default":
        return mm.band_bins(nfft, FR)
    if kind == "edge":
        return _edge_bands(nfft)
    return []


def _walk(B, n_coef, T, seed):
    """Seeded random-walk trajectories with row 0 offset to about -500, where c0 sits."""
    rng = np.random.default_rng(seed)
    M = rng.standard_normal((B, n_coef, T)).cumsum(axis=-1) * 0.5
    M[:, 0] -= 500.0
    return M.astype(np.float32)


# ---------------------------------------------------------------------------
# the case matrix: expected path and instantiation read off the dispatch predicates
# ---------------------------------------------------------------------------


class Case(NamedTuple):
    id: str
    n_coef: int
    T: int
    win: int
    hop: int
    nfft: int
    bands: str  # "default" (mm.band_bins), "edge" (_edge_bands) or "none"
    path: str
    inst: int  # KS for tc, NFFT for clip / fast, nfft for generic
    B: int = 2


CASES = [
    # tc: KS = ceil(win / 16) from 1 to 8; items n_win * n_coef either side of the 128-row MMA block
    Case("tc_ks1_win2_hop1_items127", 1, 128, 2, 1, 128, "default", "tc", 1),
    Case("tc_ks1_win16_items128", 1, 143, 16, 1, 128, "edge", "tc", 1),
    Case("tc_ks2_win17_hop_eq_win_tail_items129", 1, 17 * 129 + 10, 17, 17, 128, "default", "tc", 2),
    Case("tc_ks3_win40_gaps_chunked_items257", 1, 40 + 256 * 45, 40, 45, 128, "default", "tc", 3),
    Case("tc_ks4_win64_coef7", 7, 244, 64, 10, 128, "default", "tc", 4),
    Case("tc_ks5_win77_coef13", 13, 1001, 77, 13, 128, "default", "tc", 5),
    Case("tc_ks6_win90_coef13_bands16", 13, 360, 90, 30, 128, "edge", "tc", 6),
    Case("tc_ks7_win100_coef40_bands16", 40, 115, 100, 5, 128, "edge", "tc", 7),
    Case("tc_ks7_win100_hop1_chunked", 13, 1001, 100, 1, 128, "default", "tc", 7),
    Case("tc_ks8_win128_single_window", 13, 128, 128, 1, 128, "default", "tc", 8),
    Case("tc_ks8_win128_hop1_chunked", 13, 1001, 128, 1, 128, "edge", "tc", 8),
    # clip: every NFFT, win == nfft and win << nfft, win = 1, odd n_coef, several chunks per clip
    Case("clip_32_win_eq_nfft", 13, 400, 32, 8, 32, "default", "clip", 32),
    Case("clip_32_win1_zero", 3, 50, 1, 1, 32, "edge", "clip", 32),
    Case("clip_64_coef7_bands16", 7, 300, 50, 25, 64, "edge", "clip", 64),
    Case("clip_256_win_eq_nfft", 13, 1001, 256, 50, 256, "default", "clip", 256),
    Case("clip_256_coef41_hop1_chunks", 41, 1001, 200, 1, 256, "default", "clip", 256),
    Case("clip_512_coef5", 5, 1001, 300, 100, 512, "edge", "clip", 512),
    Case("clip_1024_win_eq_nfft", 3, 1500, 1024, 100, 1024, "default", "clip", 1024),
    Case("clip_1024_win100", 13, 1001, 100, 50, 1024, "edge", "clip", 1024),
    # fast: the clip kernel declines once n_coef * win * 4 bytes pass its budget
    Case("fast_1024_coef40_win1000", 40, 1200, 1000, 50, 1024, "default", "fast", 1024),
    Case("fast_256_coef128_win250_bands16", 128, 400, 250, 50, 256, "edge", "fast", 256),
    # generic: nfft 2048 and 4096
    Case("generic_2048_win1500", 3, 2500, 1500, 250, 2048, "default", "generic", 2048),
    Case("generic_2048_win2048_bands16", 2, 2048, 2048, 1, 2048, "edge", "generic", 2048),
    Case("generic_4096_win3000", 2, 4000, 3000, 500, 4096, "default", "generic", 4096),
    Case("generic_4096_win4096_bands16", 2, 4096 + 700, 4096, 350, 4096, "edge", "generic", 4096),
]
TC_CASES = [c for c in CASES if c.path == "tc"]

# one geometry per path for the properties that do not need the whole matrix
PATH_GEOMETRY = {
    # name: (n_coef, T, win, hop, nfft, path, inst)
    "tc": (13, 300, 100, 50, 128, "tc", 7),
    "clip": (13, 300, 50, 10, 64, "clip", 64),
    "fast": (40, 1200, 1000, 50, 1024, "fast", 1024),
    "generic2048": (3, 2500, 1500, 250, 2048, "generic", 2048),
    "generic4096": (2, 4000, 3000, 500, 4096, "generic", 4096),
}

_TOKENS = {"modspec_tc_kernel": "tc", "modspec_clip_kernel": "clip", "modspec_fast_kernel": "fast",
           "modspec_kernel": "generic"}


def _k6_kernels(names):
    """(path, instantiation) of every K6 kernel among profiler kernel names (demangled or mangled)."""
    out = []
    for name in names:
        for tok, path in _TOKENS.items():
            if tok not in name:
                continue
            args = re.search(tok + r"<\s*(\d+)\s*(?:,\s*(\w+))?", name) or re.search(tok + r"ILi(\d+)E(?:Li(\d+)E)?", name)
            if path == "tc":
                inst = int(args.group(2)) if args else None
            elif path in ("clip", "fast"):
                inst = int(args.group(1)) if args else None
            else:
                inst = None
            out.append((path, inst))
    return out


def _plan(flags=0):
    cfg = mm.MfccConfig(16000, 512, 400, 160, 40, 13, 0.0, 8000.0, flags=flags)
    return mm.get_plan(cfg)


def _probe(fn):
    """Run ``fn`` under torch.profiler with CUDA activity; return (result, K6 kernels that ran, launch count delta)."""
    torch = _torch()
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    n0 = _lib.lib().mmf_launch_count(0)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    launches = _lib.lib().mmf_launch_count(0) - n0
    names = [e.name for e in prof.events()]
    assert names, "the profiler saw no kernels at all: the path probe cannot tell which K6 kernel ran"
    return res, _k6_kernels(names), launches


def _expect_path(ran, path, inst, launches, n_launches=1):
    want = (path, inst if path != "generic" else None)
    assert ran and all(k == want for k in ran), f"expected only {want}, K6 kernels that ran: {ran}"
    assert len(ran) == n_launches and launches == n_launches, (ran, launches)


def _check(mag, band, M, win, hop, nfft, bins, path, record=None):
    rmag, rband, e_win = _ref_modspec(M, win, hop, nfft, bins)
    assert mag.shape == rmag.shape
    em = _mag_err(mag, rmag)
    eb = _band_err(band, rband, e_win) if bins else 0.0
    if record is not None:
        record("mag_err", em)
        record("band_err", eb)
    assert em <= RTOL_MAG[path], f"magnitude error {em:.3g} > {RTOL_MAG[path]:.3g}"
    assert eb <= RTOL_BAND[path], f"band energy error {eb:.3g} > {RTOL_BAND[path]:.3g}"


# ---------------------------------------------------------------------------
# CPU: the reference and the bounds
# ---------------------------------------------------------------------------


@pytest.mark.parametrize("win_s,hop_s,T", [(1.0, 0.5, 1001), (1.0, 0.01, 400), (0.77, 0.13, 1001), (2.0, 0.5, 700)])
def test_reference_agrees_with_oracle(win_s, hop_s, T):
    """On geometries both can express, ``_ref_modspec`` rounds to exactly the oracle's float32 output: the oracle
    computes in float64 and casts, so this is the float64 agreement the cast leaves visible (a relative difference
    above 2^-24 would change a rounded value somewhere in these arrays)."""
    M = _walk(1, 13, T, 5)[0]
    Lw, Hw, nfft, n_win = oracle.modspec_sizes(T, FR, win_s, hop_s)
    bins = mm.band_bins(nfft, FR)
    om, ob, _ = oracle.modulation_spectrum(M, FR, mod_win_s=win_s, mod_hop_s=hop_s)
    rm, rb, _ = _ref_modspec(M, Lw, Hw, nfft, bins)
    assert rm.shape == om.shape and rb.shape == ob.shape
    assert np.array_equal(rm.astype(np.float32), om)
    assert np.array_equal(rb.astype(np.float32), ob)


def test_case_matrix_reaches_every_kernel_instantiation():
    """The case table names every K6 kernel and instantiation: TC for KS 1..8, clip for nfft 32..1024, fast, and
    the generic kernel at 2048 and 4096 (each GPU case then proves with the probe that it ran there)."""
    got = {(c.path, c.inst) for c in CASES}
    want = {("tc", k) for k in range(1, 9)} | {("clip", n) for n in (32, 64, 256, 512, 1024)}
    want |= {("generic", 2048), ("generic", 4096)}
    assert want <= got
    assert any(c.path == "fast" for c in CASES)
    for c in CASES:
        if c.path == "tc":
            assert c.inst == -(-c.win // 16) and c.nfft == 128 and 2 <= c.win <= 128
    # the TC cases rerun with MMF_FLAG_NO_TC_MODSPEC cover clip at nfft 128
    assert all(c.nfft == 128 for c in TC_CASES)


_MISTAKES = ["late_window", "symmetric_hann", "no_mean", "band_hi_included", "shifted_bin"]


@pytest.mark.parametrize("mistake", _MISTAKES)
def test_tolerances_catch_plausible_mistakes(mistake):
    """Each plausible implementation mistake misses the reference by more than 10x the bound of every path, on
    the fixtures of the GPU cases (float32 output, as the kernels write it)."""
    worst = {}
    for c in CASES:
        if c.win == 1 or (mistake == "shifted_bin" and c.win == 2):
            continue  # all zero, and Hann(2) = [0, 1]: flat spectra that no bin shift changes
        if mistake == "band_hi_included" and c.bands == "none":
            continue
        T = min(c.T, c.win + 4 * c.hop)
        M = _walk(1, min(c.n_coef, 16), T, 1)
        bins = _bands(c.bands, c.nfft)
        rm, rb, e_win = _ref_modspec(M, c.win, c.hop, c.nfft, bins)
        wm, wb, _ = _ref_modspec(M, c.win, c.hop, c.nfft, bins, mistake=mistake)
        if mistake == "band_hi_included":
            # only bands that stop short of nfft/2 + 1 can take one more bin
            keep = [i for i, (lo, hi) in enumerate(bins) if lo < hi <= c.nfft // 2 and rb[..., i].max() > 0]
            miss = _band_err(wb[..., keep].astype(np.float32), rb[..., keep], e_win)
            bound = RTOL_BAND[c.path]
        else:
            miss = _mag_err(wm.astype(np.float32), rm)
            bound = RTOL_MAG[c.path]
        worst[c.id] = miss / bound
    assert worst and min(worst.values()) > 10.0, min(worst.items(), key=lambda kv: kv[1])


def test_reference_known_answers():
    """The reference itself: a constant row gives exactly zero, and a cosine on bin k0 with win == nfft gives
    A*win/4 at k0 and A*win/8 at k0 +- 1."""
    nfft, k0, A = 256, 9, 1.5
    n = np.arange(nfft)
    M = np.stack([np.full(nfft, -500.25), A * np.cos(2 * np.pi * k0 * n / nfft)]).astype(np.float32)
    mag, _, _ = _ref_modspec(M, nfft, 1, nfft, [])
    assert np.all(mag[0] == 0.0)
    assert abs(mag[1, 0, k0] - A * nfft / 4) < 1e-5
    assert abs(mag[1, 0, k0 - 1] - A * nfft / 8) < 1e-5 and abs(mag[1, 0, k0 + 1] - A * nfft / 8) < 1e-5


# ---------------------------------------------------------------------------
# GPU: the case matrix
# ---------------------------------------------------------------------------


# with MMF_FLAG_NO_TC_MODSPEC the TC cases land on the clip kernel at nfft 128
_RUNS = [(c, 0) for c in CASES] + [(c, _lib.MMF_FLAG_NO_TC_MODSPEC) for c in TC_CASES]


@pytest.mark.gpu
@pytest.mark.parametrize("case,flags", _RUNS, ids=[c.id + ("_no_tc" if f else "") for c, f in _RUNS])
def test_modspec_path_matches_reference(case, flags, cuda_device, record_property):
    torch = _torch()
    path, inst = (case.path, case.inst) if not flags else ("clip", 128)
    M = _walk(case.B, case.n_coef, case.T, 100 + case.win)
    bins = _bands(case.bands, case.nfft)
    plan = _plan(flags)
    x = torch.as_tensor(M).to(cuda_device)
    (mag, band), ran, launches = _probe(lambda: plan.modspec(x, case.win, case.hop, case.nfft, bins))
    _expect_path(ran, path, inst, launches)
    mag = mag.cpu().numpy()
    band = band.cpu().numpy() if band is not None else None
    _check(mag, band, M, case.win, case.hop, case.nfft, bins, path, record_property)
    if case.win == 1:  # mean removed and Hann(1) = 0: exactly zero
        assert np.all(mag == 0.0) and np.all(band == 0.0)


@pytest.mark.gpu
def test_generic_grid_y_fold(cuda_device):
    """65 537 clips: the generic kernel folds grid.y (limit 65 535) into two launches; clips either side of the fold
    match the reference."""
    torch = _torch()
    B, T, win, nfft = 65537, 1500, 1500, 2048
    gen = torch.Generator(device=cuda_device).manual_seed(7)
    x = torch.randn((B, 1, T), device=cuda_device, generator=gen).cumsum_(-1).mul_(0.5)
    bins = mm.band_bins(nfft, FR)
    plan = _plan()
    (mag, band), ran, launches = _probe(lambda: plan.modspec(x, win, 1, nfft, bins))
    _expect_path(ran, "generic", None, launches, n_launches=2)
    pick = [0, 1, 65533, 65534, 65535, 65536]
    M = x[pick].cpu().numpy()
    _check(mag[pick].cpu().numpy(), band[pick].cpu().numpy(), M, win, 1, nfft, bins, "generic")
    del x, mag, band
    torch.cuda.empty_cache()


# ---------------------------------------------------------------------------
# GPU: known answers that do not depend on the reference
# ---------------------------------------------------------------------------


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(PATH_GEOMETRY))
def test_known_answers(name, cuda_device):
    """Per path, with win == nfft: constant rows give exactly 0.0 (the pivot subtraction is exact, and so is the
    fp64 mean of equal floats); a cosine on bin k0 gives A*win/4 at k0, A*win/8 at k0 +- 1 and ~0 elsewhere;
    adding a constant to a trajectory leaves the outputs unchanged within the path's bounds."""
    torch = _torch()
    n_coef, _, _, _, nfft, path, inst = PATH_GEOMETRY[name]
    if path == "tc":
        inst = 8
    win, hop, T = nfft, nfft // 4, nfft + 2 * (nfft // 4)
    bins = mm.band_bins(nfft, FR)
    plan = _plan()
    run = lambda M: _probe(lambda: plan.modspec(torch.as_tensor(M).to(cuda_device), win, hop, nfft, bins))  # noqa: E731

    const = np.broadcast_to(np.linspace(-500.25, 37.5, n_coef, dtype=np.float32)[None, :, None], (1, n_coef, T)).copy()
    (mag, band), ran, launches = run(const)
    _expect_path(ran, path, inst, launches)
    assert torch.count_nonzero(mag).item() == 0 and torch.count_nonzero(band).item() == 0

    k0 = 5
    A = (1.0 + np.arange(n_coef)) / n_coef
    t = np.arange(T)
    cos = (A[None, :, None] * np.cos(2 * np.pi * k0 * t / nfft)[None, None, :]).astype(np.float32)
    (mag, _), _, _ = run(cos)
    mag = mag.cpu().numpy()[0].astype(np.float64)  # [C, n_win, nb]
    peak = (A * win / 4)[:, None]
    tol = 4 * RTOL_MAG[path] * peak  # the float32 cosine itself carries ~1e-7 relative
    assert np.all(np.abs(mag[..., k0] - peak) <= tol)
    assert np.all(np.abs(mag[..., k0 - 1] - peak / 2) <= tol)
    assert np.all(np.abs(mag[..., k0 + 1] - peak / 2) <= tol)
    rest = np.delete(mag, [k0 - 1, k0, k0 + 1], axis=-1)
    assert np.all(rest <= tol[..., None])

    # trajectories on a 2^-10 grid: adding 512 is exact in float32, so only the kernel can change the output
    M = np.round(_walk(1, n_coef, T, 3).astype(np.float64) * 1024) / 1024
    (m0, b0), _, _ = run(M.astype(np.float32))
    (m1, b1), _, _ = run((M + 512.0).astype(np.float32))
    e_win = _ref_modspec(M.astype(np.float32), win, hop, nfft, bins)[2]
    assert _mag_err(m1.cpu().numpy(), m0.cpu().numpy().astype(np.float64)) <= RTOL_MAG[path]
    assert _band_err(b1.cpu().numpy(), b0.cpu().numpy().astype(np.float64), e_win) <= RTOL_BAND[path]


# ---------------------------------------------------------------------------
# GPU: output selection, determinism and batch independence
# ---------------------------------------------------------------------------


def _geometry_batch(name, B=64):
    n_coef, T, win, hop, nfft, path, inst = PATH_GEOMETRY[name]
    return _walk(B, n_coef, T, 40), win, hop, nfft, path, inst


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(PATH_GEOMETRY))
def test_output_selection_is_bit_identical(name, cuda_device):
    """A magnitude-only call, a band-only call (as CorpusRunner makes them) and a call with both give bit-identical
    magnitudes and band energies where they overlap, on the intended path."""
    torch = _torch()
    M, win, hop, nfft, path, inst = _geometry_batch(name)
    bins = mm.band_bins(nfft, FR)
    plan = _plan()
    x = torch.as_tensor(M).to(cuda_device)
    (mag, band), ran, launches = _probe(lambda: plan.modspec(x, win, hop, nfft, bins))
    _expect_path(ran, path, inst, launches)
    (mag_only, none), ran, launches = _probe(lambda: plan.modspec(x, win, hop, nfft, None))
    _expect_path(ran, path, inst, launches)
    assert none is None
    (no_mag, band_only), ran, launches = _probe(lambda: plan.modspec(x, win, hop, nfft, bins, want_mag=False))
    _expect_path(ran, path, inst, launches)
    assert no_mag is None
    assert torch.equal(mag_only, mag)
    assert torch.equal(band_only, band)


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(PATH_GEOMETRY))
def test_repeatable_and_batch_independent(name, cuda_device):
    """The same call twice gives identical bits, and clip i gives the same bits alone, inside a batch of 64 and
    after the batch is permuted (DESIGN.md section 2: a clip's features never depend on its batch)."""
    torch = _torch()
    M, win, hop, nfft, path, inst = _geometry_batch(name)
    bins = mm.band_bins(nfft, FR)
    plan = _plan()
    x = torch.as_tensor(M).to(cuda_device)
    (mag, band), ran, launches = _probe(lambda: plan.modspec(x, win, hop, nfft, bins))
    _expect_path(ran, path, inst, launches)
    for _ in range(3):
        m2, b2 = plan.modspec(x, win, hop, nfft, bins)
        assert torch.equal(m2, mag) and torch.equal(b2, band), "the same call gave different bits"
    for i in (0, 17, 63):
        mi, bi = plan.modspec(x[i : i + 1], win, hop, nfft, bins)
        assert torch.equal(mi[0], mag[i]) and torch.equal(bi[0], band[i]), f"clip {i} alone differs from the batch"
    perm = torch.as_tensor(np.random.default_rng(9).permutation(M.shape[0])).to(cuda_device)
    mp, bp = plan.modspec(x[perm].contiguous(), win, hop, nfft, bins)
    assert torch.equal(mp, mag[perm]) and torch.equal(bp, band[perm]), "a permuted batch changed a clip's bits"


# ---------------------------------------------------------------------------
# GPU: the host-buffer bundle with every modulation geometry
# ---------------------------------------------------------------------------

HOST_GEOMETRY = {
    # name: (mod_win_s, mod_hop_s, seconds, nfft, path) at 100 frames/s
    "tc": (1.0, 0.5, 10.0, 128, "tc"),
    "clip32": (0.2, 0.1, 10.0, 32, "clip"),
    "clip64": (0.5, 0.25, 10.0, 64, "clip"),
    "generic2048": (15.0, 5.0, 40.0, 2048, "generic"),
    "generic4096": (30.0, 10.0, 60.0, 4096, "generic"),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(HOST_GEOMETRY))
def test_host_bundle_modulation_geometries(name, cuda_device, record_property):
    """``mmf_features_host`` (``FeatureExtractor.host_call``) is bit-identical to the device-resident call for
    every modulation geometry, and within bounds of ``oracle.mfcc_features`` with the default bands."""
    torch = _torch()
    win_s, hop_s, secs, nfft, path = HOST_GEOMETRY[name]
    sr = 16000
    y = synth_batch(61, 2, int(sr * secs), sr)
    fx = mm.FeatureExtractor(sr, mod_win_s=win_s, mod_hop_s=hop_s)
    T = fx.plan.num_frames(y.shape[-1])
    assert fx.modspec_geometry(T)[2] == nfft
    want = ("totChange", "mfcc", "modspec", "band_energy")
    dev, ran, _ = _probe(lambda: fx(torch.as_tensor(y).to(cuda_device), want_logmel=False))
    assert ran and {p for p, _ in ran} == {path}, ran
    host = fx.host_call(y, want=want)
    for k in want:
        assert np.array_equal(host[k], dev[k].cpu().numpy()), k
    ref = oracle.mfcc_features(y[0], sr, mod_win_s=win_s, mod_hop_s=hop_s)
    assert host["modspec"][0].shape == ref["modspec"].shape
    # MFCC differences of up to 1e-3 enter every window sample: the magnitudes' error grows with the window
    # (a Hann window sums to win / 2), so the north_star 1e-3 holds up to win 100 frames and scales beyond
    win = int(round(win_s * FR))
    err = float(np.max(np.abs(host["modspec"][0] - ref["modspec"])))
    record_property("modspec_abs_err", err)
    assert err < ABS_TOL * max(1.0, win / 100.0), err
    assert np.allclose(host["band_energy"][0], ref["band_energy"], rtol=1e-4, atol=1e-3 * max(1.0, win / 100.0))


@pytest.mark.gpu
def test_modulation_windows_of_16_frames_or_fewer_are_rejected(cuda_device):
    """nfft < 32 stays unsupported: a FeatureExtractor whose modulation window is 16 frames or fewer raises, on the
    device-resident call and on the host-buffer bundle alike."""
    torch = _torch()
    sr = 16000
    y = synth_batch(62, 1, sr * 2, sr)
    fx = mm.FeatureExtractor(sr, mod_win_s=0.16, mod_hop_s=0.08)
    assert fx.modspec_geometry(200)[:3] == (16, 8, 16)
    with pytest.raises(mm.MmfError) as e:
        fx(torch.as_tensor(y).to(cuda_device), want_logmel=False)
    assert e.value.code == _lib.MMF_ERR_UNSUPPORTED
    with pytest.raises(mm.MmfError) as e:
        fx.host_call(y)
    assert e.value.code == _lib.MMF_ERR_UNSUPPORTED


# ---------------------------------------------------------------------------
# GPU: argument validation
# ---------------------------------------------------------------------------

_BAD_ARGS = [
    # (id, win, hop, nfft, bins, code)
    ("nfft16", 16, 4, 16, None, _lib.MMF_ERR_UNSUPPORTED),
    ("nfft8192", 5000, 100, 8192, None, _lib.MMF_ERR_UNSUPPORTED),
    ("nfft_not_pow2", 100, 50, 192, None, _lib.MMF_ERR_UNSUPPORTED),
    ("win_gt_nfft", 129, 50, 128, None, _lib.MMF_ERR_UNSUPPORTED),
    ("hop0", 100, 0, 128, None, _lib.MMF_ERR_UNSUPPORTED),
    ("bands17", 100, 50, 128, [(1, 3)] * 17, _lib.MMF_ERR_UNSUPPORTED),
    ("lo_gt_hi", 100, 50, 128, [(1, 3), (9, 4)], _lib.MMF_ERR_INVALID),
    ("hi_past_nyquist", 100, 50, 128, [(1, 3), (60, 66)], _lib.MMF_ERR_INVALID),
    ("lo_negative", 100, 50, 128, [(-1, 3)], _lib.MMF_ERR_INVALID),
]


@pytest.mark.gpu
@pytest.mark.parametrize("win,hop,nfft,bins,code", [a[1:] for a in _BAD_ARGS], ids=[a[0] for a in _BAD_ARGS])
def test_invalid_arguments_raise_and_launch_nothing(win, hop, nfft, bins, code, cuda_device):
    torch = _torch()
    plan = _plan()
    x = torch.zeros((2, 3, 6000), device=cuda_device)
    torch.cuda.synchronize()
    n0 = _lib.lib().mmf_launch_count(0)
    with pytest.raises(mm.MmfError) as e:
        plan.modspec(x, win, hop, nfft, bins)
    assert e.value.code == code, e.value
    assert _lib.lib().mmf_launch_count(0) == n0


@pytest.mark.gpu
@pytest.mark.parametrize("bins", [[(1, 3), (9, 4)], [(60, 66)]], ids=["lo_gt_hi", "hi_past_nyquist"])
def test_host_bundle_rejects_bad_bands(bins, cuda_device):
    """The host-buffer bundle validates band ranges as ``mmf_modspec`` does, before anything is queued."""
    sr = 16000
    y = synth_batch(63, 1, sr * 2, sr)
    fx = mm.FeatureExtractor(sr)
    n0 = _lib.lib().mmf_launch_count(0)
    with pytest.raises(mm.MmfError) as e:
        fx.plan.features_host(y, fx.prm, (100, 50, 128, bins), want=("totChange", "band_energy"))
    assert e.value.code == _lib.MMF_ERR_INVALID, e.value
    assert _lib.lib().mmf_launch_count(0) == n0
