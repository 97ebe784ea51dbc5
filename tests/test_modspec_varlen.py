"""Variable-length batches of the modulation spectrum (mmf_modspec_varlen, Plan.modspec_varlen,
FeatureExtractor.varlen, mfcc_features_many).

The contract: windows [0, n_win_i) of clip i are bit-identical to mmf_modspec on that clip alone (its T_i frames,
rows contiguous), every output element at a window >= n_win_i is exactly 0, and no frame >= T_i affects any output.
Each clip runs on the kernel its own call runs on; the tcgen05 and clip-resident kernels take the whole batch in one
launch each.
"""

from typing import NamedTuple

import numpy as np
import pytest

import oracle
import modulation_mfcc_b200 as mm
from modulation_mfcc_b200 import _lib
from modulation_mfcc_b200.synth import synth_clip
from test_modspec_paths import ABS_TOL, FR, RTOL_BAND, RTOL_MAG, _band_err, _edge_bands, _mag_err, _probe, _ref_modspec


def _torch():
    import torch

    return torch


class Route(NamedTuple):
    id: str
    n_coef: int
    win: int
    hop: int
    nfft: int
    bands: str  # "default" (mm.band_bins), "edge" (16 edge bands) or "none"
    path: str  # the kernel the batch's clips take (with flags 0)
    inst: int
    t_max: int  # longest random clip (frames)


ROUTES = [
    # FeatureExtractor's default at 10 ms: 1 s / 0.5 s windows, 13 coefficients (a few window counts -- 37, 43, ...
    # -- leave the tcgen05 kernel for the clip kernel, in the batch as alone: test_mixed_routes)
    Route("tc_ks7_default", 13, 100, 50, 128, "default", "tc", 7, 1800),
    Route("tc_ks2_coef1_items127_129", 1, 20, 7, 128, "edge", "tc", 2, 1200),
    Route("tc_ks3_coef5", 5, 40, 3, 128, "edge", "tc", 3, 700),
    Route("tc_ks8_hop1_chunked", 13, 128, 1, 128, "none", "tc", 8, 1200),
    Route("clip_32", 13, 32, 8, 32, "default", "clip", 32, 600),
    Route("clip_64_bands16", 7, 50, 25, 64, "edge", "clip", 64, 900),
    # FeatureExtractor's default at 5 ms: 2 s / 1 s windows -> win 200, nfft 256
    Route("clip_256_default_5ms", 13, 200, 100, 256, "default", "clip", 256, 3000),
    Route("clip_256_coef41_hop1_chunks", 41, 200, 1, 256, "none", "clip", 256, 600),
    Route("clip_1024", 3, 1000, 100, 1024, "edge", "clip", 1024, 3000),
    Route("fast_1024", 40, 1000, 50, 1024, "default", "fast", 1024, 1500),
    Route("generic_2048", 3, 1500, 250, 2048, "edge", "generic", 2048, 2600),
]
TC_ROUTES = [r for r in ROUTES if r.path == "tc"]
_RUNS = [(r, 0) for r in ROUTES] + [(r, _lib.MMF_FLAG_NO_TC_MODSPEC) for r in TC_ROUTES]


def _bands(kind, nfft):
    if kind == "default":
        return mm.band_bins(nfft, FR)
    if kind == "edge":
        return _edge_bands(nfft)
    return []


def _lengths(r, n_clips=40, seed=0):
    """Frame counts covering the edges the kernels care about, the rest random in [0, t_max]."""
    win, hop = r.win, r.hop
    T = [0, win - 1, win]  # no windows (T = 0 included), no windows, exactly one
    for k in (1, 3, 8):  # either side of a window-count step
        T += [win + k * hop - 1, win + k * hop, win + k * hop + hop - 1]
    for rows in (127, 128, 129):  # n_win * n_coef around the 128-row MMA block
        if rows % r.n_coef == 0:
            T.append(win + (rows // r.n_coef - 1) * hop)
    T.append(r.t_max)  # the most windows: several chunks where the route chunks
    rng = np.random.default_rng(seed)
    T += [int(t) for t in rng.integers(0, r.t_max + 1, max(0, n_clips - len(T)))]
    return np.asarray(T, np.int64)


def _walk_ragged(T, n_coef, seed, fill=None):
    """Random-walk trajectories (row 0 near -500, where c0 sits) in [B, n_coef, max T]; frames >= T_i get ``fill``."""
    rng = np.random.default_rng(seed)
    P = int(T.max())
    M = (rng.standard_normal((len(T), n_coef, P)).cumsum(axis=-1) * 0.5).astype(np.float32)
    M[:, 0] -= 500.0
    if fill is not None:
        for i, t in enumerate(T):
            M[i, :, t:] = fill
    return M


def _plan(flags=0):
    return mm.get_plan(mm.MfccConfig(16000, 512, 400, 160, 40, 13, 0.0, 8000.0, flags=flags))


def _solo_parity(plan, x, T, win, hop, nfft, bins, want_mag=True):
    """Every clip of the ragged call against plan.modspec on that clip alone; returns the call's outputs."""
    torch = _torch()
    (mag, band, windows), ran, _ = _probe(lambda: plan.modspec_varlen(x, T, win, hop, nfft, bins, want_mag=want_mag))
    assert list(windows) == [1 + (t - win) // hop if t >= win else 0 for t in T]
    W = int(windows.max())
    B, n_coef = x.shape[:2]
    nb = nfft // 2 + 1
    assert mag is None if not want_mag else mag.shape == (B, n_coef, W, nb)
    assert band is None if not bins else band.shape == (B, W, len(bins))
    some = [i for i in range(B) if windows[i] > 0]  # a clip without windows has no solo call to compare with
    solo, ran_solo, _ = _probe(
        lambda: [plan.modspec(x[i : i + 1, :, : T[i]].contiguous(), win, hop, nfft, bins, want_mag=want_mag) for i in some]
    )
    # the same kernels and instantiations as the clips' own calls, nothing else
    assert set(ran) == set(ran_solo), (ran, ran_solo)
    for i in range(B):
        w = int(windows[i])
        m1, b1 = solo[some.index(i)] if w else (None, None)
        if mag is not None:
            if w:
                assert torch.equal(mag[i, :, :w], m1[0]), f"clip {i} (T {T[i]}): magnitudes differ from its own call"
            assert torch.count_nonzero(mag[i, :, w:]).item() == 0, f"clip {i}: non-zero magnitude tail"
        if band is not None:
            if w:
                assert torch.equal(band[i, :w], b1[0]), f"clip {i} (T {T[i]}): band energies differ from its own call"
            assert torch.count_nonzero(band[i, w:]).item() == 0, f"clip {i}: non-zero band tail"
    return mag, band, windows, ran


# ---------------------------------------------------------------------------
# GPU: every route, bit for bit against the single-clip call
# ---------------------------------------------------------------------------


@pytest.mark.gpu
@pytest.mark.parametrize("r,flags", _RUNS, ids=[r.id + ("_no_tc" if f else "") for r, f in _RUNS])
def test_varlen_matches_solo_calls(r, flags, cuda_device):
    torch = _torch()
    T = _lengths(r, seed=r.win)
    M = _walk_ragged(T, r.n_coef, 100 + r.win)
    bins = _bands(r.bands, r.nfft)
    plan = _plan(flags)
    _, _, _, ran = _solo_parity(plan, torch.as_tensor(M).to(cuda_device), T, r.win, r.hop, r.nfft, bins)
    want = (r.path, r.inst) if not flags else ("clip", 128)
    if r.path == "generic":
        want = ("generic", None)
    assert want in ran, ran


@pytest.mark.gpu
@pytest.mark.parametrize("r", [ROUTES[0], ROUTES[6], ROUTES[9]], ids=lambda r: r.id)
def test_output_selection(r, cuda_device):
    """Magnitude-only and band-only calls: each clip still equals its own call, tails 0."""
    torch = _torch()
    T = _lengths(r, seed=3)
    x = torch.as_tensor(_walk_ragged(T, r.n_coef, 7)).to(cuda_device)
    plan = _plan()
    bins = mm.band_bins(r.nfft, FR)
    mag, none, _, _ = _solo_parity(plan, x, T, r.win, r.hop, r.nfft, None)
    assert none is None
    no_mag, band, _, _ = _solo_parity(plan, x, T, r.win, r.hop, r.nfft, bins, want_mag=False)
    assert no_mag is None
    both_m, both_b, _ = plan.modspec_varlen(x, T, r.win, r.hop, r.nfft, bins)
    assert torch.equal(both_m, mag) and torch.equal(both_b, band)


@pytest.mark.gpu
def test_against_the_reference(cuda_device, record_property):
    """The tcgen05 route's valid windows against the float64 reference, within the single-clip bounds."""
    torch = _torch()
    r = ROUTES[0]
    T = _lengths(r, n_clips=24, seed=5)
    M = _walk_ragged(T, r.n_coef, 11)
    bins = _bands(r.bands, r.nfft)
    mag, band, windows = _plan().modspec_varlen(torch.as_tensor(M).to(cuda_device), T, r.win, r.hop, r.nfft, bins)
    mag, band = mag.cpu().numpy(), band.cpu().numpy()
    worst_m = worst_b = 0.0
    for i, t in enumerate(T):
        w = int(windows[i])
        if not w:
            continue
        rm, rb, e_win = _ref_modspec(M[i, :, :t], r.win, r.hop, r.nfft, bins)
        worst_m = max(worst_m, _mag_err(mag[i, :, :w], rm))
        worst_b = max(worst_b, _band_err(band[i, :w], rb, e_win))
    record_property("mag_err", worst_m)
    record_property("band_err", worst_b)
    assert worst_m <= RTOL_MAG["tc"] and worst_b <= RTOL_BAND["tc"], (worst_m, worst_b)


@pytest.mark.gpu
def test_mixed_routes(cuda_device):
    """At FeatureExtractor's default geometry (13 coefficients, win 100, hop 50, nfft 128) a clip of 37 or 43
    windows is cut into two chunks whose last one does not fit the tcgen05 kernel's staging buffer, so its own call
    takes the clip kernel: a batch that holds such clips runs both kernels, each clip on its own one."""
    torch = _torch()
    r = ROUTES[0]
    n_win = [3, 37, 12, 43, 36, 38, 1, 0, 42, 44, 37]
    T = np.asarray([r.win + (w - 1) * r.hop + (w % 3) * 7 if w else 60 for w in n_win], np.int64)
    x = torch.as_tensor(_walk_ragged(T, r.n_coef, 13)).to(cuda_device)
    _, _, _, ran = _solo_parity(_plan(), x, T, r.win, r.hop, r.nfft, mm.band_bins(r.nfft, FR))
    assert set(ran) == {("tc", 7), ("clip", 128)}, ran


@pytest.mark.gpu
@pytest.mark.parametrize("r", [ROUTES[0], ROUTES[6]], ids=lambda r: r.id)
def test_launch_count_does_not_grow_with_the_batch(r, cuda_device):
    """On the batched routes 400 clips take as many launches as 40: the route's kernel and the tails."""
    torch = _torch()
    plan = _plan()
    bins = mm.band_bins(r.nfft, FR)
    rng = np.random.default_rng(17)
    counts = []
    for n_clips in (40, 400):
        # up to 36 windows at the 10 ms default: every clip on the tcgen05 kernel (test_mixed_routes)
        T = rng.integers(0, min(r.t_max, r.win + 35 * r.hop) + 1, n_clips).astype(np.int64)
        x = torch.zeros((n_clips, r.n_coef, int(T.max())), device=cuda_device)
        plan.modspec_varlen(x, T, r.win, r.hop, r.nfft, bins)  # warm-up (workspace growth)
        torch.cuda.synchronize()
        _, ran, launches = _probe(lambda: plan.modspec_varlen(x, T, r.win, r.hop, r.nfft, bins))
        assert {p for p, _ in ran} == {r.path}, ran
        counts.append(launches)
    assert counts[0] == counts[1] and counts[0] <= 2, counts


# ---------------------------------------------------------------------------
# GPU: ragged-batch properties
# ---------------------------------------------------------------------------

_PROPERTY_ROUTES = [ROUTES[0], ROUTES[4], ROUTES[9], ROUTES[10]]


@pytest.mark.gpu
@pytest.mark.parametrize("r", _PROPERTY_ROUTES, ids=lambda r: r.id)
@pytest.mark.parametrize("fill", [np.nan, 1e30], ids=["nan", "1e30"])
def test_frames_past_a_clip_do_not_matter(r, fill, cuda_device):
    torch = _torch()
    T = _lengths(r, n_clips=24, seed=19)
    bins = _bands(r.bands, r.nfft)
    plan = _plan()
    clean = plan.modspec_varlen(torch.as_tensor(_walk_ragged(T, r.n_coef, 23, fill=0.0)).to(cuda_device), T, r.win,
                                r.hop, r.nfft, bins)
    dirty = plan.modspec_varlen(torch.as_tensor(_walk_ragged(T, r.n_coef, 23, fill=fill)).to(cuda_device), T, r.win,
                                r.hop, r.nfft, bins)
    assert torch.equal(clean[0], dirty[0]) and torch.equal(clean[1], dirty[1])


@pytest.mark.gpu
@pytest.mark.parametrize("r", _PROPERTY_ROUTES, ids=lambda r: r.id)
def test_equal_lengths_equal_the_batch_call(r, cuda_device):
    torch = _torch()
    T = np.full(24, r.t_max - 3, np.int64)
    x = torch.as_tensor(_walk_ragged(T, r.n_coef, 29)).to(cuda_device)
    bins = _bands(r.bands, r.nfft)
    plan = _plan()
    mag, band, _ = plan.modspec_varlen(x, T, r.win, r.hop, r.nfft, bins)
    m1, b1 = plan.modspec(x, r.win, r.hop, r.nfft, bins)
    assert torch.equal(mag, m1)
    assert (band is None and b1 is None) or torch.equal(band, b1)


@pytest.mark.gpu
@pytest.mark.parametrize("r", _PROPERTY_ROUTES, ids=lambda r: r.id)
def test_permuting_clips_permutes_outputs(r, cuda_device):
    torch = _torch()
    T = _lengths(r, n_clips=24, seed=31)
    M = _walk_ragged(T, r.n_coef, 37, fill=0.0)
    perm = np.random.default_rng(2).permutation(len(T))
    bins = _bands(r.bands, r.nfft)
    plan = _plan()
    a = plan.modspec_varlen(torch.as_tensor(M).to(cuda_device), T, r.win, r.hop, r.nfft, bins)
    b = plan.modspec_varlen(torch.as_tensor(M[perm]).to(cuda_device), T[perm], r.win, r.hop, r.nfft, bins)
    p = torch.as_tensor(perm).to(cuda_device)
    assert torch.equal(a[0][p], b[0])
    assert (a[1] is None and b[1] is None) or torch.equal(a[1][p], b[1])


@pytest.mark.gpu
def test_no_windows_at_all(cuda_device):
    """Every clip shorter than the window: empty outputs, nothing launched."""
    torch = _torch()
    plan = _plan()
    x = torch.zeros((3, 13, 90), device=cuda_device)
    torch.cuda.synchronize()
    n0 = _lib.lib().mmf_launch_count(0)
    mag, band, windows = plan.modspec_varlen(x, [90, 0, 99 - 10], 100, 50, 128, mm.band_bins(128, FR))
    assert mag.shape == (3, 13, 0, 65) and band.shape == (3, 0, 5) and list(windows) == [0, 0, 0]
    assert _lib.lib().mmf_launch_count(0) == n0


# ---------------------------------------------------------------------------
# GPU: end to end
# ---------------------------------------------------------------------------

_SR = 16000


def _e2e_clips(seed):
    # shorter than 1 s (no modulation windows), exactly 1 s, and longer clips with odd sample counts
    lengths = [int(_SR * 0.7), _SR, int(_SR * 2.3) + 17, _SR * 5 + 123, int(_SR * 3.7) + 1, _SR * 7 - 5]
    return [synth_clip(seed + i, n, _SR).astype(np.float32) for i, n in enumerate(lengths)]


def _same(a, b):
    if hasattr(a, "cpu"):
        a = a.cpu().numpy()
    if hasattr(b, "cpu"):
        b = b.cpu().numpy()
    return a.shape == b.shape and np.array_equal(a, b)


@pytest.mark.gpu
@pytest.mark.parametrize("tStep,path", [(0.01, "tc"), (0.005, "clip")])
def test_features_many_matches_single_clip_calls(tStep, path, cuda_device):
    torch = _torch()
    clips = _e2e_clips(41)
    fx = mm.FeatureExtractor(_SR, tStep=tStep)
    many, ran, _ = _probe(lambda: mm.mfcc_features_many(clips, _SR, tStep=tStep))
    assert path in {p for p, _ in ran}, ran
    dev = mm.mfcc_features_many([torch.as_tensor(c).to(cuda_device) for c in clips], _SR, tStep=tStep)
    for i, c in enumerate(clips):
        one = mm.mfcc_features_batch(c[None], _SR, tStep=tStep)
        assert set(many[i]) == set(one) == set(dev[i]), (set(many[i]), set(one))
        for k, v in one.items():
            v = v if k == "T" else v[0]
            assert isinstance(many[i][k], np.ndarray) and _same(many[i][k], v), (i, k)
            if k != "T":
                assert dev[i][k].is_cuda, (i, k)
            assert _same(dev[i][k], v), (i, k)
    assert many[0]["modspec"].shape[1] == 0 and many[0]["band_energy"].shape[0] == 0  # 0.7 s: no windows
    # FeatureExtractor.varlen on the padded batch: the padded dict, clip by clip the same bits
    lengths = [len(c) for c in clips]
    pcm = np.zeros((len(clips), max(lengths)), np.float32)
    for i, c in enumerate(clips):
        pcm[i, : len(c)] = c
    res = fx.varlen(torch.as_tensor(pcm).to(cuda_device), lengths)
    assert {"frames", "windows", "totChange", "logmel", "mfcc", "delta", "modspec", "band_energy"} <= set(res)
    for i in range(len(clips)):
        T, W = int(res["frames"][i]), int(res["windows"][i])
        assert _same(res["modspec"][i, :, :W], many[i]["modspec"]) and _same(res["band_energy"][i, :W], many[i]["band_energy"])
        assert _same(res["mfcc"][i, :, :T], many[i]["mfcc"])
        assert not res["modspec"][i, :, W:].any() and not res["band_energy"][i, W:].any()


@pytest.mark.gpu
def test_features_many_against_the_oracle(cuda_device, record_property):
    clips = _e2e_clips(43)
    many = mm.mfcc_features_many(clips, _SR)
    ref = oracle.mfcc_features(clips[3], _SR)
    got = many[3]
    assert got["modspec"].shape == ref["modspec"].shape
    err = float(np.max(np.abs(got["modspec"] - ref["modspec"])))
    record_property("modspec_abs_err", err)
    assert err < ABS_TOL, err
    assert np.allclose(got["band_energy"], ref["band_energy"], rtol=1e-4, atol=1e-3)


@pytest.mark.gpu
def test_too_short_clip_names_its_index(cuda_device):
    clips = _e2e_clips(47)
    clips[2] = clips[2][: 160 * 10]
    with pytest.raises(ValueError) as single:
        mm.mfcc_features_batch(clips[2][None], _SR)
    _lib.lib().mmf_launch_count(1)
    with pytest.raises(ValueError, match="clip 2") as many:
        mm.mfcc_features_many(clips, _SR)
    assert str(single.value) in str(many.value)
    assert _lib.lib().mmf_launch_count(1) == 0


@pytest.mark.gpu
def test_bad_lengths_launch_nothing(cuda_device):
    torch = _torch()
    plan = _plan()
    x = torch.zeros((3, 13, 500), device=cuda_device)
    torch.cuda.synchronize()
    for T, named in (([500, 501, 200], "clip 1"), ([500, 200, -1], "clip 2")):
        n0 = _lib.lib().mmf_launch_count(0)
        with pytest.raises(mm.MmfError) as e:
            plan.modspec_varlen(x, T, 100, 50, 128, mm.band_bins(128, FR))
        assert e.value.code == _lib.MMF_ERR_INVALID and named in e.value.msg, e.value
        assert _lib.lib().mmf_launch_count(0) == n0


# ---- argument checks that fail before any CUDA call (no GPU needed) ----------------------------------------------


def _call(T, n_clips=None, pitch=100, win=10, hop=5, nfft=32, n_coef=3, bands=None, band_out=None):
    Th = np.ascontiguousarray(T, dtype=np.int64) if T is not None else None
    lo = hi = None
    if bands:
        lo = np.ascontiguousarray([b[0] for b in bands], np.int32)
        hi = np.ascontiguousarray([b[1] for b in bands], np.int32)
    return _lib.lib().mmf_modspec_varlen(
        None, None, len(T) if n_clips is None else n_clips, n_coef, Th.ctypes.data if Th is not None else None, pitch,
        win, hop, nfft, None, band_out, lo.ctypes.data if lo is not None else None,
        hi.ctypes.data if hi is not None else None, len(bands) if bands else 0, None)


@pytest.mark.parametrize(
    "args, code, named",
    [
        (dict(T=None, n_clips=2), _lib.MMF_ERR_INVALID, None),
        (dict(T=[10, 20], n_clips=0), _lib.MMF_ERR_INVALID, None),
        (dict(T=[10, 20], n_coef=0), _lib.MMF_ERR_INVALID, None),
        (dict(T=[10, -1]), _lib.MMF_ERR_INVALID, "clip 1"),
        (dict(T=[10, 20, 101]), _lib.MMF_ERR_INVALID, "clip 2"),
        (dict(T=[10, 20], nfft=16, win=10), _lib.MMF_ERR_UNSUPPORTED, None),
        (dict(T=[10, 20], hop=0), _lib.MMF_ERR_UNSUPPORTED, None),
        (dict(T=[10, 20], win=40, nfft=32), _lib.MMF_ERR_UNSUPPORTED, None),
        (dict(T=[10, 20], bands=[(3, 2)], band_out=1), _lib.MMF_ERR_INVALID, None),
        (dict(T=[10, 20], bands=[(1, 3)] * 17), _lib.MMF_ERR_UNSUPPORTED, None),
        (dict(T=[10, 20]), _lib.MMF_ERR_INVALID, None),  # lengths and geometry fine: NULL plan and input
    ],
)
def test_invalid_arguments_without_a_device(args, code, named):
    assert _call(**args) == code
    if named:
        assert named in _lib.lib().mmf_last_error().decode()


def test_varlen_modspec_symbol_is_bound():
    assert "mmf_modspec_varlen" in _lib.exported_symbols()
    assert callable(mm.mfcc_features_many) and callable(mm.FeatureExtractor.varlen)
    assert callable(mm.Plan.modspec_varlen)
