"""Packed clips of different lengths through the host-buffer bundle (mmf_features_host_varlen[_pcm16],
mmf_features_varlen_sizes, Plan.features_host_varlen, FeatureExtractor.host_varlen / host_many).

The contract: each clip's packed blocks are bit-identical to mmf_features_host on that clip alone, whatever chunk it
lands in and whoever its neighbours are, and nothing outside [offsets[0], offsets[n]) is read.
"""

import ctypes as C

import numpy as np
import pytest

import oracle
import modulation_mfcc_b200 as mm
from modulation_mfcc_b200 import _lib
from modulation_mfcc_b200.synth import synth_clip

ABS_TOL = 1e-3
ALL = ("totChange", "mfcc", "delta", "modspec", "band_energy")
CONFIGS = {
    # name: (sr, n_fft, winLen, tStep, n_mels, n_mfcc, fmin, fmax)
    "cfg1_16k": (16000, 512, 0.025, 0.01, 40, 13, 0.0, 8000.0),  # tcgen05 mel, tcgen05 K6
    "gui_default": (10000, 512, 0.025, 0.005, 128, 13, 100.0, 10000.0),
    "cfg3_44k": (44100, 2048, 0.025, 0.01, 128, 20, 0.0, 22050.0),  # CUDA-core K1
    "n400": (16000, 400, 0.025, 0.01, 40, 13, 0.0, 8000.0),  # generic n_fft: every clip on the single-clip route
}
FUSED_MAX_T = 12 * 32 * 9  # longest row the fused per-clip kernel takes


def _fx(name, flags=0):
    sr, n_fft, winLen, tStep, n_mels, n_mfcc, fmin, fmax = CONFIGS[name]
    return mm.FeatureExtractor(sr, tStep=tStep, winLen=winLen, n_fft=n_fft, n_mels=n_mels, n_mfcc=n_mfcc, fmin=fmin,
                               fmax=fmax, flags=flags)


def _lengths(fx, seed=0):
    """Sample counts covering the edges: the shortest legal clip, the 32/64/128/256-frame tiles, a clip past the fused
    kernel, clips without a modulation window, and 37, 43, 51 windows at the extractor's modulation geometry.  The
    extra samples cycle through every residue mod 4, so the clip starts do too."""
    hop = fx.plan.cfg.hop_length
    Lw, Hw, _, _ = fx.modspec_geometry(0)
    padlen = mm.sos_zi(mm.api._butter_sos(6, 12 / ((1 / fx.tStep) / 2), "low"))[1]
    frames = [padlen + 1, 31, 32, 33, 64, 65, 127, 128, 129, 255, 256, 257, FUSED_MAX_T + 40, Lw - 1, Lw,
              (36 * Hw) + Lw, (42 * Hw) + Lw, (50 * Hw) + Lw]
    rng = np.random.default_rng(seed)
    frames += [int(t) for t in rng.integers(padlen + 2, 900, 6)]
    return [int((T - 1) * hop + (i % 4) + (hop // 2 if i % 3 == 0 else 0)) for i, T in enumerate(frames)]


def _clips(lengths, sr, seed=0, pcm16=False):
    clips = [synth_clip(seed + i, n, sr).astype(np.float32) for i, n in enumerate(lengths)]
    if pcm16:
        clips = [np.clip(np.round(c * 32768.0), -32768, 32767).astype(np.int16) for c in clips]
    return clips


def _pack(clips, lead=3, tail=5):
    """Clips back to back after `lead` poison samples (NaN for float32), `tail` more after the last."""
    dt = clips[0].dtype
    poison = np.nan if dt == np.float32 else 32767
    n = sum(len(c) for c in clips)
    buf = np.full(lead + n + tail, poison, dt)
    offsets = np.zeros(len(clips) + 1, np.int64)
    offsets[0] = lead
    for i, c in enumerate(clips):
        offsets[i + 1] = offsets[i] + len(c)
        buf[offsets[i] : offsets[i + 1]] = c
    return buf, offsets


def _blocks(res, fx, i):
    """Clip i's packed blocks, shaped as features_host returns one clip."""
    nm = fx.plan.cfg.n_mfcc
    _, _, nfft, bins = fx.modspec_geometry(0)
    nb, n_bands = nfft // 2 + 1, len(bins)
    f0, f1 = int(res["frame_offsets"][i]), int(res["frame_offsets"][i + 1])
    w0, w1 = int(res["window_offsets"][i]), int(res["window_offsets"][i + 1])
    T, W = f1 - f0, w1 - w0
    out = {"totChange": res["totChange"][f0:f1].reshape(1, T)}
    for k in ("mfcc", "delta"):
        if k in res:
            out[k] = res[k][nm * f0 : nm * f1].reshape(1, nm, T)
    if "modspec" in res:
        out["modspec"] = res["modspec"][nm * nb * w0 : nm * nb * w1].reshape(1, nm, W, nb)
    if "band_energy" in res:
        out["band_energy"] = res["band_energy"][n_bands * w0 : n_bands * w1].reshape(1, W, n_bands)
    return out


def _chunks(lengths, pcm16):
    """The chunk policy of features_host_varlen_impl, for checking that a test spans the chunks it means to."""
    budget = (96 if pcm16 else 32) << 20
    cuts, c0 = [], 0
    while c0 < len(lengths):
        c1, real, n_max = c0 + 1, lengths[c0], lengths[c0]
        while c1 < len(lengths):
            m = max(n_max, lengths[c1])
            if (real + lengths[c1]) * 4 > budget or (c1 + 1 - c0) * ((m + 3) & ~3) * 4 > 2 * budget:
                break
            real, n_max, c1 = real + lengths[c1], m, c1 + 1
        cuts.append((c0, c1))
        c0 = c1
    return cuts


# ---- GPU -----------------------------------------------------------------------------------------------------------


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CONFIGS))
@pytest.mark.parametrize("flags", [0, _lib.MMF_FLAG_NO_TC_MEL, _lib.MMF_FLAG_NO_TMA, _lib.MMF_FLAG_NO_TC_MODSPEC])
def test_packed_matches_solo_host_calls(name, flags, cuda_device):
    """Every clip's packed blocks equal features_host on that clip alone, bit for bit: float32 and int16, for the
    full bundle, the bundle without delta (the folded route) and totChange alone."""
    fx = _fx(name, flags)
    lengths = _lengths(fx, seed=len(name) + flags)
    for pcm16 in (False, True):
        clips = _clips(lengths, fx.plan.cfg.sample_rate, seed=7, pcm16=pcm16)
        buf, offsets = _pack(clips)
        for want in (ALL, ("totChange", "mfcc", "modspec", "band_energy"), ("totChange",)):
            res = fx.host_varlen(buf, offsets, want=want)
            assert list(res["frames"]) == [fx.plan.num_frames(n) for n in lengths]
            for i, c in enumerate(clips):
                one = fx.host_call(c[None], want=want)
                got = _blocks(res, fx, i)
                for k in want:
                    assert np.array_equal(got[k], one[k]), (pcm16, want, k, i)


@pytest.mark.gpu
@pytest.mark.parametrize("pcm16", [False, True])
def test_equal_lengths_equal_the_padded_batch(pcm16, cuda_device):
    fx = _fx("cfg1_16k")
    n = 16000 * 3 + 77
    clips = _clips([n] * 40, 16000, seed=3, pcm16=pcm16)
    batch = np.stack(clips)
    ref = fx.host_call(batch, want=ALL)
    res = fx.host_varlen(batch.reshape(-1), np.arange(41, dtype=np.int64) * n, want=ALL)
    for k in ALL:
        assert res[k].tobytes() == ref[k].tobytes(), k


@pytest.mark.gpu
@pytest.mark.parametrize("pcm16", [False, True])
def test_multi_chunk_matches_device_varlen_and_oracle(pcm16, cuda_device):
    """Three chunks or more: a medium clip caps its chunk through the padded-footprint budget, and one clip longer
    than the float32 budget forms a chunk alone.  Every clip equals FeatureExtractor.varlen on the device (itself
    bit-identical to the solo calls); the clips on either side of each chunk boundary are checked against the
    oracle."""
    torch = pytest.importorskip("torch")
    sr = 16000
    fx = _fx("cfg1_16k")
    short = [48000 + 13 * i for i in range(7)]
    medium = 6_000_000 if pcm16 else 2_000_000
    long = 26_000_000 if pcm16 else 9_000_000  # over the input type's budget (96 MiB / 32 MiB of float32)
    lengths = short[:3] + [medium] + short[3:] + [long] + short[:3] + [medium] + short[3:]
    cuts = _chunks(lengths, pcm16)
    assert len(cuts) >= 3 and (lengths.index(long), lengths.index(long) + 1) in cuts, cuts
    clips = _clips(lengths, sr, seed=40, pcm16=pcm16)
    buf, offsets = _pack(clips)
    res = fx.host_varlen(buf, offsets, want=ALL)
    n_max = max(lengths)
    pad = torch.zeros((len(clips), (n_max + 3) // 4 * 4), dtype=torch.float32)
    for i, c in enumerate(clips):
        pad[i, : len(c)] = torch.as_tensor(c.astype(np.float32) / 32768.0 if pcm16 else c)
    dev = fx.varlen(pad.to(cuda_device), lengths, want_logmel=False)
    dev = {k: (v.cpu().numpy() if hasattr(v, "cpu") else v) for k, v in dev.items() if v is not None}
    for i in range(len(clips)):
        got = _blocks(res, fx, i)
        T, W = int(dev["frames"][i]), int(dev["windows"][i])
        assert np.array_equal(got["totChange"][0], dev["totChange"][i, :T]), i
        assert np.array_equal(got["mfcc"][0], dev["mfcc"][i, :, :T]), i
        assert np.array_equal(got["delta"][0], dev["delta"][i, :, :T]), i
        assert np.array_equal(got["modspec"][0], dev["modspec"][i, :, :W]), i
        assert np.array_equal(got["band_energy"][0], dev["band_energy"][i, :W]), i
    edges = sorted({j for c0, c1 in cuts for j in (c0 - 1, c0, c1 - 1, c1) if 0 <= j < len(clips)})
    for i in edges:
        y = clips[i].astype(np.float32) / 32768.0 if pcm16 else clips[i]
        ref = oracle.mfcc_features(y, sr)
        got = _blocks(res, fx, i)
        for k in ("mfcc", "totChange", "modspec"):
            assert np.max(np.abs(got[k][0] - ref[k])) < ABS_TOL, (k, i)


@pytest.mark.gpu
def test_launches_do_not_grow_with_the_clips(cuda_device):
    """One chunk of default-route clips takes a fixed number of launches.  Both batches hold 32 clips or more, so
    both take the batched output filter of the ragged change path."""
    fx = _fx("cfg1_16k")
    rng = np.random.default_rng(5)
    counts = []
    for n_clips in (40, 64):
        lengths = [int(n) for n in rng.integers(30000, 160000, n_clips)]
        buf, offsets = _pack(_clips(lengths, 16000, seed=n_clips))
        fx.host_varlen(buf, offsets, want=ALL)  # warm-up (workspace growth)
        _lib.lib().mmf_launch_count(1)
        fx.host_varlen(buf, offsets, want=ALL)
        counts.append(_lib.lib().mmf_launch_count(1))
    assert counts[0] == counts[1], counts


@pytest.mark.gpu
def test_device_call_in_flight_does_not_disturb_host_call(cuda_device):
    torch = pytest.importorskip("torch")
    sr = 16000
    fx = _fx("cfg1_16k")
    lengths = [int(n) for n in np.random.default_rng(8).integers(40000, 200000, 60)]
    clips = _clips(lengths, sr, seed=60)
    buf, offsets = _pack(clips)
    ref = fx.host_varlen(buf, offsets, want=ALL)
    pcm = mm.synth_batch_device(64, 160000, sr, seed=99, device=cuda_device)
    dev = fx(pcm, want_logmel=False)
    # a device call queued on the caller's stream, then a host call on the same plan, then the reverse
    dev2 = fx(pcm, want_logmel=False)
    res = fx.host_varlen(buf, offsets, want=ALL)
    res2 = fx.host_varlen(buf, offsets, want=ALL)
    dev3 = fx(pcm, want_logmel=False)
    for k in ALL:
        assert np.array_equal(res[k], ref[k]) and np.array_equal(res2[k], ref[k]), k
        assert torch.equal(dev2[k], dev[k]) and torch.equal(dev3[k], dev[k]), k


@pytest.mark.gpu
def test_host_many_matches_mfcc_features_batch(cuda_device):
    sr = 16000
    fx = _fx("cfg1_16k")
    lengths = [32001, 50003, 16000 * 3 + 2, 20011]
    clips = _clips(lengths, sr, seed=70)
    many = fx.host_many(clips)
    assert len(many) == len(clips)
    for c, d in zip(clips, many):
        one = mm.mfcc_features_batch(c[None], sr, tStep=0.01, winLen=0.025, n_fft=512, n_mels=40, n_mfcc=13,
                                     fmax=8000.0)
        for k in ALL:
            assert np.array_equal(d[k], one[k][0]), k
        assert np.array_equal(d["T"], one["T"])
    assert fx.host_many([]) == []


@pytest.mark.gpu
def test_too_short_clip_fails_before_anything_runs(cuda_device):
    fx = _fx("cfg1_16k")
    clips = _clips([16000, 20000, 800, 16000], 16000, seed=1)
    buf, offsets = _pack(clips)
    _lib.lib().mmf_launch_count(1)
    with pytest.raises(ValueError, match="clip 2"):
        fx.host_varlen(buf, offsets)
    assert _lib.lib().mmf_launch_count(1) == 0


# ---- no GPU needed -------------------------------------------------------------------------------------------------


def _sizes(cfg, offsets, mod=None):
    offs = np.ascontiguousarray(offsets, dtype=np.int64)
    n = len(offs) - 1
    fo, wo = np.zeros(max(n, 0) + 1, np.int64), np.zeros(max(n, 0) + 1, np.int64)
    mp = None
    if mod is not None:
        mp = _lib.mmf_modspec_params()
        mp.win, mp.hop, mp.nfft = mod
    rc = _lib.lib().mmf_features_varlen_sizes(C.byref(cfg.to_c()), C.byref(mp) if mp is not None else None, n,
                                              offs.ctypes.data, fo.ctypes.data, wo.ctypes.data)
    return rc, fo, wo


@pytest.mark.parametrize("mod", [None, (100, 50, 128), (0, 50, 128), (37, 11, 64)])
def test_sizes_match_the_frame_and_window_formulas(mod):
    cfg = mm.MfccConfig(16000, 512, 400, 160, 40, 13, 0.0, 8000.0)
    rng = np.random.default_rng(2)
    lengths = rng.integers(1, 400000, 200)
    offsets = np.concatenate([[17], 17 + np.cumsum(lengths)])
    rc, fo, wo = _sizes(cfg, offsets, mod)
    assert rc == 0
    T = np.array([mm.num_frames(int(n), 512, 160) for n in lengths])
    assert np.array_equal(fo, np.concatenate([[0], np.cumsum(T)]))
    if mod is None or mod[0] == 0:
        assert not wo.any()
    else:
        win, hop, _ = mod
        n_win = np.where(T >= win, 1 + (T - win) // hop, 0)
        assert np.array_equal(wo, np.concatenate([[0], np.cumsum(n_win)]))


def _host_varlen_call(offsets, n_clips=None):
    offs = np.ascontiguousarray(offsets, dtype=np.int64) if offsets is not None else None
    p = _lib.mmf_change_params()
    tot = np.zeros(8, np.float64)
    return [
        fn(None, None, len(offsets) - 1 if n_clips is None else n_clips, offs.ctypes.data if offs is not None else None,
           C.byref(p), None, tot.ctypes.data, None, None, None, None)
        for fn in (_lib.lib().mmf_features_host_varlen, _lib.lib().mmf_features_host_varlen_pcm16)
    ]


@pytest.mark.parametrize(
    "offsets, clip",
    [([-1, 10, 20], 0), ([0, 10, 10, 30], 1), ([0, 10, 20, 15], 2), ([5, 4], 0), ([0, 100, 200, 300, 299], 3)],
)
def test_bad_offsets_fail_before_any_plan_or_device(offsets, clip):
    lib = _lib.lib()
    for rc in _host_varlen_call(offsets):
        assert rc == _lib.MMF_ERR_INVALID
        assert f"clip {clip}" in lib.mmf_last_error().decode()
    rc, _, _ = _sizes(mm.MfccConfig(16000, 512, 400, 160, 40, 13, 0.0, 8000.0), offsets)
    assert rc == _lib.MMF_ERR_INVALID and f"clip {clip}" in lib.mmf_last_error().decode()


def test_null_offsets_and_empty_batches_fail():
    lib = _lib.lib()
    for rc in _host_varlen_call(None, n_clips=2):
        assert rc == _lib.MMF_ERR_INVALID and "offsets is NULL" in lib.mmf_last_error().decode()
    for rc in _host_varlen_call([0], n_clips=0):
        assert rc == _lib.MMF_ERR_INVALID
    # valid offsets, no plan: the NULL plan is reported only after the offsets passed
    for rc in _host_varlen_call([0, 10, 20]):
        assert rc == _lib.MMF_ERR_INVALID and "NULL argument" in lib.mmf_last_error().decode()
