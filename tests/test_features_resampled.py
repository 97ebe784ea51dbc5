"""Packed clips at their own sample rates through the host-buffer bundle (mmf_features_host_varlen_resampled,
mmf_resample_varlen, Plan.features_host_varlen(rates=), FeatureExtractor.host_varlen / host_many(rates=) / host_files).

The contract: clip i's packed blocks are bit-identical to
    features_host(resample_poly(pcm16_to_f32(x_i) or x_i, up, down, "hq"))
on that clip alone, with (up, down) = resample_ratio(rate_i, sr), whatever chunk it lands in and whoever its
neighbours are; a clip at the plan's rate is staged as the plan-rate packed call stages it.
"""

import ctypes as C
import math
from fractions import Fraction

import numpy as np
import pytest

import oracle
import modulation_mfcc_b200 as mm
from modulation_mfcc_b200 import _lib
from modulation_mfcc_b200.plan import RESAMPLE_CLIP, design_resample_filter, resample_descriptors, resample_ratio
from modulation_mfcc_b200.synth import synth_clip

ALL = ("totChange", "mfcc", "delta", "modspec", "band_energy")
CONFIGS = {
    # name: (sr, n_fft, winLen, tStep, n_mels, n_mfcc, fmin, fmax), source rates of the clips
    "cfg1_16k": ((16000, 512, 0.025, 0.01, 40, 13, 0.0, 8000.0), (44100, 48000, 8000, 44056, 16000)),
    "gui_default": ((10000, 512, 0.025, 0.005, 128, 13, 100.0, 10000.0), (22050, 11025, 10000)),
    "cfg3_44k": ((44100, 2048, 0.025, 0.01, 128, 20, 0.0, 22050.0), (48000, 16000, 44100)),
}


def _fx(name):
    sr, n_fft, winLen, tStep, n_mels, n_mfcc, fmin, fmax = CONFIGS[name][0]
    return mm.FeatureExtractor(sr, tStep=tStep, winLen=winLen, n_fft=n_fft, n_mels=n_mels, n_mfcc=n_mfcc, fmin=fmin,
                               fmax=fmax)


def _clip(seed, n, rate, pcm16):
    c = synth_clip(seed, n, rate).astype(np.float32)
    return np.clip(np.round(c * 32768.0), -32768, 32767).astype(np.int16) if pcm16 else c


def _solo(fx, plan, x, rate, want):
    """The three-step reference of the contract for one clip."""
    up, down = resample_ratio(rate, fx.sr)
    y = plan.pcm16_to_f32(x) if x.dtype == np.int16 else x
    y = plan.resample_poly(y, up, down, "hq")
    y = y.cpu().numpy() if hasattr(y, "cpu") else np.asarray(y, np.float32)
    return fx.host_call(np.ascontiguousarray(y)[None], want=want)


def _blocks(res, fx, i):
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


def _packed(clips, lead=3, tail=5):
    """Clips back to back after `lead` poison samples (NaN / 32767), `tail` more after the last."""
    poison = np.nan if clips[0].dtype == np.float32 else 32767
    n = sum(len(c) for c in clips)
    buf = np.full(lead + n + tail, poison, clips[0].dtype)
    offsets = np.zeros(len(clips) + 1, np.int64)
    offsets[0] = lead
    for i, c in enumerate(clips):
        offsets[i + 1] = offsets[i] + len(c)
        buf[offsets[i] : offsets[i + 1]] = c
    return buf, offsets


def _padlen(fx):
    return mm.sos_zi(mm.api._butter_sos(6, 12 / ((1 / fx.tStep) / 2), "low"))[1]


def _shortest(fx, rate):
    """Fewest samples at `rate` whose resampled clip has more frames than the filters' padlen."""
    up, down = resample_ratio(rate, fx.sr)
    need = _padlen(fx) * fx.plan.cfg.hop_length  # T = 1 + n // hop > padlen
    n = need * down // up
    while -(-(n * up) // down) < need:
        n += 1
    while n > 1 and -(-((n - 1) * up) // down) >= need:
        n -= 1
    return n


# ---- GPU -----------------------------------------------------------------------------------------------------------


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CONFIGS))
@pytest.mark.parametrize("pcm16", [False, True])
def test_mixed_rates_match_solo_resample_then_host_call(name, pcm16, cuda_device):
    """Every rate of the configuration in one batch, twice over (different lengths, unaligned starts covering every
    residue mod 4): each clip's blocks equal the three-step reference, bit for bit, for the whole bundle and for
    totChange alone."""
    fx = _fx(name)
    rates = list(CONFIGS[name][1]) * 2
    lengths = [int(r * (1.3 + 0.37 * i)) + i for i, r in enumerate(rates)]
    clips = [_clip(11 + i, n, r, pcm16) for i, (n, r) in enumerate(zip(lengths, rates))]
    buf, offsets = _packed(clips)
    assert sorted(set(o % 4 for o in offsets[:-1])) == [0, 1, 2, 3]
    for want in (ALL, ("totChange",)):
        res = fx.host_varlen(buf, offsets, want=want, rates=rates)
        for i, (c, r) in enumerate(zip(clips, rates)):
            one = _solo(fx, fx.plan, c, r, want)
            got = _blocks(res, fx, i)
            for k in want:
                assert np.array_equal(got[k], one[k]), (want, k, i, r)


@pytest.mark.gpu
def test_plan_rate_clips_equal_the_plan_rate_call(cuda_device):
    fx = _fx("cfg1_16k")
    clips = [_clip(i, 16000 + 1234 * i, 16000, True) for i in range(5)]
    buf, offsets = _packed(clips)
    ref = fx.host_varlen(buf, offsets, want=ALL)
    res = fx.host_varlen(buf, offsets, want=ALL, rates=[16000] * 5)
    for k in ALL:
        assert res[k].tobytes() == ref[k].tobytes(), k


@pytest.mark.gpu
@pytest.mark.parametrize("pcm16", [False, True])
def test_shortest_legal_clip_and_one_sample_less(pcm16, cuda_device):
    """The shortest clip at each rate that is legal after resampling runs (and matches its reference) among poison;
    one sample less fails with the too-short error naming its index before anything is launched."""
    fx = _fx("cfg1_16k")
    rates = [44100, 8000, 48000, 16000]
    lengths = [_shortest(fx, r) for r in rates]
    clips = [_clip(30 + i, n, r, pcm16) for i, (n, r) in enumerate(zip(lengths, rates))]
    buf, offsets = _packed(clips)
    res = fx.host_varlen(buf, offsets, want=ALL, rates=rates)
    for i, (c, r) in enumerate(zip(clips, rates)):
        assert int(res["frames"][i]) == _padlen(fx) + 1
        one = _solo(fx, fx.plan, c, r, ALL)
        for k in ALL:
            assert np.array_equal(_blocks(res, fx, i)[k], one[k]), (k, i)
    for j in range(len(clips)):
        short = list(clips)
        short[j] = clips[j][:-1]
        b2, o2 = _packed(short)
        _lib.lib().mmf_launch_count(1)
        with pytest.raises(ValueError, match=f"clip {j}"):
            fx.host_varlen(b2, o2, want=ALL, rates=rates)
        assert _lib.lib().mmf_launch_count(1) == 0


def _chunks(len_in, len_out, pcm16):
    """The chunk policy of features_host_varlen_impl: native samples against the budget, staged rows (resampled
    lengths) against twice it."""
    budget = (96 if pcm16 else 32) << 20
    cuts, c0 = [], 0
    while c0 < len(len_in):
        c1, real, n_max = c0 + 1, len_in[c0], len_out[c0]
        while c1 < len(len_in):
            m = max(n_max, len_out[c1])
            if (real + len_in[c1]) * 4 > budget or (c1 + 1 - c0) * ((m + 3) & ~3) * 4 > 2 * budget:
                break
            real, n_max, c1 = real + len_in[c1], m, c1 + 1
        cuts.append((c0, c1))
        c0 = c1
    return cuts


@pytest.mark.gpu
def test_long_48k_clip_among_short_clips_over_several_chunks(cuda_device):
    """A 48 kHz clip over the float32 budget forms a chunk alone, between chunks of short clips at mixed rates; every
    clip matches its reference, bit for bit."""
    fx = _fx("cfg1_16k")
    rates = [44100, 16000, 8000] * 3 + [48000] + [22050, 16000, 44100] * 3
    len_in = [int(r * 2.1) + 7 * i for i, r in enumerate(rates)]
    len_in[9] = 9_000_000  # 187.5 s at 48 kHz: 36 MB of float32 crosses PCIe, 12 MB is staged
    rs, _ = resample_descriptors(len_in, rates, 16000)
    cuts = _chunks(len_in, [int(n) for n in rs["n_out"]], False)
    assert (9, 10) in cuts and len(cuts) >= 3, cuts
    clips = [_clip(50 + i, n, r, False) for i, (n, r) in enumerate(zip(len_in, rates))]
    buf, offsets = _packed(clips)
    res = fx.host_varlen(buf, offsets, want=ALL, rates=rates)
    for i, (c, r) in enumerate(zip(clips, rates)):
        one = _solo(fx, fx.plan, c, r, ALL)
        for k in ALL:
            assert np.array_equal(_blocks(res, fx, i)[k], one[k]), (k, i)


@pytest.mark.gpu
def test_permuting_the_clips_permutes_the_blocks(cuda_device):
    fx = _fx("cfg1_16k")
    rates = [44100, 48000, 8000, 16000, 44056, 22050]
    clips = [_clip(70 + i, int(r * (1.5 + 0.2 * i)), r, True) for i, r in enumerate(rates)]
    many = fx.host_many(clips, rates=rates)
    perm = [3, 0, 5, 1, 4, 2]
    many_p = fx.host_many([clips[p] for p in perm], rates=[rates[p] for p in perm])
    for j, p in enumerate(perm):
        for k in ALL + ("T",):
            assert np.array_equal(many_p[j][k], many[p][k]), (k, j)


@pytest.mark.gpu
def test_one_staging_launch_per_chunk_whatever_the_rates(cuda_device):
    """A one-chunk batch of mixed rates takes as many launches as the plan-rate call on the same clips resampled
    beforehand: the resampling adds no launch to the staging one."""
    fx = _fx("cfg1_16k")
    rates = [44100, 48000, 8000, 16000, 22050, 11025] * 6
    clips = [_clip(90 + i, int(r * (2 + 0.1 * i)), r, True) for i, r in enumerate(rates)]
    resampled = [np.ascontiguousarray(_solo_signal(fx, c, r)) for c, r in zip(clips, rates)]
    b_nat, o_nat = _packed(clips)
    b_res, o_res = _packed(resampled)
    counts = []
    for call in (lambda: fx.host_varlen(b_nat, o_nat, want=ALL, rates=rates),
                 lambda: fx.host_varlen(b_res, o_res, want=ALL)):
        call()  # warm-up (workspace growth)
        _lib.lib().mmf_launch_count(1)
        call()
        counts.append(_lib.lib().mmf_launch_count(1))
    assert counts[0] == counts[1], counts


def _solo_signal(fx, x, rate):
    up, down = resample_ratio(rate, fx.sr)
    y = fx.plan.pcm16_to_f32(x) if x.dtype == np.int16 else x
    y = fx.plan.resample_poly(y, up, down, "hq")
    return y.cpu().numpy() if hasattr(y, "cpu") else np.asarray(y, np.float32)


def _resample_varlen(plan, x_packed, offsets, rs, h, y_stride):
    torch = pytest.importorskip("torch")
    x = torch.as_tensor(x_packed).to(plan.device)
    y = torch.full((len(rs), y_stride), float("nan"), device=plan.device)
    offs = np.ascontiguousarray(offsets, np.int64)
    _lib.check(_lib.lib().mmf_resample_varlen(plan._h, x.data_ptr(), len(rs), offs.ctypes.data, rs.ctypes.data,
                                              h.ctypes.data if len(h) else None, len(h), y.data_ptr(), y_stride,
                                              int(torch.cuda.current_stream(plan.device).cuda_stream)))
    return y.cpu().numpy()


@pytest.mark.gpu
def test_resample_varlen_matches_resample_poly_and_upfirdn(cuda_device):
    """The resampling stage alone: each row bit for bit against Plan.resample_poly on the clip, and within 2e-6 of
    upfirdn in float64 with the same taps; a plan-rate clip is copied; the row past n_out is not written."""
    import scipy.signal

    plan = _fx("cfg1_16k").plan
    rates = [44100, 48000, 8000, 44056, 16000, 22050, 11025]
    clips = [_clip(110 + i, int(r * 0.9) + 3 * i, r, False) for i, r in enumerate(rates)]
    buf, offsets = _packed(clips)
    rs, h = resample_descriptors([len(c) for c in clips], rates, 16000)
    stride = int(rs["n_out"].max()) + 5
    y = _resample_varlen(plan, buf, offsets, rs, h, stride)
    for i, (c, r) in enumerate(zip(clips, rates)):
        n_out = int(rs[i]["n_out"])
        up, down = resample_ratio(r, 16000)
        ref = plan.resample_poly(c, up, down, "hq").cpu().numpy() if (up, down) != (1, 1) else c
        assert np.array_equal(y[i, :n_out], ref), i
        assert np.isnan(y[i, n_out:]).all(), i
        if (up, down) != (1, 1):
            taps, n_pre, _ = design_resample_filter(len(c), up, down, "hq")
            full = scipy.signal.upfirdn(taps.astype(np.float64), c.astype(np.float64), up, down)
            assert np.max(np.abs(y[i, :n_out] - full[n_pre : n_pre + n_out])) < 2e-6, i


def _write_wavs(tmp_path):
    from scipy.io import wavfile

    files = []
    for i, (rate, kind) in enumerate([(44100, "int16_stereo"), (48000, "float32_mono"), (8000, "int16_stereo"),
                                      (16000, "float32_mono"), (22050, "int16_mono")]):
        n = int(rate * (2.2 + 0.3 * i))
        a, b = synth_clip(200 + i, n, rate), synth_clip(300 + i, n, rate)
        if kind == "int16_stereo":
            data = np.stack([a, b], axis=1)
            data = np.clip(np.round(data * 32768.0), -32768, 32767).astype(np.int16)
        elif kind == "int16_mono":
            data = np.clip(np.round(a * 32768.0), -32768, 32767).astype(np.int16)
        else:
            data = a.astype(np.float32)
        p = str(tmp_path / f"f{i}.wav")
        wavfile.write(p, rate, data)
        files.append(p)
    return files


@pytest.mark.gpu
@pytest.mark.parametrize("channel", [0, 1])
def test_host_files_match_the_loader_and_get_mfccs_change(channel, cuda_device, tmp_path):
    sr = 16000
    fx = _fx("cfg1_16k")
    files = _write_wavs(tmp_path)
    many = fx.host_files(files, channel=channel)
    tot_only = fx.host_files(files, channel=channel, want=("totChange",))
    assert len(many) == len(files)
    for p, d, t in zip(files, many, tot_only):
        y = mm.api._read_audio(p, sr)
        y = y[channel] if y.ndim > 1 else y
        one = fx.host_call(np.ascontiguousarray(y)[None], want=ALL)
        for k in ALL:
            assert np.array_equal(d[k], one[k][0]), (p, k)
        tot, _ = mm.get_MFCCS_change(p, sr, channelN=channel, tStep=0.01, winLen=0.025, n_mfcc=13, n_fft=512,
                                     minFreq=0.0, maxFreq=8000.0, removeFirst=1, filtCutoff=12, filtOrd=6,
                                     diffMethod="grad", outFilter=None, n_mels=40)
        assert np.array_equal(t["totChange"], tot), p
    # the oracle on the device-resampled signal of the 44.1 kHz stereo file
    y = mm.api._read_audio(files[0], sr)[channel]
    ref = oracle.mfcc_features(y, sr)
    assert np.max(np.abs(many[0]["mfcc"] - ref["mfcc"])) < 1e-3


@pytest.mark.gpu
def test_host_files_rejects_what_is_not_a_wav(cuda_device, tmp_path):
    p = tmp_path / "not.wav"
    p.write_bytes(b"OggS" + bytes(100))
    with pytest.raises(ValueError, match="not.wav"):
        _fx("cfg1_16k").host_files([str(p)])


# ---- no GPU needed -------------------------------------------------------------------------------------------------


def test_resample_clip_layout_matches_the_library():
    assert _lib.lib().mmf_abi_sizeof(3) == RESAMPLE_CLIP.itemsize == C.sizeof(_lib.mmf_resample_clip)
    for name in RESAMPLE_CLIP.names:
        assert RESAMPLE_CLIP.fields[name][1] == getattr(_lib.mmf_resample_clip, name).offset, name


@pytest.mark.parametrize("sr_in, sr", [(44100, 16000), (48000, 16000), (8000, 16000), (22050, 10000),
                                       (11025, 10000), (44056, 16000), (16000, 16000), (16001, 16000), (96000, 44100)])
def test_ratio_helper_is_the_loaders_fraction(sr_in, sr):
    up, down = resample_ratio(sr_in, sr)
    if float(sr_in) == float(sr):
        assert (up, down) == (1, 1)
        return
    fr = Fraction(float(sr) / float(sr_in)).limit_denominator(1000)
    g = math.gcd(fr.numerator, fr.denominator)
    assert (up, down) == (fr.numerator // g, fr.denominator // g)
    assert math.gcd(up, down) == 1
    if (sr_in, sr) == (44056, 16000):
        assert (up, down) == (357, 983)


def test_rates_bookkeeping():
    """One table entry per distinct ratio; each clip's len_h, n_pre_remove and n_out are design_resample_filter's for
    its own length, its taps a prefix of its entry (the rest zeros); plan-rate clips are up = down = 1, n_out = len."""
    rates = [44100, 48000, 44100, 16000, 8000, 44100, 48000]
    lengths = [44100 * 2 + 17, 48000 + 5, 44100 * 3 + 1, 16000 * 2, 8000 * 3 + 3, 44100 + 440, 48000 * 2 + 1]
    rs, h = resample_descriptors(lengths, rates, 16000)
    ratios = {resample_ratio(r, 16000) for r in rates} - {(1, 1)}
    assert len({int(t) for t, (u, d) in zip(rs["tap0"], zip(rs["up"], rs["down"])) if (u, d) != (1, 1)}) == len(ratios)
    for i, (n, r) in enumerate(zip(lengths, rates)):
        up, down = resample_ratio(r, 16000)
        assert (int(rs[i]["up"]), int(rs[i]["down"])) == (up, down)
        if (up, down) == (1, 1):
            assert int(rs[i]["n_out"]) == n
            continue
        taps, n_pre, n_out = design_resample_filter(n, up, down, "hq")
        t0, L = int(rs[i]["tap0"]), int(rs[i]["len_h"])
        assert (L, int(rs[i]["n_pre_remove"]), int(rs[i]["n_out"])) == (len(taps), n_pre, n_out)
        assert np.array_equal(h[t0 : t0 + L], taps)
    # sizes of the prefix sums of n_out are the frames and windows at the plan's rate
    cfg = mm.MfccConfig(16000, 512, 400, 160, 40, 13, 0.0, 8000.0)
    offs = np.concatenate([[0], np.cumsum(rs["n_out"])]).astype(np.int64)
    fo, wo = np.zeros(len(rs) + 1, np.int64), np.zeros(len(rs) + 1, np.int64)
    assert _lib.lib().mmf_features_varlen_sizes(C.byref(cfg.to_c()), None, len(rs), offs.ctypes.data, fo.ctypes.data,
                                                wo.ctypes.data) == 0
    assert list(np.diff(fo)) == [mm.num_frames(int(n), 512, 160) for n in rs["n_out"]]


def _rs(*clips):
    rs = np.zeros(len(clips), RESAMPLE_CLIP)
    for i, c in enumerate(clips):
        for k, v in c.items():
            rs[i][k] = v
    return rs


GOOD = dict(up=160, down=441, tap0=0, len_h=100, n_pre_remove=3, n_out=-(-1000 * 160 // 441))
SAME = dict(up=1, down=1, n_out=1000)


@pytest.mark.parametrize(
    "bad, what",
    [
        (dict(GOOD, up=0), "up and down"),
        (dict(GOOD, down=-1), "up and down"),
        (dict(GOOD, n_out=GOOD["n_out"] + 1), "ceil(len * up / down)"),
        (dict(SAME, n_out=999), "plan's rate"),
        (dict(GOOD, tap0=60), "tap table"),
        (dict(GOOD, tap0=-1), "tap table"),
        (dict(GOOD, len_h=0), "len_h"),
        (dict(GOOD, n_pre_remove=-2), "n_pre_remove"),
    ],
)
def test_bad_descriptors_fail_before_any_plan_or_device(bad, what):
    lib = _lib.lib()
    offsets = np.array([0, 1000, 2000, 3000], np.int64)
    h = np.zeros(150, np.float32)
    p = _lib.mmf_change_params()
    tot = np.zeros(8, np.float64)
    for j in range(3):
        clips = [GOOD, SAME, GOOD]
        clips[j] = bad
        rs = _rs(*clips)
        rc = lib.mmf_features_host_varlen_resampled(None, None, 1, 3, offsets.ctypes.data, rs.ctypes.data,
                                                    h.ctypes.data, len(h), C.byref(p), None, tot.ctypes.data, None,
                                                    None, None, None)
        msg = lib.mmf_last_error().decode()
        assert rc == _lib.MMF_ERR_INVALID and f"clip {j}:" in msg and what in msg, msg
        rc = lib.mmf_resample_varlen(None, None, 3, offsets.ctypes.data, rs.ctypes.data, h.ctypes.data, len(h), None,
                                     2000, None)
        msg = lib.mmf_last_error().decode()
        assert rc == _lib.MMF_ERR_INVALID and f"clip {j}:" in msg and what in msg, msg
    # valid descriptors, no plan: the NULL plan is reported only after they passed; bad offsets come first
    rs = _rs(GOOD, SAME, GOOD)
    rc = lib.mmf_features_host_varlen_resampled(None, None, 0, 3, offsets.ctypes.data, rs.ctypes.data, h.ctypes.data,
                                                len(h), C.byref(p), None, tot.ctypes.data, None, None, None, None)
    assert rc == _lib.MMF_ERR_INVALID and "NULL argument" in lib.mmf_last_error().decode()
    bad_offsets = np.array([0, 1000, 900, 3000], np.int64)
    rc = lib.mmf_resample_varlen(None, None, 3, bad_offsets.ctypes.data, rs.ctypes.data, h.ctypes.data, len(h), None,
                                 2000, None)
    assert rc == _lib.MMF_ERR_INVALID and "clip 1" in lib.mmf_last_error().decode()
    # a plan-rate-only batch needs no taps
    rs = _rs(SAME, SAME, SAME)
    rc = lib.mmf_resample_varlen(None, None, 3, offsets.ctypes.data, rs.ctypes.data, None, 0, None, 2000, None)
    assert rc == _lib.MMF_ERR_INVALID and "NULL argument" in lib.mmf_last_error().decode()
