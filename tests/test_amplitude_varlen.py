"""The RMS amplitude envelope of packed clips (rms_varlen_kernel): mmf_rms, mmf_rms_varlen, mmf_amp_varlen_sizes,
mmf_features_host_varlen_amp, Plan.rms_varlen, FeatureExtractor(want=(..., "amplitude")) and
calculate_amplitude_envelope_many.

The contract: clip i's envelope block is bit-identical to
    calculate_amplitude_envelope(x_i, rate_i, winLen, hopLen, center, outFilter=None | 'iir')
on that clip alone, x_i its native samples as float32 (int16: x * (1/32768), as pcm16_to_f32_kernel scales it) and
rate_i its own rate, whatever chunk it lands in and whoever its neighbours are.
"""

import ctypes as C
import os

import numpy as np
import pytest

import modulation_mfcc_b200 as mm
from modulation_mfcc_b200 import _lib
from modulation_mfcc_b200.plan import amp_sizes, make_amp_params, resample_descriptors
from modulation_mfcc_b200.synth import synth_clip

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "rms_bits.npz")
ALL = ("totChange", "mfcc", "delta", "modspec", "band_energy")


def _fx(sr=16000, **amp):
    return mm.FeatureExtractor(sr, tStep=0.01, winLen=0.025, n_fft=512, n_mels=40, n_mfcc=13, fmin=0.0,
                               fmax=sr / 2, **amp)


def _clip(seed, n, rate, pcm16):
    c = synth_clip(seed, n, rate).astype(np.float32)
    return np.clip(np.round(c * 32768.0), -32768, 32767).astype(np.int16) if pcm16 else c


def _as_f32(x):
    """The clip as the device sees it: int16 scaled by 1/32768 (an exact power of two) in float32."""
    return x.astype(np.float32) * np.float32(1.0 / 32768.0) if x.dtype == np.int16 else x


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


def _amp_kw(fx, filt):
    kw = dict(winLen=fx.amp_winLen, hopLen=fx.amp_hopLen, center=fx.amp_center)
    return dict(kw, outFilter="iir", outFiltCutOff=[12], outFiltLen=6, outFiltType="low") if filt else kw


def _solo(fx, x, rate, filt):
    return mm.calculate_amplitude_envelope(_as_f32(x), rate, **_amp_kw(fx, filt))


def _block(res, i):
    a0, a1 = int(res["amp_offsets"][i]), int(res["amp_offsets"][i + 1])
    return res["amplitude"][a0:a1]


def _amp_fx(filt, sr=16000, **kw):
    return _fx(sr, amp_outFilter="iir" if filt else None, **kw)


# ---- GPU -----------------------------------------------------------------------------------------------------------


@pytest.mark.gpu
@pytest.mark.parametrize("pcm16", [False, True])
@pytest.mark.parametrize("filt", [False, True])
@pytest.mark.parametrize("center", [True, False])
@pytest.mark.parametrize("mode", ["plan_rate", "rates"])
def test_bundle_envelope_matches_the_single_call(mode, center, filt, pcm16, cuda_device):
    """Each clip's envelope equals calculate_amplitude_envelope on that clip at its own rate, bit for bit: raw and
    'iir', float32 and int16, plan-rate clips (even frame_length 1600 and odd 401) and 44.1, 48, 22.05, 8 and
    44.056 kHz clips (frame_length 4410, 4800, 2205, 800 and 4405)."""
    if mode == "plan_rate":
        cases = [(_amp_fx(filt, amp_center=center), None), (_amp_fx(filt, amp_center=center, amp_winLen=0.0251), None)]
        rates = [16000] * 7
    else:
        cases = [(_amp_fx(filt, amp_center=center), True)]
        rates = [44100, 48000, 22050, 8000, 44056, 16000, 44100]
    lengths = [int(r * (1.1 + 0.43 * i)) + 3 * i for i, r in enumerate(rates)]
    clips = [_clip(40 + i, n, r, pcm16) for i, (n, r) in enumerate(zip(lengths, rates))]
    buf, offsets = _packed(clips)
    for fx, with_rates in cases:
        res = fx.host_varlen(buf, offsets, want=("totChange", "amplitude"), rates=rates if with_rates else None)
        assert res["amplitude"].dtype == (np.float64 if filt else np.float32)
        for i, (c, r) in enumerate(zip(clips, rates)):
            amp, ampT = _solo(fx, c, r, filt)
            assert np.array_equal(_block(res, i), amp), (i, r)
            assert len(ampT) == len(amp)


@pytest.mark.gpu
@pytest.mark.parametrize("filt", [False, True])
def test_frames_over_the_shared_memory_span(filt, cuda_device):
    """winLen = 1 s at 48 and 44.1 kHz: frames longer than the staged span are read from global memory in the same
    order, and still equal the single call."""
    fx = _amp_fx(filt, amp_winLen=1.0)
    rates = [48000, 44100, 16000]
    clips = [_clip(60 + i, int(r * 3.3) + i, r, False) for i, r in enumerate(rates)]
    buf, offsets = _packed(clips)
    res = fx.host_varlen(buf, offsets, want=("totChange", "amplitude"), rates=rates)
    for i, (c, r) in enumerate(zip(clips, rates)):
        assert np.array_equal(_block(res, i), _solo(fx, c, r, filt)[0]), i
    amp, off = fx.plan.rms_varlen(buf, offsets, [(48000, 480), (44100, 441), (16000, 160)], True)
    for i, c in enumerate(clips):
        one = mm.calculate_amplitude_envelope(c, rates[i], winLen=1.0)[0]
        assert np.array_equal(amp[off[i] : off[i + 1]].cpu().numpy(), one), i


@pytest.mark.gpu
@pytest.mark.parametrize("filt", [False, True])
def test_raw_int16_relation(filt, cuda_device):
    """The GUI passes raw int16 (main.py:843-849): the bundle's envelope of an int16 clip times 32768 equals
    calculate_amplitude_envelope of the raw samples, bit for bit (a power-of-two scale is exact through fmaf, the
    division, sqrtf and the float64 filter)."""
    fx = _amp_fx(filt)
    rates = [44100, 16000, 22050]
    clips = [_clip(80 + i, int(r * (2 + 0.5 * i)), r, True) for i, r in enumerate(rates)]
    buf, offsets = _packed(clips)
    res = fx.host_varlen(buf, offsets, want=("totChange", "amplitude"), rates=rates)
    for i, (c, r) in enumerate(zip(clips, rates)):
        raw = mm.calculate_amplitude_envelope(c, r, **_amp_kw(fx, filt))[0]
        assert np.array_equal(_block(res, i) * 32768, raw), i


@pytest.mark.gpu
@pytest.mark.parametrize("pcm16", [False, True])
def test_poison_never_reaches_an_output(pcm16, cuda_device):
    """Poison (NaN / 32767) before the first clip, after the last and as a whole clip between two others: every
    other clip's envelope equals its single call."""
    fx = _amp_fx(True)
    poison = np.full(5000, 32767 if pcm16 else np.nan, np.int16 if pcm16 else np.float32)
    clips = [_clip(90, 17001, 16000, pcm16), poison, _clip(91, 23456, 16000, pcm16), poison.copy(),
             _clip(92, 16000, 16000, pcm16)]
    buf, offsets = _packed(clips, lead=4801, tail=4801)
    for filt in (False, True):
        fx = _amp_fx(filt)
        res = fx.host_varlen(buf, offsets, want=("totChange", "amplitude"))
        for i in (0, 2, 4):
            got = _block(res, i)
            assert np.isfinite(got).all(), i
            assert np.array_equal(got, _solo(fx, clips[i], 16000, filt)[0]), i


@pytest.mark.gpu
def test_long_clip_over_several_chunks(cuda_device):
    """A 187.5 s clip at 48 kHz forms a chunk alone among chunks of short clips; its 18 750-frame envelope takes the
    long-row filter route, the short ones the chunk-parallel kernel.  Every envelope equals its single call, and the
    MFCC-side outputs are byte-identical to the call without the envelope."""
    fx = _amp_fx(True)
    rates = [44100, 16000, 8000] * 3 + [48000] + [22050, 16000, 44100] * 3
    len_in = [int(r * 2.1) + 7 * i for i, r in enumerate(rates)]
    len_in[9] = 9_000_000
    clips = [_clip(50 + i, n, r, False) for i, (n, r) in enumerate(zip(len_in, rates))]
    buf, offsets = _packed(clips)
    res = fx.host_varlen(buf, offsets, want=ALL + ("amplitude",), rates=rates)
    ref = fx.host_varlen(buf, offsets, want=ALL, rates=rates)
    for k in ALL:
        assert res[k].tobytes() == ref[k].tobytes(), k
    assert int(res["amp_offsets"][10] - res["amp_offsets"][9]) == 18751
    for i, (c, r) in enumerate(zip(clips, rates)):
        assert np.array_equal(_block(res, i), _solo(fx, c, r, True)[0]), (i, r)


@pytest.mark.gpu
def test_permuting_the_clips_permutes_the_blocks(cuda_device):
    fx = _amp_fx(True)
    rates = [44100, 48000, 8000, 16000, 44056, 22050]
    clips = [_clip(70 + i, int(r * (1.5 + 0.2 * i)), r, True) for i, r in enumerate(rates)]
    want = ALL + ("amplitude",)
    many = fx.host_many(clips, want=want, rates=rates)
    perm = [3, 0, 5, 1, 4, 2]
    many_p = fx.host_many([clips[p] for p in perm], want=want, rates=[rates[p] for p in perm])
    for j, p in enumerate(perm):
        for k in want + ("T", "ampT"):
            assert np.array_equal(many_p[j][k], many[p][k]), (k, j)


def _call_amp(fx, buf, offsets, rs, h, amp, geom, outs):
    """mmf_features_host_varlen_amp with explicit buffers; returns the launch count of the call."""
    p = fx.plan
    mp = mm.plan._modspec_params(fx.modspec_geometry(0))
    _lib.lib().mmf_launch_count(1)
    _lib.check(_lib.lib().mmf_features_host_varlen_amp(
        p._h, buf.ctypes.data, 1 if buf.dtype == np.int16 else 0, len(offsets) - 1, offsets.ctypes.data,
        rs.ctypes.data if rs is not None else None, h.ctypes.data if h is not None and len(h) else None,
        len(h) if h is not None else 0, C.byref(fx.prm), C.byref(mp), C.byref(amp) if amp is not None else None,
        geom.ctypes.data if geom is not None else None, *[o.ctypes.data if o is not None else None for o in outs]))
    return _lib.lib().mmf_launch_count(1)


def _outs(fx, offsets, rs, amp_off, filt):
    B = len(offsets) - 1
    fo, wo = np.zeros(B + 1, np.int64), np.zeros(B + 1, np.int64)
    mp = mm.plan._modspec_params(fx.modspec_geometry(0))
    out_offs = np.concatenate([[0], np.cumsum(rs["n_out"])]).astype(np.int64)
    _lib.check(_lib.lib().mmf_features_varlen_sizes(C.byref(fx.plan.cfg.to_c()), C.byref(mp), B, out_offs.ctypes.data,
                                                    fo.ctypes.data, wo.ctypes.data))
    nm, nb, n_bands = 13, mp.nfft // 2 + 1, mp.n_bands
    F, W = int(fo[-1]), int(wo[-1])
    outs = [np.full(F, 7.0), np.full(nm * F, 7.0, np.float32), np.full(nm * F, 7.0, np.float32),
            np.full(nm * W * nb, 7.0, np.float32), np.full(W * n_bands, 7.0, np.float32)]
    if amp_off is None:
        return outs + [None, None]
    A = int(amp_off[-1])
    return outs + [None if filt else np.full(A, 7.0, np.float32), np.full(A, 7.0) if filt else None]


@pytest.mark.gpu
def test_launches_without_and_with_the_envelope(cuda_device):
    """amp = NULL queues exactly what mmf_features_host_varlen_resampled queues, with byte-identical outputs; with
    the envelope (raw or filtered), a chunk takes a fixed number of extra launches whatever its clip count."""
    fx = _amp_fx(True)
    mp = mm.plan._modspec_params(fx.modspec_geometry(0))
    extra = {}
    for n in (6, 24):
        rates = [44100, 48000, 8000, 16000, 22050, 11025] * (n // 6)
        clips = [_clip(100 + i, int(r * (2 + 0.1 * i)), r, True) for i, r in enumerate(rates)]
        buf, offsets = _packed(clips)
        rs, h = resample_descriptors(np.diff(offsets), rates, fx.sr)
        geom = np.ascontiguousarray([(int(0.1 * r), int(0.01 * r)) for r in rates], np.int32)
        _, _, amp_off = amp_sizes(offsets, geom, True)
        ref = _outs(fx, offsets, rs, None, False)
        _lib.lib().mmf_launch_count(1)
        for _ in range(2):  # (the second call after the workspace has grown)
            _lib.lib().mmf_launch_count(1)
            _lib.check(_lib.lib().mmf_features_host_varlen_resampled(
                fx.plan._h, buf.ctypes.data, 1, n, offsets.ctypes.data, rs.ctypes.data, h.ctypes.data, len(h),
                C.byref(fx.prm), C.byref(mp), *[o.ctypes.data for o in ref[:5]]))
            base = _lib.lib().mmf_launch_count(1)
        got = _outs(fx, offsets, rs, None, False)
        assert _call_amp(fx, buf, offsets, rs, h, None, None, got) == base
        for a, b in zip(ref[:5], got[:5]):
            assert a.tobytes() == b.tobytes()
        for filt in (False, True):
            amp = make_amp_params(True, fx.amp_sos if filt else None)
            outs = _outs(fx, offsets, rs, amp_off, filt)
            extra[(n, filt)] = _call_amp(fx, buf, offsets, rs, h, amp, geom, outs) - base
            for a, b in zip(ref[:5], outs[:5]):
                assert a.tobytes() == b.tobytes()
    assert extra[(6, False)] == extra[(24, False)] == 1, extra
    assert extra[(6, True)] == extra[(24, True)] == 2, extra


@pytest.mark.gpu
def test_mmf_rms_reproduces_the_previous_kernel(cuda_device):
    """tests/golden/rms_bits.npz holds inputs and the outputs of the previous one-warp-per-frame mmf_rms kernel: center
    on and off, odd and even frame_length, a clip shorter than its frame, loud int16-range values and a frame over the
    staged span."""
    g = np.load(GOLDEN)
    plan = _fx().plan
    n_cases = int(g["n_cases"])
    assert n_cases >= 5
    for k in range(n_cases):
        x = g[f"x{k}"]
        fl, hop, center = (int(v) for v in g[f"p{k}"])
        got = plan.rms(x, fl, hop, bool(center)).cpu().numpy()
        assert got.tobytes() == g[f"y{k}"].tobytes(), k


@pytest.mark.gpu
def test_rms_varlen_equals_per_row_rms(cuda_device):
    plan = _fx().plan
    rng = np.random.default_rng(5)
    lengths = [1, 50, 399, 400, 401, 16000, 44101, 7]
    geom = [(400, 160), (33, 7), (400, 160), (401, 100), (1600, 160), (441, 147), (4410, 441), (8, 1)]
    clips = [rng.standard_normal(n).astype(np.float32) for n in lengths]
    buf, offsets = _packed(clips)
    for center in (True, False):
        keep = [i for i, n in enumerate(lengths) if center or n >= geom[i][0]]
        sub = [clips[i] for i in keep]
        b, o = _packed(sub)
        amp, off = plan.rms_varlen(b, o, [geom[i] for i in keep], center)
        amp = amp.cpu().numpy()
        for j, i in enumerate(keep):
            one = plan.rms(clips[i], geom[i][0], geom[i][1], center).cpu().numpy()[0]
            assert np.array_equal(amp[off[j] : off[j + 1]], one), (center, i)
    assert len(buf) == offsets[-1] + 5


@pytest.mark.gpu
@pytest.mark.parametrize("filt", [None, "iir", "fir"])
def test_many_clips_equal_the_single_call(filt, cuda_device):
    rates = [44100, 16000, 8000, 22050]
    clips = [_clip(120 + i, int(r * (1.2 + 0.3 * i)), r, False) for i, r in enumerate(rates)]
    kw = dict(outFilter=filt, outFiltCutOff=[12]) if filt else {}
    many = mm.calculate_amplitude_envelope_many(clips, rates, **kw)
    for (amp, ampT), c, r in zip(many, clips, rates):
        one, oneT = mm.calculate_amplitude_envelope(c, r, **kw)
        assert np.array_equal(amp, one) and np.array_equal(ampT, oneT), r
    one_rate = mm.calculate_amplitude_envelope_many(clips, 16000)
    for (amp, _), c in zip(one_rate, clips):
        assert np.array_equal(amp, mm.calculate_amplitude_envelope(c, 16000)[0])


def _write_wavs(tmp_path):
    from scipy.io import wavfile

    files = []
    for i, (rate, kind) in enumerate([(44100, "int16_stereo"), (48000, "float32_mono"), (8000, "int16_mono"),
                                      (16000, "float32_mono")]):
        n = int(rate * (2.2 + 0.3 * i))
        a, b = synth_clip(200 + i, n, rate), synth_clip(300 + i, n, rate)
        if kind == "int16_stereo":
            data = np.clip(np.round(np.stack([a, b], axis=1) * 32768.0), -32768, 32767).astype(np.int16)
        elif kind == "int16_mono":
            data = np.clip(np.round(a * 32768.0), -32768, 32767).astype(np.int16)
        else:
            data = a.astype(np.float32)
        p = str(tmp_path / f"f{i}.wav")
        wavfile.write(p, rate, data)
        files.append(p)
    return files


@pytest.mark.gpu
@pytest.mark.parametrize("filt", [False, True])
def test_host_files_match_the_gui_envelope(filt, cuda_device, tmp_path):
    """host_files' envelope of each file equals calculate_amplitude_envelope(wavfile data of the channel, file_sr):
    float files directly, 16-bit files times 32768 (the GUI passes raw int16).  Mixed int16 / float corpora and all
    int16 corpora both hold."""
    from scipy.io import wavfile

    fx = _amp_fx(filt)
    files = _write_wavs(tmp_path)
    for group in (files, [files[0], files[2]]):
        many = fx.host_files(group, channel=0, want=("totChange", "amplitude"))
        for p, d in zip(group, many):
            file_sr, data = wavfile.read(p)
            x = data[:, 0] if data.ndim > 1 else data
            ref, refT = mm.calculate_amplitude_envelope(np.ascontiguousarray(x), file_sr, **_amp_kw(fx, filt))
            got = d["amplitude"] * 32768 if x.dtype == np.int16 else d["amplitude"]
            assert np.array_equal(got, ref), p
            assert np.array_equal(d["ampT"], refT), p


# ---- no GPU needed -------------------------------------------------------------------------------------------------


def test_amp_params_layout_matches_the_library():
    assert _lib.lib().mmf_abi_sizeof(4) == C.sizeof(_lib.mmf_amp_params)
    for name, off in (("center", 0), ("out_n_sections", 4), ("out_sos", 8)):
        assert getattr(_lib.mmf_amp_params, name).offset == off, name


@pytest.mark.parametrize("center", [True, False])
def test_sizes_follow_the_reference_formula(center):
    rates = [44100, 48000, 22050, 8000, 44056, 16000]
    lengths = [44100 * 2 + 17, 4800, 2205, 800 * 3 + 1, 44056 + 440, 16000 * 5]
    offsets = np.concatenate([[11], 11 + np.cumsum(lengths)]).astype(np.int64)
    geom = [(int(0.1 * r), int(0.01 * r)) for r in rates]
    _, g, amp_off = amp_sizes(offsets, geom, center)
    assert g.dtype == np.int32 and g.shape == (6, 2)
    for i, (n, (fl, hop)) in enumerate(zip(lengths, geom)):
        pad = fl // 2 if center else 0
        assert amp_off[i + 1] - amp_off[i] == 1 + (n + 2 * pad - fl) // hop, i  # calc.py:326-331


def _sizes_rc(offsets, geom, center):
    lib = _lib.lib()
    offsets = np.ascontiguousarray(offsets, np.int64)
    geom = np.ascontiguousarray(geom, np.int32)
    amp_off = np.zeros(len(offsets), np.int64)
    rcs = [lib.mmf_amp_varlen_sizes(len(offsets) - 1, offsets.ctypes.data, geom.ctypes.data, center,
                                    amp_off.ctypes.data)]
    msgs = [lib.mmf_last_error().decode()]
    rcs.append(lib.mmf_rms_varlen(None, None, len(offsets) - 1, offsets.ctypes.data, geom.ctypes.data, center, None,
                                  None))
    msgs.append(lib.mmf_last_error().decode())
    amp = make_amp_params(center)
    tot = np.zeros(8)
    a = np.zeros(8, np.float32)
    rcs.append(lib.mmf_features_host_varlen_amp(None, None, 0, len(offsets) - 1, offsets.ctypes.data, None, None, 0,
                                                C.byref(_lib.mmf_change_params()), None, C.byref(amp),
                                                geom.ctypes.data, tot.ctypes.data, None, None, None, None,
                                                a.ctypes.data, None))
    msgs.append(lib.mmf_last_error().decode())
    return rcs, msgs


@pytest.mark.parametrize(
    "bad, center, code, what",
    [
        ((0, 160), 1, _lib.MMF_ERR_INVALID, "frame_length"),
        ((400, 0), 1, _lib.MMF_ERR_INVALID, "hop"),
        ((-3, 10), 0, _lib.MMF_ERR_INVALID, "frame_length"),
        ((1001, 10), 0, _lib.MMF_ERR_TOO_SHORT, "Input is too short"),
    ],
)
def test_bad_geometry_fails_naming_the_clip_before_any_plan_or_device(bad, center, code, what):
    offsets = [0, 1000, 2000, 3000]
    for j in range(3):
        geom = [(400, 160)] * 3
        geom[j] = bad
        rcs, msgs = _sizes_rc(offsets, geom, center)
        for rc, msg in zip(rcs, msgs):
            assert rc == code and f"clip {j}:" in msg and what in msg, msg


def test_other_checks_before_any_plan_or_device():
    lib = _lib.lib()
    # bad offsets come first, named by clip
    rcs, msgs = _sizes_rc([0, 1000, 900, 3000], [(400, 160)] * 3, 1)
    assert all(rc == _lib.MMF_ERR_INVALID and "clip 1" in m for rc, m in zip(rcs, msgs)), msgs
    # good geometry: the NULL plan is reported only after it passed; center lets a clip be shorter than its frame
    rcs, msgs = _sizes_rc([0, 1000, 1300, 3000], [(400, 160), (1001, 10), (400, 160)], 1)
    assert rcs[0] == 0
    assert all(rc == _lib.MMF_ERR_INVALID and "NULL argument" in m for rc, m in zip(rcs[1:], msgs[1:])), msgs
    # a filtered envelope of at most padlen frames fails naming the clip
    sos = mm.api._design_iir(100.0, [12], 6, "low")
    padlen = mm.sos_zi(sos)[1]
    offsets = np.array([0, 16000, 16000 + 160 * (padlen - 1), 40000], np.int64)  # clip 1: padlen frames (center)
    geom = np.array([(1600, 160), (1600, 160), (1600, 160)], np.int32)
    assert int(np.diff(amp_sizes(offsets, geom, True)[2])[1]) == padlen
    amp = make_amp_params(True, sos)
    f = np.zeros(8)
    rc = lib.mmf_features_host_varlen_amp(None, None, 0, 3, offsets.ctypes.data, None, None, 0,
                                          C.byref(_lib.mmf_change_params()), None, C.byref(amp), geom.ctypes.data,
                                          f.ctypes.data, None, None, None, None, None, f.ctypes.data)
    msg = lib.mmf_last_error().decode()
    assert rc == _lib.MMF_ERR_TOO_SHORT and "clip 1:" in msg and f"padlen, which is {padlen}" in msg, msg
    # filtered output without a filter; amplitude outputs without parameters
    rc = lib.mmf_features_host_varlen_amp(None, None, 0, 3, offsets.ctypes.data, None, None, 0,
                                          C.byref(_lib.mmf_change_params()), None, C.byref(make_amp_params(True)),
                                          geom.ctypes.data, f.ctypes.data, None, None, None, None, None, f.ctypes.data)
    assert rc == _lib.MMF_ERR_INVALID and "out_n_sections" in lib.mmf_last_error().decode()
    rc = lib.mmf_features_host_varlen_amp(None, None, 0, 3, offsets.ctypes.data, None, None, 0,
                                          C.byref(_lib.mmf_change_params()), None, None, geom.ctypes.data,
                                          f.ctypes.data, None, None, None, None, f.ctypes.data, None)
    assert rc == _lib.MMF_ERR_INVALID and "without parameters" in lib.mmf_last_error().decode()


def _raised(fn):
    try:
        fn()
    except Exception as e:  # noqa: BLE001 -- the reference raises bare Exception
        return type(e), str(e)
    return None


@pytest.mark.parametrize(
    "kw",
    [
        dict(amp_outFiltCutOff=[60]),
        dict(amp_outFiltCutOff=[20, 10], amp_outFiltType="band"),
        dict(amp_outFiltType="notch"),
        dict(amp_outFiltCutOff=[5, 10], amp_outFiltType="low"),
        dict(amp_outFiltCutOff=None),
    ],
)
def test_feature_extractor_validates_the_envelope_filter_as_apply_filter_does(kw):
    """The 'iir' envelope filter is validated at construction, before any device work, with the exception the
    single call's applyFilter raises for the same arguments."""
    args = dict(amp_outFiltCutOff=[12], amp_outFiltLen=6, amp_outFiltType="low") | kw
    got = _raised(lambda: _fx(amp_outFilter="iir", **args))
    want = _raised(lambda: mm.api._design_iir(100.0, args["amp_outFiltCutOff"], args["amp_outFiltLen"],
                                              args["amp_outFiltType"]))
    assert want is not None and got == want, (got, want)


@pytest.mark.parametrize("filt", ["fir", "sg"])
def test_feature_extractor_takes_only_none_or_iir(filt):
    with pytest.raises(ValueError, match="None or 'iir'"):
        _fx(amp_outFilter=filt)
