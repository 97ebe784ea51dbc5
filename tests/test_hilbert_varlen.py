"""The Hilbert envelope ('Hilb', script/calc.py:284-286) of packed clips: mmf_hilbert_envelope on the batched
Bluestein kernels, mmf_hilbert_varlen, mmf_env_varlen_sizes, mmf_features_host_varlen_env, Plan.hilbert_varlen,
calculate_amplitude_envelope_many(method='Hilb') and FeatureExtractor(amp_method='Hilb').

The contract: clip i's envelope is bit-identical to mmf_hilbert_envelope on that clip alone (whose bytes
tests/golden/hilbert_bits.npz pins), then, with an output filter, to mmf_sosfiltfilt on that envelope, whatever batch,
sub-batch or chunk the clip lands in.
"""

import ctypes as C
import hashlib
import os

import numpy as np
import pytest
import scipy.signal

import modulation_mfcc_b200 as mm
from modulation_mfcc_b200 import _lib
from modulation_mfcc_b200.plan import env_sizes, make_env_params
from modulation_mfcc_b200.synth import synth_clip

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "hilbert_bits.npz")
ALL = ("totChange", "mfcc", "delta", "modspec", "band_energy")


def _fx(sr=16000, **kw):
    return mm.FeatureExtractor(sr, tStep=0.01, winLen=0.025, n_fft=512, n_mels=40, n_mfcc=13, fmin=0.0, fmax=sr / 2,
                               amp_method="Hilb", **kw)


def _clip(seed, n, rate, pcm16):
    c = synth_clip(seed, n, rate).astype(np.float32)
    return np.clip(np.round(c * 32768.0), -32768, 32767).astype(np.int16) if pcm16 else c


def _as_f32(x):
    return x.astype(np.float32) * np.float32(1.0 / 32768.0) if x.dtype == np.int16 else x


def _packed(clips, lead=3, tail=5):
    """Clips back to back after `lead` poison samples (NaN / 32767), `tail` more after the last."""
    poison = np.nan if clips[0].dtype == np.float32 else 32767
    buf = np.full(lead + sum(len(c) for c in clips) + tail, poison, clips[0].dtype)
    offsets = np.zeros(len(clips) + 1, np.int64)
    offsets[0] = lead
    for i, c in enumerate(clips):
        offsets[i + 1] = offsets[i] + len(c)
        buf[offsets[i] : offsets[i + 1]] = c
    return buf, offsets


def _ragged_lengths(seed=7, n=64):
    rng = np.random.default_rng(seed)
    lengths = [int(v) for v in rng.integers(1, 300_001, n - 16)]
    lengths += [1, 2, 17, 4095, 4096, 4097, 4099, 65537, 100003, 160000, 160000, 4097, 5000, 5000, 262144, 262145]
    rng.shuffle(lengths)
    return lengths


def _solo(plan, c):
    return plan.hilbert_envelope(c).cpu().numpy()


# ---- GPU -----------------------------------------------------------------------------------------------------------


@pytest.mark.gpu
def test_single_call_reproduces_the_previous_kernels(cuda_device):
    """hilbert_bits.npz holds SHA-256 digests of mmf_hilbert_envelope outputs from the one-launch-per-pass kernels:
    even, odd and prime n, powers of two, 4097, batches of several rows, both sides of the two / three pass-group
    boundary and lengths up to 2^26."""
    g = np.load(GOLDEN)
    plan = _fx().plan
    sr = int(g["sr"])
    assert len(g["cases"]) >= 15
    for (seed, n, n_clips), want in zip(g["cases"], g["sha256"]):
        x = np.stack([synth_clip(int(seed) + i, int(n), sr) for i in range(int(n_clips))])
        got = plan.hilbert_envelope(x).cpu().numpy()
        assert hashlib.sha256(got.tobytes()).hexdigest().encode() == want, (seed, n, n_clips)


@pytest.mark.gpu
def test_ragged_equals_solo_and_scipy(cuda_device):
    """64 packed clips of 1 .. 300 000 samples (short ones on the direct route, primes, repeated lengths): every
    block equals the single call on the clip alone, and lies within 2e-6 of scipy; NaN poison around the clips
    never reaches an output.  Permuting the clips permutes the blocks, and splitting them across calls changes
    nothing."""
    plan = _fx().plan
    lengths = _ragged_lengths()
    clips = [_clip(500 + i, n, 16000, False) for i, n in enumerate(lengths)]
    buf, offsets = _packed(clips, lead=4097, tail=4099)
    amp, off = plan.hilbert_varlen(buf, offsets)
    amp = amp.cpu().numpy()
    assert np.array_equal(off, offsets - offsets[0])
    solo = [_solo(plan, c) for c in clips]
    for i, c in enumerate(clips):
        blk = amp[off[i] : off[i + 1]]
        assert np.isfinite(blk).all(), i
        assert blk.tobytes() == solo[i].tobytes(), (i, len(c))
        ref = np.abs(scipy.signal.hilbert(c.astype(np.float64)))
        assert np.max(np.abs(blk - ref)) < (2e-6 if len(c) > 4096 else 1e-4), (i, len(c))
    perm = np.random.default_rng(3).permutation(len(clips))
    b2, o2 = _packed([clips[p] for p in perm])
    a2, f2 = plan.hilbert_varlen(b2, o2)
    a2 = a2.cpu().numpy()
    for j, p in enumerate(perm):
        assert a2[f2[j] : f2[j + 1]].tobytes() == solo[p].tobytes(), (j, p)
    for part in (slice(0, 20), slice(20, 21), slice(21, None)):
        b3, o3 = _packed(clips[part])
        a3, f3 = plan.hilbert_varlen(b3, o3)
        a3 = a3.cpu().numpy()
        for j, i in enumerate(range(len(clips))[part]):
            assert a3[f3[j] : f3[j + 1]].tobytes() == solo[i].tobytes(), i


@pytest.mark.gpu
def test_several_sub_batches(cuda_device):
    """40 clips of about a million samples (M = 2^21, 64 MB of work buffers each) need more scratch than one
    sub-batch holds: every block still equals the single call."""
    plan = _fx().plan
    lengths = [1_000_003 + 17 * i for i in range(40)]
    clips = [_clip(900 + i, n, 16000, False) for i, n in enumerate(lengths)]
    buf, offsets = _packed(clips)
    amp, off = plan.hilbert_varlen(buf, offsets)
    amp = amp.cpu().numpy()
    for i, c in enumerate(clips):
        assert amp[off[i] : off[i + 1]].tobytes() == _solo(plan, c).tobytes(), i


@pytest.mark.gpu
def test_launch_count_does_not_grow_with_the_clips(cuda_device):
    """A ragged call over clips of more than 4096 samples: the same launches for 8 and for 512 clips, at most the
    chirp and twiddle tables plus 5 transforms x 3 pass groups."""
    plan = _fx().plan
    counts = []
    for B in (8, 512):
        rng = np.random.default_rng(B)
        lengths = [int(v) for v in rng.integers(4097, 8193, B)]  # (512 of them fit one sub-batch)
        lengths[0] = (1 << 21) + 1  # one three-group clip in each
        x = np.concatenate([_clip(i, n, 16000, False) for i, n in enumerate(lengths)])
        offsets = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
        plan.hilbert_varlen(x, offsets)
        _lib.lib().mmf_launch_count(1)
        plan.hilbert_varlen(x, offsets)
        counts.append(_lib.lib().mmf_launch_count(1))
    assert counts[0] == counts[1] <= 2 + 5 * 3, counts


@pytest.mark.gpu
@pytest.mark.parametrize("filt", [None, "iir"])
def test_many_clips_equal_the_single_call(filt, cuda_device):
    rates = [44100, 16000, 8000, 22050, 16000]
    lengths = [int(r * (1.2 + 0.3 * i)) for i, r in enumerate(rates)] + [3000]
    rates.append(16000)
    clips = [_clip(120 + i, n, r, False) for i, (n, r) in enumerate(zip(lengths, rates))]
    kw = dict(outFilter=filt, outFiltCutOff=[12]) if filt else {}
    many = mm.calculate_amplitude_envelope_many(clips, rates, method="Hilb", **kw)
    for (amp, ampT), c, r in zip(many, clips, rates):
        one, oneT = mm.calculate_amplitude_envelope(c, r, method="Hilb", **kw)
        assert np.array_equal(amp, one) and np.array_equal(ampT, oneT), r


def _solo_env(fx, x, rate):
    kw = dict(hopLen=fx.amp_hopLen)
    if fx.amp_sos is not None:
        kw |= dict(outFilter="iir", outFiltCutOff=[12], outFiltLen=6, outFiltType="low")
    return mm.calculate_amplitude_envelope(_as_f32(x), rate, method="Hilb", **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("pcm16", [False, True])
@pytest.mark.parametrize("filt", [False, True])
@pytest.mark.parametrize("mode", ["plan_rate", "rates"])
def test_bundle_envelope_matches_the_single_call(mode, filt, pcm16, cuda_device):
    """Each clip's Hilbert envelope from host_varlen equals calculate_amplitude_envelope(method='Hilb') on that clip
    at its own rate, bit for bit, raw and 'iir', float32 and int16, plan-rate and mixed-rate clips (one of them on
    the direct route); the MFCC-side blocks equal the call without the envelope."""
    fx = _fx(amp_outFilter="iir" if filt else None)
    rates = [16000] * 6 if mode == "plan_rate" else [44100, 48000, 22050, 8000, 16000, 44100]
    lengths = [int(r * (1.1 + 0.43 * i)) + 3 * i for i, r in enumerate(rates)]
    lengths[3] = 3500
    clips = [_clip(40 + i, n, r, pcm16) for i, (n, r) in enumerate(zip(lengths, rates))]
    buf, offsets = _packed(clips)
    with_rates = rates if mode == "rates" else None
    res = fx.host_varlen(buf, offsets, want=ALL + ("amplitude",), rates=with_rates)
    ref = mm.FeatureExtractor(16000, tStep=0.01, winLen=0.025, n_fft=512, n_mels=40, n_mfcc=13, fmin=0.0,
                              fmax=8000).host_varlen(buf, offsets, want=ALL, rates=with_rates)
    for k in ALL:
        assert res[k].tobytes() == ref[k].tobytes(), k
    assert res["amplitude"].dtype == (np.float64 if filt else np.float32)
    assert np.array_equal(np.diff(res["amp_offsets"]), lengths)
    for i, (c, r) in enumerate(zip(clips, rates)):
        a0, a1 = int(res["amp_offsets"][i]), int(res["amp_offsets"][i + 1])
        assert np.array_equal(res["amplitude"][a0:a1], _solo_env(fx, c, r)[0]), (i, r)


@pytest.mark.gpu
def test_multi_chunk_batch_and_host_many(cuda_device):
    """int16 clips spread over several chunks (a 187.5 s clip forms one alone): host_many's amplitude and ampT
    equal the single call for each clip."""
    fx = _fx(amp_outFilter="iir")
    rates = [44100, 16000, 8000, 48000, 22050, 16000]
    lengths = [int(r * 2.1) + 7 * i for i, r in enumerate(rates)]
    lengths[3] = 9_000_000
    clips = [_clip(50 + i, n, r, True) for i, (n, r) in enumerate(zip(lengths, rates))]
    many = fx.host_many(clips, want=("totChange", "amplitude"), rates=rates)
    for d, c, r in zip(many, clips, rates):
        amp, ampT = _solo_env(fx, c, r)
        assert np.array_equal(d["amplitude"], amp) and np.array_equal(d["ampT"], ampT), r


@pytest.mark.gpu
def test_host_files_int16_relation(cuda_device, tmp_path):
    """host_files: a 16-bit file's envelope times 32768 equals the Hilbert envelope of its raw int16 samples (a
    power-of-two scale is exact through the float64 transforms); a float file's equals its own."""
    from scipy.io import wavfile

    files = []
    for i, (rate, dt) in enumerate([(44100, np.int16), (48000, np.float32), (8000, np.int16), (16000, np.int16)]):
        a = synth_clip(200 + i, int(rate * (2.2 + 0.3 * i)), rate)
        data = np.clip(np.round(a * 32768.0), -32768, 32767).astype(np.int16) if dt == np.int16 else a
        files.append(str(tmp_path / f"f{i}.wav"))
        wavfile.write(files[-1], rate, data)
    fx = _fx()
    for group in (files, [files[0], files[2], files[3]]):
        many = fx.host_files(group, want=("totChange", "amplitude"))
        for p, d in zip(group, many):
            file_sr, x = wavfile.read(p)
            ref = mm.calculate_amplitude_envelope(x, file_sr, method="Hilb")[0]
            got = d["amplitude"] * 32768 if x.dtype == np.int16 else d["amplitude"]
            assert np.array_equal(got, ref), p


# ---- no GPU needed -------------------------------------------------------------------------------------------------


def test_env_params_layout_matches_the_library():
    assert _lib.lib().mmf_abi_sizeof(5) == C.sizeof(_lib.mmf_env_params)
    for name, off in (("method", 0), ("center", 4), ("out_n_sections", 8), ("out_sos", 16)):
        assert getattr(_lib.mmf_env_params, name).offset == off, name


def test_env_sizes():
    offsets = np.array([11, 1011, 1012, 5000, 405000], np.int64)
    assert np.array_equal(env_sizes(offsets, make_env_params("Hilb")), [0, 1000, 1001, 4989, 404989])
    geom = [(1600, 160)] * 4
    rms = env_sizes(offsets, make_env_params("RMS", True), geom)
    assert np.array_equal(rms, mm.plan.amp_sizes(offsets, geom, True)[2])


def _rc(fn):
    rc = fn()
    return rc, _lib.lib().mmf_last_error().decode()


def test_checks_fail_naming_the_clip_before_anything_is_queued():
    lib = _lib.lib()
    hil = make_env_params("Hilb")
    f = np.zeros(8)
    a = np.zeros(8, np.float32)
    # bad offsets
    bad = np.array([0, 1000, 900, 3000], np.int64)
    for rc, msg in (_rc(lambda: lib.mmf_hilbert_varlen(None, None, 3, bad.ctypes.data, None, None)),
                    _rc(lambda: lib.mmf_env_varlen_sizes(3, bad.ctypes.data, C.byref(hil), None, f.ctypes.data))):
        assert rc == _lib.MMF_ERR_INVALID and "clip 1" in msg, msg
    # a clip over 2^26 samples
    big = np.array([0, 1000, 1000 + (1 << 26) + 1, 3 * (1 << 26)], np.int64)
    for rc, msg in (_rc(lambda: lib.mmf_hilbert_varlen(None, None, 3, big.ctypes.data, None, None)),
                    _rc(lambda: lib.mmf_env_varlen_sizes(3, big.ctypes.data, C.byref(hil), None, f.ctypes.data))):
        assert rc == _lib.MMF_ERR_UNSUPPORTED and "clip 1:" in msg and "2^26" in msg, msg
    # an unknown method
    unknown = make_env_params("Hilb")
    unknown.method = 7
    ok = np.array([0, 1000, 2000], np.int64)
    rc, msg = _rc(lambda: lib.mmf_env_varlen_sizes(2, ok.ctypes.data, C.byref(unknown), None, f.ctypes.data))
    assert rc == _lib.MMF_ERR_INVALID and "unknown envelope method 7" in msg, msg
    rc, msg = _rc(lambda: lib.mmf_features_host_varlen_env(None, None, 0, 2, ok.ctypes.data, None, None, 0,
                                                            C.byref(_lib.mmf_change_params()), None, C.byref(unknown),
                                                            None, f.ctypes.data, None, None, None, None, a.ctypes.data,
                                                            None))
    assert rc == _lib.MMF_ERR_INVALID and "unknown envelope method" in msg, msg
    # good arguments: the NULL plan is reported only after every check passed
    rc, msg = _rc(lambda: lib.mmf_hilbert_varlen(None, None, 2, ok.ctypes.data, None, None))
    assert rc == _lib.MMF_ERR_INVALID and "NULL argument" in msg, msg
    # a filtered envelope of at most padlen samples
    sos = mm.api._design_iir(100.0, [12], 6, "low")
    padlen = mm.sos_zi(sos)[1]
    offs = np.array([0, 16000, 16000 + padlen, 40000], np.int64)
    env = make_env_params("Hilb", True, sos)
    rc, msg = _rc(lambda: lib.mmf_features_host_varlen_env(None, None, 0, 3, offs.ctypes.data, None, None, 0,
                                                            C.byref(_lib.mmf_change_params()), None, C.byref(env),
                                                            None, f.ctypes.data, None, None, None, None, None,
                                                            f.ctypes.data))
    assert rc == _lib.MMF_ERR_TOO_SHORT and "clip 1:" in msg and f"padlen, which is {padlen}" in msg, msg


def test_feature_extractor_validates_the_method():
    with pytest.raises(ValueError, match="'RMS' or 'Hilb'"):
        mm.FeatureExtractor(16000, amp_method="RMSpraat")
    with pytest.raises(ValueError, match="'RMS' or 'Hilb'"):
        mm.calculate_amplitude_envelope_many([np.zeros(100, np.float32)], 16000, method="hilb")


def test_no_source_names_the_batched_copy_family():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    bad = "cudaMemcpy" + "BatchAsync", "cudaMemcpy3D" + "BatchAsync", "cuMemcpy" + "BatchAsync"
    for sub in ("modulation_mfcc_b200", "tools", "tests"):
        for dirpath, _, names in os.walk(os.path.join(root, sub)):
            for name in names:
                if name.endswith((".cu", ".cuh", ".h", ".cpp", ".py", ".sh")):
                    with open(os.path.join(dirpath, name), errors="ignore") as fh:
                        text = fh.read()
                    assert not any(b in text for b in bad), name
