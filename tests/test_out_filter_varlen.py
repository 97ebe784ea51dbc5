"""The 'fir' and 'sg' output filters over rows of any lengths: mmf_filter_varlen / Plan.filter_varlen, the batched
get_MFCCS_change_many and calculate_amplitude_envelope_many, and FeatureExtractor(diffMethod=, outFilter=, ...).

The contract: every row's output is bit-identical to mmf_fir_filtfilt / mmf_stencil on that row alone (whose bytes
tests/golden/filter_bits.npz pins), whatever batch, layout, input type or chunk the row lands in.
"""

import ctypes as C
import importlib.util
import os
import wave

import numpy as np
import pytest
import scipy.signal

import modulation_mfcc_b200 as mm
from modulation_mfcc_b200 import _lib
from modulation_mfcc_b200.api import _savgol_stencil, _findiff_stencil
from modulation_mfcc_b200.synth import synth_clip

HERE = os.path.dirname(__file__)
GOLDEN = os.path.join(HERE, "golden", "filter_bits.npz")
ALL = ("totChange", "mfcc", "delta", "modspec", "band_energy")
SR = 16000


def _bits_module():
    spec = importlib.util.spec_from_file_location("make_filter_bits", os.path.join(HERE, "golden", "make_filter_bits.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def _plan():
    return mm.get_plan(mm.MfccConfig(16000.0))


def _filters():
    """(name, OutFilter, single-row call) for FIR taps 1, 7, 64 and 513 and for savgol / gradient / findiff stencils."""
    out = []
    rng = np.random.default_rng(5)
    for n in (1, 7, 64, 513):
        b = rng.standard_normal(n)
        b /= np.abs(b).sum()
        out.append((f"fir{n}", mm.fir_filter(b), lambda p, x, b=b: p.fir_filtfilt(x, b)))
    grad = (np.array([-0.5, 0.0, 0.5]), np.array([[-1.0, 1.0]]), np.array([[-1.0, 1.0]]))
    for name, st in [("sg5", _savgol_stencil(5, 2, 0)), ("sg11", _savgol_stencil(11, 3, 0)),
                     ("sg31", _savgol_stencil(31, 4, 0)), ("sg6", _savgol_stencil(6, 2, 0)),
                     ("grad", grad), ("findiff", _findiff_stencil(2, 4))]:
        out.append((name, mm.stencil_filter(*st), lambda p, x, st=st: p.stencil(x, *st)))
    return out


def _min_len(f):
    c = f.c
    return 3 * c.n_taps + 1 if c.kind == _lib.MMF_FILT_FIR else max(c.n_edge_in, 2 * c.n_edge, 1)


def _lengths(f, seed):
    """Mixed lengths from the shortest the filter takes, across the 256-output item boundaries."""
    m = _min_len(f)
    ext = 6 * f.c.n_taps if f.c.kind == _lib.MMF_FILT_FIR else 0
    base = [m, m + 1, 255, 256, 257, 511, 512, 513, 768 - ext, 769 - ext, 1000, 3001]
    rng = np.random.default_rng(seed)
    base += [int(v) for v in rng.integers(m, 5000, 12)]
    return [max(v, m) for v in base]


# ---------------------------------------------------------------------------------------------------------------
# the kernels
# ---------------------------------------------------------------------------------------------------------------


@pytest.mark.gpu
def test_single_calls_reproduce_the_previous_kernels(cuda_device):
    """filter_bits.npz holds SHA-256 digests of the fixed-length kernels' outputs: FIR taps 1 to 4096, savgol windows
    3 to 31, get_velocity's gradient / findiff / savgol stencils, float32 inputs and one 360 001-sample row."""
    m = _bits_module()
    g = np.load(GOLDEN)
    names = [n for n in g["names"]]
    assert names == [m.case_name(c) for c in m.cases()]
    plan = _plan()
    bad = [name for name, c, want in zip(names, m.cases(), g["sha256"]) if m.digest(m.run_case(plan, c)) != want]
    assert not bad, bad


@pytest.mark.gpu
@pytest.mark.parametrize("f32", [False, True])
def test_ragged_rows_equal_the_single_call(f32, cuda_device):
    """Packed rows between NaN poison and padded rows with NaN padding, in buffer order and permuted: each row equals
    the single call on that row alone (the single call reads float64: float32 rows are widened first), and no NaN
    reaches an output."""
    import torch

    plan = _plan()
    dt = torch.float32 if f32 else torch.float64
    for k, (name, f, solo) in enumerate(_filters()):
        lengths = _lengths(f, k)
        rows = [synth_clip(300 + k * 50 + i, n, 100).astype(np.float32 if f32 else np.float64)
                for i, n in enumerate(lengths)]
        ref = [solo(plan, torch.as_tensor(r.astype(np.float64))[None].to(cuda_device))[0].cpu().numpy() for r in rows]
        for perm in (np.arange(len(rows)), np.random.default_rng(k).permutation(len(rows))):
            rs = [rows[i] for i in perm]
            offsets = np.zeros(len(rs) + 1, np.int64)
            offsets[0] = 3
            np.cumsum([len(r) for r in rs], out=offsets[1:])
            offsets[1:] += 3
            buf = np.full(int(offsets[-1]) + 5, np.nan)
            for i, r in enumerate(rs):
                buf[offsets[i]: offsets[i + 1]] = r
            y = plan.filter_varlen(torch.as_tensor(buf).to(cuda_device, dt), offsets, f).cpu().numpy()
            pad = np.full((len(rs), max(lengths) + 7), np.nan)
            for i, r in enumerate(rs):
                pad[i, : len(r)] = r
            yp = plan.filter_varlen(torch.as_tensor(pad).to(cuda_device, dt), [len(r) for r in rs], f).cpu().numpy()
            for i, j in enumerate(perm):
                got = y[offsets[i]: offsets[i + 1]]
                assert got.tobytes() == ref[j].tobytes(), (name, i)
                assert yp[i, : len(rs[i])].tobytes() == ref[j].tobytes(), (name, i)
                assert not np.any(yp[i, len(rs[i]):]), name  # the padding is 0


@pytest.mark.gpu
def test_more_rows_than_one_grid_dimension(cuda_device):
    """70 000 rows (the single calls take at most 65 535): each equals the single call over its length group."""
    import torch

    plan = _plan()
    rng = np.random.default_rng(11)
    lengths = rng.integers(31, 90, 70_000)
    x = torch.as_tensor(rng.standard_normal(int(lengths.sum()))).to(cuda_device)
    offsets = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
    for f, solo in [(mm.fir_filter([0.25, 0.5, 0.25]), lambda r: plan.fir_filtfilt(r, [0.25, 0.5, 0.25])),
                    (mm.stencil_filter(*_savgol_stencil(31, 3, 0)), lambda r: plan.stencil(r, *_savgol_stencil(31, 3, 0)))]:
        y = plan.filter_varlen(x, offsets, f)
        for n in (31, 57, 89):
            idx = np.nonzero(lengths == n)[0]
            rows = torch.stack([x[offsets[i]: offsets[i + 1]] for i in idx])
            got = torch.stack([y[offsets[i]: offsets[i + 1]] for i in idx])
            assert torch.equal(solo(rows), got), n


@pytest.mark.gpu
def test_launch_count_does_not_grow_with_the_rows(cuda_device):
    import torch

    plan = _plan()
    for f, want in [(mm.fir_filter(np.ones(21) / 21), 2), (mm.stencil_filter(*_savgol_stencil(11, 3, 0)), 1)]:
        for B in (8, 4096):
            lengths = np.random.default_rng(B).integers(64, 2000, B)
            offsets = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
            x = torch.randn(int(offsets[-1]), device=cuda_device, dtype=torch.float64)
            _lib.lib().mmf_launch_count(1)
            plan.filter_varlen(x, offsets, f)
            assert _lib.lib().mmf_launch_count(1) == want, B


@pytest.mark.gpu
def test_accuracy_against_scipy(cuda_device):
    import torch

    plan = _plan()
    rng = np.random.default_rng(3)
    rows = [rng.standard_normal(n) for n in (200, 1001, 4097)]
    offsets = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)
    x = torch.as_tensor(np.concatenate(rows)).to(cuda_device)
    b = scipy.signal.firwin(31, 12 / 50, window=("kaiser", 7.4))
    y = plan.filter_varlen(x, offsets, mm.fir_filter(b)).cpu().numpy()
    s = plan.filter_varlen(x, offsets, mm.stencil_filter(*_savgol_stencil(11, 3, 0))).cpu().numpy()
    for i, r in enumerate(rows):
        np.testing.assert_allclose(y[offsets[i]: offsets[i + 1]], scipy.signal.filtfilt(b, 1, r), rtol=0, atol=1e-12)
        np.testing.assert_allclose(s[offsets[i]: offsets[i + 1]], scipy.signal.savgol_filter(r, 11, 3, mode="interp"),
                                   rtol=0, atol=1e-12)


# ---------------------------------------------------------------------------------------------------------------
# the Python drop-ins
# ---------------------------------------------------------------------------------------------------------------

OUT = {
    "fir": dict(outFilter="fir", outFiltCutOff=[60], outFiltLen=31),
    "sg": dict(outFilter="sg", outFiltCutOff=[12], outFiltLen=11, outFiltPolyOrd=3),
}


@pytest.mark.gpu
@pytest.mark.parametrize("filt", ["fir", "sg"])
def test_change_many_equals_the_single_call(filt, cuda_device):
    import torch

    lengths = [SR * 2 + 17, SR // 2, SR * 5, 3 * SR + 5]
    clips = [synth_clip(70 + i, n, SR) for i, n in enumerate(lengths)]
    clips[1] = torch.as_tensor(clips[1]).to(cuda_device)
    many = mm.get_MFCCS_change_many(clips, SR, **OUT[filt])
    for i, ((tot, T), c) in enumerate(zip(many, clips)):
        one, oneT = mm.get_MFCCS_change(c.cpu().numpy() if isinstance(c, torch.Tensor) else c, SR, **OUT[filt])
        got = tot.cpu().numpy() if isinstance(tot, torch.Tensor) else tot
        assert isinstance(tot, torch.Tensor) == isinstance(c, torch.Tensor)
        assert got.tobytes() == one.tobytes() and np.array_equal(T, oneT), i


@pytest.mark.gpu
@pytest.mark.parametrize("method", ["RMS", "Hilb"])
@pytest.mark.parametrize("filt", ["fir", "sg"])
def test_envelope_many_equals_the_single_call(filt, method, cuda_device):
    rates = [16000, 44100, 8000, 22050]
    clips = [synth_clip(90 + i, int(r * (1.5 + i)), r).astype(np.float32) for i, r in enumerate(rates)]
    kw = dict(OUT[filt], outFiltCutOff=[12] if filt == "sg" else [20])
    many = mm.calculate_amplitude_envelope_many(clips, rates, method=method, **kw)
    for (amp, ampT), c, r in zip(many, clips, rates):
        one, oneT = mm.calculate_amplitude_envelope(c, r, method=method, **kw)
        assert amp.tobytes() == one.tobytes() and np.array_equal(ampT, oneT), r


@pytest.mark.gpu
def test_too_short_names_the_clip(cuda_device):
    clips = [synth_clip(1, SR, SR), synth_clip(2, SR // 20, SR)]  # the second: a 51-frame curve at 1 kHz
    for kw in (dict(outFilter="fir", outFiltCutOff=[60], outFiltLen=31), dict(outFilter="sg", outFiltCutOff=[12],
                                                                                outFiltLen=61)):
        with pytest.raises(ValueError) as one:
            mm.get_MFCCS_change(clips[1], SR, **kw)
        with pytest.raises(ValueError, match="clip 1: ") as many:
            mm.get_MFCCS_change_many(clips, SR, **kw)
        assert str(many.value) == "clip 1: " + str(one.value)


def _fx(sr=SR, **kw):
    return mm.FeatureExtractor(sr, tStep=0.01, winLen=0.025, n_fft=512, n_mels=40, n_mfcc=13, fmin=0.0, fmax=sr / 2,
                               **kw)


def _solo(clip, sr, kw):
    """get_MFCCS_change with the extractor's settings"""
    return mm.get_MFCCS_change(clip, sr, tStep=0.01, winLen=0.025, n_fft=512, n_mels=40, n_mfcc=13, minFreq=0.0,
                               maxFreq=sr / 2, **kw)[0]


SETTINGS = {
    "none": dict(outFilter=None),
    "iir": dict(outFilter="iir", outFiltCutOff=[8], outFiltLen=4),
    "fir": dict(outFilter="fir", outFiltCutOff=[10], outFiltLen=21),
    "sg": dict(outFilter="sg", outFiltCutOff=[12], outFiltLen=11, outFiltPolyOrd=3),
}


def _write_wav(path, x, rate):
    with wave.open(str(path), "wb") as w:
        w.setnchannels(1)
        w.setsampwidth(2)
        w.setframerate(rate)
        w.writeframes(x.astype("<i2").tobytes())


@pytest.mark.gpu
@pytest.mark.parametrize("diff", ["grad", "sg"])
@pytest.mark.parametrize("setting", list(SETTINGS))
def test_feature_extractor_curve_equals_the_single_call(setting, diff, cuda_device, tmp_path):
    """Every clip's totChange from host_many, host_varlen(rates=...), host_files, __call__, varlen and host_call
    equals get_MFCCS_change on that clip with the same settings, bit for bit."""
    import torch

    kw = dict(SETTINGS[setting], diffMethod=diff)
    fx = _fx(**kw)
    lengths = [int(SR * 1.7), SR * 3 + 11, int(SR * 0.9), SR * 2]
    clips = [synth_clip(200 + i, n, SR).astype(np.float32) for i, n in enumerate(lengths)]
    want = [_solo(c, SR, kw) for c in clips]
    for d, w in zip(fx.host_many(clips, want=ALL), want):
        assert d["totChange"].tobytes() == w.tobytes()
    pcm = torch.zeros((len(clips), max(lengths)), device=cuda_device)
    for i, c in enumerate(clips):
        pcm[i, : len(c)] = torch.as_tensor(c)
    res = fx.varlen(pcm, lengths)
    for i, w in enumerate(want):
        assert res["totChange"][i, : res["frames"][i]].cpu().numpy().tobytes() == w.tobytes()
    eq = np.stack([clips[3], clips[3] * np.float32(0.5)])
    weq = [want[3], _solo(eq[1], SR, kw)]
    for got in (fx(torch.as_tensor(eq).to(cuda_device))["totChange"].cpu().numpy(), fx.host_call(eq, want=ALL)["totChange"]):
        assert got[0].tobytes() == weq[0].tobytes() and got[1].tobytes() == weq[1].tobytes()
    # int16 WAV files at mixed rates: host_files and host_varlen(rates=) against the file-path single call
    rates = [44100, 8000, 22050, 16000]
    paths, raw = [], []
    for i, r in enumerate(rates):
        x = np.clip(np.round(synth_clip(220 + i, int(r * (1.2 + 0.5 * i)), r) * 20000), -32768, 32767).astype(np.int16)
        paths.append(tmp_path / f"c{i}.wav")
        _write_wav(paths[-1], x, r)
        raw.append(x)
    want_f = [_solo(str(p), SR, kw) for p in paths]
    for d, w in zip(fx.host_files([str(p) for p in paths], want=ALL), want_f):
        assert d["totChange"].tobytes() == w.tobytes()
    offsets = np.concatenate([[0], np.cumsum([len(x) for x in raw])]).astype(np.int64)
    res = fx.host_varlen(np.concatenate(raw), offsets, want=ALL, rates=rates)
    for i, w in enumerate(want_f):
        f0, f1 = res["frame_offsets"][i], res["frame_offsets"][i + 1]
        assert res["totChange"][f0:f1].tobytes() == w.tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("setting", ["fir", "sg"])
def test_feature_extractor_multi_chunk_batch(setting, cuda_device):
    """Float32 clips of 2.5 to 3.3 M samples spread over several chunks; the MFCC-side blocks equal the call without
    the filter, and the filter adds a fixed number of launches per chunk."""
    kw = SETTINGS[setting]
    fx, ref = _fx(**kw), _fx()
    lengths = [2_500_000 + 200_000 * i for i in range(5)]
    clips = [synth_clip(400 + i, n, SR).astype(np.float32) for i, n in enumerate(lengths)]
    many = fx.host_many(clips, want=ALL)
    base = ref.host_many(clips, want=ALL)
    for i, (d, b, c) in enumerate(zip(many, base, clips)):
        assert d["totChange"].tobytes() == _solo(c, SR, kw).tobytes(), i
        for k in ALL[1:]:
            assert d[k].tobytes() == b[k].tobytes(), (i, k)
    # launches: the filter's per chunk, on top of the same raw-curve call without it
    offsets = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
    buf = np.concatenate(clips)
    counts = []
    for f in (fx.change_out, None):
        _lib.lib().mmf_launch_count(1)
        fx.plan.features_host_varlen(buf, offsets, fx.prm, change_out=f)
        counts.append(_lib.lib().mmf_launch_count(1))
    per = 2 if setting == "fir" else 1
    assert (counts[0] - counts[1]) % per == 0 and 2 * per <= counts[0] - counts[1] <= 5 * per, counts


@pytest.mark.gpu
def test_bundle_too_short_names_the_clip(cuda_device):
    fx = _fx(outFilter="fir", outFiltCutOff=[10], outFiltLen=21)  # padlen 63: curves of at most 63 frames fail
    clips = [synth_clip(1, SR, SR).astype(np.float32), synth_clip(2, 9000, SR).astype(np.float32)]
    with pytest.raises(ValueError, match="^clip 1: The length of the input vector x must be greater than padlen, "
                                         "which is 63.$"):
        fx.host_many(clips)


# ---------------------------------------------------------------------------------------------------------------
# host-only
# ---------------------------------------------------------------------------------------------------------------


def test_out_filter_layout_matches_the_library():
    assert C.sizeof(_lib.mmf_out_filter) == _lib.lib().mmf_abi_sizeof(6)
    assert [f for f, _ in _lib.mmf_out_filter._fields_] == [
        "kind", "n_taps", "taps", "half", "coef", "n_edge", "n_edge_in", "edge_l", "edge_r"]


def _err(fn, *args):
    rc = fn(*args)
    return rc, _lib.lib().mmf_last_error().decode()


def test_checks_fail_naming_the_clip_before_any_device_work():
    L = _lib.lib()
    T = np.array([100, 64, 63, 10], np.int64)
    fir = mm.fir_filter(np.ones(21) / 21)
    assert _err(L.mmf_filter_varlen_check, C.byref(fir.c), 4, T.ctypes.data) == (
        _lib.MMF_ERR_TOO_SHORT, "clip 2: The length of the input vector x must be greater than padlen, which is 63.")
    sg = mm.stencil_filter(*_savgol_stencil(11, 3, 0))
    T2 = np.array([11, 10], np.int64)
    assert _err(L.mmf_filter_varlen_check, C.byref(sg.c), 2, T2.ctypes.data) == (
        _lib.MMF_ERR_TOO_SHORT, "clip 1: input shorter than the stencil's edge window")
    assert L.mmf_filter_varlen_check(C.byref(sg.c), 1, T2.ctypes.data) == 0
    bad = mm.fir_filter(np.ones(3))
    bad.c.n_taps = 0
    assert L.mmf_filter_varlen_check(C.byref(bad.c), 1, T.ctypes.data) == _lib.MMF_ERR_UNSUPPORTED
    bad.c.n_taps, bad.c.kind = 3, 7
    assert L.mmf_filter_varlen_check(C.byref(bad.c), 1, T.ctypes.data) == _lib.MMF_ERR_INVALID
    edge = mm.stencil_filter(*_savgol_stencil(5, 2, 0))
    edge.c.edge_l = None
    assert _err(L.mmf_filter_varlen_check, C.byref(edge.c), 1, T.ctypes.data) == (
        _lib.MMF_ERR_INVALID, "edge matrices are NULL")
    # the device call runs the same checks first: no plan is touched
    x = np.zeros(4, np.int64)
    assert _err(L.mmf_filter_varlen, None, C.byref(fir.c), None, 0, 4, x.ctypes.data, T.ctypes.data, None,
                x.ctypes.data, None)[1].startswith("clip 2: ")
    # the bundle: a bad filter, or a change stage that already filters the curve, fails before the plan is needed
    offs = np.array([0, 1000], np.int64)
    prm_raw = mm.make_change_params(scipy.signal.butter(6, 0.24, output="sos"), out_sos=None)
    prm_iir = mm.make_change_params(scipy.signal.butter(6, 0.24, output="sos"), out_sos=scipy.signal.butter(
        6, 0.24, output="sos"))
    pcm = np.zeros(1000, np.float32)
    tot = np.zeros(8, np.float64)
    args = lambda prm, f: (None, pcm.ctypes.data, 0, 1, offs.ctypes.data, None, None, 0, C.byref(prm), None, None, None,
                           C.byref(f.c), tot.ctypes.data, None, None, None, None, None, None)  # noqa: E731
    assert _err(L.mmf_features_host_varlen_out, *args(prm_iir, fir)) == (
        _lib.MMF_ERR_INVALID, "change_out needs prm->out_kind == 1 (the raw curve)")
    assert L.mmf_features_host_varlen_out(*args(prm_raw, bad)) == _lib.MMF_ERR_INVALID
    assert _err(L.mmf_features_host_varlen_out, *args(prm_raw, fir)) == (_lib.MMF_ERR_INVALID, "NULL argument")


@pytest.mark.parametrize("kw", [
    dict(outFilter="fir", outFiltCutOff=[12], outFiltLen=0),
    dict(outFilter="fir", outFiltCutOff=[12], outFiltLen=4, outFiltType="high"),
    dict(outFilter="fir", outFiltCutOff=[60]),
    dict(outFilter="fir", outFiltCutOff=[20, 10], outFiltType="band"),
    dict(outFilter="fir", outFiltCutOff=[10, 20], outFiltType="low"),
    dict(outFilter="sg", outFiltCutOff=[12], outFiltLen=3, outFiltPolyOrd=5),
    dict(outFilter="sg", outFiltCutOff=[10, 20], outFiltType="band"),
    dict(outFilter="sg", outFiltCutOff=[12], outFiltType="xyz"),
    dict(outFilter="sg", outFiltCutOff=None),
    dict(outFilter="iir", outFiltCutOff=[12], outFiltType="band"),
])
def test_feature_extractor_raises_what_apply_filter_raises(kw):
    """Checked on construction with no device: the exception applyFilter's validation and filter design raise (the
    design's own errors come from scipy: firwin, savgol_coeffs)."""
    from modulation_mfcc_b200.api import _design_filter

    post = dict(filt=kw["outFilter"], cutOff=kw.get("outFiltCutOff", [12]), filtLen=kw.get("outFiltLen", 6),
                filtType=kw.get("outFiltType", "low"), polyOrd=kw.get("outFiltPolyOrd", 3))
    with pytest.raises(Exception) as ref:
        _design_filter(100.0, **post)
    with pytest.raises(type(ref.value)) as got:
        mm.FeatureExtractor(16000, tStep=0.01, **kw)
    assert str(got.value) == str(ref.value)


def test_feature_extractor_rejects_an_unknown_filter():
    with pytest.raises(ValueError, match="outFilter must be None, 'iir', 'fir' or 'sg'"):
        mm.FeatureExtractor(16000, outFilter="median", outFiltCutOff=[12])
