"""Variable-length batches of the MFCC-change path (mmf_mfcc_change_varlen, Plan.mfcc_change_varlen,
get_MFCCS_change_many).

The contract: frames [0, T_i) of clip i are bit-identical to mmf_mfcc_change on that clip alone, every output
element at a frame >= T_i is exactly 0, and nothing past a clip's length is ever read as anything but zero.
"""

import ctypes as C

import numpy as np
import pytest
import scipy.signal

import oracle
import modulation_mfcc_b200 as mm
from modulation_mfcc_b200 import _lib
from modulation_mfcc_b200.synth import synth_clip

ABS_TOL = 1e-3

CONFIGS = {
    # name: (sr, n_fft, winLen, tStep, n_mels, n_mfcc, fmin, fmax)
    "gui_default": (10000, 512, 0.025, 0.005, 128, 13, 100.0, 10000.0),  # tcgen05 mel, empty top bands
    "cfg1_16k": (16000, 512, 0.025, 0.01, 40, 13, 0.0, 8000.0),
    "cfg3_44k": (44100, 2048, 0.025, 0.01, 128, 20, 0.0, 22050.0),  # CUDA-core K1
    "n400": (16000, 400, 0.025, 0.01, 40, 13, 0.0, 8000.0),  # generic n_fft: every clip on the single-clip path
}
FUSED_MAX_T = 12 * 32 * 9  # longest row the fused per-clip kernel takes


def _torch():
    import torch

    return torch


def _cfg(name, flags=0):
    sr, n_fft, winLen, tStep, n_mels, n_mfcc, fmin, fmax = CONFIGS[name]
    win, hop = mm.frame_sizes(sr, winLen, tStep)
    return mm.MfccConfig(sr, n_fft, win, hop, n_mels, n_mfcc, fmin, fmax, flags=flags), tStep


def _params(tStep, out_filter, remove_first=1, diff_method=0):
    sos = scipy.signal.butter(6, 12 / ((1 / tStep) / 2), "low", output="sos")
    out = {"none": sos, "iir": scipy.signal.butter(6, 10 / ((1 / tStep) / 2), "low", output="sos"), "raw": None}
    return mm.make_change_params(sos, remove_first=remove_first, diff_method=diff_method, out_sos=out[out_filter]), sos


def _lengths_for(cfg, padlen, n_clips=40, seed=0):
    """Clip lengths (samples) covering the edges the kernels care about, the rest random."""
    hop = cfg.hop_length
    T_of = lambda T, extra=0: (T - 1) * hop + extra  # noqa: E731  (1 + n // hop == T for extra < hop)
    rng = np.random.default_rng(seed)
    special = [T_of(padlen + 1), T_of(padlen + 1, hop - 1)]  # the shortest legal clip, both ends of its hop
    for edge in (32, 64, 128, 256):  # TF tiles, 64-frame tiles, 128-frame blocks
        special += [T_of(edge - 1, 3), T_of(edge, 1), T_of(edge + 1, hop // 2)]
    special += [T_of(FUSED_MAX_T + 40, 7)]  # longer than the fused kernel: the single-clip path in the same batch
    n_rand = max(0, n_clips - len(special))
    special += [T_of(int(T), int(x)) for T, x in zip(rng.integers(padlen + 2, 700, n_rand), rng.integers(0, hop, n_rand))]
    return [int(n) for n in special]


def _clips(lengths, sr, seed=0):
    return [synth_clip(seed + i, n, sr).astype(np.float32) for i, n in enumerate(lengths)]


def _padded(clips, fill=0.0, stride=None, offset=0):
    torch = _torch()
    n_max = max(len(c) for c in clips)
    stride = stride or (n_max + 3) // 4 * 4  # 16-byte rows: the TMA loader (offset 1 breaks that: the plain loader)
    buf = np.full((len(clips), stride + offset), fill, np.float32)
    for i, c in enumerate(clips):
        buf[i, offset : offset + len(c)] = c
    dev = torch.as_tensor(buf).cuda()
    return dev[:, offset : offset + n_max] if offset else dev


def _host(res):
    return {k: (v.cpu().numpy() if hasattr(v, "cpu") else v) for k, v in res.items() if v is not None}


def _check_against_solo(plan, clips, prm, want_delta, want_feats=True):
    torch = _torch()
    lengths = [len(c) for c in clips]
    vr = plan.mfcc_change_varlen(_padded(clips), lengths, prm, want_logmel=want_feats, want_mfcc=want_feats,
                                 want_delta=want_delta)
    v = _host(vr)
    frames = v["frames"]
    assert list(frames) == [plan.num_frames(n) for n in lengths]
    assert v["totChange"].shape == (len(clips), frames.max())
    for i, c in enumerate(clips):
        one = _host(plan.mfcc_change(torch.as_tensor(c[None]).cuda(), prm, want_logmel=want_feats, want_mfcc=want_feats,
                                     want_delta=want_delta))
        T = frames[i]
        for k in ("totChange", "logmel", "mfcc", "delta"):
            if k not in one:
                assert k not in v, k
                continue
            assert np.array_equal(v[k][i, ..., :T], one[k][0]), (k, i, T)
            assert not np.any(v[k][i, ..., T:]), (k, i, T)
    return v


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CONFIGS))
@pytest.mark.parametrize("flags", [0, _lib.MMF_FLAG_NO_TC_MEL, _lib.MMF_FLAG_NO_TMA, _lib.MMF_FLAG_FOLD_MFCC])
@pytest.mark.parametrize("want_delta", [False, True])
def test_varlen_matches_solo_calls(name, flags, want_delta, cuda_device):
    """Every clip of a 40-clip batch (so the batched output filter runs) equals its own single-clip call."""
    cfg, tStep = _cfg(name, flags)
    plan = mm.get_plan(cfg)
    # cycle remove_first, diff_method and the output filter over the cases
    k = list(CONFIGS).index(name) + flags.bit_length() + int(want_delta)
    out_filter = ("iir", "none", "raw")[k % 3]
    prm, sos = _params(tStep, out_filter, remove_first=k % 2, diff_method=(k // 2) % 2)
    padlen = max(mm.sos_zi(sos)[1], 21)
    clips = _clips(_lengths_for(cfg, padlen), cfg.sample_rate, seed=11 * k)
    _check_against_solo(plan, clips, prm, want_delta)


@pytest.mark.gpu
@pytest.mark.parametrize("out_filter", ["none", "iir", "raw"])
@pytest.mark.parametrize("remove_first", [0, 1])
@pytest.mark.parametrize("diff_method", [0, 1])
def test_varlen_change_parameters(out_filter, remove_first, diff_method, cuda_device):
    cfg, tStep = _cfg("cfg1_16k")
    plan = mm.get_plan(cfg)
    prm, sos = _params(tStep, out_filter, remove_first, diff_method)
    clips = _clips(_lengths_for(cfg, mm.sos_zi(sos)[1], n_clips=36, seed=3), cfg.sample_rate, seed=5)
    _check_against_solo(plan, clips, prm, want_delta=diff_method == 1)
    _check_against_solo(plan, clips[:10], prm, want_delta=False, want_feats=False)  # fewer than 32: per-CTA output filter


@pytest.mark.gpu
@pytest.mark.parametrize(
    "name, flags",
    # cfg1: the tcgen05 kernel's hop-160 instantiation, and the CUDA-core kernel; the GUI default (hop 50): the
    # tcgen05 kernel's general TMA branch
    [("cfg1_16k", 0), ("cfg1_16k", _lib.MMF_FLAG_NO_TC_MEL), ("gui_default", 0)],
)
@pytest.mark.parametrize("fill", [np.nan, 1e6])
def test_padding_contents_do_not_matter(name, flags, fill, cuda_device):
    cfg, tStep = _cfg(name, flags)
    plan = mm.get_plan(cfg)
    prm, sos = _params(tStep, "iir")
    clips = _clips(_lengths_for(cfg, mm.sos_zi(sos)[1], n_clips=34, seed=9)[:-1], cfg.sample_rate, seed=2)
    lengths = [len(c) for c in clips]
    kw = dict(want_logmel=True, want_mfcc=True, want_delta=True)
    ref = _host(plan.mfcc_change_varlen(_padded(clips), lengths, prm, **kw))
    for offset in (0, 1):  # offset 1: the base is not 16-byte aligned -> the plain loader instead of the TMA
        got = _host(plan.mfcc_change_varlen(_padded(clips, fill, offset=offset), lengths, prm, **kw))
        for k in ("totChange", "logmel", "mfcc", "delta"):
            assert np.array_equal(got[k], ref[k]), (k, offset)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["gui_default", "cfg3_44k"])
def test_equal_lengths_equal_the_batch_call(name, cuda_device):
    torch = _torch()
    cfg, tStep = _cfg(name)
    plan = mm.get_plan(cfg)
    prm, _ = _params(tStep, "iir")
    n = int(cfg.sample_rate * 2.3) + 17
    pcm = torch.as_tensor(np.stack(_clips([n] * 40, cfg.sample_rate, seed=4))).cuda()
    kw = dict(want_logmel=True, want_mfcc=True, want_delta=True)
    v = _host(plan.mfcc_change_varlen(pcm, [n] * 40, prm, **kw))
    b = _host(plan.mfcc_change(pcm, prm, **kw))
    for k in ("totChange", "logmel", "mfcc", "delta"):
        assert np.array_equal(v[k], b[k]), k


@pytest.mark.gpu
def test_permuting_clips_permutes_outputs(cuda_device):
    cfg, tStep = _cfg("gui_default")
    plan = mm.get_plan(cfg)
    prm, sos = _params(tStep, "iir")
    clips = _clips(_lengths_for(cfg, mm.sos_zi(sos)[1], seed=6), cfg.sample_rate, seed=8)
    perm = np.random.default_rng(1).permutation(len(clips))
    kw = dict(want_logmel=True, want_mfcc=True, want_delta=False)
    a = _host(plan.mfcc_change_varlen(_padded(clips), [len(c) for c in clips], prm, **kw))
    pc = [clips[j] for j in perm]
    b = _host(plan.mfcc_change_varlen(_padded(pc), [len(c) for c in pc], prm, **kw))
    for k in ("totChange", "logmel", "mfcc"):
        assert np.array_equal(a[k][perm], b[k]), k


@pytest.mark.gpu
@pytest.mark.parametrize(
    "name, max_frames",
    # the longest rows whose float64 row buffers fit the fused kernel's shared memory at these shapes (12 or 19 kept
    # coefficients); longer rows leave the fused kernel in the single-clip call too
    [("cfg1_16k", 2001), ("gui_default", 2101), ("cfg3_44k", 1301)],
)
@pytest.mark.parametrize("want_delta", [False, True])
def test_one_launch_per_stage(name, max_frames, want_delta, cuda_device):
    """No clip on the single-clip path: 400 clips take as many launches as 40, with and without a delta output
    (cfg3's 20 coefficients take the separate MFCC kernel even without one, as its single-clip call does)."""
    cfg, tStep = _cfg(name)
    plan = mm.get_plan(cfg)
    prm, sos = _params(tStep, "iir")
    rng = np.random.default_rng(12)
    hop = cfg.hop_length
    counts = []
    for n_clips in (40, 400):
        lengths = [int((T - 1) * hop + x) for T, x in zip(rng.integers(200, max_frames + 1, n_clips), rng.integers(0, hop, n_clips))]
        pcm = _torch().zeros((n_clips, max(lengths)), device="cuda")
        kw = dict(want_logmel=True, want_mfcc=True, want_delta=want_delta)
        plan.mfcc_change_varlen(pcm, lengths, prm, **kw)  # warm-up (workspace growth)
        _lib.lib().mmf_launch_count(1)
        plan.mfcc_change_varlen(pcm, lengths, prm, **kw)
        counts.append(_lib.lib().mmf_launch_count(1))
    assert counts[0] == counts[1], counts
    assert counts[0] <= 7, counts


@pytest.mark.gpu
def test_many_matches_single_calls_and_oracle(cuda_device):
    torch = _torch()
    sr = 16000
    kw = dict(tStep=0.01, winLen=0.025, n_mfcc=13, n_fft=512, minFreq=0, maxFreq=8000, n_mels=40, outFiltCutOff=[12])
    lengths = [sr * 2 + 77, sr * 3 + 5, int(sr * 2.5), sr * 4 - 1]
    clips = _clips(lengths, sr, seed=21)
    many = mm.get_MFCCS_change_many(clips, sr, **kw)
    for i, c in enumerate(clips):
        tot, T = many[i]
        one, T1 = mm.get_MFCCS_change(c, sr, **kw)
        assert isinstance(tot, np.ndarray) and np.array_equal(tot, one) and np.array_equal(T, T1)
        ref, rT = oracle.get_MFCCS_change(c, sr, **kw)
        assert np.array_equal(T, rT) and np.max(np.abs(tot - ref)) < ABS_TOL
    # CUDA in -> CUDA out; features per clip
    dev = [torch.as_tensor(c).cuda() for c in clips]
    many_d = mm.get_MFCCS_change_many(dev, sr, return_features=True, **kw)
    for i, c in enumerate(clips):
        tot, T, feats = many_d[i]
        one, _, f1 = mm.get_MFCCS_change(c, sr, return_features=True, **kw)
        assert tot.is_cuda and np.array_equal(tot.cpu().numpy(), one)
        for k in ("logmel", "mfcc", "delta"):
            assert np.array_equal(feats[k].cpu().numpy(), f1[k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("outFilter", ["fir", "sg"])
def test_many_output_filters(outFilter, cuda_device):
    sr = 16000
    kw = dict(tStep=0.01, n_mels=40, maxFreq=8000, outFilter=outFilter, outFiltCutOff=[12], outFiltLen=21)
    clips = _clips([sr * 3 + 11, sr * 5, sr * 2 + 160 * 7 + 3], sr, seed=31)
    many = mm.get_MFCCS_change_many(clips, sr, **kw)
    for i, c in enumerate(clips):
        one, T1 = mm.get_MFCCS_change(c, sr, **kw)
        assert np.array_equal(many[i][0], one) and np.array_equal(many[i][1], T1)


@pytest.mark.gpu
@pytest.mark.parametrize("outFilter", ["fir", "sg"])
def test_too_short_for_the_output_filter_names_its_index(outFilter, cuda_device):
    """Long enough for the Butterworth cascade, too short for a 61-tap output filter."""
    sr = 16000
    kw = dict(tStep=0.01, n_mels=40, maxFreq=8000, outFilter=outFilter, outFiltCutOff=[12], outFiltLen=61)
    clips = _clips([sr * 3, 160 * 50, sr * 2], sr, seed=41)
    with pytest.raises(ValueError) as single:
        mm.get_MFCCS_change(clips[1], sr, **kw)
    with pytest.raises(ValueError, match="clip 1") as many:
        mm.get_MFCCS_change_many(clips, sr, **kw)
    assert str(single.value) in str(many.value)


@pytest.mark.gpu
def test_too_short_clip_names_its_index(cuda_device):
    sr = 16000
    clips = _clips([sr * 2, sr * 3, 160 * 10, sr], sr)
    with pytest.raises(ValueError) as single:
        mm.get_MFCCS_change(clips[2], sr, tStep=0.01, n_mels=40, maxFreq=8000, outFiltCutOff=[12])
    with pytest.raises(ValueError, match="clip 2") as many:
        mm.get_MFCCS_change_many(clips, sr, tStep=0.01, n_mels=40, maxFreq=8000, outFiltCutOff=[12])
    assert str(single.value) in str(many.value)
    cfg, tStep = _cfg("cfg1_16k")
    plan = mm.get_plan(cfg)
    prm, _ = _params(tStep, "iir")
    _lib.lib().mmf_launch_count(1)
    with pytest.raises(mm.MmfError) as e:
        plan.mfcc_change_varlen(_padded(clips), [len(c) for c in clips], prm)
    assert e.value.code == _lib.MMF_ERR_TOO_SHORT and "clip 2" in e.value.msg
    assert _lib.lib().mmf_launch_count(1) == 0


@pytest.mark.gpu
def test_bad_lengths_with_a_plan(cuda_device):
    cfg, tStep = _cfg("cfg1_16k")
    plan = mm.get_plan(cfg)
    prm, _ = _params(tStep, "iir")
    pcm = _torch().zeros((3, 16000), device="cuda")
    for lengths in ([16000, 0, 8000], [16000, 16001, 8000], [-5, 16000, 16000]):
        with pytest.raises(mm.MmfError) as e:
            plan.mfcc_change_varlen(pcm, lengths, prm)
        assert e.value.code == _lib.MMF_ERR_INVALID


# ---- argument checks that fail before any CUDA call (no GPU needed) ----------------------------------------------


def _call(lengths, n_clips=None, stride=100, plan=None, pcm=None, prm=True, tot=None):
    lens = np.ascontiguousarray(lengths, dtype=np.int64) if lengths is not None else None
    p = _lib.mmf_change_params()
    return _lib.lib().mmf_mfcc_change_varlen(
        plan, pcm, len(lengths) if n_clips is None else n_clips, lens.ctypes.data if lens is not None else None,
        stride, C.byref(p) if prm else None, tot, None, None, None, None)


@pytest.mark.parametrize(
    "args, named",
    [
        (dict(lengths=None, n_clips=2), None),
        (dict(lengths=[10, 20], n_clips=0), None),
        (dict(lengths=[10, 0]), "clip 1"),
        (dict(lengths=[10, 20, 101]), "clip 2"),
        (dict(lengths=[-1]), "clip 0"),
        (dict(lengths=[10, 20]), None),  # lengths fine: NULL plan, pcm and tot
    ],
)
def test_invalid_arguments_without_a_device(args, named):
    assert _call(**args) == _lib.MMF_ERR_INVALID
    if named:
        assert named in _lib.lib().mmf_last_error().decode()


def test_varlen_symbol_is_bound():
    assert "mmf_mfcc_change_varlen" in _lib.exported_symbols()
    assert callable(mm.get_MFCCS_change_many)
