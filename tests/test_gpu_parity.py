"""GPU parity tests: every CUDA entry point, called through the C ABI, against the
CPU oracle on the same seeded inputs.

Tolerances (BASELINE.json north_star / SURVEY.md section 8d):
  * log-mel: relative error of the linear mel power <= 1e-4 for bins above the
    amin floor (== 4.3e-4 dB absolute);
  * MFCC, delta, modulation magnitudes, totChange: <= 1e-3 absolute;
  * time anchors T: exact.
"""

import numpy as np
import pytest
import scipy.signal

import oracle
import modulation_mfcc_b200 as mm
from modulation_mfcc_b200 import _lib
from modulation_mfcc_b200.synth import synth_batch, synth_clip

pytestmark = pytest.mark.gpu

LOGMEL_REL = 1e-4  # on linear mel power
ABS_TOL = 1e-3


def _torch():
    import torch

    return torch


CONFIGS = {
    # name: (sr, n_fft, winLen, tStep, n_mels, n_mfcc, fmin, fmax, seconds)
    "cfg1_16k": (16000, 512, 0.025, 0.01, 40, 13, 0.0, 8000.0, 10.0),
    "gui_default": (10000, 512, 0.025, 0.005, 128, 13, 100.0, 10000.0, 4.0),
    "cfg3_44k": (44100, 2048, 0.025, 0.01, 128, 20, 0.0, 22050.0, 3.0),
    "n1024": (22050, 1024, 0.04, 0.0125, 64, 16, 50.0, 11025.0, 2.0),
    "n256": (8000, 256, 0.025, 0.01, 32, 12, 0.0, 4000.0, 2.0),
    "n4096": (48000, 4096, 0.08, 0.02, 96, 24, 20.0, 24000.0, 2.0),
}


def _cfg(name, **over):
    sr, n_fft, winLen, tStep, n_mels, n_mfcc, fmin, fmax, secs = CONFIGS[name]
    win, hop = mm.frame_sizes(sr, winLen, tStep)
    cfg = mm.MfccConfig(sr, n_fft, win, hop, n_mels, n_mfcc, fmin, fmax, **over)
    return cfg, secs


def _mel_rel_err(logmel_gpu, logmel_ref_unclamped):
    """Relative error in linear mel power for bins above the amin floor."""
    ok = logmel_ref_unclamped > -99.0
    d = np.abs(logmel_gpu - logmel_ref_unclamped)[ok]
    return float(np.max(np.abs(10.0 ** (d / 10.0) - 1.0))) if d.size else 0.0


def _oracle_unclamped(y, cfg):
    M, inter = oracle.mfcc(
        y, cfg.sample_rate, n_mfcc=cfg.n_mfcc, win_length=cfg.win_length, hop_length=cfg.hop_length, n_fft=cfg.n_fft,
        fmin=cfg.fmin, fmax=cfg.fmax, n_mels=cfg.n_mels, return_intermediates=True)
    unclamped = oracle.power_to_db(inter["melspec"], top_db=None)
    return M, inter, unclamped


@pytest.mark.parametrize("name", list(CONFIGS))
@pytest.mark.parametrize("flags", [0, _lib.MMF_FLAG_NO_TMA])
def test_stft_power(name, flags, cuda_device):
    cfg, secs = _cfg(name, flags=flags)
    y = synth_batch(0, 3, int(cfg.sample_rate * secs) + 37, cfg.sample_rate)
    plan = mm.get_plan(cfg)
    P = plan.stft_power(y).cpu().numpy()
    for i in range(y.shape[0]):
        ref = oracle.stft_power(y[i], cfg.n_fft, cfg.hop_length, cfg.win_length)
        assert P[i].shape == ref.shape
        # fp32 FFT: error relative to the frame's spectral peak
        peak = ref.max(axis=0, keepdims=True)
        assert np.max(np.abs(P[i] - ref) / peak) < 2e-6, name


@pytest.mark.parametrize("name", ["cfg1_16k", "gui_default"])
def test_stft_power_tensor_core_transform(name, cuda_device):
    """MMF_FLAG_TC_FFT: the 512-point transform as tcgen05.mma kind::f16 GEMM stages (fp16 x3 operand
    split, accumulators in tensor memory) against the oracle, same bound as the FP32 kernel, and
    against the FP32 kernel itself; ragged frame counts, a silent clip and a loud one included."""
    cfg, secs = _cfg(name, flags=_lib.MMF_FLAG_TC_FFT)
    n = int(cfg.sample_rate * secs) + 37
    y = synth_batch(0, 5, n, cfg.sample_rate)
    y[3] = 0.0
    y[4] *= 1000.0
    P = mm.get_plan(cfg).stft_power(y).cpu().numpy()
    Q = mm.get_plan(mm.plan.replace(cfg, flags=0)).stft_power(y).cpu().numpy()
    assert P.shape == Q.shape
    assert np.all(P[3] == 0.0)
    for i in (0, 1, 2, 4):
        ref = oracle.stft_power(y[i], cfg.n_fft, cfg.hop_length, cfg.win_length)
        peak = ref.max(axis=0, keepdims=True)
        assert np.max(np.abs(P[i] - ref) / peak) < 2e-6, (name, i)
        assert np.max(np.abs(P[i] - Q[i]) / peak) < 2e-6, (name, i)


def test_stft_power_split_variants_agree(cuda_device):
    cfg, secs = _cfg("cfg1_16k")
    y = synth_batch(5, 2, 16000 * 2, 16000)
    a = mm.get_plan(cfg).stft_power(y).cpu().numpy()
    b = mm.get_plan(mm.plan.replace(cfg, flags=_lib.MMF_FLAG_SPLIT_SMEM)).stft_power(y).cpu().numpy()
    assert np.array_equal(a, b)  # same arithmetic, different data path


@pytest.mark.parametrize("name", list(CONFIGS))
def test_logmel_mfcc_delta(name, cuda_device):
    cfg, secs = _cfg(name)
    y = synth_batch(10, 2, int(cfg.sample_rate * secs), cfg.sample_rate)
    plan = mm.get_plan(cfg)
    lm, cmax = plan.logmel(y)
    lm_unclamped = lm.cpu().numpy().copy()
    mf, dl = plan.mfcc(lm, cmax, delta=True, clamp_in_place=True)
    lm_c, mf, dl = lm.cpu().numpy(), mf.cpu().numpy(), dl.cpu().numpy()
    for i in range(y.shape[0]):
        M, inter, unclamped = _oracle_unclamped(y[i], cfg)
        assert _mel_rel_err(lm_unclamped[i], unclamped) < LOGMEL_REL, name
        assert np.max(np.abs(lm_c[i] - inter["logmel"])) < 4.4e-4, name  # clamped log-mel, dB
        assert np.max(np.abs(mf[i] - M)) < ABS_TOL, name
        assert np.max(np.abs(dl[i] - np.gradient(M, axis=1))) < ABS_TOL, name


@pytest.mark.parametrize("name", list(CONFIGS))
def test_mfcc_fp32_and_tensor_core_kernels_agree(name, cuda_device):
    """MMF_FLAG_TC_DCT (clamp + DCT-II as a tcgen05 GEMM with fp16 operand pairs; the FP32 FMA kernel for
    shapes it declines) against the default FP32 FMA kernel and the oracle: MFCC, delta, clamped log-mel."""
    cfg, secs = _cfg(name)
    y = synth_batch(21, 3, int(cfg.sample_rate * secs) + 11, cfg.sample_rate)
    out = []
    for flags in (_lib.MMF_FLAG_TC_DCT, 0):
        plan = mm.get_plan(mm.plan.replace(cfg, flags=flags))
        lm, cmax = plan.logmel(y)
        mf, dl = plan.mfcc(lm, cmax, delta=True, clamp_in_place=True)
        mf2 = plan.mfcc(lm, cmax, delta=False, clamp_in_place=False)  # no halo, already clamped input
        out.append((lm.cpu().numpy(), mf.cpu().numpy(), dl.cpu().numpy(), mf2.cpu().numpy()))
    assert np.array_equal(out[0][0], out[1][0]), name  # the clamp itself is exact in both
    assert np.max(np.abs(out[0][1] - out[1][1])) < 2e-4, name
    assert np.max(np.abs(out[0][2] - out[1][2])) < 2e-4, name
    assert np.max(np.abs(out[0][3] - out[0][1])) < 2e-4, name
    for i in range(y.shape[0]):
        M, inter, _ = _oracle_unclamped(y[i], cfg)
        assert np.max(np.abs(out[0][1][i] - M)) < ABS_TOL, name
        assert np.max(np.abs(out[0][2][i] - np.gradient(M, axis=1))) < ABS_TOL, name


@pytest.mark.parametrize("name", ["cfg1_16k", "gui_default", "cfg3_44k", "n256"])
def test_mfcc_tensor_core_variant(name, cuda_device):
    """MMF_FLAG_MMA_DCT: clamp + DCT-II (+ delta) through mma.sync TF32 x3 instead of FP32 FMAs."""
    cfg, secs = _cfg(name, flags=_lib.MMF_FLAG_MMA_DCT)
    y = synth_batch(60, 2, int(cfg.sample_rate * secs), cfg.sample_rate)
    plan = mm.get_plan(cfg)
    lm, cmax = plan.logmel(y)
    mf, dl = plan.mfcc(lm, cmax, delta=True)
    lm, mf, dl = lm.cpu().numpy(), mf.cpu().numpy(), dl.cpu().numpy()
    for i in range(2):
        M, inter, _ = _oracle_unclamped(y[i], cfg)
        assert np.max(np.abs(mf[i] - M)) < ABS_TOL
        assert np.max(np.abs(dl[i] - np.gradient(M, axis=1))) < ABS_TOL
        assert np.max(np.abs(lm[i] - inter["logmel"])) < 4.4e-4  # clamped in place


GENERIC_NFFT = {
    # name: (sr, n_fft, win_length, hop, n_mels, n_mfcc, fmin, fmax, seconds): sizes the register FFT does not cover
    "nfft400_win_eq": (16000, 400, 400, 160, 40, 13, 0.0, 8000.0, 2.0),
    "nfft500_gui_rate": (10000, 500, 250, 50, 128, 13, 100.0, 10000.0, 2.0),
    "nfft401_odd": (16000, 401, 321, 160, 40, 13, 0.0, 8000.0, 1.0),
    "nfft128_small": (8000, 128, 100, 40, 24, 12, 0.0, 4000.0, 1.0),
    "nfft1200": (44100, 1200, 1102, 441, 64, 20, 20.0, 22050.0, 1.0),
    "nfft3000": (48000, 3000, 2400, 480, 80, 13, 0.0, 24000.0, 0.5),
}


@pytest.mark.parametrize("name", list(GENERIC_NFFT))
def test_generic_n_fft_matrix_product_dft(name, cuda_device):
    """librosa.stft takes any n_fft (script/mfcc.py:387; the GUI field is free text): everything that is not a
    power of two in [256, 4096] runs the FP32 matrix-product DFT + the sparse mel walk."""
    sr, n_fft, win, hop, n_mels, n_mfcc, fmin, fmax, secs = GENERIC_NFFT[name]
    cfg = mm.MfccConfig(sr, n_fft, win, hop, n_mels, n_mfcc, fmin, fmax)
    y = synth_batch(50, 3, int(sr * secs), sr)
    plan = mm.get_plan(cfg)
    P = plan.stft_power(y).cpu().numpy()
    for i in range(3):
        ref = oracle.stft_power(y[i], n_fft, hop, win)
        assert P[i].shape == ref.shape
        assert np.max(np.abs(P[i] - ref) / ref.max(axis=0, keepdims=True)) < 1e-5
    lm, cmax = plan.logmel(y)
    mf, d = plan.mfcc(lm.clone(), cmax, delta=True)
    for i in range(3):
        M, inter, unclamped = _oracle_unclamped(y[i], cfg)
        assert _mel_rel_err(lm[i].cpu().numpy(), unclamped) < LOGMEL_REL
        assert np.max(np.abs(mf[i].cpu().numpy() - M)) < ABS_TOL
        assert np.max(np.abs(d[i].cpu().numpy() - np.gradient(M, axis=1))) < ABS_TOL
    if name == "nfft500_gui_rate":  # through the reference-facing call
        kw = dict(KW_GUI)
        kw["n_fft"] = 500
        tot, T = mm.get_MFCCS_change(y[0], sr, **kw)
        rtot, rT = oracle.get_MFCCS_change(y[0], sr, **kw)
        assert np.array_equal(T, rT) and np.max(np.abs(tot - rtot)) < ABS_TOL


def test_rejected_plan_leaves_the_next_plan_working(cuda_device):
    """A hop so long that no tile of frames fits in shared memory is rejected when the plan is built. The failed
    construction releases what it allocated, and a valid plan built next in the same process computes log-mel."""
    cfg, secs = _cfg("cfg1_16k")
    with pytest.raises(mm.MmfError) as ei:
        mm.Plan(mm.plan.replace(cfg, hop_length=2000))
    assert ei.value.code == _lib.MMF_ERR_UNSUPPORTED
    assert ei.value.msg == "hop_length/n_fft combination needs more shared memory than one SM has"
    y = synth_batch(12, 2, int(cfg.sample_rate * secs), cfg.sample_rate)
    plan = mm.Plan(cfg)
    try:
        lm = plan.logmel(y)[0].cpu().numpy()
    finally:
        plan.close()
    for i in range(y.shape[0]):
        _, _, unclamped = _oracle_unclamped(y[i], cfg)
        assert _mel_rel_err(lm[i], unclamped) < LOGMEL_REL


def test_clamp_is_active_on_gui_default(cuda_device):
    """fmax above Nyquist leaves empty mel filters at -100 dB, so top_db=80 always clamps."""
    cfg, secs = _cfg("gui_default")
    y = synth_clip(3, int(cfg.sample_rate * secs), cfg.sample_rate)
    plan = mm.get_plan(cfg)
    lm, cmax = plan.logmel(y)
    raw = lm.cpu().numpy()[0].copy()
    plan.mfcc(lm, cmax, clamp_in_place=True)
    clamped = lm.cpu().numpy()[0]
    assert raw.min() == pytest.approx(-100.0)
    assert clamped.min() == pytest.approx(raw.max() - 80.0, abs=1e-4)
    assert (clamped > raw).any()


def test_edge_clips(cuda_device):
    cfg, _ = _cfg("cfg1_16k")
    n = 16000
    plan = mm.get_plan(cfg)
    clips = np.zeros((5, n), np.float32)
    clips[1] = 0.25                                   # DC
    t = np.arange(n) / 16000.0
    clips[2] = 0.5 * np.sin(2 * np.pi * (16000 / 512 * 20) * t)  # tone on bin 20
    clips[3, 0] = 1.0                                 # impulse at the first sample
    clips[4, -1] = 1.0                                # impulse at the last sample
    lm, cmax = plan.logmel(clips)
    raw = lm.cpu().numpy().copy()
    mf = plan.mfcc(lm, cmax).cpu().numpy()
    P = plan.stft_power(clips).cpu().numpy()
    assert np.all(raw[0] == -100.0)                   # all-zero clip: amin floor, no clamp effect
    assert np.argmax(P[2][:, 50]) == 20
    for i in range(5):
        M, inter, unclamped = _oracle_unclamped(clips[i], cfg)
        ref_p = inter["power"]
        assert np.max(np.abs(P[i] - ref_p)) <= 2e-6 * max(ref_p.max(), 1e-30)
        # impulses make most mel bins tiny but non-zero: compare in dB with an absolute bound
        assert np.max(np.abs(mf[i] - M)) < ABS_TOL


@pytest.mark.parametrize("x_dtype", ["f32", "f64"])
@pytest.mark.parametrize("order,wn", [(6, 0.24), (6, 0.12), (2, 0.3), (4, 0.048)])
def test_sosfiltfilt(order, wn, x_dtype, cuda_device):
    torch = _torch()
    rng = np.random.default_rng(7)
    x = rng.standard_normal((5, 12, 333)).cumsum(axis=-1)
    if x_dtype == "f32":
        x = x.astype(np.float32)
    sos = scipy.signal.butter(order, wn, output="sos")
    plan = mm.get_plan(_cfg("cfg1_16k")[0])
    y = plan.sosfiltfilt(torch.as_tensor(x).cuda(), sos).cpu().numpy()
    ref = scipy.signal.sosfiltfilt(sos, x)
    assert y.dtype == np.float64
    assert np.max(np.abs(y - ref)) < 1e-9 * max(1.0, np.abs(ref).max())


def test_sosfiltfilt_bandpass_and_too_short(cuda_device):
    torch = _torch()
    rng = np.random.default_rng(8)
    x = rng.standard_normal((3, 400))
    sos = scipy.signal.butter(4, [0.1, 0.3], btype="bandpass", output="sos")
    plan = mm.get_plan(_cfg("cfg1_16k")[0])
    y = plan.sosfiltfilt(torch.as_tensor(x).cuda(), sos).cpu().numpy()
    assert np.max(np.abs(y - scipy.signal.sosfiltfilt(sos, x))) < 1e-9
    sos6 = scipy.signal.butter(6, 0.24, output="sos")
    ok = plan.sosfiltfilt(torch.as_tensor(x[:, :22]).cuda(), sos6).cpu().numpy()  # T = 22: shortest legal
    assert np.max(np.abs(ok - scipy.signal.sosfiltfilt(sos6, x[:, :22]))) < 1e-9
    with pytest.raises(mm.MmfError) as ei:
        plan.sosfiltfilt(torch.as_tensor(x[:, :21]).cuda(), sos6)
    assert ei.value.code == _lib.MMF_ERR_TOO_SHORT
    assert "greater than padlen, which is 21" in ei.value.msg


@pytest.mark.parametrize("name", ["cfg1_16k", "gui_default", "cfg3_44k", "n1024"])
@pytest.mark.parametrize("flags", [_lib.MMF_FLAG_SCALAR_FFT, _lib.MMF_FLAG_MMA_MEL,
                                   _lib.MMF_FLAG_SCALAR_FFT | _lib.MMF_FLAG_MMA_MEL])
def test_logmel_kernel_variants(name, flags, cuda_device):
    """The non-default code paths of the fused kernel: one frame per thread group on
    scalar FP32 (default: two frames on packed FFMA2/FADD2) and the mel projection on
    the tensor cores (mma.sync TF32 x3; default: sparse FP32 walk)."""
    cfg, secs = _cfg(name, flags=flags)
    y = synth_batch(70, 3, int(cfg.sample_rate * secs), cfg.sample_rate)
    plan = mm.get_plan(cfg)
    lm, cmax = plan.logmel(y)
    lm = lm.cpu().numpy()
    for i in range(3):
        _, _, unclamped = _oracle_unclamped(y[i], cfg)
        assert _mel_rel_err(lm[i], unclamped) <= LOGMEL_REL, (name, flags)


@pytest.mark.parametrize("T", [22, 45, 333, 1001, 2001, 2038, 2039, 5000, 6071, 7000, 40000])
@pytest.mark.parametrize("order", [2, 6, 8, 10])
def test_sosfiltfilt_chunk_parallel_and_sequential_paths(T, order, cuda_device):
    """Rows with T + 2*padlen <= 6112 and <= 4 sections take the chunk-parallel
    kernel (one warp per row, exact state carry across 32 chunks); longer rows the
    super-block scan (state / carry / apply kernels); more than 4 sections the
    sequential kernel.  All must equal scipy."""
    torch = _torch()
    rng = np.random.default_rng(100 + T + order)
    x = (rng.standard_normal((7, T)).cumsum(axis=-1) + 3.0).astype(np.float32)
    sos = scipy.signal.butter(order, 0.24, output="sos")
    plan = mm.get_plan(_cfg("cfg1_16k")[0])
    padlen = 3 * (2 * len(sos) + 1 - min((sos[:, 2] == 0).sum(), (sos[:, 5] == 0).sum()))
    if T <= padlen:
        with pytest.raises(mm.MmfError):
            plan.sosfiltfilt(torch.as_tensor(x).cuda(), sos)
        return
    y = plan.sosfiltfilt(torch.as_tensor(x).cuda(), sos).cpu().numpy()
    ref = scipy.signal.sosfiltfilt(sos, x)
    assert np.max(np.abs(y - ref)) < 1e-9 * max(1.0, np.abs(ref).max())


def test_fused_change_kernel_equals_unfused(cuda_device):
    """change_fused_kernel (rows resident in shared memory) against the separate
    filter / derivative / filter kernels (MMF_FLAG_UNFUSED_CHANGE) and the oracle."""
    sr = 16000
    y = synth_batch(40, 5, sr * 10, sr)
    kw = dict(tStep=0.01, winLen=0.025, n_mfcc=13, n_fft=512, minFreq=0, maxFreq=8000, outFiltCutOff=[12], n_mels=40)
    for over in (dict(), dict(outFilter=None), dict(diffMethod="sg"), dict(removeFirst=0), dict(filtOrd=4, outFiltLen=4),
                 dict(filtOrd=8, outFiltLen=8), dict(outFiltLen=2)):
        k = {**kw, **over}
        fused, T = mm.get_MFCCS_change_batch(y, sr, **k)
        unfused, _ = mm.get_MFCCS_change_batch(y, sr, flags=_lib.MMF_FLAG_UNFUSED_CHANGE, **k)
        assert np.max(np.abs(fused - unfused)) < 1e-11, over
        for i in (0, 4):
            ref, Tref = oracle.get_MFCCS_change(y[i], sr, **k)
            assert np.array_equal(T, Tref)
            assert np.max(np.abs(fused[i] - ref)) < ABS_TOL, over


@pytest.mark.parametrize("name", ["cfg1_16k", "gui_default", "n256"])
@pytest.mark.parametrize("remove_first,clamp", [(1, True), (0, False)])
def test_per_clip_kernel_from_logmel_is_bit_identical(name, remove_first, clamp, cuda_device):
    """The per-clip kernel with clamp + DCT-II folded in (MMF_FLAG_FOLD_MFCC; the default when no
    delta is requested) against the separate MFCC kernel followed by the per-clip kernel
    (MMF_FLAG_SEPARATE_MFCC): same FMA order, so MFCC, delta, the clamped log-mel written back
    and the curve must be bit-identical."""
    cfg, secs = _cfg(name)
    y = synth_batch(77, 3, int(cfg.sample_rate * max(secs, 1.0)), cfg.sample_rate)
    sos = scipy.signal.butter(6, 12.0, "low", fs=cfg.sample_rate / cfg.hop_length, output="sos")
    prm = mm.plan.make_change_params(sos, remove_first=remove_first, diff_method=0, out_sos=sos)
    res = []
    for flags in (_lib.MMF_FLAG_FOLD_MFCC, _lib.MMF_FLAG_SEPARATE_MFCC):
        plan = mm.get_plan(mm.plan.replace(cfg, flags=flags))
        lm, cmax = plan.logmel(y)
        out = plan.change_from_logmel(lm, cmax, prm, want_delta=True, clamp_in_place=clamp)
        res.append({k: v.cpu().numpy() for k, v in out.items()} | {"logmel": lm.cpu().numpy()})
        # no delta requested: the default folds (one launch fewer than with the separate kernel)
        lm2, cmax2 = plan.logmel(y)
        n0 = _lib.lib().mmf_launch_count(0)
        out2 = plan.change_from_logmel(lm2, cmax2, prm, want_delta=False, clamp_in_place=clamp)
        res[-1]["launches"] = _lib.lib().mmf_launch_count(0) - n0
        assert np.array_equal(out2["totChange"].cpu().numpy(), res[-1]["totChange"])
        assert np.array_equal(out2["mfcc"].cpu().numpy(), res[-1]["mfcc"])
    for k in ("logmel", "mfcc", "delta", "totChange"):
        assert np.array_equal(res[0][k], res[1][k]), (name, k)
    assert (res[0]["launches"], res[1]["launches"]) == (1, 2)


KW_GUI = dict(channelN=0, tStep=0.005, winLen=0.025, n_mfcc=13, n_fft=512, minFreq=100, maxFreq=10000, removeFirst=1,
              filtCutoff=12, filtOrd=6, diffMethod="grad", outFilter="iir", outFiltType="low", outFiltCutOff=[12],
              outFiltLen=6, outFiltPolyOrd=3)


def test_get_MFCCS_change_gui_call(cuda_device):
    """The exact call of script/main.py:750-769."""
    y = synth_clip(1, 40000, 10000)
    tot, T = mm.get_MFCCS_change(y, 10000, **KW_GUI)
    ref, Tref = oracle.get_MFCCS_change(y, 10000, **KW_GUI)
    assert tot.dtype == np.float64 and T.dtype == np.float64
    assert np.array_equal(T, Tref)
    assert np.max(np.abs(tot - ref)) < ABS_TOL


@pytest.mark.parametrize(
    "over",
    [
        dict(outFilter=None),
        dict(diffMethod="sg"),
        dict(removeFirst=0),
        dict(outFilter="fir", outFiltLen=11, outFiltCutOff=[12]),
        dict(outFilter="sg", outFiltLen=7, outFiltPolyOrd=3, outFiltCutOff=[12]),
        dict(outFilter="iir", outFiltType="band", outFiltCutOff=[2, 20], outFiltLen=4),
        dict(outFilter="iir", outFiltType="high", outFiltCutOff=[5], outFiltLen=3),
        dict(tStep=0.01, n_fft=1024, winLen=0.04),
    ],
)
def test_get_MFCCS_change_variants(over, cuda_device):
    y = synth_clip(2, 30000, 10000)
    kw = dict(KW_GUI)
    kw.update(over)
    tot, T = mm.get_MFCCS_change(y, 10000, **kw)
    ref, Tref = oracle.get_MFCCS_change(y, 10000, **kw)
    assert np.array_equal(T, Tref)
    assert np.max(np.abs(tot - ref)) < ABS_TOL, over


def test_get_MFCCS_change_multichannel_and_features(cuda_device):
    y2 = np.stack([synth_clip(3, 20000, 10000), synth_clip(4, 20000, 10000)])
    kw = dict(KW_GUI)
    kw["channelN"] = 1
    tot, T, feats = mm.get_MFCCS_change(y2, 10000, return_features=True, **kw)
    ref, Tref, rf = oracle.get_MFCCS_change(y2, 10000, return_features=True, **kw)
    assert np.max(np.abs(tot - ref)) < ABS_TOL
    assert np.max(np.abs(feats["mfcc"] - rf["mfcc"])) < ABS_TOL
    assert np.max(np.abs(feats["logmel"] - rf["logmel"])) < 4.4e-4


def test_get_MFCCS_change_errors(cuda_device):
    y = synth_clip(2, 30000, 10000)
    kw = dict(KW_GUI)
    with pytest.raises(TypeError):  # signature default outFiltCutOff=[None] (script/mfcc.py:308, :93)
        mm.get_MFCCS_change(y, 10000, **{**kw, "outFiltCutOff": [None]})
    with pytest.raises(Exception, match="Cut off frequencies must be smaller"):
        mm.get_MFCCS_change(y, 10000, **{**kw, "outFiltCutOff": [200]})
    with pytest.raises(Exception, match="filtType must be one among"):
        mm.get_MFCCS_change(y, 10000, **{**kw, "outFiltType": "notch"})
    with pytest.raises(ValueError, match="greater than padlen"):  # 21 frames
        mm.get_MFCCS_change(y[: 50 * 20], 10000, **kw)
    with pytest.raises(ValueError):  # win_length > n_fft
        mm.get_MFCCS_change(y, 10000, **{**kw, "winLen": 0.1})


def test_batch_equals_single_and_host_call(cuda_device):
    """Batched clips give bit-identical results to one-at-a-time calls, through both
    the device API and the host-buffer C entry point."""
    sr = 16000
    y = synth_batch(20, 9, sr * 2, sr)
    kw = dict(tStep=0.01, winLen=0.025, n_mfcc=13, n_fft=512, minFreq=0, maxFreq=8000, outFiltCutOff=[12], n_mels=40)
    tot_b, T = mm.get_MFCCS_change_batch(y, sr, **kw)
    for i in (0, 4, 8):
        tot_1, _ = mm.get_MFCCS_change(y[i], sr, **kw)
        assert np.array_equal(tot_b[i], tot_1)
        ref, Tref = oracle.get_MFCCS_change(y[i], sr, **kw)
        assert np.max(np.abs(tot_b[i] - ref)) < ABS_TOL
        assert np.array_equal(T, Tref)
    torch = _torch()
    tot_d, _ = mm.get_MFCCS_change_batch(torch.as_tensor(y).cuda(), sr, **kw)
    assert np.array_equal(tot_d.cpu().numpy(), tot_b)


def test_feature_bundle_and_modspec(cuda_device):
    sr = 16000
    y = synth_batch(30, 3, sr * 10, sr)
    res = mm.mfcc_features_batch(y, sr, tStep=0.01, winLen=0.025, n_fft=512, n_mels=40, n_mfcc=13)
    for i in range(3):
        ref = oracle.mfcc_features(y[i], sr)
        assert np.max(np.abs(res["mfcc"][i] - ref["mfcc"])) < ABS_TOL
        assert np.max(np.abs(res["delta"][i] - ref["delta"])) < ABS_TOL
        assert np.max(np.abs(res["logmel"][i] - ref["logmel"])) < 4.4e-4
        assert np.max(np.abs(res["totChange"][i] - ref["totChange"])) < ABS_TOL
        assert res["modspec"][i].shape == ref["modspec"].shape == (13, 19, 65)
        assert np.max(np.abs(res["modspec"][i] - ref["modspec"])) < ABS_TOL  # north_star: 1e-3 absolute
        assert np.allclose(res["band_energy"][i], ref["band_energy"], rtol=1e-4, atol=1e-3)
        assert np.array_equal(res["T"], ref["T"])


def test_modspec_kernel_alone(cuda_device):
    """The trajectory FFT itself, on identical float32 input: <= 1e-3 absolute."""
    torch = _torch()
    rng = np.random.default_rng(11)
    M = (rng.standard_normal((4, 13, 1001)).cumsum(axis=-1) * 0.5).astype(np.float32)
    plan = mm.get_plan(_cfg("cfg1_16k")[0])
    for (win_s, hop_s, fr) in [(1.0, 0.5, 100.0), (1.0, 0.01, 100.0), (2.0, 0.5, 200.0), (10.01, 1.0, 100.0)]:
        Lw, Hw, nfft, n_win = mm.modspec_sizes(1001, fr, win_s, hop_s)
        bins = mm.band_bins(nfft, fr)
        mag, band = plan.modspec(torch.as_tensor(M).cuda(), Lw, Hw, nfft, bins)
        mag, band = mag.cpu().numpy(), band.cpu().numpy()
        for i in range(4):
            rm, rb, _ = oracle.modulation_spectrum(M[i], fr, mod_win_s=win_s, mod_hop_s=hop_s)
            assert mag[i].shape == rm.shape
            assert np.max(np.abs(mag[i] - rm)) < ABS_TOL
            assert np.allclose(band[i], rb, rtol=2e-6, atol=1e-6)


@pytest.mark.parametrize("flags", [0, _lib.MMF_FLAG_NO_TC_MODSPEC])
def test_modspec_tensor_core_gemm(flags, cuda_device):
    """Default for win <= 128, nfft = 128: windowing + DFT of 128 trajectory windows at a time as one
    tcgen05.mma kind::f16 GEMM (fp16 operand pairs, accumulators in tensor memory); MMF_FLAG_NO_TC_MODSPEC
    selects the FP32 register FFT.  Same bounds for both against the oracle on identical float32 input,
    including a trajectory with a large offset (c0 sits near -500), chunked clips (hop 1), and shapes the
    GEMM path declines (they fall through to the FP32 kernel)."""
    torch = _torch()
    rng = np.random.default_rng(12)
    M = (rng.standard_normal((5, 13, 1001)).cumsum(axis=-1) * 0.5).astype(np.float32)
    M[:, 0] -= 500.0
    cfg = mm.plan.replace(_cfg("cfg1_16k")[0], flags=flags)
    plan = mm.get_plan(cfg)
    for (win_s, hop_s, fr) in [(1.0, 0.5, 100.0), (1.0, 0.01, 100.0), (0.77, 0.13, 100.0), (1.28, 0.5, 100.0),
                               (2.0, 0.5, 200.0)]:
        Lw, Hw, nfft, n_win = mm.modspec_sizes(1001, fr, win_s, hop_s)
        bins = mm.band_bins(nfft, fr)
        n0 = _lib.lib().mmf_launch_count(0)
        mag, band = plan.modspec(torch.as_tensor(M).cuda(), Lw, Hw, nfft, bins)
        assert _lib.lib().mmf_launch_count(0) - n0 == 1
        mag, band = mag.cpu().numpy(), band.cpu().numpy()
        for i in range(M.shape[0]):
            rm, rb, _ = oracle.modulation_spectrum(M[i], fr, mod_win_s=win_s, mod_hop_s=hop_s)
            assert mag[i].shape == rm.shape
            assert np.max(np.abs(mag[i] - rm)) < ABS_TOL, (win_s, hop_s)
            assert np.allclose(band[i], rb, rtol=2e-6, atol=1e-6), (win_s, hop_s)


def test_get_velocity_and_filters(cuda_device):
    rng = np.random.default_rng(5)
    x = rng.standard_normal(777).cumsum()
    for kw in [dict(method="gradient", difference=1), dict(method="gradient", difference=2),
               dict(method="sg", difference=1, width=5, polyOrder=2), dict(method="sg", difference=2, width=7, polyOrder=3),
               dict(method="finDiff", difference=1, accOrder=2), dict(method="finDiff", difference=2, accOrder=2),
               dict(method="finDiff", difference=1, accOrder=4)]:
        for sr in (1.0, 200.0):
            got = mm.get_velocity(x, sr, **kw)
            ref = oracle.get_velocity(x, sr, **kw)
            assert got.dtype == np.float64
            assert np.max(np.abs(got - ref)) <= 1e-9 * max(1.0, np.abs(ref).max()), kw
    with pytest.raises(ValueError, match="Méthode inconnue"):
        mm.get_velocity(x, 1.0, method="nope")
    for kw in [dict(filt="iir", cutOff=[12], filtLen=6), dict(filt="fir", cutOff=[12], filtLen=21),
               dict(filt="fir", cutOff=[5, 30], filtLen=31, filtType="band"), dict(filt="sg", cutOff=[12], filtLen=9, polyOrd=3),
               dict(filt="iir", cutOff=[20], filtLen=4, filtType="high")]:
        got = mm.applyFilter(x, 200.0, **kw)
        ref = oracle.applyFilter(x, 200.0, **kw)
        assert np.max(np.abs(got - ref)) < 1e-9 * max(1.0, np.abs(ref).max()), kw
    assert mm.applyFilter(x, 200.0, filt="unknown", cutOff=[12]) is None


def test_rms_envelope(cuda_device):
    sr = 16000
    y = synth_clip(6, sr * 3, sr)
    amp, t = mm.calculate_amplitude_envelope(y, sr)
    ramp, rt = oracle.calculate_amplitude_envelope(y, sr)
    assert amp.dtype == np.float32 and amp.shape == ramp.shape
    assert np.array_equal(t, rt)
    assert np.allclose(amp, ramp, rtol=1e-4, atol=1e-7)
    # raw int16 PCM, as script/main.py:843-849 passes it
    yi = (y * 32767).astype(np.int16)
    amp, _ = mm.calculate_amplitude_envelope(yi, sr, winLen=0.05, hopLen=0.005, center=False, outFilter="iir", outFiltCutOff=[12])
    ramp, _ = oracle.calculate_amplitude_envelope(yi.astype(np.float32), sr, winLen=0.05, hopLen=0.005, center=False, outFilter="iir", outFiltCutOff=[12])
    assert np.allclose(amp, ramp, rtol=1e-4, atol=1e-3)


def test_preemphasis_extension(cuda_device):
    cfg, _ = _cfg("cfg1_16k", preemph=0.97)
    y = synth_clip(8, 16000, 16000)
    yp = y.copy()
    yp[1:] = y[1:] - np.float32(0.97) * y[:-1]
    P = mm.get_plan(cfg).stft_power(y).cpu().numpy()[0]
    ref = oracle.stft_power(yp, cfg.n_fft, cfg.hop_length, cfg.win_length)
    assert np.max(np.abs(P - ref) / ref.max(axis=0, keepdims=True)) < 2e-6


def test_full_size_properties(cuda_device):
    """BASELINE cfg 2 at full size (1024 x 10 s): size-independent properties."""
    torch = _torch()
    sr, n = 16000, 160000
    pcm = mm.synth_batch_device(1024, n, sr, seed=1234, device=cuda_device)
    fx = mm.FeatureExtractor(sr, tStep=0.01, winLen=0.025, n_fft=512, n_mels=40, n_mfcc=13)
    res = fx(pcm)
    assert res["mfcc"].shape == (1024, 13, 1001) and res["modspec"].shape == (1024, 13, 19, 65)
    for v in res.values():
        assert bool(torch.isfinite(v).all())
    # (1) host-recomputed parity sample
    idx = [0, 511, 1023]
    host = pcm[idx].cpu().numpy()
    for j, i in enumerate(idx):
        ref = oracle.mfcc_features(host[j], sr)
        assert np.max(np.abs(res["mfcc"][i].cpu().numpy() - ref["mfcc"])) < ABS_TOL
        assert np.max(np.abs(res["totChange"][i].cpu().numpy() - ref["totChange"])) < ABS_TOL
    # (2) batch position independence: the same clip anywhere in the batch gives identical bits
    perm = torch.randperm(1024, device=cuda_device, generator=torch.Generator(device=cuda_device).manual_seed(1))
    res_p = fx(pcm[perm].contiguous())
    assert torch.equal(res_p["mfcc"], res["mfcc"][perm])
    assert torch.equal(res_p["totChange"], res["totChange"][perm])
    # (3) gain linearity: x2 amplitude -> +20*log10(2) dB on every unclamped log-mel bin, c0 shifts, c1.. unchanged
    plan = fx.plan
    lm1, _ = plan.logmel(pcm[:64])
    lm2, _ = plan.logmel(pcm[:64] * 0.5)
    assert float((lm1 - lm2 - 20 * np.log10(2.0)).abs().max()) < 2e-4
    # (4) Parseval on the power spectrum: sum_k c_k |X_k|^2 == n_fft * sum_n (w x)^2
    P = plan.stft_power(pcm[:8])
    w = torch.as_tensor(oracle.padded_hann(400, 512), device=cuda_device)
    xp = torch.nn.functional.pad(pcm[:8].double(), (256, 256))
    fr = xp.unfold(1, 512, 160) * w
    lhs = 2 * P.double().sum(dim=1) - P[:, 0].double() - P[:, -1].double()
    rhs = 512 * (fr**2).sum(dim=-1)
    assert float(((lhs - rhs).abs() / rhs).max()) < 1e-5


def test_host_path_multi_chunk_equals_device_path(cuda_device):
    """The e2e entry point the bench times (``mmf_features_host``: 32 MB chunks over two streams and two
    workspace slots) over 5 chunks (float32) / 2 chunks (int16), against the device-resident call and the oracle."""
    torch = _torch()
    sr, n, B = 16000, 160000, 256  # 52 clips per chunk -> 5 chunks (int16: 157 -> 2), the last one ragged
    pcm = mm.synth_batch_device(B, n, sr, seed=4321, device=cuda_device)
    fx = mm.FeatureExtractor(sr, tStep=0.01, winLen=0.025, n_fft=512, n_mels=40, n_mfcc=13)
    dev = fx(pcm, want_logmel=False)
    want = ("totChange", "mfcc", "delta", "modspec", "band_energy")
    host_in = pcm.cpu().numpy()
    out = fx.host_call(host_in, want=want)
    for k in want:
        assert np.array_equal(out[k], dev[k].cpu().numpy()), k
    # a device-resident call in flight on the caller's stream must not disturb a host call on the same plan
    dev2 = fx(pcm[:64], want_logmel=False)
    out2 = fx.host_call(host_in[100:180], want=want)
    for k in want:
        assert np.array_equal(out2[k], out[k][100:180]), k
        assert torch.equal(dev2[k], dev[k][:64]), k
    for i in (0, 51, 52, 233, 255):  # both sides of a chunk boundary, first and last clip
        ref = oracle.mfcc_features(host_in[i], sr)
        assert np.max(np.abs(out["mfcc"][i] - ref["mfcc"])) < ABS_TOL
        assert np.max(np.abs(out["totChange"][i] - ref["totChange"])) < ABS_TOL
        assert np.max(np.abs(out["modspec"][i] - ref["modspec"])) < ABS_TOL
    # int16 ingest: 96 MB chunks (157 clips), samples scaled by 1/32768 on the device
    q = torch.clamp(torch.round(pcm * 32768.0), -32768, 32767).to(torch.int16)
    out16 = fx.host_call(q.cpu().numpy(), want=want)
    devq = fx(q.to(torch.float32) / 32768.0, want_logmel=False)
    for k in want:
        assert np.array_equal(out16[k], devq[k].cpu().numpy()), k
    # strided host rows (clip_stride > n_samples) take the 2-D copy path
    wide = np.zeros((160, n + 64), np.float32)
    wide[:, :n] = host_in[:160]
    out_s = fx.host_call(wide[:, :n], want=("totChange", "mfcc"))
    assert np.array_equal(out_s["totChange"], out["totChange"][:160])
    assert np.array_equal(out_s["mfcc"], out["mfcc"][:160])


def test_integer_audio_semantics(cuda_device):
    """librosa rejects integer audio (valid_audio under script/mfcc.py:387); the host-buffer C entry points
    take int16 explicitly and scale by 1/32768."""
    sr = 16000
    f32 = synth_batch(40, 3, sr * 2, sr)
    pcm16 = np.clip(np.round(f32 * 32768.0), -32768, 32767).astype(np.int16)
    kw = dict(tStep=0.01, winLen=0.025, n_mfcc=13, n_fft=512, minFreq=0, maxFreq=8000, outFiltCutOff=[12], n_mels=40)
    with pytest.raises(mm.ParameterError, match="floating-point"):
        mm.get_MFCCS_change(pcm16[0], sr, **kw)
    with pytest.raises(mm.ParameterError, match="floating-point"):
        mm.get_MFCCS_change_batch(pcm16, sr, **kw)
    with pytest.raises(mm.ParameterError, match="floating-point"):
        mm.get_MFCCS_change_batch(_torch().as_tensor(pcm16).cuda(), sr, **kw)
    # Plan.mfcc_change_host: int16 goes to mmf_features_host_pcm16 (no float reinterpretation of the buffer)
    from modulation_mfcc_b200.api import _butter_sos, _change_setup

    plan = _change_setup(sr, 0.01, 0.025, 13, 512, 0, 8000, 40, 0.0, None)
    sos = _butter_sos(6, 12 / 50.0, "low")
    prm = mm.make_change_params(sos, out_sos=sos)
    a, ma = plan.mfcc_change_host(pcm16, prm, want_mfcc=True)
    b, mb = plan.mfcc_change_host(pcm16.astype(np.float32) / 32768.0, prm, want_mfcc=True)
    assert np.array_equal(a, b) and np.array_equal(ma, mb)
    c = plan.mfcc_change_host(np.ascontiguousarray(np.pad(pcm16, ((0, 0), (0, 6))))[:, : pcm16.shape[1]], prm)  # strided rows
    assert np.array_equal(c, a)
    ref, _ = oracle.get_MFCCS_change(pcm16[1].astype(np.float32) / 32768.0, sr, **kw)
    assert np.max(np.abs(a[1] - ref)) < ABS_TOL


def test_cfg4_one_hour_recording_full_size(cuda_device):
    """BASELINE configs[3] at its stated size: one 1-hour 16 kHz recording (57.6 M samples, T = 360 001 frames),
    MFCC-change curve through the long-row zero-phase filters and the modulation spectrum over 1 s windows at
    0.5 s hop and at a one-frame hop, against the oracle run on the same hour of audio."""
    sr, secs = 16000, 3600
    n = sr * secs
    rng = np.random.default_rng(77)
    t = np.arange(n, dtype=np.float64) / sr
    # speech-rate AM/FM carrier + noise with slowly drifting level, so windows an hour apart differ
    y = (0.08 * (1.0 + 0.5 * np.sin(2 * np.pi * t / 600.0)) * rng.standard_normal(n)
         + 0.3 * np.sin(2 * np.pi * (200.0 + 50.0 * np.sin(2 * np.pi * 3.0 * t)) * t) * (0.6 + 0.4 * np.sin(2 * np.pi * 4.0 * t)))
    y = np.clip(y, -1.0, 1.0).astype(np.float32)
    del t
    res = mm.mfcc_features_batch(y[None, :], sr, tStep=0.01, winLen=0.025, n_fft=512, n_mels=40, n_mfcc=13)
    T = 360001
    assert res["mfcc"].shape == (1, 13, T) and res["totChange"].shape == (1, T)
    ref = oracle.mfcc_features(y, sr)
    assert np.array_equal(res["T"], ref["T"])
    assert np.max(np.abs(res["logmel"][0] - ref["logmel"])) < 4.4e-4
    assert np.max(np.abs(res["mfcc"][0] - ref["mfcc"])) < ABS_TOL
    assert np.max(np.abs(res["delta"][0] - ref["delta"])) < ABS_TOL
    assert np.max(np.abs(res["totChange"][0] - ref["totChange"])) < ABS_TOL
    assert res["modspec"].shape[1:] == ref["modspec"].shape == (13, 7199, 65)
    assert np.max(np.abs(res["modspec"][0] - ref["modspec"])) < ABS_TOL
    assert np.allclose(res["band_energy"][0], ref["band_energy"], rtol=1e-4, atol=1e-3)
    # one-frame hop (359 902 windows): a slice of windows from the start, the middle and the end of the hour
    torch = _torch()
    fx = mm.FeatureExtractor(sr, tStep=0.01, winLen=0.025, n_fft=512, n_mels=40, n_mfcc=13, mod_hop_s=0.01)
    mfcc_dev = torch.as_tensor(ref["mfcc"][None]).cuda()  # identical input on both sides
    Lw, Hw, nfft, bins = fx.modspec_geometry(T)
    assert (Lw, Hw, nfft) == (100, 1, 128)
    mag, band = fx.plan.modspec(mfcc_dev, Lw, Hw, nfft, bins)
    assert mag.shape == (1, 13, T - Lw + 1, 65)
    for j0 in (0, 180000, T - Lw - 63):
        seg = ref["mfcc"][:, j0 : j0 + Lw + 63]
        rmag, rband, _ = oracle.modulation_spectrum(seg, 100.0, mod_win_s=1.0, mod_hop_s=0.01)
        assert np.max(np.abs(mag[0, :, j0 : j0 + 64].cpu().numpy() - rmag)) < ABS_TOL
        assert np.allclose(band[0, j0 : j0 + 64].cpu().numpy(), rband, rtol=2e-4, atol=1e-3)


def test_pcm16_host_path_is_bit_identical(cuda_device):
    """int16 PCM in (scaled by 1/32768 on the device) == the float32 call on x/32768."""
    sr = 16000
    rng = np.random.default_rng(5)
    pcm16 = np.clip(np.round(synth_batch(80, 5, sr * 3, sr) * 32768.0), -32768, 32767).astype(np.int16)
    pcm16[0, :10] = [-32768, 32767, 0, 1, -1, 2, -2, 100, -100, 5]
    f32 = pcm16.astype(np.float32) / 32768.0
    fx = mm.FeatureExtractor(sr, tStep=0.01, winLen=0.025, n_fft=512, n_mels=40, n_mfcc=13)
    want = ("totChange", "mfcc", "delta", "modspec", "band_energy")
    a = {k: v.copy() for k, v in fx.host_call(pcm16, want=want).items()}
    b = fx.host_call(f32, want=want)
    for k in want:
        assert np.array_equal(a[k], b[k]), k
    ref = oracle.mfcc_features(f32[2], sr)
    assert np.max(np.abs(a["mfcc"][2] - ref["mfcc"])) < ABS_TOL
    torch = _torch()
    y = fx.plan.pcm16_to_f32(torch.as_tensor(pcm16).cuda()).cpu().numpy()
    assert np.array_equal(y, f32)


@pytest.mark.parametrize("up,down,n", [(160, 441, 44100), (1, 2, 10001), (3, 1, 5000), (441, 160, 8000), (2, 3, 97), (1000, 997, 6000)])
def test_resample_poly_matches_scipy(up, down, n, cuda_device):
    rng = np.random.default_rng(up * 1000 + down)
    x = rng.standard_normal((3, n)).astype(np.float32)
    plan = mm.get_plan(_cfg("cfg1_16k")[0])
    y = plan.resample_poly(x, up, down).cpu().numpy()
    ref = scipy.signal.resample_poly(x.astype(np.float64), up, down, axis=-1)
    assert y.shape == ref.shape
    assert np.max(np.abs(y - ref)) < 2e-5 * max(1.0, np.abs(ref).max())


def test_load_channel_wav_pcm16_and_resample(cuda_device, tmp_path):
    """load_channel: WAV parse on the host, PCM16 scaling and rate conversion on the device."""
    from scipy.io import wavfile

    sr_file, sr = 44100, 16000
    y = synth_clip(7, sr_file * 2, sr_file)
    pcm = np.clip(np.round(y * 32767.0), -32768, 32767).astype(np.int16)
    path = str(tmp_path / "clip.wav")
    wavfile.write(path, sr_file, pcm)
    got = mm.load_channel(path, sr)
    # the loader converts the rate with libsoxr HQ's band limits (what librosa.load applies at script/mfcc.py:373);
    # the device kernel against the same taps applied by scipy's upfirdn in float64
    from modulation_mfcc_b200.plan import design_resample_filter

    h, n_pre, n_out = design_resample_filter(len(pcm), 160, 441, "hq")
    want = scipy.signal.upfirdn(h.astype(np.float64), pcm.astype(np.float64) / 32768.0, 160, 441)[n_pre : n_pre + n_out]
    assert got.dtype == np.float32 and got.shape == want.shape
    assert np.max(np.abs(got - want)) < 2e-6
    # ... and a pure tone below the band edge against the ideal resampling (through the 16-bit file: 2^-16 rounding)
    tone = np.sin(2 * np.pi * 5000.0 * np.arange(sr_file) / sr_file) * 0.5
    wavfile.write(str(tmp_path / "tone.wav"), sr_file, np.round(tone * 32767.0).astype(np.int16))
    got_t = mm.load_channel(str(tmp_path / "tone.wav"), sr)
    ideal = np.sin(2 * np.pi * 5000.0 * np.arange(len(got_t)) / sr) * 0.5 * 32767.0 / 32768.0
    assert np.max(np.abs(got_t - ideal)[800:-800]) < 4e-5
    same = mm.load_channel(path, sr_file)
    assert np.array_equal(same, pcm.astype(np.float32) / 32768.0)
    # a path goes straight through get_MFCCS_change like an array does (script/mfcc.py:372-380)
    tot_p, T_p = mm.get_MFCCS_change(path, sr, **{**KW_GUI, "tStep": 0.01, "maxFreq": 8000, "minFreq": 0})
    tot_a, T_a = mm.get_MFCCS_change(got, sr, **{**KW_GUI, "tStep": 0.01, "maxFreq": 8000, "minFreq": 0})
    assert np.array_equal(T_p, T_a) and np.array_equal(tot_p, tot_a)


def test_find_peaks_matches_scipy(cuda_device):
    """Landmarks of the curve (script/main.py:1566, :1601): default scipy.signal.find_peaks."""
    rng = np.random.default_rng(12)
    x = rng.standard_normal((6, 777)).cumsum(axis=-1)
    x[1] = np.round(x[1])            # flat tops and flat valleys
    x[2, 100:140] = x[2, 100]        # a long plateau
    x[3] = 0.0                       # constant row: no peaks
    x[4, :] = np.arange(777)         # monotone: no peaks
    sr = 16000
    y = synth_batch(90, 2, sr * 10, sr)
    tot, _ = mm.get_MFCCS_change_batch(y, sr, tStep=0.01, winLen=0.025, n_mfcc=13, n_fft=512, minFreq=0, maxFreq=8000,
                                       outFiltCutOff=[12], n_mels=40)
    plan = mm.get_plan(_cfg("cfg1_16k")[0])
    for data in (x, tot):
        for minima in (False, True):
            idx, cnt = plan.find_peaks(data, minima=minima)
            idx, cnt = idx.cpu().numpy(), cnt.cpu().numpy()
            for r in range(data.shape[0]):
                ref, _ = scipy.signal.find_peaks(-data[r] if minima else data[r])
                assert cnt[r] == len(ref)
                assert np.array_equal(idx[r, : cnt[r]], ref)
    idx, cnt = plan.find_peaks(x[0], max_peaks=3)
    ref, _ = scipy.signal.find_peaks(x[0])
    assert int(cnt[0]) == len(ref) and np.array_equal(idx[0].cpu().numpy(), ref[:3])


GOLDEN_DIR = __import__("os").path.join(__import__("os").path.dirname(__import__("os").path.abspath(__file__)), "golden")
GOLDEN_CASES = {
    # name: (seed, sr, seconds, kwargs) -- the recipe of tests/golden/make_golden.py
    "cfg1_16k_40mel": (0, 16000, 2.0, dict(tStep=0.01, winLen=0.025, n_fft=512, n_mels=40, n_mfcc=13)),
    "cfg3_44k_128mel": (1, 44100, 1.0, dict(tStep=0.01, winLen=0.025, n_fft=2048, n_mels=128, n_mfcc=20)),
    "gui_default_10k": (2, 10000, 2.0, dict(tStep=0.005, winLen=0.025, n_fft=512, n_mels=128, n_mfcc=13, fmin=100, fmax=10000)),
    "cfg4_long_hop": (3, 16000, 4.0, dict(tStep=0.01, winLen=0.025, n_fft=512, n_mels=40, n_mfcc=13, mod_hop_s=0.01)),
}


@pytest.mark.parametrize("name", list(GOLDEN_CASES))
def test_cuda_path_against_committed_golden_vectors(name, cuda_device):
    """The CUDA path against the committed fixtures themselves (no oracle call at test time)."""
    import os

    seed, sr, secs, kw = GOLDEN_CASES[name]
    g = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    y = synth_clip(seed, int(sr * secs), sr)
    assert np.array_equal(y[:64], g["y_head"]) and len(y) == int(g["n"])
    res = mm.mfcc_features_batch(y[None, :], sr, **kw)
    assert np.array_equal(res["T"], g["T"])
    # clamped log-mel: absolute dB bound equivalent to 1e-4 relative on linear power
    assert np.max(np.abs(res["logmel"][0] - g["logmel"])) < 4.4e-4
    assert np.max(np.abs(res["mfcc"][0] - g["mfcc"])) < ABS_TOL
    assert np.max(np.abs(res["delta"][0] - g["delta"])) < ABS_TOL
    assert np.max(np.abs(res["totChange"][0] - g["totChange"])) < ABS_TOL
    step = 10 if name == "cfg4_long_hop" else 1
    ms = res["modspec"][0][:, ::step]
    assert ms.shape == g["modspec"].shape
    assert np.max(np.abs(ms - g["modspec"])) < ABS_TOL  # north_star: 1e-3 absolute on modulation magnitudes
    be = res["band_energy"][0]
    assert np.max(np.abs(be - g["band_energy"]) / np.maximum(1.0, np.abs(g["band_energy"]))) < 2e-3


def test_cuda_path_against_golden_edge_cases(cuda_device):
    import os

    g = np.load(os.path.join(GOLDEN_DIR, "edge_cases.npz"))
    n, sr = 8000, 16000
    t = np.arange(n) / sr
    z = np.zeros(n, np.float32)
    imp0, impN = z.copy(), z.copy()
    imp0[0], impN[-1] = 1.0, 1.0
    clips = {"zero": z, "dc": np.full(n, 0.25, np.float32), "tone_bin20": (0.5 * np.sin(2 * np.pi * (sr / 512 * 20) * t)).astype(np.float32),
             "impulse_first": imp0, "impulse_last": impN}
    cfg = mm.MfccConfig(sr, 512, 400, 160, 40, 13, 0.0, 8000.0)
    plan = mm.get_plan(cfg)
    for k, y in clips.items():
        lm, cmax = plan.logmel(y[None, :])
        mf = plan.mfcc(lm, cmax).cpu().numpy()[0]
        assert np.max(np.abs(mf - g[k + "_mfcc"])) < ABS_TOL, k
    y22 = synth_clip(9, 21 * 50, 10000)
    kw = dict(tStep=0.005, winLen=0.025, n_mfcc=13, n_fft=512, minFreq=100, maxFreq=10000, outFiltCutOff=[12])
    tot, T = mm.get_MFCCS_change(y22, 10000, **kw)
    assert np.array_equal(T, g["t22_T"]) and np.max(np.abs(tot - g["t22_tot"])) < ABS_TOL


@pytest.mark.parametrize("n", [160000, 16000, 12345, 4097, 4096, 1000, 100, 441000, 65537])
def test_hilbert_envelope_matches_scipy(n, cuda_device):
    """'Hilb' amplitude (script/calc.py:284-286): |scipy.signal.hilbert(x)| at the signal's own length -- even, odd,
    prime (65537), 2^k; above 4096 samples through the O(n log n) Bluestein path."""
    x = synth_clip(13, n, 16000)
    plan = mm.get_plan(_cfg("cfg1_16k")[0])
    amp = plan.hilbert_envelope(x).cpu().numpy()
    ref = np.abs(scipy.signal.hilbert(x.astype(np.float64)))
    assert amp.shape == ref.shape
    assert np.max(np.abs(amp - ref)) < (2e-6 if n > 4096 else 1e-4)
    if n == 16000:
        a, t = mm.calculate_amplitude_envelope(x, 16000, method="Hilb")
        ra, rt = oracle.calculate_amplitude_envelope(x, 16000, method="Hilb")
        assert np.max(np.abs(a - ra)) < 1e-4 and np.array_equal(t, rt)


def test_hilbert_envelope_batch_and_one_hour(cuda_device):
    torch = _torch()
    plan = mm.get_plan(_cfg("cfg1_16k")[0])
    xb = synth_batch(70, 3, 30011, 16000)
    amp = plan.hilbert_envelope(xb).cpu().numpy()
    for i in range(3):
        assert np.max(np.abs(amp[i] - np.abs(scipy.signal.hilbert(xb[i].astype(np.float64))))) < 2e-6
    # one hour at 16 kHz (57.6 M samples): analytic known answer, an amplitude-modulated carrier on an exact bin
    n = 57_600_000
    t = torch.arange(n, device=cuda_device, dtype=torch.float64)
    env = 0.6 + 0.3 * torch.cos(2 * torch.pi * 5.0 * t / n)
    x = (env * torch.cos(2 * torch.pi * 1_000_000.0 * t / n)).to(torch.float32)
    got = plan.hilbert_envelope(x)
    assert float((got.double() - env).abs().max()) < 1e-5


def _random_cases(n_cases=28, seed=2026):
    rng = np.random.default_rng(seed)
    cases = []
    for i in range(n_cases):
        sr = int(rng.choice([8000, 10000, 16000, 22050, 44100]))
        n_fft = int(rng.choice([256, 512, 512, 1024, 2048]))
        win = int(rng.integers(max(16, n_fft // 4), n_fft + 1))
        hop = int(rng.integers(max(1, win // 8), win + 1))
        n_mels = int(rng.integers(8, 161))
        n_mfcc = int(rng.integers(2, min(40, n_mels) + 1))
        fmin = float(rng.choice([0.0, 50.0, 300.0]))
        fmax = float(rng.choice([sr / 2, 0.4 * sr, 1.2 * sr]))
        frames = int(rng.integers(25, 140))
        n = frames * hop + int(rng.integers(0, hop))
        clips = int(rng.integers(1, 4))
        cases.append((i, sr, n_fft, win, hop, n_mels, n_mfcc, fmin, fmax, n, clips))
    return cases


@pytest.mark.parametrize("case", _random_cases(), ids=lambda c: f"r{c[0]}_fft{c[2]}_w{c[3]}_h{c[4]}_m{c[5]}")
def test_randomised_configurations(case, cuda_device):
    """Seeded sweep over frame geometry and filterbank shapes (odd hops and clip lengths take the
    non-vector and non-TMA loaders, win == n_fft, fmax above Nyquist, narrow and wide banks)."""
    i, sr, n_fft, win, hop, n_mels, n_mfcc, fmin, fmax, n, clips = case
    cfg = mm.MfccConfig(sr, n_fft, win, hop, n_mels, n_mfcc, fmin, fmax)
    y = synth_batch(200 + 7 * i, clips, n, sr)
    plan = mm.get_plan(cfg)
    lm, cmax = plan.logmel(y)
    lm_unclamped = lm.cpu().numpy().copy()
    mf, dl = plan.mfcc(lm, cmax, delta=True)
    mf, dl = mf.cpu().numpy(), dl.cpu().numpy()
    for c in range(clips):
        M, inter, unclamped = _oracle_unclamped(y[c], cfg)
        assert lm_unclamped[c].shape == unclamped.shape
        assert _mel_rel_err(lm_unclamped[c], unclamped) <= LOGMEL_REL
        assert np.max(np.abs(mf[c] - M)) < ABS_TOL
        assert np.max(np.abs(dl[c] - np.gradient(M, axis=1))) < ABS_TOL


def _random_change_cases(n_cases=14, seed=77):
    rng = np.random.default_rng(seed)
    out = []
    for i in range(n_cases):
        sr = int(rng.choice([10000, 16000]))
        tStep = float(rng.choice([0.005, 0.01, 0.0125]))
        kw = dict(
            tStep=tStep, winLen=0.025, n_mfcc=int(rng.integers(3, 21)), n_fft=512, minFreq=float(rng.choice([0, 100])),
            maxFreq=float(rng.choice([sr / 2, sr])), removeFirst=int(rng.integers(0, 2)),
            filtCutoff=float(rng.choice([6, 12, 18])), filtOrd=int(rng.choice([2, 4, 6, 8, 10])),
            diffMethod=str(rng.choice(["grad", "sg"])), outFilter=rng.choice([None, "iir", "fir", "sg"]),
            outFiltType=str(rng.choice(["low", "high"])), outFiltCutOff=[float(rng.choice([5, 12, 20]))],
            outFiltLen=int(rng.choice([3, 5, 6, 7, 9])), outFiltPolyOrd=2, n_mels=int(rng.choice([40, 64, 128])),
        )
        if kw["outFilter"] == "fir" and kw["outFiltType"] == "high" and kw["outFiltLen"] % 2 == 0:
            kw["outFiltLen"] += 1  # scipy refuses an even-length high-pass FIR
        secs = float(rng.choice([1.5, 4.0, 9.0, 25.0]))  # 25 s at 5 ms steps: rows beyond the shared-memory IIR
        out.append((i, sr, secs, kw))
    return out


@pytest.mark.parametrize("case", _random_change_cases(), ids=lambda c: f"c{c[0]}")
def test_randomised_change_pipeline(case, cuda_device):
    """Seeded sweep over the post-MFCC part of get_MFCCS_change: filter orders (fused kernel up to
    4 sections, sequential beyond), derivative methods, every output-filter branch, short and long rows."""
    i, sr, secs, kw = case
    y = synth_batch(300 + i, 2, int(sr * secs), sr)
    tot, T = mm.get_MFCCS_change_batch(y, sr, **kw)
    for c in range(2):
        ref, Tref = oracle.get_MFCCS_change(y[c], sr, **kw)
        assert np.array_equal(T, Tref)
        assert np.max(np.abs(tot[c] - ref)) < ABS_TOL, kw


def test_zero_phase_filter_properties_full_size(cuda_device):
    """Size-independent property of K4 at the bench's row count (12 288 rows x 1001 frames): linearity
    (odd extension, zi * x[0] start-up and both passes are linear in x), plus a scipy sample."""
    torch = _torch()
    g = torch.Generator(device=cuda_device).manual_seed(3)
    x = torch.randn((12288, 1001), device=cuda_device, dtype=torch.float64, generator=g).cumsum(dim=-1)
    y = torch.randn((12288, 1001), device=cuda_device, dtype=torch.float64, generator=g)
    sos = scipy.signal.butter(6, 0.24, output="sos")
    plan = mm.get_plan(_cfg("cfg1_16k")[0])
    fx, fy = plan.sosfiltfilt(x, sos), plan.sosfiltfilt(y, sos)
    fz = plan.sosfiltfilt(2.0 * x - 3.0 * y, sos)
    scale = float(x.abs().max())
    assert float((fz - (2.0 * fx - 3.0 * fy)).abs().max()) < 1e-9 * scale
    ref = scipy.signal.sosfiltfilt(sos, x[:3].cpu().numpy())
    assert np.max(np.abs(fx[:3].cpu().numpy() - ref)) < 1e-9 * scale


# ---------------------------------------------------------------------------------------------------
# K1 with the mel projection on the tcgen05 tensor cores (csrc/stft_mel_tc.cu)
# ---------------------------------------------------------------------------------------------------
TC_MEL_CASES = {
    # name: (sr, winLen, tStep, n_mels, fmin, fmax, seconds, preemph)
    "cfg2_40mel": (16000, 0.025, 0.01, 40, 0.0, 8000.0, 3.0, 0.0),
    "mel64_fmin": (16000, 0.032, 0.008, 64, 60.0, 7600.0, 2.0, 0.0),
    "mel26_8k": (8000, 0.03, 0.0125, 26, 0.0, 4000.0, 2.5, 0.0),
    "mel13_oddhop": (16000, 0.02, 0.0100625, 13, 0.0, 8000.0, 2.0, 0.0),  # hop 161: scalar span loads
    "mel40_preemph": (16000, 0.025, 0.01, 40, 0.0, 8000.0, 2.0, 0.97),
    # the reference GUI's default (script/main.py:739): 128 bands up to 10 kHz at a 10 kHz sampling rate -- the bands
    # above the Nyquist frequency are empty, 100 remain: 112 accumulator columns per term
    "gui_default_128": (10000, 0.025, 0.005, 128, 100.0, 10000.0, 2.0, 0.0),
    "mel96_fmax_low": (16000, 0.025, 0.01, 96, 0.0, 6000.0, 1.5, 0.0),
}


def _tc_cfg(name, flags):
    sr, winLen, tStep, n_mels, fmin, fmax, secs, pre = TC_MEL_CASES[name]
    win, hop = mm.frame_sizes(sr, winLen, tStep)
    return mm.MfccConfig(sr, 512, win, hop, n_mels, 13, fmin, fmax, preemph=pre, flags=flags), secs


def test_tcgen05_mel_plain_loader_is_bit_identical(cuda_device):
    """Unaligned input (or MMF_FLAG_NO_TMA) takes the plain span loader of the same kernel: identical bits."""
    torch = _torch()
    cfg, secs = _tc_cfg("cfg2_40mel", 0)
    y = synth_batch(303, 4, int(cfg.sample_rate * secs), cfg.sample_rate)
    a, ka = mm.get_plan(cfg).logmel(y)
    b, kb = mm.get_plan(mm.plan.replace(cfg, flags=_lib.MMF_FLAG_NO_TMA)).logmel(y)
    assert torch.equal(a, b) and torch.equal(ka, kb)
    # a row pitch that is not a multiple of 16 bytes cannot be described to the TMA unit
    wide = torch.zeros((4, y.shape[1] + 1), device=cuda_device)
    wide[:, : y.shape[1]] = torch.as_tensor(y)
    c, kc = mm.get_plan(cfg).logmel(wide[:, : y.shape[1]])
    assert torch.equal(a, c) and torch.equal(ka, kc)


@pytest.mark.parametrize("name", list(TC_MEL_CASES))
def test_logmel_tcgen05_mel_projection(name, cuda_device):
    """The default K1 of batches (mel projection as a tcgen05 GEMM over 128-frame blocks, bf16 operand pairs) against
    the oracle (north_star: 1e-4 on linear mel power) and against the CUDA-core kernel; per-clip maxima agree."""
    cfg, secs = _tc_cfg(name, 0)
    y = synth_batch(300, 5, int(cfg.sample_rate * secs), cfg.sample_rate)
    y[3] *= 1000.0  # loud clip
    y[4] *= 1e-4   # near-silent clip: most bands sit on the amin floor
    lm, cmax = mm.get_plan(cfg).logmel(y)
    cfg_ref, _ = _tc_cfg(name, _lib.MMF_FLAG_NO_TC_MEL)
    lm_ref, cmax_ref = mm.get_plan(cfg_ref).logmel(y)
    lm, lm_ref = lm.cpu().numpy(), lm_ref.cpu().numpy()
    assert np.isfinite(lm).all()
    assert _mel_rel_err(lm, lm_ref) <= LOGMEL_REL, name
    km, kr = cmax.cpu().numpy().view(np.float32), cmax_ref.cpu().numpy().view(np.float32)
    assert np.max(np.abs(km - kr)) < 4.4e-4, name  # per-clip max keys are the float bits of a non-negative-or-not dB value
    if cfg.preemph == 0.0:
        for i in range(y.shape[0]):
            _, _, unclamped = _oracle_unclamped(y[i], cfg)
            assert _mel_rel_err(lm[i], unclamped) <= LOGMEL_REL, (name, i)


@pytest.mark.parametrize("n_samples", [1, 159, 160, 10079, 10080, 10240, 20319, 20320, 20480, 20481, 40000])
def test_tcgen05_mel_ragged_lengths(n_samples, cuda_device):
    """Frame counts around the 64-frame tile and 128-frame block edges (T = 1, 63, 64, 65, 127, 128, 129, ...): blocks
    with one tile, partly filled tiles, rows beyond T never stored."""
    cfg, _ = _tc_cfg("cfg2_40mel", 0)
    y = synth_batch(301, 3, n_samples, cfg.sample_rate)
    plan = mm.get_plan(cfg)
    lm, cmax = plan.logmel(y)
    lm = lm.cpu().numpy()
    assert lm.shape[2] == 1 + n_samples // cfg.hop_length
    for i in range(3):
        _, _, unclamped = _oracle_unclamped(y[i], cfg)
        assert _mel_rel_err(lm[i], unclamped) <= LOGMEL_REL, (n_samples, i)
    ref, cref = mm.get_plan(_tc_cfg("cfg2_40mel", _lib.MMF_FLAG_NO_TC_MEL)[0]).logmel(y)
    assert np.max(np.abs(cmax.cpu().numpy().view(np.float32) - cref.cpu().numpy().view(np.float32))) < 4.4e-4


def test_tcgen05_mel_is_the_default_and_feeds_the_whole_path(cuda_device):
    """n_fft = 512 with up to 64 bands takes the tcgen05 kernel without any flag; the composite call (MFCC, delta,
    MFCC-change curve, modulation spectrum) stays within the north_star bounds of the oracle."""
    sr = 16000
    y = synth_batch(302, 160, sr * 2, sr)  # T = 201 -> 2 blocks per clip, 320 blocks
    res = mm.mfcc_features_batch(y, sr, tStep=0.01, winLen=0.025, n_fft=512, n_mels=40, n_mfcc=13)
    ref_flags = mm.mfcc_features_batch(y, sr, tStep=0.01, winLen=0.025, n_fft=512, n_mels=40, n_mfcc=13,
                                       flags=_lib.MMF_FLAG_NO_TC_MEL)
    assert not np.array_equal(res["mfcc"], ref_flags["mfcc"])  # different kernels really ran
    for i in (0, 77, 159):
        ref = oracle.mfcc_features(y[i], sr)
        assert np.max(np.abs(res["mfcc"][i] - ref["mfcc"])) < ABS_TOL
        assert np.max(np.abs(res["totChange"][i] - ref["totChange"])) < ABS_TOL
        assert np.max(np.abs(res["modspec"][i] - ref["modspec"])) < ABS_TOL


def test_batch_size_never_changes_a_clip(cuda_device):
    """Kernel selection by batch size (per-clip fused output filter below 32 clips, one launch over all clips above)
    must not change a single bit of a clip's features; neither may the position of the clip in the batch."""
    sr = 16000
    y = synth_batch(304, 40, sr * 3, sr)
    big = mm.mfcc_features_batch(y, sr, tStep=0.01, winLen=0.025, n_fft=512, n_mels=40, n_mfcc=13)
    for i in (0, 17, 39):
        one = mm.mfcc_features_batch(y[i : i + 1], sr, tStep=0.01, winLen=0.025, n_fft=512, n_mels=40, n_mfcc=13)
        for k in ("mfcc", "delta", "totChange", "modspec", "band_energy"):
            assert np.array_equal(one[k][0], big[k][i]), (k, i)
    small = mm.mfcc_features_batch(y[8:20], sr, tStep=0.01, winLen=0.025, n_fft=512, n_mels=40, n_mfcc=13)
    for k in ("mfcc", "delta", "totChange", "modspec", "band_energy"):
        assert np.array_equal(small[k], big[k][8:20]), k
    # the GUI's own call (no delta output -> MFCC stage folded into the per-clip kernel), both batch regimes
    kw = dict(KW_GUI, tStep=0.01, n_mels=40, maxFreq=8000)
    c1, T1 = mm.get_MFCCS_change(y[5], sr, **kw)
    cb, Tb = mm.get_MFCCS_change_batch(y, sr, **{k: v for k, v in kw.items() if k != "channelN"})
    assert np.array_equal(c1, cb[5]) and np.array_equal(T1, Tb)


def test_tcgen05_mel_is_deterministic_under_load(cuda_device):
    """compute-sanitizer is not available on the GPU pool, so hazards in the kernel's hand-rolled synchronisation
    (named barriers per group, TMA / MMA mbarriers, the last-arriver MMA issue, exchange buffers reused as row
    staging) are hunted the blunt way: a batch with ~14 blocks per CTA, 25 launches, every bit equal -- and equal
    to the same clips run in small batches, where each CTA sees a different block sequence."""
    torch = _torch()
    cfg, _ = _tc_cfg("cfg2_40mel", 0)
    pcm = mm.synth_batch_device(260, 16000 * 10, 16000, seed=77, device=cuda_device)
    plan = mm.get_plan(cfg)
    lm0, k0 = plan.logmel(pcm)
    lm0, k0 = lm0.clone(), k0.clone()
    for _ in range(25):
        lm, k = plan.logmel(pcm)
        assert torch.equal(lm, lm0) and torch.equal(k, k0)
    for b0 in (0, 37, 255):
        lm, k = plan.logmel(pcm[b0 : b0 + 5])
        assert torch.equal(lm, lm0[b0 : b0 + 5]) and torch.equal(k, k0[b0 : b0 + 5])


def test_cfg3_full_size_properties(cuda_device):
    """BASELINE configs[2] at its stated size (512 x 10 s at 44.1 kHz, n_fft 2048, 128 mel, 20 MFCC): an oracle
    sample, finiteness, batch-position independence and gain linearity on the whole batch."""
    torch = _torch()
    sr, n, B = 44100, 441000, 512
    pcm = mm.synth_batch_device(B, n, sr, seed=4242, device=cuda_device)
    fx = mm.FeatureExtractor(sr, tStep=0.01, winLen=0.025, n_fft=2048, n_mels=128, n_mfcc=20)
    res = fx(pcm, want_logmel=False)
    T = 1 + n // 441
    assert res["mfcc"].shape == (B, 20, T)
    for v in res.values():
        assert v is None or bool(torch.isfinite(v).all())
    for i in (0, 511):
        ref = oracle.mfcc_features(pcm[i].cpu().numpy(), sr, n_fft=2048, n_mels=128, n_mfcc=20)
        assert np.max(np.abs(res["mfcc"][i].cpu().numpy() - ref["mfcc"])) < ABS_TOL
        assert np.max(np.abs(res["totChange"][i].cpu().numpy() - ref["totChange"])) < ABS_TOL
        assert np.max(np.abs(res["modspec"][i].cpu().numpy() - ref["modspec"])) < ABS_TOL
    perm = torch.randperm(B, device=cuda_device, generator=torch.Generator(device=cuda_device).manual_seed(3))
    res_p = fx(pcm[perm].contiguous(), want_logmel=False)
    assert torch.equal(res_p["mfcc"], res["mfcc"][perm]) and torch.equal(res_p["totChange"], res["totChange"][perm])
    lm1, _ = fx.plan.logmel(pcm[:32])
    lm2, _ = fx.plan.logmel(pcm[:32] * 0.5)
    assert float((lm1 - lm2 - 20 * np.log10(2.0)).abs().max()) < 2e-4
