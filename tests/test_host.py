"""CPU tests of the host-side logic: the C-ABI library loads and exports every
symbol include/mmf.h declares, its host tables equal the oracle's, the drop-in
modules keep the reference's signatures, and the kernel-phase emulator (the exact
__host__ __device__ code of the CUDA kernel, run thread by thread on the CPU)
reproduces numpy's rfft.  No compute call needs a GPU here."""

import ctypes
import inspect
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import scipy.signal

import oracle
import modulation_mfcc_b200 as mm
from modulation_mfcc_b200 import _lib
from modulation_mfcc_b200.synth import synth_clip

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "mmf.h")).read()
    declared = set(re.findall(r"\b(mmf_[a-z0-9_]+)\s*\(", hdr))
    assert declared, "no declarations parsed"
    lib = mm.lib()
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in mmf.h but not exported"
    assert declared == set(mm.exported_symbols())
    assert lib.mmf_version() == 100
    assert lib.mmf_num_frames(160000, 512, 160) == 1001
    assert lib.mmf_num_frames(100, 512, 50) == 3


def test_flag_constants_match_header():
    """Every MMF_FLAG_* of include/mmf.h has the same value in the ctypes binding, and all are distinct bits."""
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "mmf.h")).read()
    flags = {m.group(1): int(m.group(2)) for m in re.finditer(r"#define (MMF_FLAG_\w+) (\d+)", hdr)}
    assert len(flags) >= 11
    for name, val in flags.items():
        assert getattr(_lib, name) == val, name
        assert val & (val - 1) == 0, name
    assert len(set(flags.values())) == len(flags)


def test_struct_layouts_match_header():
    lib = mm.lib()
    assert ctypes.sizeof(_lib.mmf_config) == lib.mmf_abi_sizeof(0)
    assert ctypes.sizeof(_lib.mmf_change_params) == lib.mmf_abi_sizeof(1)
    assert ctypes.sizeof(_lib.mmf_modspec_params) == lib.mmf_abi_sizeof(2)
    assert _lib.mmf_config.fmin.offset == 32 and _lib.mmf_config.amin.offset == 48


@pytest.mark.parametrize(
    "cfg",
    [
        mm.MfccConfig(16000, 512, 400, 160, 40, 13, 0.0, 8000.0),
        mm.MfccConfig(10000, 512, 250, 50, 128, 13, 100.0, 10000.0),
        mm.MfccConfig(44100, 2048, 1102, 441, 128, 20, 0.0, 22050.0),
        mm.MfccConfig(22050, 1024, 551, 220, 64, 16, 50.0, 11025.0),
    ],
)
def test_host_tables_equal_oracle(cfg):
    w, mel, dct = mm.host_tables(cfg)
    assert np.array_equal(w, oracle.padded_hann(cfg.win_length, cfg.n_fft).astype(np.float32))
    assert np.array_equal(mel, oracle.mel_filterbank(cfg.sample_rate, cfg.n_fft, cfg.n_mels, cfg.fmin, cfg.fmax))
    assert np.max(np.abs(dct - oracle.dct_ortho_matrix(cfg.n_mfcc, cfg.n_mels))) < 1e-7


def test_config_validation_without_gpu():
    lib = mm.lib()
    bad = mm.MfccConfig(16000, 8192, 400, 160, 40, 13).to_c()
    assert lib.mmf_host_tables(ctypes.byref(bad), None, None, None) == _lib.MMF_ERR_UNSUPPORTED
    assert b"n_fft must be in [16, 4096]" in lib.mmf_last_error()
    # any n_fft in range is accepted (librosa takes any; non powers of two run the matrix-product DFT)
    ok = mm.MfccConfig(16000, 500, 400, 160, 40, 13)
    w, m, d = mm.host_tables(ok)
    assert w.shape == (500,) and m.shape == (40, 251) and np.allclose(w, oracle.padded_hann(400, 500), atol=1e-7)
    assert np.max(np.abs(m - oracle.mel_filterbank(16000, 500, 40, 0.0, 8000.0))) < 3e-7
    bad = mm.MfccConfig(16000, 512, 600, 160, 40, 13).to_c()
    assert lib.mmf_host_tables(ctypes.byref(bad), None, None, None) == _lib.MMF_ERR_INVALID
    assert b"at least input size" in lib.mmf_last_error()


def test_sos_zi_and_padlen():
    for sos in (scipy.signal.butter(6, 0.24, output="sos"), scipy.signal.butter(4, [0.1, 0.3], btype="band", output="sos"),
                scipy.signal.butter(1, 0.2, output="sos"), scipy.signal.butter(5, 0.2, btype="high", output="sos")):
        zi, padlen = mm.sos_zi(sos)
        assert np.max(np.abs(zi - scipy.signal.sosfilt_zi(sos))) < 1e-12
        ntaps = 2 * sos.shape[0] + 1 - min((sos[:, 2] == 0).sum(), (sos[:, 5] == 0).sum())
        assert padlen == 3 * ntaps


def test_no_cpu_fallback():
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(mm.MmfError, match="no CUDA device"):
        mm.get_MFCCS_change(np.zeros(16000, np.float32), 16000, tStep=0.01, outFiltCutOff=[12])
    h = ctypes.c_void_p()
    cfg = mm.MfccConfig(16000).to_c()
    assert mm.lib().mmf_plan_create(ctypes.byref(h), ctypes.byref(cfg)) == _lib.MMF_ERR_CUDA


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "modulation_mfcc_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(import|from)\s+oracle\b", src, re.M), f
    for f in ("script/mfcc.py", "script/calc.py"):
        assert "oracle" not in open(os.path.join(ROOT, f)).read()
    # helper scripts under tools/ are not test infrastructure either (studies that need the oracle live in tests/studies)
    for f in os.listdir(os.path.join(ROOT, "tools")):
        if f.endswith(".py"):
            src = open(os.path.join(ROOT, "tools", f)).read()
            assert not re.search(r"^\s*(import|from)\s+oracle\b", src, re.M), f


# ---------------------------------------------------------------------------
# drop-in signatures (reference: script/mfcc.py:29-39,137-150,262-264,291-311;
# script/calc.py:23-33,221-234,593-601)
# ---------------------------------------------------------------------------

REFERENCE_SIGNATURES = {
    ("mfcc", "applyFilter"): "(x, sr, /, *, filt='iir', cutOff=[None], filtLen=6, filtType='low', polyOrd=3, coeffs=None)",
    ("mfcc", "get_amplitude"): "(x, sr, /, *, method='RMS', winLen=0.1, hopLen=0.01, center=True, outFilter=None, outFiltType='low', outFiltCutOff=[12], outFiltLen=6, outFiltPolyOrd=3)",
    ("mfcc", "load_channel"): "(file_path, signal_sample_rate=10000, channel_nb=0)",
    ("mfcc", "get_MFCCS_change"): "(audioIn, sigSr, /, *, channelN=0, tStep=0.001, winLen=0.025, n_mfcc=13, n_fft=512, minFreq=100, maxFreq=10000, removeFirst=1, filtCutoff=12, filtOrd=6, diffMethod='grad', outFilter='iir', outFiltType='low', outFiltCutOff=[None], outFiltLen=6, outFiltPolyOrd=3)",
    ("calc", "applyFilter"): "(x, sr, /, *, filt='iir', cutOff=[None], filtLen=6, filtType='low', polyOrd=3, coeffs=None)",
    ("calc", "calculate_amplitude_envelope"): "(x, sr, /, *, method='RMS', winLen=0.1, hopLen=0.01, center=True, outFilter=None, outFiltType='low', outFiltCutOff=[12], outFiltLen=6, outFiltPolyOrd=3)",
    ("calc", "get_velocity"): "(x, sr, difference=1, method='gradient', width=3, accOrder=2, polyOrder=2)",
}
ADDITIVE = {"n_mels", "preemph", "return_features", "device"}  # allowed extra keywords, reference defaults


def _load_shim(name):
    import importlib.util

    spec = importlib.util.spec_from_file_location(f"shim_{name}", os.path.join(ROOT, "script", f"{name}.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _strip(sig: inspect.Signature) -> str:
    params = [p.replace(annotation=inspect.Parameter.empty) for p in sig.parameters.values() if p.name not in ADDITIVE]
    return str(sig.replace(parameters=params, return_annotation=inspect.Signature.empty))


@pytest.mark.parametrize("key", list(REFERENCE_SIGNATURES))
def test_shim_signatures(key):
    mod = _load_shim(key[0])
    assert _strip(inspect.signature(getattr(mod, key[1]))) == REFERENCE_SIGNATURES[key]


def test_reference_signatures_table_matches_reference_source():
    """When the checkout of the original project is present, parse it and make
    sure the table above is what the reference really declares."""
    import ast

    from oracle import ref_loader

    ref = ref_loader.script_dir()
    if not ref_loader.available():
        pytest.skip(f"the original project's scripts are not under {ref} (set $MMF_REFERENCE_ROOT)")
    for (modname, fn), expect in REFERENCE_SIGNATURES.items():
        tree = ast.parse(open(os.path.join(ref, modname + ".py")).read())
        node = next(n for n in ast.walk(tree) if isinstance(n, ast.FunctionDef) and n.name == fn)
        a = node.args
        names = [x.arg for x in a.posonlyargs + a.args + a.kwonlyargs]
        exp_names = re.findall(r"([A-Za-z_][A-Za-z_0-9]*)(?==|,|\))", expect.replace("/", "").replace("*", ""))
        exp_names = [n for n in exp_names if n not in ("None", "True", "False")]
        assert names == [n for n in exp_names if n in names] and set(names) <= set(exp_names), (modname, fn)
        assert len(a.posonlyargs) == (2 if "/" in expect else 0)
        defaults = [ast.literal_eval(d) for d in a.defaults] + [ast.literal_eval(d) for d in a.kw_defaults if d is not None]
        for d in defaults:
            assert repr(d) in expect or str(d) in expect


def test_shim_modules_export_what_main_imports():
    # script/main.py:29-36 and script/ui.py:6
    m, c = _load_shim("mfcc"), _load_shim("calc")
    for n in ("load_channel", "get_MFCCS_change"):
        assert callable(getattr(m, n))
    for n in ("calc_formants", "calculate_amplitude_envelope", "get_f0", "get_velocity", "read_AG50x", "MinMaxFinder"):
        assert hasattr(c, n)
    with pytest.raises(NotImplementedError):
        c.get_f0()
    f = c.MinMaxFinder()
    t = np.linspace(0, 1, 101)
    v = np.sin(2 * np.pi * 3 * t)
    tx, vx = f.analyse_maximum(t, v, (0.0, 1.0))
    assert len(tx) == 3 and np.allclose(vx, 1.0, atol=1e-2)
    tn, vn = f.analyse_minimum(t, v, (0.0, 0.5))
    assert len(tn) == 1
    assert f.analyse_maximum(t, v, None) == ([], [])


def test_argument_validation_happens_before_any_gpu_work():
    """Reference error behaviour that must not depend on a device."""
    x = np.random.default_rng(0).standard_normal(200)
    with pytest.raises(ValueError, match="Méthode inconnue"):
        mm.get_velocity(x, 1.0, method="bogus")
    with pytest.raises(NotImplementedError):
        mm.calculate_amplitude_envelope(x, 100.0, method="RMSpraat")


def test_stencil_probing_matches_scipy():
    from modulation_mfcc_b200.api import _findiff_stencil, _savgol_stencil

    def apply(c, el, er, x):
        half, ne = (len(c) - 1) // 2, el.shape[0]
        y = np.zeros_like(x)
        for t in range(len(x)):
            if t < ne:
                y[t] = el[t] @ x[: el.shape[1]]
            elif t >= len(x) - ne:
                y[t] = er[t - (len(x) - ne)] @ x[len(x) - er.shape[1] :]
            else:
                y[t] = sum(c[o + half] * x[t + o] for o in range(-half, half + 1))
        return y

    x = np.random.default_rng(3).standard_normal(60)
    for w, p, d in [(3, 2, 1), (5, 2, 0), (7, 3, 2), (6, 3, 0), (9, 4, 1)]:
        ref = scipy.signal.savgol_filter(x, w, p, deriv=d, mode="interp")
        assert np.max(np.abs(apply(*_savgol_stencil(w, p, d), x) - ref)) < 1e-12
    for d, a in [(1, 2), (2, 2), (1, 4), (2, 4), (1, 6)]:
        ref = oracle.mfcc_oracle._findiff_apply(x, 1.0, d, a)
        assert np.max(np.abs(apply(*_findiff_stencil(d, a), x) - ref)) < 1e-11


# ---------------------------------------------------------------------------
# host emulator of the kernel phases
# ---------------------------------------------------------------------------


@pytest.fixture(scope="module")
def emu():
    so = os.path.join(ROOT, "tests", "emu", "libmmf_emu.so")
    src = os.path.join(ROOT, "tests", "emu", "emu_stft.cu")
    hdrs = [os.path.join(ROOT, "modulation_mfcc_b200", "csrc", h) for h in ("stft_core.cuh", "fft_regs.cuh")]
    stale = not os.path.exists(so) or any(os.path.getmtime(so) < os.path.getmtime(p) for p in [src] + hdrs)
    if stale:
        nvcc = "/usr/local/cuda/bin/nvcc"
        if not os.path.exists(nvcc):
            if not os.path.exists(so):
                pytest.skip("nvcc not available to build the emulator")
        else:
            subprocess.run([nvcc, "-O2", "-std=c++17", "--extended-lambda", "-shared", "-Xcompiler", "-fPIC", "-o", so, src],
                           check=True, capture_output=True)
    lib = ctypes.CDLL(so)
    fp = ctypes.POINTER(ctypes.c_float)
    lib.emu_stft_power.argtypes = [fp, ctypes.c_long, ctypes.c_int, ctypes.c_int, fp, fp, ctypes.c_long, ctypes.c_int]
    lib.emu_mel.argtypes = [fp, ctypes.c_long, ctypes.c_int, ctypes.POINTER(ctypes.c_int), fp, ctypes.c_int, ctypes.c_int, fp]
    lib.emu_mel_groups.argtypes = [fp, ctypes.c_long, ctypes.c_int, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int), fp,
                                   ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, fp]
    return lib


def _p(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_float))


def test_emulated_butterflies(emu):
    rng = np.random.default_rng(0)
    for n, fn in ((16, emu.emu_dft16), (8, emu.emu_dft8)):
        x = rng.standard_normal(2 * n).astype(np.float32)
        out = np.zeros(2 * n, np.float32)
        fn(_p(x), _p(out))
        ref = np.fft.fft(x[0::2] + 1j * x[1::2])
        assert np.max(np.abs(out[0::2] + 1j * out[1::2] - ref)) < 2e-6


@pytest.mark.parametrize("nfft,sr,win,hop", [(256, 8000, 200, 80), (512, 16000, 400, 160), (512, 10000, 250, 50),
                                             (1024, 22050, 551, 220), (2048, 44100, 1102, 441), (4096, 44100, 4096, 1000)])
def test_emulated_stft_matches_numpy(emu, nfft, sr, win, hop):
    y = synth_clip(3, sr // 2, sr)
    w = oracle.padded_hann(win, nfft).astype(np.float32)
    T = oracle.n_frames(len(y), nfft, hop)
    ref = oracle.stft_power(y, nfft, hop, win)
    # mode bit 0: split step from registers (n_fft 512 only); bit 1: two frames per thread group
    # through the packed value type (the code path of the FFMA2/FADD2 kernel)
    for mode in ([0, 1, 2, 3] if nfft == 512 else [0, 2]):
        pw = np.zeros((nfft // 2 + 1, T), np.float32)
        assert emu.emu_stft_power(_p(y), len(y), nfft, hop, _p(w), _p(pw), T, mode) == 0
        assert np.max(np.abs(pw - ref)) / ref.max() < 1e-6, mode


def _sparse_mel(cfg):
    """Python restatement of host_mel_sparse() for the emulator test."""
    _, mel, _ = mm.host_tables(cfg)
    F = cfg.n_bins
    mel_f = oracle.mel_to_hz(np.linspace(oracle.hz_to_mel(cfg.fmin), oracle.hz_to_mel(cfg.fmax), cfg.n_mels + 2))
    fk = np.fft.rfftfreq(cfg.n_fft, 1.0 / cfg.sample_rate)
    seg = np.searchsorted(mel_f, fk, side="right") - 1
    w2 = np.zeros((F, 2), np.float32)
    for k in range(F):
        for m in np.nonzero(mel[:, k])[0]:
            assert m in (seg[k] - 1, seg[k])
            w2[k, 0 if m == seg[k] - 1 else 1] = mel[m, k]
    seg_start = np.array([int(np.argmax(seg >= j)) if np.any(seg >= j) else F for j in range(cfg.n_mels + 2)], np.int32)
    return mel, seg_start, w2


@pytest.mark.parametrize("cfg,bpw", [(mm.MfccConfig(16000, 512, 400, 160, 40, 13, 0.0, 8000.0), 3),
                                     (mm.MfccConfig(10000, 512, 250, 50, 128, 13, 100.0, 10000.0), 8),
                                     (mm.MfccConfig(44100, 2048, 1102, 441, 128, 20, 0.0, 22050.0), 2)])
def test_emulated_sparse_mel_equals_dense(emu, cfg, bpw):
    mel, seg_start, w2 = _sparse_mel(cfg)
    rng = np.random.default_rng(4)
    P = rng.random((cfg.n_bins, 7)).astype(np.float32)
    out = np.zeros((cfg.n_mels, 7), np.float32)
    emu.emu_mel(_p(P), 7, cfg.n_bins, seg_start.ctypes.data_as(ctypes.POINTER(ctypes.c_int)), _p(w2), cfg.n_mels, bpw, _p(out))
    ref = mel.astype(np.float64) @ P.astype(np.float64)
    assert np.max(np.abs(out - ref)) <= 2e-6 * max(1.0, np.abs(ref).max())


def _mel_groups(cfg, pp):
    """Python restatement of host_mel_groups() (csrc/host_tables.cpp) for the emulator test."""
    mel, seg_start, w2 = _sparse_mel(cfg)
    F = cfg.n_bins
    segtab, segstep, w = [], [], []
    pos = 0
    for j in range(cfg.n_mels + 2):
        a = int(seg_start[j])
        b = int(seg_start[j + 1]) if j <= cfg.n_mels else a
        g0 = a // 4
        g1 = (b + 3) // 4 if b > a else g0
        segtab.append((g0, len(w) // 8))
        segstep.append((g1 - g0, (g0 - pos) * 2 * pp if j else 0))
        pos = g1
        for g in range(g0, g1):
            ks = [4 * g + i for i in range(4)]
            w += [float(w2[k, 0]) if a <= k < b and k < F else 0.0 for k in ks]
            w += [float(w2[k, 1]) if a <= k < b and k < F else 0.0 for k in ks]
    segstep.append((0, 0))
    return mel, np.array(segtab, np.int32), np.array(segstep, np.int32), np.array(w, np.float32)


@pytest.mark.parametrize("cfg,bpw,tf,two", [(mm.MfccConfig(16000, 512, 400, 160, 40, 13, 0.0, 8000.0), 5, 32, 1),
                                            (mm.MfccConfig(10000, 512, 250, 50, 128, 13, 100.0, 10000.0), 16, 32, 1),
                                            (mm.MfccConfig(44100, 2048, 1102, 441, 128, 20, 0.0, 22050.0), 7, 8, 1),
                                            (mm.MfccConfig(8000, 256, 200, 80, 32, 12, 0.0, 4000.0), 4, 32, 0),
                                            (mm.MfccConfig(16000, 512, 400, 160, 40, 13, 300.0, 7000.0), 40, 16, 1)])
def test_emulated_grouped_mel_equals_dense(emu, cfg, bpw, tf, two):
    """The grouped mel walk on the bin-pair power tile (the kernel's default mel phase), run on the CPU from the
    same __host__ __device__ code: equals the dense filterbank product for every band split and tile shape."""
    mel, segtab, segstep, w = _mel_groups(cfg, tf + 2)
    rng = np.random.default_rng(4)
    T = 45  # ragged last tile
    P = (rng.random((cfg.n_bins, T)) * 10.0 ** rng.uniform(-6, 3, (cfg.n_bins, 1))).astype(np.float32)
    out = np.zeros((cfg.n_mels, T), np.float32)
    ip = ctypes.POINTER(ctypes.c_int)
    rc = emu.emu_mel_groups(_p(P), T, cfg.n_bins, segtab.ctypes.data_as(ip), segstep.ctypes.data_as(ip), _p(w), cfg.n_mels, bpw, tf, two, _p(out))
    assert rc == 0
    ref = mel.astype(np.float64) @ P.astype(np.float64)
    assert np.max(np.abs(out - ref) / np.maximum(ref, 1e-30)) <= 2e-6


def test_operand_split_accuracy_study():
    """Host emulation behind the tcgen05 kernels' operand format (tests/studies/tf32_dft_study.py): single TF32
    operands miss the 1e-4 mel-power bound by far, the three-term TF32 split and the fp16 pair split (what
    tc_fft.cu / modspec_tc.cu / mfcc_tc.cu use) sit at the fp32 FFT's own error."""
    import importlib.util

    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "studies", "tf32_dft_study.py")
    spec = importlib.util.spec_from_file_location("tf32_dft_study", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    err = mod.study(n_clips=1, seconds=0.5, verbose=False)
    assert err["tf32 x1"] > 1e-4
    assert err["tf32 x3"] < 1e-5 and err["fp16 x3"] < 1e-5
    assert err["fp16 x3"] < 3 * err["fp32 FFT"]


def test_plan_cache_is_lru_and_never_closes_live_plans(monkeypatch):
    """ADVICE r1: the plan cache must evict the least recently used entry and must not close() a plan
    that another object may still hold (device memory goes with the last reference)."""
    from modulation_mfcc_b200 import plan as plan_mod

    closed = []

    class FakePlan:
        def __init__(self, cfg):
            self.cfg = cfg

        def close(self):
            closed.append(self.cfg)

    monkeypatch.setattr(plan_mod, "Plan", FakePlan)
    monkeypatch.setattr(plan_mod, "_PLANS", type(plan_mod._PLANS)())
    cfgs = [mm.MfccConfig(8000.0 + i) for i in range(plan_mod._MAX_PLANS + 3)]
    first = plan_mod.get_plan(cfgs[0])
    for c in cfgs[1 : plan_mod._MAX_PLANS]:
        plan_mod.get_plan(c)
    assert plan_mod.get_plan(cfgs[0]) is first  # refreshes cfgs[0]
    for c in cfgs[plan_mod._MAX_PLANS :]:
        plan_mod.get_plan(c)
    assert len(plan_mod._PLANS) == plan_mod._MAX_PLANS
    assert cfgs[0] in plan_mod._PLANS  # most recently used survived
    assert cfgs[1] not in plan_mod._PLANS and cfgs[2] not in plan_mod._PLANS and cfgs[3] not in plan_mod._PLANS
    assert closed == []  # evicted plans are dropped, not closed


def test_integer_audio_is_rejected_before_any_gpu_work():
    """librosa.util.valid_audio semantics under script/mfcc.py:387."""
    with pytest.raises(mm.ParameterError, match="floating-point"):
        mm.get_MFCCS_change(np.zeros(4000, np.int16), 10000, outFiltCutOff=[12])


@pytest.mark.parametrize("sr_in,sr_out", [(44100, 16000), (48000, 16000), (22050, 16000), (16000, 10000), (8000, 16000)])
def test_hq_resampler_is_transparent_below_the_band_edge(sr_in, sr_out):
    """The loader's rate conversion (``quality="hq"``: libsoxr HQ's band limits, script/mfcc.py:373 -> librosa.load)
    reproduces band-limited content below 0.9 of the lower Nyquist within 1e-5 of the ideal resampling, and removes
    content above the lower Nyquist by >= 100 dB; the scipy-compatible filter (Kaiser-5) is two decades worse in
    the pass band -- the deviation from the reference's loader that round 1 left unquantified."""
    from fractions import Fraction

    import scipy.signal

    from modulation_mfcc_b200.plan import design_resample_filter

    fr = Fraction(sr_out, sr_in)
    up, down = fr.numerator, fr.denominator
    n = sr_in
    t = np.arange(n) / sr_in
    nyq = min(sr_in, sr_out) / 2

    def run(x, quality):
        h, n_pre, n_out = design_resample_filter(n, up, down, quality)
        y = scipy.signal.upfirdn(h.astype(np.float64), x, up, down)
        return y[n_pre : n_pre + n_out]

    edge = int(0.05 * sr_out)
    for frac in (0.05, 0.5, 0.9):
        f = frac * nyq
        y = run(np.sin(2 * np.pi * f * t), "hq")
        assert len(y) == -(-n * up // down)
        ref = np.sin(2 * np.pi * f * np.arange(len(y)) / sr_out)
        assert np.max(np.abs(y - ref)[edge:-edge]) < 1e-5, (frac, np.max(np.abs(y - ref)[edge:-edge]))
    if sr_out < sr_in:  # alias rejection: a tone just above the new Nyquist must vanish
        y = run(np.sin(2 * np.pi * (1.02 * nyq) * t), "hq")
        assert np.max(np.abs(y)[edge:-edge]) < 1e-5
    y_sp = run(np.sin(2 * np.pi * 0.5 * nyq * t), "scipy")
    ref = np.sin(2 * np.pi * 0.5 * nyq * np.arange(len(y_sp)) / sr_out)
    assert 1e-4 < np.max(np.abs(y_sp - ref)[edge:-edge]) < 5e-3
    # the scipy-compatible design is scipy's own
    x = np.random.default_rng(0).standard_normal(4000)
    h, n_pre, n_out = design_resample_filter(len(x), up, down, "scipy")
    mine = scipy.signal.upfirdn(h.astype(np.float64), x, up, down)[n_pre : n_pre + n_out]
    assert np.max(np.abs(mine - scipy.signal.resample_poly(x, up, down))) < 2e-6


def test_bf16_pair_mel_projection_accuracy():
    """Host emulation of the operand format of K1's tcgen05 mel projection (csrc/stft_mel_tc.cu): power = b1 + b2
    (the fp32 value rounded half-up to bf16 -- half an ulp added to the bits, top half kept, as the kernel does --
    and the top 16 bits of the exact remainder), weights
    = w1 + w2 (round-to-nearest bf16 pair), D = b1.w1 + (b1.w2 + b2.w1) accumulated in fp32.  On the oracle's own power
    spectra the mel powers stay within 3.5e-5 of the float64 projection (north_star bound 1e-4); a single bf16 operand
    (no b2 / w2) misses the bound by two decades, which is why the kernel carries the pair."""
    sr = 16000
    rng = np.random.default_rng(5)
    worst_pair, worst_single = 0.0, 0.0
    for n_mels, fmax in ((40, 8000.0), (64, 7600.0), (128, 8000.0)):
        y = mm_synth(rng, sr)
        _, inter = oracle.mfcc(y, sr, n_mfcc=13, win_length=400, hop_length=160, n_fft=512, fmin=0.0, fmax=fmax, n_mels=n_mels,
                               return_intermediates=True)
        P = inter["power"].astype(np.float32)              # [257, T]
        W = oracle.mel_filterbank(sr, 512, n_mels, 0.0, fmax).astype(np.float32)  # [n_mels, 257]
        ref = W.astype(np.float64) @ P.astype(np.float64)

        def trunc16(x):
            return (x.view(np.uint32) & np.uint32(0xFFFF0000)).view(np.float32)

        def rn16(x):
            u = x.view(np.uint32).astype(np.uint64)
            u = (u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFF0000
            return u.astype(np.uint32).view(np.float32)

        b1 = trunc16((P.view(np.uint32) + np.uint32(0x8000)).view(np.float32))
        b2 = trunc16(P - b1)
        w1 = rn16(W)
        w2 = rn16(W - w1)
        d1 = w1 @ b1                                        # fp32 accumulation, like the tensor core's
        d2 = w2 @ b1 + w1 @ b2
        got = (d1 + d2).astype(np.float64)
        floor = ref.max() * 1e-8                            # the top_db = 80 clamp floor of the clip
        ok = ref > floor
        worst_pair = max(worst_pair, float(np.max(np.abs(got - ref)[ok] / ref[ok])))
        worst_single = max(worst_single, float(np.max(np.abs((w1 @ b1).astype(np.float64) - ref)[ok] / ref[ok])))
    assert worst_pair < 3.5e-5, worst_pair
    assert worst_single > 1e-3, worst_single


def mm_synth(rng, sr):
    t = np.arange(2 * sr) / sr
    y = 0.1 * rng.standard_normal(t.size) + 0.3 * np.sin(2 * np.pi * (200 + 50 * np.sin(2 * np.pi * 3 * t)) * t) * (0.6 + 0.4 * np.sin(2 * np.pi * 4 * t))
    return np.clip(y, -1, 1).astype(np.float32)
