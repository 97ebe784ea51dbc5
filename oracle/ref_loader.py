"""Run the reference's own ``script/mfcc.py`` and ``script/calc.py`` -- UNMODIFIED -- in this image.

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``).  The reference modules need
librosa, parselmouth, pyqtgraph, xarray and findiff at import time
(``script/mfcc.py:1-27``, ``script/calc.py:1-19``); none is installed and there is no
network.  Everything *around* those imports -- time anchors, dropping c0, ``butter`` +
``sosfiltfilt``, ``np.gradient`` / ``savgol_filter``, the norm over coefficients, the
whole of ``applyFilter``, ``get_velocity`` and the envelope driver
(``mfcc.py:29-135, 137-259, 372-427``; ``calc.py:23-129, 221-343, 593-650``) -- is plain
numpy/scipy and runs here as written once the five missing packages are replaced by
stub modules in ``sys.modules``:

* ``librosa.feature.mfcc`` -> ``oracle.mfcc`` (the restated librosa chain, SURVEY
  Appendix A.1-A.7; cross-checked against torchaudio / transformers in
  ``tests/test_oracle.py``) -- this is the one step that stays a restatement,
* ``librosa.feature.rms`` -> ``oracle.rms_frames``,
* ``librosa.load`` / ``librosa.core.load`` -> WAV reader (scipy) for files already at the
  requested rate; anything else raises (soxr is not available either),
* ``findiff.FinDiff`` -> the restated stencils (``oracle.findiff_stencils``),
* ``parselmouth``, ``pyqtgraph``, ``xarray`` -> empty stubs (Praat / GUI / EMA code paths
  are outside the hot path and raise if touched).

The modules are executed from where they lie in the checkout of the original project at
``reference_path`` of ``BASELINE.json``, or at ``$MMF_REFERENCE_ROOT`` when that is set (never
copied).  That checkout is not part of this repository, so the outputs of these functions are
committed as golden vectors (``tests/golden/ref_*.npz``, minted by
``tests/golden/make_ref_golden.py``); ``available()`` says whether the live reference can
be used in the current process.
"""

from __future__ import annotations

import importlib.util
import json
import os
import sys
import types

import numpy as np


def _baseline_reference_path() -> str:
    with open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "BASELINE.json")) as f:
        return json.load(f)["reference_path"]


REFERENCE_ROOT = os.environ.get("MMF_REFERENCE_ROOT") or _baseline_reference_path()
_loaded: dict[str, types.ModuleType] = {}


def script_dir() -> str:
    """Where the original ``script/mfcc.py`` and ``script/calc.py`` are looked for."""
    return os.path.join(REFERENCE_ROOT, "script")


def available() -> bool:
    return os.path.isfile(os.path.join(script_dir(), "mfcc.py")) and os.path.isfile(os.path.join(script_dir(), "calc.py"))


class _Untouchable(types.ModuleType):
    """Stub module: importing it works, using anything from it raises."""

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)

        def _raise(*a, **k):
            raise NotImplementedError(f"{self.__name__}.{name} is stubbed in oracle/ref_loader.py (outside the hot path)")

        return _raise


def _librosa_stub():
    from . import mfcc_oracle as o

    def mfcc(y=None, sr=22050, n_mfcc=20, **kw):
        # librosa.feature.mfcc(y=, sr=, n_mfcc=, win_length=, hop_length=, n_fft=, fmin=, fmax=) as
        # invoked at script/mfcc.py:387; n_mels is librosa's implicit 128 unless the caller passes it.
        return o.mfcc(
            np.asarray(y),
            sr,
            n_mfcc=n_mfcc,
            win_length=kw.get("win_length", kw.get("n_fft", 2048)),
            hop_length=kw.get("hop_length", 512),
            n_fft=kw.get("n_fft", 2048),
            fmin=kw.get("fmin", 0.0),
            fmax=kw.get("fmax", None),
            n_mels=kw.get("n_mels", 128),
        )

    def rms(y=None, frame_length=2048, hop_length=512, center=True, pad_mode="constant", **kw):
        assert pad_mode == "constant"
        return o.rms_frames(np.asarray(y), frame_length, hop_length, center)[None, :]

    def load(path, sr=22050, mono=True, **kw):
        import scipy.io.wavfile

        fs, data = scipy.io.wavfile.read(path)
        if sr is not None and fs != sr:
            raise NotImplementedError("stub librosa.load: resampling (soxr_hq) is not available in this image")
        if data.dtype.kind == "i":
            data = data.astype(np.float32) / float(2 ** (8 * data.dtype.itemsize - 1))
        else:
            data = data.astype(np.float32)
        data = data.T  # [channels, n]
        if mono and data.ndim > 1:
            data = data.mean(axis=0)
        return data, fs

    def fft_frequencies(sr=22050, n_fft=2048):
        return np.fft.rfftfreq(n_fft, 1.0 / sr)

    lib = types.ModuleType("librosa")
    feature = types.ModuleType("librosa.feature")
    core = types.ModuleType("librosa.core")
    convert = types.ModuleType("librosa.core.convert")
    feature.mfcc, feature.rms = mfcc, rms
    core.load, core.convert = load, convert
    convert.fft_frequencies = fft_frequencies
    lib.feature, lib.core, lib.load = feature, core, load
    untouch = _Untouchable("librosa")
    lib.pyin, lib.stft = untouch.pyin, untouch.stft
    return {"librosa": lib, "librosa.feature": feature, "librosa.core": core, "librosa.core.convert": convert}


def _findiff_stub():
    from . import mfcc_oracle as o

    class FinDiff:
        """``FinDiff(axis, spacing, deriv, acc=)`` for axis 0 (the only use: script/calc.py:636)."""

        def __init__(self, axis, h, deriv=1, acc=2):
            assert axis == 0
            self.h, self.deriv, self.acc = h, deriv, acc

        def __call__(self, x):
            return o._findiff_apply(np.asarray(x), self.h, self.deriv, self.acc)

    m = types.ModuleType("findiff")
    m.FinDiff = FinDiff
    return {"findiff": m}


def _stubs():
    mods = {}
    mods.update(_librosa_stub())
    mods.update(_findiff_stub())
    pm = _Untouchable("parselmouth")
    praat = _Untouchable("parselmouth.praat")
    pm.praat = praat
    pm.Sound = type("Sound", (), {})  # used as an annotation at script/calc.py:132
    mods.update({"parselmouth": pm, "parselmouth.praat": praat})
    mods["pyqtgraph"] = _Untouchable("pyqtgraph")
    mods["xarray"] = _Untouchable("xarray")
    return mods


def load(name: str) -> types.ModuleType:
    """Import ``<REFERENCE_ROOT>/script/<name>.py`` (``'mfcc'`` or ``'calc'``) unmodified, with the
    stubs visible only while its top-level imports run."""
    if name in _loaded:
        return _loaded[name]
    if not available():
        raise FileNotFoundError(f"reference scripts not found under {script_dir()} (BASELINE.json reference_path; $MMF_REFERENCE_ROOT overrides it)")
    stubs = _stubs()
    saved = {k: sys.modules.get(k) for k in stubs}
    sys.modules.update(stubs)
    try:
        spec = importlib.util.spec_from_file_location(f"_mmf_reference_{name}", os.path.join(script_dir(), name + ".py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    _loaded[name] = mod
    return mod


def ref_mfcc() -> types.ModuleType:
    return load("mfcc")


def ref_calc() -> types.ModuleType:
    return load("calc")
