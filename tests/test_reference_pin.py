"""Parity pin to the reference's OWN code.

``tests/golden/ref_outputs.npz`` holds what the original project's ``script/mfcc.py`` and ``script/calc.py`` --
executed unmodified through ``oracle/ref_loader.py`` -- return for every case of ``tests/ref_cases.py``.

* CPU (``-m "not gpu"``): the oracle restatement must reproduce those outputs bit for bit and raise the error
  cases' exceptions, and, when the checkout of the original project is present (``reference_path`` of
  ``BASELINE.json``, or ``$MMF_REFERENCE_ROOT``), the live reference must still produce the committed vectors and
  raise the same exceptions as the oracle.
* GPU (``-m gpu``): the CUDA path, through the reference-facing Python mirror and the C ABI, must match the
  reference outputs within north_star's tolerances (1e-3 absolute on curves derived from MFCCs, 1e-9 relative
  for the float64 filters and stencils, exact time axes).
"""

import os

import numpy as np
import pytest

import oracle
from oracle import ref_loader

import ref_cases

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_outputs.npz")


@pytest.fixture(scope="module")
def golden():
    with np.load(GOLDEN) as z:
        return {k: z[k] for k in z.files}


def _expected(golden, name):
    out = []
    while f"{name}__{len(out)}" in golden:
        out.append(golden[f"{name}__{len(out)}"])
    assert out, name
    return out


ORACLE_MODS = {"mfcc": oracle, "calc": oracle}
NO_REFERENCE = f"the original project's scripts are not under {ref_loader.script_dir()} (set $MMF_REFERENCE_ROOT)"


def test_every_case_has_a_golden_vector(golden):
    names = {k.rsplit("__", 1)[0] for k in golden}
    assert names == set(ref_cases.CASES)


@pytest.mark.parametrize("name", list(ref_cases.CASES))
def test_oracle_reproduces_reference_outputs(name, golden):
    got = ref_cases.run_case(ORACLE_MODS, name)
    exp = _expected(golden, name)
    assert len(got) == len(exp)
    for g, e in zip(got, exp):
        assert g.dtype == e.dtype and g.shape == e.shape
        assert np.array_equal(g, e), (name, float(np.max(np.abs(g - e))))


@pytest.mark.skipif(not ref_loader.available(), reason=NO_REFERENCE)
@pytest.mark.parametrize("name", list(ref_cases.CASES))
def test_live_reference_still_produces_the_golden_vectors(name, golden):
    mods = {"mfcc": ref_loader.ref_mfcc(), "calc": ref_loader.ref_calc()}
    got = ref_cases.run_case(mods, name)
    for g, e in zip(got, _expected(golden, name)):
        assert np.array_equal(g, e), name


# the top-level imports of the original script/mfcc.py and script/calc.py that the loader stubs
_REFERENCE_IMPORTS = "import librosa\nimport parselmouth\nimport pyqtgraph as pg\nimport xarray\nfrom findiff import FinDiff\n"


def test_reference_modules_are_loaded_from_the_reference_tree(tmp_path, monkeypatch):
    """The loader executes the scripts where they lie, with its stubs, on a stand-in tree of the reference
    (the same imports at the top of each module) when the real checkout is not present."""
    if not ref_loader.available():
        (tmp_path / "script").mkdir()
        for name in ("mfcc", "calc"):
            (tmp_path / "script" / f"{name}.py").write_text(_REFERENCE_IMPORTS + "MFCC = librosa.feature.mfcc\n")
        monkeypatch.setattr(ref_loader, "REFERENCE_ROOT", str(tmp_path))
        monkeypatch.setattr(ref_loader, "_loaded", {})
    m = ref_loader.ref_mfcc()
    assert os.path.realpath(m.__file__).startswith(os.path.realpath(ref_loader.REFERENCE_ROOT))
    # the loader leaves no stub behind
    import sys

    for k in ("librosa", "parselmouth", "pyqtgraph", "xarray", "findiff"):
        mod = sys.modules.get(k)
        assert mod is None or getattr(mod, "__file__", None) is not None


@pytest.mark.skipif(not ref_loader.available(), reason=NO_REFERENCE)
@pytest.mark.parametrize("case", ref_cases.ERROR_CASES, ids=lambda c: c[0])
def test_oracle_raises_what_the_reference_raises(case):
    _, module, func, make_x, args, kwargs, etype, frag = case
    mods = {"mfcc": ref_loader.ref_mfcc(), "calc": ref_loader.ref_calc()}
    with pytest.raises(etype) as ref_exc:
        getattr(mods[module], func)(make_x(), *args, **kwargs)
    with pytest.raises(etype) as ora_exc:
        getattr(oracle, func)(make_x(), *args, **kwargs)
    assert type(ref_exc.value) is type(ora_exc.value)
    assert str(ref_exc.value) == str(ora_exc.value)
    assert frag in str(ref_exc.value)


@pytest.mark.parametrize("case", ref_cases.ERROR_CASES, ids=lambda c: c[0])
def test_oracle_raises_the_reference_error_cases(case):
    _, module, func, make_x, args, kwargs, etype, frag = case
    with pytest.raises(etype) as exc:
        getattr(oracle, func)(make_x(), *args, **kwargs)
    assert frag in str(exc.value)


# ------------------------------------------------------------------------------------------------------------
# GPU: the CUDA path against the reference's outputs
# ------------------------------------------------------------------------------------------------------------


def _tolerance(name, e):
    if name.startswith(("change_",)):
        return 1e-3  # north_star: <= 1e-3 absolute on MFCC-derived magnitudes
    if name.startswith("env_rms"):
        return 1e-4 * max(1.0, float(np.abs(e).max()))
    if name.startswith("env_hilb"):
        return 1e-4
    return 1e-9 * max(1.0, float(np.abs(e).max()))  # float64 filters / stencils


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(ref_cases.CASES))
def test_cuda_path_matches_reference_outputs(name, golden, cuda_device):
    import modulation_mfcc_b200 as mm

    mods = {"mfcc": mm, "calc": mm}
    got = ref_cases.run_case(mods, name)
    exp = _expected(golden, name)
    assert len(got) == len(exp)
    # values
    g, e = got[0], exp[0]
    assert g.shape == e.shape and g.dtype == e.dtype, (name, g.shape, e.shape, g.dtype, e.dtype)
    err = float(np.max(np.abs(g.astype(np.float64) - e.astype(np.float64))))
    assert err <= _tolerance(name, e), (name, err)
    # time axis (second return value): exact
    if len(exp) > 1:
        assert got[1].dtype == exp[1].dtype
        assert np.array_equal(got[1], exp[1]), name


@pytest.mark.gpu
@pytest.mark.parametrize("case", ref_cases.ERROR_CASES, ids=lambda c: c[0])
def test_cuda_path_raises_what_the_reference_raises(case, cuda_device):
    import modulation_mfcc_b200 as mm

    _, module, func, make_x, args, kwargs, etype, frag = case
    with pytest.raises(etype) as exc:
        getattr(mm, func)(make_x(), *args, **kwargs)
    assert frag in str(exc.value)
