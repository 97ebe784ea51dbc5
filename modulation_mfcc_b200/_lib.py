"""ctypes binding of ``libmmf_b200.so`` (C ABI declared in ``include/mmf.h``).

The library is built in-tree by :func:`build` (``nvcc`` for sm_100a).  There is no
CPU fallback anywhere in this package: if the shared object is missing it is an
ImportError-grade failure, and every compute entry point raises when no CUDA
device is present.
"""

from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess
from pathlib import Path

PKG_DIR = Path(__file__).resolve().parent
CSRC = PKG_DIR / "csrc"
LIB_PATH = PKG_DIR / "libmmf_b200.so"
SOURCES = ["stft_mel.cu", "stft_mel_tc.cu", "post_kernels.cu", "change_fused.cu", "modspec_fast.cu", "modspec_tc.cu", "mfcc_tc.cu", "tc_fft.cu", "dft_generic.cu", "hilbert_fft.cu", "c_api.cu", "host_tables.cpp"]
HEADERS = ["fft_regs.cuh", "stft_core.cuh", "sos_par.cuh", "mmf_internal.h", "../../include/mmf.h"]

NVCC_FLAGS = [
    "-gencode",
    "arch=compute_100a,code=sm_100a",
    "-lineinfo",
    "-O3",
    "-std=c++17",
    "--extended-lambda",
    "-Xcompiler",
    "-fPIC",
    "-shared",
]


class MmfError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"[mmf {code}] {msg}")
        self.code = code
        self.msg = msg


MMF_ERR_INVALID = -1
MMF_ERR_UNSUPPORTED = -2
MMF_ERR_CUDA = -3
MMF_ERR_TOO_SHORT = -4
MMF_ERR_NOMEM = -5

MMF_FLAG_NO_TMA = 1
MMF_FLAG_SPLIT_SMEM = 2
MMF_FLAG_UNFUSED_CHANGE = 4
MMF_FLAG_SCALAR_FFT = 8
MMF_FLAG_MMA_MEL = 16
MMF_FLAG_MMA_DCT = 32
MMF_FLAG_SEPARATE_MFCC = 64
MMF_FLAG_FOLD_MFCC = 128
MMF_FLAG_TC_FFT = 256
MMF_FLAG_NO_TC_MODSPEC = 512
MMF_FLAG_TC_DCT = 1024
MMF_FLAG_MEL_WALK = 2048
MMF_FLAG_NO_TC_MEL = 4096


class mmf_config(C.Structure):
    _fields_ = [
        ("sample_rate", C.c_double),
        ("n_fft", C.c_int32),
        ("win_length", C.c_int32),
        ("hop_length", C.c_int32),
        ("n_mels", C.c_int32),
        ("n_mfcc", C.c_int32),
        ("fmin", C.c_double),
        ("fmax", C.c_double),
        ("amin", C.c_float),
        ("top_db", C.c_float),
        ("preemph", C.c_float),
        ("device", C.c_int32),
        ("flags", C.c_int32),
    ]


class mmf_change_params(C.Structure):
    _fields_ = [
        ("remove_first", C.c_int32),
        ("diff_method", C.c_int32),
        ("n_sections", C.c_int32),
        ("sos", C.c_double * 96),
        ("out_kind", C.c_int32),
        ("out_n_sections", C.c_int32),
        ("out_sos", C.c_double * 96),
    ]


class mmf_modspec_params(C.Structure):
    _fields_ = [
        ("win", C.c_int32),
        ("hop", C.c_int32),
        ("nfft", C.c_int32),
        ("n_bands", C.c_int32),
        ("band_lo", C.c_int32 * 16),
        ("band_hi", C.c_int32 * 16),
    ]


class mmf_resample_clip(C.Structure):
    _fields_ = [
        ("up", C.c_int32),
        ("down", C.c_int32),
        ("tap0", C.c_int64),
        ("len_h", C.c_int32),
        ("n_pre_remove", C.c_int64),
        ("n_out", C.c_int64),
    ]


class mmf_amp_params(C.Structure):
    _fields_ = [
        ("center", C.c_int32),
        ("out_n_sections", C.c_int32),
        ("out_sos", C.c_double * 96),
    ]


OBJ_DIR = PKG_DIR / "build"


def _stale(target: Path, deps) -> bool:
    if not target.exists():
        return True
    t = target.stat().st_mtime
    return any(p.exists() and p.stat().st_mtime > t for p in deps)


def needs_build() -> bool:
    return _stale(LIB_PATH, [(CSRC / f).resolve() for f in SOURCES + HEADERS] + [Path(__file__).resolve()])


def build(force: bool = False, verbose: bool = False) -> Path:
    """Compile every CUDA source of the package for sm_100a into ``libmmf_b200.so``.

    One object per source (compiled in parallel, rebuilt only when the source or a
    header is newer), then one link step."""
    if not force and not needs_build():
        return LIB_PATH
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not Path(nvcc).exists():
        if LIB_PATH.exists():  # GPU box without a toolkit: use the prebuilt file that travelled with the repo
            return LIB_PATH
        raise RuntimeError("nvcc not found and libmmf_b200.so is missing")
    from concurrent.futures import ThreadPoolExecutor

    OBJ_DIR.mkdir(exist_ok=True)
    headers = [(CSRC / h).resolve() for h in HEADERS]
    compile_flags = [f for f in NVCC_FLAGS if f != "-shared"]

    def compile_one(src: str):
        obj = OBJ_DIR / (Path(src).stem + ".o")
        if not force and not _stale(obj, [CSRC / src, *headers]):
            return obj, ""
        cmd = [nvcc, *compile_flags, *(["-Xptxas", "-v"] if verbose else []), "-c", "-o", str(obj), str(CSRC / src)]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n" + res.stdout + res.stderr)
        return obj, res.stderr

    with ThreadPoolExecutor(max_workers=min(len(SOURCES), os.cpu_count() or 1)) as pool:
        results = list(pool.map(compile_one, SOURCES))
    if verbose:
        print("".join(log for _, log in results))
    cmd = [nvcc, "-shared", "-o", str(LIB_PATH), *[str(o) for o, _ in results]]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc link failed:\n" + res.stdout + res.stderr)
    return LIB_PATH


_lib = None

_i64, _i32, _vp = C.c_int64, C.c_int32, C.c_void_p
_SIGNATURES = {
    "mmf_version": (C.c_int, []),
    "mmf_last_error": (C.c_char_p, []),
    "mmf_num_frames": (_i64, [_i64, _i32, _i32]),
    "mmf_host_tables": (C.c_int, [C.POINTER(mmf_config), _vp, _vp, _vp]),
    "mmf_sos_zi": (C.c_int, [_vp, _i32, _vp, C.POINTER(_i32)]),
    "mmf_plan_create": (C.c_int, [C.POINTER(_vp), C.POINTER(mmf_config)]),
    "mmf_plan_destroy": (C.c_int, [_vp]),
    "mmf_stft_power": (C.c_int, [_vp, _vp, _i64, _i64, _i64, _vp, _vp]),
    "mmf_logmel": (C.c_int, [_vp, _vp, _i64, _i64, _i64, _vp, _vp, _vp]),
    "mmf_mfcc": (C.c_int, [_vp, _vp, _vp, _i64, _i64, _vp, _vp, _i32, _vp]),
    "mmf_sosfiltfilt": (C.c_int, [_vp, _vp, _i32, _i64, _i64, _i64, _vp, _i32, _vp, _i64, _vp]),
    "mmf_delta_norm": (C.c_int, [_vp, _vp, _i64, _i32, _i64, _i32, _vp, _vp]),
    "mmf_fir_filtfilt": (C.c_int, [_vp, _vp, _i64, _i64, _vp, _i32, _vp, _vp, _vp]),
    "mmf_stencil": (C.c_int, [_vp, _vp, _i64, _i64, _vp, _i32, _vp, _vp, _i32, _i32, _vp, _vp]),
    "mmf_modspec": (C.c_int, [_vp, _vp, _i64, _i32, _i64, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _i32, _vp]),
    "mmf_modspec_varlen": (C.c_int, [_vp, _vp, _i64, _i32, _vp, _i64, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _i32, _vp]),
    "mmf_rms": (C.c_int, [_vp, _vp, _i64, _i64, _i64, _i32, _i32, _i32, _vp, _vp]),
    "mmf_mfcc_change": (
        C.c_int,
        [_vp, _vp, _i64, _i64, _i64, C.POINTER(mmf_change_params), _vp, _vp, _vp, _vp, _vp],
    ),
    "mmf_mfcc_change_varlen": (
        C.c_int,
        [_vp, _vp, _i64, _vp, _i64, C.POINTER(mmf_change_params), _vp, _vp, _vp, _vp, _vp],
    ),
    "mmf_mfcc_change_host": (C.c_int, [_vp, _vp, _i64, _i64, _i64, C.POINTER(mmf_change_params), _vp, _vp]),
    "mmf_change_from_logmel": (
        C.c_int,
        [_vp, _vp, _vp, _i64, _i64, C.POINTER(mmf_change_params), _vp, _vp, _vp, _i32, _vp],
    ),
    "mmf_features_host": (
        C.c_int,
        [_vp, _vp, _i64, _i64, _i64, C.POINTER(mmf_change_params), C.POINTER(mmf_modspec_params), _vp, _vp, _vp, _vp, _vp],
    ),
    "mmf_features_host_pcm16": (
        C.c_int,
        [_vp, _vp, _i64, _i64, _i64, C.POINTER(mmf_change_params), C.POINTER(mmf_modspec_params), _vp, _vp, _vp, _vp, _vp],
    ),
    "mmf_features_varlen_sizes": (
        C.c_int,
        [C.POINTER(mmf_config), C.POINTER(mmf_modspec_params), _i64, _vp, _vp, _vp],
    ),
    "mmf_features_host_varlen": (
        C.c_int,
        [_vp, _vp, _i64, _vp, C.POINTER(mmf_change_params), C.POINTER(mmf_modspec_params), _vp, _vp, _vp, _vp, _vp],
    ),
    "mmf_features_host_varlen_pcm16": (
        C.c_int,
        [_vp, _vp, _i64, _vp, C.POINTER(mmf_change_params), C.POINTER(mmf_modspec_params), _vp, _vp, _vp, _vp, _vp],
    ),
    "mmf_features_host_varlen_resampled": (
        C.c_int,
        [_vp, _vp, _i32, _i64, _vp, _vp, _vp, _i64, C.POINTER(mmf_change_params), C.POINTER(mmf_modspec_params),
         _vp, _vp, _vp, _vp, _vp],
    ),
    "mmf_resample_varlen": (C.c_int, [_vp, _vp, _i64, _vp, _vp, _vp, _i64, _vp, _i64, _vp]),
    "mmf_features_host_varlen_amp": (
        C.c_int,
        [_vp, _vp, _i32, _i64, _vp, _vp, _vp, _i64, C.POINTER(mmf_change_params), C.POINTER(mmf_modspec_params),
         C.POINTER(mmf_amp_params), _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp],
    ),
    "mmf_amp_varlen_sizes": (C.c_int, [_i64, _vp, _vp, _i32, _vp]),
    "mmf_rms_varlen": (C.c_int, [_vp, _vp, _i64, _vp, _vp, _i32, _vp, _vp]),
    "mmf_pcm16_to_f32": (C.c_int, [_vp, _vp, _i64, _vp, _vp]),
    "mmf_hilbert_envelope": (C.c_int, [_vp, _vp, _i64, _i64, _i64, _vp, _i64, _vp]),
    "mmf_find_peaks": (C.c_int, [_vp, _vp, _i64, _i64, _i64, _i32, _i32, _vp, _vp, _vp]),
    "mmf_resample_poly": (C.c_int, [_vp, _vp, _i64, _i64, _i64, _vp, _i32, _i32, _i32, _i64, _i64, _vp, _i64, _vp]),
    "mmf_abi_sizeof": (C.c_int, [_i32]),
    "mmf_launch_count": (_i64, [_i32]),
}


def exported_symbols() -> list[str]:
    return list(_SIGNATURES)


def lib() -> C.CDLL:
    """Load (building if necessary) the shared library; raises if it cannot be had."""
    global _lib
    if _lib is None:
        if needs_build():
            build()
        if not LIB_PATH.exists():
            raise ImportError(f"{LIB_PATH} is missing: the CUDA extension is required (no CPU fallback)")
        l = C.CDLL(str(LIB_PATH))
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        raise MmfError(rc, lib().mmf_last_error().decode("utf-8", "replace"))
