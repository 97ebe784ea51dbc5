"""B200-native MFCC / cepstral-modulation hot path of aaron-randreth/modulation-mfcc.

Python host code (this package) -> C ABI (``include/mmf.h``, ``libmmf_b200.so``) ->
hand-written sm_100a CUDA kernels (``csrc/``).  No CPU fallback: importing works
anywhere, computing requires a Blackwell GPU.
"""

from ._lib import MmfError, build, exported_symbols, lib  # noqa: F401
from .plan import (  # noqa: F401
    MfccConfig,
    OutFilter,
    Plan,
    clear_plans,
    fir_filter,
    frame_sizes,
    get_plan,
    host_tables,
    make_change_params,
    num_frames,
    resample_descriptors,
    resample_ratio,
    sos_zi,
    stencil_filter,
)
from .api import (  # noqa: F401
    MODULATION_BANDS_HZ,
    FeatureExtractor,
    ParameterError,
    applyFilter,
    band_bins,
    calculate_amplitude_envelope,
    calculate_amplitude_envelope_many,
    get_amplitude,
    get_MFCCS_change,
    get_MFCCS_change_batch,
    get_MFCCS_change_many,
    get_velocity,
    load_channel,
    mfcc_features_batch,
    mfcc_features_many,
    modspec_sizes,
)
from .shard import PeerGather, gather_features, shard_range, shard_sizes  # noqa: F401
from .corpus import CorpusRunner  # noqa: F401
from .synth import synth_batch, synth_batch_device, synth_clip  # noqa: F401

__version__ = "0.1.0"
