"""frequensee -- Python host side of the B200-native FrequenSee propagation core.

`capi` binds the C-ABI (include/frequensee.h, CUDA only, no CPU fallback); `scenes` holds the
seeded procedural scenes of the benchmark configs; `distributed` shards the work range over
torch.distributed ranks.  The C++ mirror of the reference's UFrequenSeeAudioComponent /
UAudioRayTracingSubsystem / FFrequenSeeAudioReverbPlugin interface is include/frequensee.hpp.
"""
from . import capi, scenes  # noqa: F401
from .capi import Context, MultiContext, FrequenSeeError, default_config, load_float_array, save_float_array, allocate_paths  # noqa: F401
from .capi import directivity_polar, OMNI  # noqa: F401
from .capi import OcclusionSource, OcclusionResult  # noqa: F401
from .capi import AcousticParams, AcousticSlot, DecayFit  # noqa: F401
from .capi import DIFFRACTION_DTYPE  # noqa: F401
