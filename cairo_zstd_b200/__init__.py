"""cairo_zstd_b200 -- B200-native zstd decoder behind the FrameDecoder surface of NethermindEth/cairo_zstd.

The product is the C-ABI shared library built from csrc/ (include/cairo_zstd_b200.h).  This package
holds the build recipe, a ctypes binding of that ABI, the Python mirror of the reference's
FrameDecoder traits, and the seeded input generators.  There is no CPU decode path here: without
the CUDA library (or without a GPU) every decode call raises.
"""
from .api import (  # noqa: F401
    Context,
    MultiContext,
    CzbError,
    FrameDesc,
    FrameResult,
    MAX_FRAME_OUTPUT,
    STATUS_NAMES,
    find_frame_end,
    frame_header_info,
    load_library,
    partition_frames,
    split_frames,
    status_name,
)
from .frame_decoder import (  # noqa: F401
    BlockDecodingStrategy,
    FrameDecoder,
    FrameDecoderError,
    FrameDecoderState,
)
