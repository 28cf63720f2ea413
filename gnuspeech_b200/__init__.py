"""gnuspeech_b200 -- B200-native Tube Resonance Model (TRM) synthesis: the hot path of grrrr/GnuSpeech's
Tube.framework as hand-written sm_100a CUDA kernels behind the reference's TRM interface.

    from gnuspeech_b200 import TRMDataList, TRMTubeModel, TRMInputParameters, TRMBatch

The native libraries (gnuspeech_b200/lib/libtrm.so, libtrm_cuda.so) must be built first
(`python -m gnuspeech_b200.build`); there is no CPU fallback.
"""
from ._native import (TRM_PRECISION_FP32, TRM_PRECISION_FP64, TRM_PRECISION_FP64_STRICT, TRM_STAGE_PCM, TRM_STAGE_SRC, TRM_STAGE_TUBE,  # noqa: F401
                      TRM_FRAMES_F32, TRM_FRAMES_F64, TRMError)
from .api import (EVENT_DTYPE, MMSynthesisParameters, PinnedArray, TRMBatch, TRMFrameGeneration, TRMStream, TRMStreamPool, event_list_frame_count, make_events, TRMDataList, TRMInputParameters, TRMParameters, TRMResident,  # noqa: F401
                  TRMSynthesizer, TRMTubeModel, derive, pcm_checksum, snapshot_info, sweep_synthesize)

__all__ = ["EVENT_DTYPE", "TRMStream", "TRMStreamPool", "TRMFrameGeneration", "event_list_frame_count", "make_events", "MMSynthesisParameters", "TRMBatch", "TRMDataList", "TRMInputParameters", "TRMParameters", "TRMResident", "TRMSynthesizer",
           "TRMTubeModel", "TRMError", "PinnedArray", "derive", "TRM_PRECISION_FP64", "TRM_PRECISION_FP32", "TRM_PRECISION_FP64_STRICT",
           "TRM_STAGE_TUBE", "TRM_STAGE_SRC", "TRM_STAGE_PCM", "TRM_FRAMES_F32", "TRM_FRAMES_F64", "sweep_synthesize", "pcm_checksum", "snapshot_info"]
