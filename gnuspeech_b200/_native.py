"""ctypes bindings to libtrm.so (include/trm.h).  Loading fails loudly if the library has not been
built; there is no Python or CPU fallback for the synthesis path."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# TRM_LIB_DIR selects a profiling variant built by `python -m gnuspeech_b200.build --variant <tag> ...` (tools/ only)
LIB_DIR = os.environ.get("TRM_LIB_DIR") or os.path.join(_HERE, "lib")
LIBTRM_PATH = os.path.join(LIB_DIR, "libtrm.so")
LIBTRM_CUDA_PATH = os.path.join(LIB_DIR, "libtrm_cuda.so")

TRM_OK = 0
TRM_ERR_TUBE_LENGTH, TRM_ERR_FIR, TRM_ERR_NOMEM, TRM_ERR_PARAM = -1, -2, -3, -4
TRM_ERR_CUDA, TRM_ERR_IO, TRM_ERR_STATE, TRM_ERR_SILENT = -5, -6, -7, -8
TRM_PRECISION_FP64, TRM_PRECISION_FP32, TRM_PRECISION_FP64_STRICT = 0, 1, 2
TRM_STAGE_TUBE, TRM_STAGE_SRC, TRM_STAGE_PCM = 0, 1, 2
TRM_FRAMES_F64, TRM_FRAMES_F32 = 0, 1


class TRMInputParametersStruct(C.Structure):
    """TRMInputParameters (include/trm.h; reference TRMInputParameters.h:26-54)."""
    _fields_ = [
        ("outputFileFormat", C.c_int32), ("outputRate", C.c_float), ("controlRate", C.c_float),
        ("volume", C.c_double), ("channels", C.c_int32), ("balance", C.c_double), ("waveform", C.c_int32),
        ("tp", C.c_double), ("tnMin", C.c_double), ("tnMax", C.c_double), ("breathiness", C.c_double),
        ("length", C.c_double), ("temperature", C.c_double), ("lossFactor", C.c_double), ("apScale", C.c_double),
        ("mouthCoef", C.c_double), ("noseCoef", C.c_double), ("noseRadius", C.c_double * 6),
        ("throatCutoff", C.c_double), ("throatVol", C.c_double), ("usesModulation", C.c_int32),
        ("mixOffset", C.c_double),
    ]


class TRMSynthesisParametersStruct(C.Structure):
    """TRMSynthesisParameters (include/trm.h; reference MMSynthesisParameters.h:22-52)."""
    _fields_ = [(n, C.c_double) for n in (
        "masterVolume", "vocalTractLength", "temperature", "balance", "breathiness", "lossFactor", "pitch",
        "throatCutoff", "throatVolume", "apertureScaling", "mouthCoef", "noseCoef", "mixOffset",
        "n1", "n2", "n3", "n4", "n5", "tp", "tnMin", "tnMax")] + [
        ("glottalPulseShape", C.c_int32), ("shouldUseNoiseModulation", C.c_int32), ("samplingRate", C.c_int32),
        ("outputChannels", C.c_int32)]


class TRMFrameGenerationStruct(C.Structure):
    """TRMFrameGeneration (include/trm.h; MMIntonation.m:74-80, EventList.m:983)."""
    _fields_ = [("useMacroIntonation", C.c_int32), ("useMicroIntonation", C.c_int32), ("useSmoothIntonation", C.c_int32),
                ("useDrift", C.c_int32), ("driftDeviation", C.c_double), ("driftCutoff", C.c_double), ("pitch", C.c_double),
                ("driftSeed", C.c_float), ("reserved", C.c_int32)]


class TRMDerivedValuesStruct(C.Structure):
    _fields_ = [("controlPeriod", C.c_int32), ("sampleRate", C.c_int32), ("actualTubeLength", C.c_double),
                ("padSize", C.c_int32), ("timeRegisterIncrement", C.c_uint32), ("tubeSamples", C.c_int64),
                ("numberSamples", C.c_int32)]


class TRMBatchLayoutStruct(C.Structure):
    _fields_ = [("total_frames", C.c_int64), ("total_pcm_samples", C.c_int64), ("total_out_samples", C.c_int64),
                ("audio_seconds", C.c_double), ("tube_samples", C.c_int64), ("out_samples", C.c_int64)]


class TRMStreamSnapshotInfoStruct(C.Structure):
    _fields_ = [("precision", C.c_int32), ("channels", C.c_int32), ("voice", TRMInputParametersStruct),
                ("frames_pushed", C.c_int64), ("samples_returned", C.c_int64), ("bytes", C.c_int64)]


class TRMStreamSnapshotEventInfoStruct(C.Structure):
    _fields_ = [("from_events", C.c_int32), ("n_events", C.c_int64), ("list_frames", C.c_int64),
                ("frames_generated", C.c_int64), ("fg", TRMFrameGenerationStruct)]


_lib = None


def lib():
    """Returns the loaded libtrm.so; raises if it is missing (build with `python -m gnuspeech_b200.build`)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIBTRM_PATH) or not os.path.exists(LIBTRM_CUDA_PATH):
        raise ImportError(
            "gnuspeech_b200 native libraries are missing (%s). Build them with `python -m gnuspeech_b200.build` "
            "or __graft_entry__.build(); there is no CPU fallback." % LIB_DIR)
    C.CDLL(LIBTRM_CUDA_PATH, mode=C.RTLD_GLOBAL)
    L = C.CDLL(LIBTRM_PATH)
    vp, i32, i64, dbl, sz = C.c_void_p, C.c_int32, C.c_int64, C.c_double, C.c_size_t
    P = C.POINTER

    def sig(name, res, *args):
        f = getattr(L, name)
        f.restype = res
        f.argtypes = list(args)

    sig("TRMLastErrorMessage", C.c_char_p)
    sig("TRMInputParametersSetDefaults", None, P(TRMInputParametersStruct), C.c_float)
    sig("TRMDeriveValues", C.c_int, P(TRMInputParametersStruct), sz, P(TRMDerivedValuesStruct))
    sig("TRMDataListCreate", vp)
    sig("TRMDataListCreateWithContentsOfFile", vp, C.c_char_p, P(C.c_int))
    sig("TRMDataListFree", None, vp)
    sig("TRMDataListInputParameters", P(TRMInputParametersStruct), vp)
    sig("TRMDataListAddParameters", C.c_int, vp, vp)
    sig("TRMDataListAddParametersArray", C.c_int, vp, vp, sz)
    sig("TRMDataListRemoveAllParameters", None, vp)
    sig("TRMDataListCount", sz, vp)
    sig("TRMDataListValues", vp, vp)
    sig("TRMDataListWriteToFile", C.c_int, vp, C.c_char_p)
    sig("TRMTubeModelCreate", vp, vp, P(C.c_int))
    sig("TRMTubeModelFree", None, vp)
    sig("TRMTubeModelSetPrecision", C.c_int, vp, C.c_int)
    sig("TRMTubeModelSetDevice", C.c_int, vp, C.c_int)
    sig("TRMTubeModelSynthesize", C.c_int, vp)
    sig("TRMTubeModelNumberSamples", i32, vp)
    sig("TRMTubeModelChannels", i32, vp)
    sig("TRMTubeModelHitsReferenceFlushBug", C.c_int, vp)
    sig("TRMReferenceFlushBug", C.c_int, P(TRMInputParametersStruct), sz)
    sig("TRMBatchReferenceFlushBugFlags", vp, vp)
    sig("TRMTubeModelMaximumSampleValue", dbl, vp)
    sig("TRMTubeModelResampledData", vp, vp)
    sig("TRMTubeModelTubeSignal", vp, vp, P(i64))
    sig("TRMTubeModelGetDerivedValues", None, vp, P(TRMDerivedValuesStruct))
    sig("TRMTubeModelPullPCM16", i64, vp, vp, sz, C.c_int)
    sig("TRMTubeModelGenerateWAVData", vp, vp, P(sz), P(C.c_int))
    sig("TRMTubeModelSaveOutputToFile", C.c_int, vp, C.c_char_p)
    sig("TRMFree", None, vp)
    sig("TRMSynthesisParametersRestoreDefaults", None, vp)
    sig("TRMSynthesisParametersForVoice", C.c_int, C.c_char_p, vp)
    sig("TRMInputParametersFromSynthesisParameters", None, vp, C.c_int32, vp)
    sig("TRMSynthesisParametersString", vp, vp)
    sig("TRMBatchCreate", vp, C.c_int, vp, C.c_int, vp, vp, C.c_int, P(C.c_int))
    sig("TRMBatchFree", None, vp)
    sig("TRMBatchGetLayout", None, vp, P(TRMBatchLayoutStruct))
    sig("TRMBatchNumberSamples", vp, vp)
    sig("TRMBatchPCMOffsets", vp, vp)
    sig("TRMBatchOutOffsets", vp, vp)
    sig("TRMBatchTubeOffsets", vp, vp)
    sig("TRMBatchTubeElements", i64, vp)
    sig("TRMBatchMaximumSampleValues", vp, vp)
    sig("TRMBatchKernelLaunches", i64, vp)
    sig("TRMBatchSynthesize", C.c_int, vp, vp, vp, vp, vp, C.c_int)
    sig("TRMBatchSynthesizeDebug", C.c_int, vp, vp, vp, vp, vp, C.c_int)
    sig("TRMFrameGenerationSetDefaults", None, vp)
    sig("TRMEventListFrameCount", i64, vp, i64)
    sig("TRMBatchGenerateFrames", C.c_int, vp, vp, vp, vp, vp, C.c_int, vp, vp, C.c_int)
    sig("TRMBatchSynthesizeEvents", C.c_int, vp, vp, vp, vp, vp, C.c_int, vp, vp, C.c_int)
    sig("TRMStreamCreate", vp, C.c_int, vp, C.c_int, C.c_int, C.c_int, vp)
    sig("TRMStreamCapacity", i64, vp)
    sig("TRMStreamPush", C.c_int, vp, vp, C.c_int, C.c_int, vp, vp)
    sig("TRMStreamSetVoice", C.c_int, vp, vp, vp, vp)
    sig("TRMStreamFree", None, vp)
    sig("TRMStreamPoolCreate", vp, C.c_int, C.c_int, C.c_int, C.c_int, P(C.c_int))
    sig("TRMStreamPoolOpen", C.c_int, vp, vp)
    sig("TRMStreamPoolOpenEvents", C.c_int, vp, vp, vp, i64, vp, P(i64))
    sig("TRMStreamPoolClose", C.c_int, vp, C.c_int)
    sig("TRMStreamPoolSlotCapacity", i64, vp)
    sig("TRMStreamPoolPush", C.c_int, vp, C.c_int, vp, vp, vp, vp, vp, vp)
    sig("TRMStreamPoolPushPCM16", C.c_int, vp, C.c_int, vp, vp, vp, vp, vp, vp, vp, vp)
    sig("TRMStreamPoolSetVoice", C.c_int, vp, C.c_int, vp, vp, vp, vp)
    sig("TRMStreamPoolFree", None, vp)
    sig("TRMStreamPoolSave", C.c_int, vp, C.c_int, vp, vp, i64, vp)
    sig("TRMStreamPoolRestore", C.c_int, vp, C.c_int, vp, vp, vp)
    sig("TRMStreamPoolSnapshotInfo", C.c_int, vp, i64, P(TRMStreamSnapshotInfoStruct))
    sig("TRMStreamPoolSaveAny", C.c_int, vp, C.c_int, vp, vp, i64, vp)
    sig("TRMStreamPoolSnapshotEventInfo", C.c_int, vp, i64, P(TRMStreamSnapshotEventInfoStruct))
    sig("TRMBatchSynthesizeAsync", vp, vp, vp, vp, vp, vp, C.c_int, vp)
    sig("TRMBatchWait", C.c_int, vp)
    sig("TRMBatchMakeResident", vp, vp, vp, C.c_int, P(C.c_int))
    sig("TRMResidentRunStage", C.c_int, vp, C.c_int, vp)
    sig("TRMResidentRun", C.c_int, vp, vp)
    sig("TRMResidentFetch", C.c_int, vp, vp, vp, vp, vp)
    sig("TRMResidentFree", None, vp)
    sig("TRMResidentFetchUtterance", C.c_int, vp, C.c_int, vp, vp, vp)
    sig("TRMBatchSetFrameFormat", C.c_int, vp, C.c_int)
    sig("TRMCopyProbe", C.c_int, C.c_int, vp, sz, vp, sz, C.c_int, P(C.c_double))
    sig("TRMHostAlloc", vp, sz)
    sig("TRMHostFree", None, vp)
    sig("TRMWorkloadStaticVowel", None, C.c_int, dbl, sz, vp)
    sig("TRMWorkloadRandomWalk", None, C.c_uint64, C.c_uint64, sz, vp)
    sig("TRMWorkloadRandomWalkBatch", None, C.c_uint64, C.c_uint64, sz, sz, vp, C.c_int)
    sig("TRMWorkloadGridPoint", None, C.c_uint64, sz, vp)
    sig("TRMWorkloadWalk2", None, C.c_uint64, C.c_uint64, sz, vp)
    sig("TRMSweepSynthesize", C.c_int, P(TRMInputParametersStruct), i32, C.c_uint64, C.c_uint64, i64, C.c_int, C.c_int, vp, vp, i64, vp,
        vp, i64, P(i32), P(i64), P(C.c_double))
    _lib = L
    return L


class TRMError(RuntimeError):
    def __init__(self, code, where=""):
        msg = lib().TRMLastErrorMessage()
        self.code = code
        super().__init__("%s failed with code %d: %s" % (where or "TRM call", code, (msg or b"").decode("utf-8", "replace")))


def check(code, where=""):
    if code != TRM_OK:
        raise TRMError(code, where)
    return code
