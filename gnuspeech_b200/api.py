"""Python mirror of the reference's Tube.framework interface, over the C API (include/trm.h).

Same names, argument meaning and error behaviour as the Objective-C classes so that callers (and the
parity tests) read like the reference's callers (TRMSynthesizer.m:38-136, Frameworks/Tube/main.m:12-67):

    TRMInputParameters / TRMParameters / TRMDataList / TRMTubeModel  -> Frameworks/Tube/Tube.h:7-10
    TRMSynthesizer                                                    -> Frameworks/GnuSpeech/Tube/TRMSynthesizer.h
    TRMBatch                                                          -> batched entry point (new)

Everything numerical happens in libtrm / libtrm_cuda on the GPU; this file only marshals buffers.
"""
import ctypes as C

import numpy as np

from . import _native as N
from ._native import TRMError, check  # noqa: F401

FRAME_FIELDS = ("glottalPitch", "glottalVolume", "aspirationVolume", "fricationVolume", "fricationPosition",
                "fricationCenterFrequency", "fricationBandwidth", "r1", "r2", "r3", "r4", "r5", "r6", "r7", "r8",
                "velum")


class TRMInputParameters(N.TRMInputParametersStruct):
    """Utterance-rate parameters (TRMInputParameters.h:26-54); defaults = Monet's male voice, mono."""

    def __init__(self, outputRate=44100.0, **kw):
        super().__init__()
        N.lib().TRMInputParametersSetDefaults(C.byref(self), C.c_float(outputRate))
        for k, v in kw.items():
            if k == "noseRadius":
                for i, x in enumerate(v):
                    self.noseRadius[i] = x
            else:
                setattr(self, k, v)

    def copy(self):
        o = TRMInputParameters()
        C.memmove(C.byref(o), C.byref(self), C.sizeof(self))
        return o


class MMSynthesisParameters(N.TRMSynthesisParametersStruct):
    """Utterance-rate voice parameters as Monet keeps them (MMSynthesisParameters.m:160-310): the registered defaults
    (male voice), the named voices of Other/voices.config, the TRM header they map to and its text form."""

    def __init__(self, voice=None):
        super().__init__()
        if voice is None:
            N.lib().TRMSynthesisParametersRestoreDefaults(C.byref(self))
        else:
            check(N.lib().TRMSynthesisParametersForVoice(voice.encode(), C.byref(self)), "TRMSynthesisParametersForVoice")

    def restoreDefaultValues(self):
        N.lib().TRMSynthesisParametersRestoreDefaults(C.byref(self))

    @property
    def sampleRate(self):
        return 22050.0 if self.samplingRate == 0 else 44100.0

    def inputParameters(self, fileFormat=0):
        """What -[TRMSynthesizer setupSynthesisParameters:] writes into the TRM header (TRMSynthesizer.m:38-65)."""
        ip = TRMInputParameters()
        N.lib().TRMInputParametersFromSynthesisParameters(C.byref(self), fileFormat, C.byref(ip))
        return ip

    @property
    def parameterString(self):
        p = N.lib().TRMSynthesisParametersString(C.byref(self))
        try:
            return C.string_at(p).decode()
        finally:
            N.lib().TRMFree(p)


EVENT_DTYPE = np.dtype([("time", np.int64), ("value", np.float64, (36,))])   # TRMEvent (include/trm.h; Event.h)


class TRMFrameGeneration(N.TRMFrameGenerationStruct):
    """Intonation switches, drift and base pitch of the control-frame generator (MMIntonation.m:74-80)."""

    def __init__(self, **kw):
        super().__init__()
        N.lib().TRMFrameGenerationSetDefaults(C.byref(self))
        for k, v in kw.items():
            setattr(self, k, v)


def make_events(times, values):
    """Structured TRMEvent array from times (ms) and an (n, 36) value array (NaN = no value at that event)."""
    ev = np.zeros(len(times), EVENT_DTYPE)
    ev["time"] = times
    ev["value"] = values
    return ev


def event_list_frame_count(events):
    """Number of frames -generateOutputInTimeRange: emits for an event list (TRMEventListFrameCount)."""
    events = np.ascontiguousarray(events, dtype=EVENT_DTYPE)
    return int(N.lib().TRMEventListFrameCount(events.ctypes.data_as(C.c_void_p), len(events)))


class TRMParameters(object):
    """One control frame (TRMParameters.h:9-17)."""

    def __init__(self, glottalPitch=0.0, glottalVolume=0.0, aspirationVolume=0.0, fricationVolume=0.0,
                 fricationPosition=0.0, fricationCenterFrequency=0.0, fricationBandwidth=0.0, radius=(0.0,) * 8,
                 velum=0.0):
        self.values = np.array([glottalPitch, glottalVolume, aspirationVolume, fricationVolume, fricationPosition,
                                fricationCenterFrequency, fricationBandwidth] + list(radius) + [velum], dtype=np.float64)
        assert self.values.shape == (16,)

    @property
    def valuesString(self):
        """TRMParameters.m:26-45."""
        return " ".join("%.3f" % v for v in self.values)


def derive(ip, n_frames):
    """controlPeriod / sampleRate / numberSamples ... without synthesizing (TRMTubeModel.m:196-203)."""
    dv = N.TRMDerivedValuesStruct()
    check(N.lib().TRMDeriveValues(C.byref(ip), n_frames, C.byref(dv)), "TRMDeriveValues")
    return dv


class TRMDataList(object):
    """TRMDataList.h:8-18: `inputParameters` plus the growing list of frames (`values`)."""

    def __init__(self, path=None):
        L = N.lib()
        if path is None:
            self._h = L.TRMDataListCreate()
            if not self._h:
                raise MemoryError()
            L.TRMInputParametersSetDefaults(L.TRMDataListInputParameters(self._h), C.c_float(44100.0))
        else:
            err = C.c_int(0)
            self._h = L.TRMDataListCreateWithContentsOfFile(path.encode(), C.byref(err))
            if not self._h:
                raise TRMError(err.value, "TRMDataList initWithContentsOfFile")

    @classmethod
    def initWithContentsOfFile(cls, path):
        return cls(path)

    def __del__(self):
        if getattr(self, "_h", None):
            N.lib().TRMDataListFree(self._h)
            self._h = None

    @property
    def inputParameters(self):
        return N.lib().TRMDataListInputParameters(self._h).contents

    def setInputParameters(self, ip):
        C.memmove(N.lib().TRMDataListInputParameters(self._h), C.byref(ip), C.sizeof(ip))

    def addParameters(self, frame):
        v = frame.values if isinstance(frame, TRMParameters) else np.ascontiguousarray(frame, dtype=np.float64)
        if v.ndim == 1:
            assert v.shape[0] == 16
            check(N.lib().TRMDataListAddParameters(self._h, v.ctypes.data_as(C.c_void_p)), "addParameters")
        else:
            assert v.shape[1] == 16
            check(N.lib().TRMDataListAddParametersArray(self._h, v.ctypes.data_as(C.c_void_p), v.shape[0]), "addParameters")

    def removeAllParameters(self):
        N.lib().TRMDataListRemoveAllParameters(self._h)

    @property
    def count(self):
        return int(N.lib().TRMDataListCount(self._h))

    @property
    def values(self):
        n = self.count
        if n == 0:
            return np.zeros((0, 16))
        p = N.lib().TRMDataListValues(self._h)
        return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_double)), (n, 16)).copy()

    def writeToFile(self, path):
        check(N.lib().TRMDataListWriteToFile(self._h, path.encode()), "TRMDataListWriteToFile")


class TRMTubeModel(object):
    """TRMTubeModel.h:29-40.  `initWithInputData` returns None where the reference returns nil."""

    def __init__(self, inputData, precision=N.TRM_PRECISION_FP64, device=0):
        err = C.c_int(0)
        self._h = N.lib().TRMTubeModelCreate(inputData._h, C.byref(err))
        if not self._h:
            raise TRMError(err.value, "TRMTubeModel initWithInputData")
        check(N.lib().TRMTubeModelSetPrecision(self._h, precision), "TRMTubeModelSetPrecision")
        N.lib().TRMTubeModelSetDevice(self._h, device)
        self.precision = precision

    @classmethod
    def initWithInputData(cls, inputData, **kw):
        try:
            return cls(inputData, **kw)
        except TRMError as e:
            if e.code in (N.TRM_ERR_TUBE_LENGTH, N.TRM_ERR_FIR, N.TRM_ERR_NOMEM):
                return None
            raise

    def __del__(self):
        if getattr(self, "_h", None):
            N.lib().TRMTubeModelFree(self._h)
            self._h = None

    def synthesize(self):
        check(N.lib().TRMTubeModelSynthesize(self._h), "TRMTubeModel synthesize")

    @property
    def numberSamples(self):
        return int(N.lib().TRMTubeModelNumberSamples(self._h))

    @property
    def maximumSampleValue(self):
        return float(N.lib().TRMTubeModelMaximumSampleValue(self._h))

    @property
    def derived(self):
        dv = N.TRMDerivedValuesStruct()
        N.lib().TRMTubeModelGetDerivedValues(self._h, C.byref(dv))
        return dv

    @property
    def resampledData(self):
        n = self.numberSamples
        p = N.lib().TRMTubeModelResampledData(self._h)
        if n == 0 or not p:
            return np.zeros(0)
        return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_double)), (n,)).copy()

    @property
    def tubeSignal(self):
        cnt = C.c_int64(0)
        p = N.lib().TRMTubeModelTubeSignal(self._h, C.byref(cnt))
        if cnt.value == 0 or not p:
            return np.zeros(0)
        return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_double)), (cnt.value,)).copy()

    @property
    def channels(self):
        return int(N.lib().TRMTubeModelChannels(self._h))

    @property
    def hitsReferenceFlushBug(self):
        return bool(N.lib().TRMTubeModelHitsReferenceFlushBug(self._h))

    def pcm16(self, file_variant=False, channels=None):
        """Interleaved PCM16; the buffer is sized from the MODEL's channel count (the C call writes n * channels)."""
        n = self.numberSamples
        if channels is not None and channels != self.channels:
            raise ValueError("this model has %d channel(s)" % self.channels)
        channels = self.channels
        out = np.zeros(max(n, 1) * channels, dtype=np.int16)
        got = N.lib().TRMTubeModelPullPCM16(self._h, out.ctypes.data_as(C.c_void_p), n, int(bool(file_variant)))
        if got < 0:
            raise TRMError(int(got), "TRMTubeModelPullPCM16")
        return out[: got * channels]

    def generateWAVData(self):
        ln, err = C.c_size_t(0), C.c_int(0)
        p = N.lib().TRMTubeModelGenerateWAVData(self._h, C.byref(ln), C.byref(err))
        if not p:
            raise TRMError(err.value, "generateWAVData")
        data = C.string_at(p, ln.value)
        N.lib().TRMFree(p)
        return data

    def saveOutputToFile(self, filename):
        check(N.lib().TRMTubeModelSaveOutputToFile(self._h, filename.encode()), "saveOutputToFile")
        return True


class TRMSynthesizer(object):
    """The adapter Monet drives (Frameworks/GnuSpeech/Tube/TRMSynthesizer.m:38-136): set the voice, add frames,
    synthesize; output goes to a sound file or comes back as WAV bytes (the reference plays them)."""

    def __init__(self, precision=N.TRM_PRECISION_FP64, device=0):
        self._inputData = TRMDataList()
        self._inputData.inputParameters.outputFileFormat = 0
        self.shouldSaveToSoundFile = False
        self.filename = None
        self.precision, self.device = precision, device
        self.lastWAVData = None
        self.lastTube = None

    def setupSynthesisParameters(self, ip):
        """TRMSynthesizer.m:38-65; `ip` is a TRMInputParameters (the MMSynthesisParameters equivalent)."""
        fmt = self._inputData.inputParameters.outputFileFormat
        self._inputData.setInputParameters(ip)
        self._inputData.inputParameters.controlRate = 250
        self._inputData.inputParameters.outputFileFormat = fmt
        self._inputData.inputParameters.noseRadius[0] = 0

    def removeAllParameters(self):
        self._inputData.removeAllParameters()

    def addParameters(self, parameters):
        self._inputData.addParameters(parameters)

    @property
    def fileType(self):
        return self._inputData.inputParameters.outputFileFormat

    @fileType.setter
    def fileType(self, v):
        self._inputData.inputParameters.outputFileFormat = v

    def synthesize(self):
        tube = TRMTubeModel.initWithInputData(self._inputData, precision=self.precision, device=self.device)
        if tube is None:
            return None          # "Warning: Failed to create tube model." (TRMSynthesizer.m:121-124)
        tube.synthesize()
        if self.shouldSaveToSoundFile:
            tube.saveOutputToFile(self.filename)
        else:
            self.lastWAVData = tube.generateWAVData()
        self.lastTube = tube
        return tube


class PinnedArray(object):
    """numpy view over page-locked host memory from TRMHostAlloc."""

    def __init__(self, shape, dtype):
        self.dtype = np.dtype(dtype)
        self.shape = tuple(int(s) for s in (shape if isinstance(shape, (tuple, list)) else (shape,)))
        n = int(np.prod(self.shape)) if len(self.shape) else 1
        self.nbytes = max(n, 1) * self.dtype.itemsize
        self._p = N.lib().TRMHostAlloc(self.nbytes)
        if not self._p:
            raise TRMError(N.TRM_ERR_CUDA, "TRMHostAlloc")
        buf = (C.c_char * self.nbytes).from_address(self._p)
        self.array = np.frombuffer(buf, dtype=self.dtype, count=n).reshape(self.shape)

    @property
    def ptr(self):
        return C.c_void_p(self._p)

    def free(self):
        if self._p:
            self.array = None
            N.lib().TRMHostFree(self._p)
            self._p = None

    def __del__(self):
        try:
            self.free()
        except TypeError:       # interpreter shutdown: module globals are already gone, the process frees the memory
            pass


def _ptr(a):
    if a is None:
        return None
    if isinstance(a, PinnedArray):
        return a.ptr
    return a.ctypes.data_as(C.c_void_p)


class TRMBatch(object):
    """Batched entry point: n independent utterances, one shared or n individual TRMInputParameters."""

    def __init__(self, ip, n_frames, frame_offset=None, precision=N.TRM_PRECISION_FP64):
        self.n_frames = np.ascontiguousarray(n_frames, dtype=np.int32)
        self.n = int(self.n_frames.shape[0])
        if frame_offset is None:
            frame_offset = np.concatenate(([0], np.cumsum(self.n_frames[:-1], dtype=np.int64))) if self.n else np.zeros(0, np.int64)
        self.frame_offset = np.ascontiguousarray(frame_offset, dtype=np.int64)
        self.precision = precision
        if isinstance(ip, (list, tuple)):
            assert len(ip) == self.n
            arr = (N.TRMInputParametersStruct * max(self.n, 1))()
            for i, p in enumerate(ip):
                C.memmove(C.byref(arr[i]), C.byref(p), C.sizeof(p))
            self._ip, shared = arr, 0
        else:
            self._ip, shared = ip, 1
        err = C.c_int(0)
        self._h = N.lib().TRMBatchCreate(self.n, C.cast(C.byref(self._ip) if shared else self._ip, C.c_void_p), shared,
                                         _ptr(self.frame_offset), _ptr(self.n_frames), precision, C.byref(err))
        if not self._h:
            raise TRMError(err.value, "TRMBatchCreate")
        self.layout = N.TRMBatchLayoutStruct()
        N.lib().TRMBatchGetLayout(self._h, C.byref(self.layout))
        self.sample_dtype = np.float64 if precision != N.TRM_PRECISION_FP32 else np.float32

    def __del__(self):
        if getattr(self, "_h", None):
            try:
                N.lib().TRMBatchFree(self._h)
            except TypeError:   # interpreter shutdown
                pass
            self._h = None

    def _arr(self, fn, ctype, dtype):
        if self.n == 0:
            return np.zeros(0, dtype)
        p = getattr(N.lib(), fn)(self._h)
        return np.ctypeslib.as_array(C.cast(p, C.POINTER(ctype)), (self.n,)).copy()

    @property
    def numberSamples(self):
        return self._arr("TRMBatchNumberSamples", C.c_int32, np.int32)

    @property
    def pcmOffsets(self):
        return self._arr("TRMBatchPCMOffsets", C.c_int64, np.int64)

    @property
    def outOffsets(self):
        return self._arr("TRMBatchOutOffsets", C.c_int64, np.int64)

    @property
    def tubeOffsets(self):
        return self._arr("TRMBatchTubeOffsets", C.c_int64, np.int64)

    @property
    def tubeElements(self):
        return int(N.lib().TRMBatchTubeElements(self._h))

    @property
    def maximumSampleValues(self):
        return self._arr("TRMBatchMaximumSampleValues", C.c_double, np.float64)

    @property
    def referenceFlushBugFlags(self):
        """Per utterance: the reference's streaming converter would append spurious samples here (include/trm.h)."""
        return self._arr("TRMBatchReferenceFlushBugFlags", C.c_uint8, np.uint8).astype(bool)

    @property
    def kernelLaunches(self):
        return int(N.lib().TRMBatchKernelLaunches(self._h))

    def synthesize(self, frames, pcm_out=None, samples_out=None, devices=None):
        """frames: (total_frames,16) float64 array or PinnedArray.  Blocking; returns None."""
        devs = None
        nd = 1
        if devices is not None:
            devs = np.ascontiguousarray(devices, dtype=np.int32)
            nd = int(devs.shape[0])
        check(N.lib().TRMBatchSynthesize(self._h, _ptr(frames), _ptr(pcm_out), _ptr(samples_out), _ptr(devs), nd),
              "TRMBatchSynthesize")

    def synthesize_async(self, frames, pcm_out=None, samples_out=None, devices=None):
        """Non-blocking form (TRMBatchSynthesizeAsync): returns a ticket; ticket.wait() blocks until the outputs are in
        the host buffers.  Two tickets per device overlap (copy-out of one call behind the kernels of the next); use one
        TRMBatch object per ticket in flight."""
        devs = None
        nd = 1
        if devices is not None:
            devs = np.ascontiguousarray(devices, dtype=np.int32)
            nd = int(devs.shape[0])
        err = C.c_int(0)
        h = N.lib().TRMBatchSynthesizeAsync(self._h, _ptr(frames), _ptr(pcm_out), _ptr(samples_out), _ptr(devs), nd, C.byref(err))
        if not h:
            check(err.value or N.TRM_ERR_CUDA, "TRMBatchSynthesizeAsync")
        return TRMBatchTicket(h, (frames, pcm_out, samples_out, devs, self))

    def _event_args(self, events, n_events, fg):
        events = np.ascontiguousarray(events, dtype=EVENT_DTYPE)
        cnt = np.ascontiguousarray(n_events, dtype=np.int32)
        off = np.concatenate(([0], np.cumsum(cnt)[:-1])).astype(np.int64)
        if isinstance(fg, (list, tuple)):
            arr = (N.TRMFrameGenerationStruct * len(fg))(*fg)
            return events, off, cnt, arr, 0
        return events, off, cnt, fg, 1

    def generate_frames(self, events, n_events, fg, device=0):
        """Control frames of every utterance from its event list, generated on the GPU (TRMBatchGenerateFrames).
        events: the utterances' TRMEvent lists back to back; n_events: events per utterance; fg: one TRMFrameGeneration
        for all, or a list with one per utterance.  Returns (frames (total_frames, 16), drift seeds at exit)."""
        events, off, cnt, fga, shared = self._event_args(events, n_events, fg)
        frames = np.zeros((max(1, int(self.layout.total_frames)), 16), np.float64)
        seeds = np.zeros(max(1, len(cnt)), np.float32)
        check(N.lib().TRMBatchGenerateFrames(self._h, _ptr(events), _ptr(off), _ptr(cnt), C.cast(C.byref(fga) if shared else fga, C.c_void_p),
                                             shared, _ptr(frames), _ptr(seeds), device), "TRMBatchGenerateFrames")
        return frames[:int(self.layout.total_frames)], seeds[:len(cnt)]

    def synthesize_events(self, events, n_events, fg, pcm_out=None, samples_out=None, device=0):
        """Event lists in, PCM out (TRMBatchSynthesizeEvents): the frames never exist on the host."""
        events, off, cnt, fga, shared = self._event_args(events, n_events, fg)
        check(N.lib().TRMBatchSynthesizeEvents(self._h, _ptr(events), _ptr(off), _ptr(cnt), C.cast(C.byref(fga) if shared else fga, C.c_void_p),
                                               shared, _ptr(pcm_out), _ptr(samples_out), device), "TRMBatchSynthesizeEvents")

    def synthesize_debug(self, frames, pcm_out=None, samples_out=None, tube_out=None, device=0):
        check(N.lib().TRMBatchSynthesizeDebug(self._h, _ptr(frames), _ptr(pcm_out), _ptr(samples_out), _ptr(tube_out),
                                              device), "TRMBatchSynthesizeDebug")

    def make_resident(self, frames, device=0):
        return TRMResident(self, frames, device)

    def set_frame_format(self, fmt):
        """N.TRM_FRAMES_F64 (TRMParameters rows, default) or N.TRM_FRAMES_F32 (rows of 16 floats: half the upload,
        identical results -- Monet's frames are floats)."""
        check(N.lib().TRMBatchSetFrameFormat(self._h, fmt), "TRMBatchSetFrameFormat")


class TRMStream(object):
    """Streaming synthesis of n voices at once (TRMStreamCreate / TRMStreamPush): push control frames as they arrive,
    get the un-normalised output-rate samples that became computable; pushes concatenate to exactly the one-shot
    result.  TRAcT's mode of use (Applications/TRAcT/tube.c:1096-1191), batched."""

    def __init__(self, n_streams, ip, precision=N.TRM_PRECISION_FP64, max_frames_per_push=64, device=0):
        err = C.c_int(0)
        self._ip = ip
        self.n = n_streams
        self.dtype = np.float64 if precision != N.TRM_PRECISION_FP32 else np.float32
        self._h = N.lib().TRMStreamCreate(n_streams, C.byref(ip), precision, max_frames_per_push, device, C.byref(err))
        if not self._h:
            check(err.value or N.TRM_ERR_CUDA, "TRMStreamCreate")
        self.capacity = int(N.lib().TRMStreamCapacity(self._h))
        self._buf = np.zeros((n_streams, self.capacity), self.dtype)

    def push(self, frames, flush=False):
        """frames: (n_streams, m, 16) float64 (m may be 0 with flush).  Returns (n_streams, k) samples."""
        frames = np.ascontiguousarray(frames, dtype=np.float64).reshape(self.n, -1, 16)
        m = frames.shape[1]
        k = C.c_int64(0)
        check(N.lib().TRMStreamPush(self._h, _ptr(frames) if m else None, m, 1 if flush else 0, _ptr(self._buf), C.byref(k)),
              "TRMStreamPush")
        return self._buf[:, :k.value].copy()

    def set_voice(self, ip):
        """Every stream continues with voice `ip` from the next push, its state kept (TRMStreamSetVoice; the rules of
        TRMStreamPool.set_voice).  Returns (tube_sample, output_sample), the same for every stream."""
        ts, os_ = C.c_int64(0), C.c_int64(0)
        check(N.lib().TRMStreamSetVoice(self._h, C.byref(ip), C.byref(ts), C.byref(os_)), "TRMStreamSetVoice")
        self._ip = ip
        return int(ts.value), int(os_.value)

    def free(self):
        if self._h:
            N.lib().TRMStreamFree(self._h)
            self._h = None

    def __del__(self):
        self.free()


class TRMStreamPool(object):
    """Streaming slots that open, advance and end independently, each with its own voice (TRMStreamPoolCreate / Open /
    Push / Close): a server's requests arrive at different times with different voices, and one push advances any subset
    of them, each by its own number of frames, with one waveguide and one resampler launch.  Each slot's pushes,
    concatenated, equal the one-shot synthesis of its utterance bit for bit.  A slot opened with open_events generates
    its frames on the device from a Monet event list as it advances.  Used by one thread at a time."""

    def __init__(self, capacity, precision=N.TRM_PRECISION_FP64, max_frames_per_push=64, device=0):
        err = C.c_int(0)
        self.capacity = capacity
        self.max_frames_per_push = max_frames_per_push
        self.dtype = np.float64 if precision != N.TRM_PRECISION_FP32 else np.float32
        self._h = N.lib().TRMStreamPoolCreate(capacity, precision, max_frames_per_push, device, C.byref(err))
        if not self._h:
            check(err.value or N.TRM_ERR_CUDA, "TRMStreamPoolCreate")

    def open(self, ip):
        """Opens a free slot with voice `ip` (a TRMInputParameters); returns the slot number."""
        slot = N.lib().TRMStreamPoolOpen(self._h, C.byref(ip))
        if slot < 0:
            check(slot, "TRMStreamPoolOpen")
        return slot

    def open_events(self, ip, events, fg=None):
        """Opens a free slot with voice `ip` whose frames are generated on the device from `events` (a TRMEvent array)
        with settings `fg` (None: TRMFrameGeneration() defaults) as the slot advances (TRMStreamPoolOpenEvents).  Push
        it with an int: the number of frames to generate.  Returns (slot, frames the list expands to)."""
        events = np.ascontiguousarray(events, dtype=EVENT_DTYPE)
        fg = TRMFrameGeneration() if fg is None else fg
        nf = C.c_int64(0)
        slot = N.lib().TRMStreamPoolOpenEvents(self._h, C.byref(ip), _ptr(events), len(events), C.byref(fg), C.byref(nf))
        if slot < 0:
            check(slot, "TRMStreamPoolOpenEvents")
        return slot, int(nf.value)

    def close(self, slot):
        """Abandons an open slot without its tail; the slot becomes free."""
        check(N.lib().TRMStreamPoolClose(self._h, slot), "TRMStreamPoolClose")

    def slot_capacity(self):
        return int(N.lib().TRMStreamPoolSlotCapacity(self._h))

    @staticmethod
    def _entries(frames, flush):
        """The push's entries as the C call takes them: slots, frame counts, frames back to back, flush flags.  An int
        value is the number of frames an event slot generates; it adds no frames."""
        slots = list(frames.keys()) + [s for s in flush if s not in frames]
        gen = {s: int(frames[s]) for s in slots if isinstance(frames.get(s), (int, np.integer))}
        parts = [np.zeros((0, 16)) if s in gen else
                 np.ascontiguousarray(frames.get(s, np.zeros((0, 16))), dtype=np.float64).reshape(-1, 16) for s in slots]
        slot_a = np.array(slots, dtype=np.int32)
        nf_a = np.array([gen[s] if s in gen else p.shape[0] for s, p in zip(slots, parts)], dtype=np.int32)
        fl = set(flush)
        flush_a = np.array([1 if s in fl else 0 for s in slots], dtype=np.uint8)
        allf = np.concatenate(parts) if parts else np.zeros((0, 16))
        return slots, slot_a, nf_a, (allf if allf.shape[0] else None), flush_a

    def push(self, frames, flush=()):
        """frames: {slot: (m, 16) float64} (m may be 0), or {slot: m} for a slot opened with open_events; flush: slots
        that end with this push.  Returns {slot: samples} for every slot named in `frames` or `flush`."""
        slots, slot_a, nf_a, fr, flush_a = self._entries(frames, flush)
        n = len(slots)
        out = np.zeros(max(1, n * self.slot_capacity()), self.dtype)
        off = np.zeros(n + 1, np.int64)
        check(N.lib().TRMStreamPoolPush(self._h, n, _ptr(slot_a), _ptr(nf_a), _ptr(fr), _ptr(flush_a), _ptr(out), _ptr(off)),
              "TRMStreamPoolPush")
        return {s: out[off[i]:off[i + 1]].copy() for i, s in enumerate(slots)}

    def push_pcm16(self, frames, peak, flush=()):
        """As push, but each slot's new output comes back as 16-bit PCM scaled against `peak` (a float for every slot,
        or {slot: float}): rint(y * (32767 / peak) * amplitude(volume)), times the stereo gains for a 2-channel voice,
        saturated to the int16 range (TRMStreamPoolPushPCM16).  Returns {slot: (pcm, max)}: pcm is flat interleaved
        int16 as TRMTubeModel.pcm16 returns it, max is max |y| over the samples this push produced (0.0 if none)."""
        slots, slot_a, nf_a, fr, flush_a = self._entries(frames, flush)
        n = len(slots)
        peak_a = np.array([peak[s] if isinstance(peak, dict) else peak for s in slots], dtype=np.float64)
        pcm = np.zeros(max(1, 2 * n * self.slot_capacity()), np.int16)
        off = np.zeros(n + 1, np.int64)
        mx = np.zeros(max(1, n), np.float64)
        check(N.lib().TRMStreamPoolPushPCM16(self._h, n, _ptr(slot_a), _ptr(nf_a), _ptr(fr), _ptr(flush_a), _ptr(peak_a),
                                             _ptr(pcm), _ptr(off), _ptr(mx)), "TRMStreamPoolPushPCM16")
        return {s: (pcm[off[i]:off[i + 1]].copy(), float(mx[i])) for i, s in enumerate(slots)}

    def set_voice(self, voices):
        """voices: {slot: TRMInputParameters}.  Each open slot continues with its new voice from the next push, every
        piece of its state kept (TRMStreamPoolSetVoice): any field may change as long as the control period, tube rate,
        converter and channels stay.  Returns {slot: (tube_sample, output_sample)}: the tube-rate sample from which the
        new voice is synthesized, and the output sample from which PCM pushes use its volume and balance.  All or
        nothing: a refused call changes no slot."""
        slots = [int(s) for s in voices]
        n = len(slots)
        slot_a = np.array(slots, dtype=np.int32)
        arr = (N.TRMInputParametersStruct * max(1, n))()
        for i, s in enumerate(slots):
            C.memmove(C.byref(arr[i]), C.byref(voices[s]), C.sizeof(N.TRMInputParametersStruct))
        ts = np.zeros(max(1, n), np.int64)
        os_ = np.zeros(max(1, n), np.int64)
        check(N.lib().TRMStreamPoolSetVoice(self._h, n, _ptr(slot_a), arr, _ptr(ts), _ptr(os_)), "TRMStreamPoolSetVoice")
        return {s: (int(ts[i]), int(os_[i])) for i, s in enumerate(slots)}

    def save(self, slots, event_slots=False):
        """Snapshots of open slots (TRMStreamPoolSave): {slot: bytes}.  Each restores into any pool of this precision
        and continues the stream bit for bit; the saved slots are not changed.  Slots opened with open_events are
        refused unless event_slots is True (TRMStreamPoolSaveAny): they are then saved as format version 2, with their
        event list and generator state; frame-fed slots give the same bytes either way."""
        fn = "TRMStreamPoolSaveAny" if event_slots else "TRMStreamPoolSave"
        save = getattr(N.lib(), fn)
        slots = [int(s) for s in slots]
        slot_a = np.array(slots, dtype=np.int32)
        off = np.zeros(len(slots) + 1, np.int64)
        check(save(self._h, len(slots), _ptr(slot_a), None, 0, _ptr(off)), fn)
        blob = np.zeros(max(1, int(off[-1])), np.uint8)
        check(save(self._h, len(slots), _ptr(slot_a), _ptr(blob), blob.size, _ptr(off)), fn)
        return {s: blob[off[i]:off[i + 1]].tobytes() for i, s in enumerate(slots)}

    def restore(self, snapshots):
        """Opens one free slot per snapshot (bytes from save, in this or any other pool of the same precision; an event
        slot's snapshot restores as an event slot); returns the slots in order.  All or nothing (TRMStreamPoolRestore)."""
        snapshots = [bytes(b) for b in snapshots]
        off = np.zeros(len(snapshots) + 1, np.int64)
        off[1:] = np.cumsum([len(b) for b in snapshots])
        blob = np.frombuffer(b"".join(snapshots) or b"\0", np.uint8)
        out = np.zeros(max(1, len(snapshots)), np.int32)
        check(N.lib().TRMStreamPoolRestore(self._h, len(snapshots), _ptr(blob), _ptr(off), _ptr(out)), "TRMStreamPoolRestore")
        return [int(s) for s in out[:len(snapshots)]]

    def free(self):
        if self._h:
            N.lib().TRMStreamPoolFree(self._h)
            self._h = None

    def __del__(self):
        self.free()


def snapshot_info(snapshot):
    """What a stream pool snapshot holds, after the checks a restore makes apart from the destination pool
    (TRMStreamPoolSnapshotInfo; needs no device): {precision, channels, voice (TRMInputParameters), frames_pushed,
    samples_returned, bytes, events}.  events is None for a frame-fed slot's snapshot, or for an event slot's
    (TRMStreamPoolSnapshotEventInfo) {n_events, list_frames, frames_generated, fg (TRMFrameGeneration)}.  Raises
    TRMError for a snapshot a restore would refuse on its own."""
    b = bytes(snapshot)
    buf = C.create_string_buffer(b, max(1, len(b)))
    info = N.TRMStreamSnapshotInfoStruct()
    check(N.lib().TRMStreamPoolSnapshotInfo(buf, len(b), C.byref(info)), "TRMStreamPoolSnapshotInfo")
    ev = N.TRMStreamSnapshotEventInfoStruct()
    check(N.lib().TRMStreamPoolSnapshotEventInfo(buf, len(b), C.byref(ev)), "TRMStreamPoolSnapshotEventInfo")
    voice = TRMInputParameters()
    C.memmove(C.byref(voice), C.byref(info.voice), C.sizeof(voice))
    events = None
    if ev.from_events:
        fg = TRMFrameGeneration()
        C.memmove(C.byref(fg), C.byref(ev.fg), C.sizeof(fg))
        events = {"n_events": ev.n_events, "list_frames": ev.list_frames, "frames_generated": ev.frames_generated, "fg": fg}
    return {"precision": info.precision, "channels": info.channels, "voice": voice, "frames_pushed": info.frames_pushed,
            "samples_returned": info.samples_returned, "bytes": info.bytes, "events": events}


class TRMBatchTicket(object):
    """Handle of an asynchronous TRMBatch call; keeps the call's buffers alive until wait() returns."""

    def __init__(self, handle, keep):
        self._h = handle
        self._keep = keep

    def wait(self):
        if self._h:
            h, self._h = self._h, None
            rc = N.lib().TRMBatchWait(h)
            self._keep = None
            check(rc, "TRMBatchWait")

    def __del__(self):
        try:
            self.wait()
        except Exception:
            pass


class TRMResident(object):
    """Frames resident in HBM; stages launched on a caller-provided CUDA stream (bench `value`, roofline)."""

    def __init__(self, batch, frames, device=0):
        err = C.c_int(0)
        self.batch = batch
        self._h = N.lib().TRMBatchMakeResident(batch._h, _ptr(frames), device, C.byref(err))
        if not self._h:
            raise TRMError(err.value, "TRMBatchMakeResident")

    def run_stage(self, stage, stream=0):
        check(N.lib().TRMResidentRunStage(self._h, stage, C.c_void_p(stream)), "TRMResidentRunStage")

    def run(self, stream=0):
        check(N.lib().TRMResidentRun(self._h, C.c_void_p(stream)), "TRMResidentRun")

    def fetch(self, pcm_out=None, samples_out=None, maxima=None, tube_out=None):
        check(N.lib().TRMResidentFetch(self._h, _ptr(pcm_out), _ptr(samples_out), _ptr(maxima), _ptr(tube_out)),
              "TRMResidentFetch")

    def fetch_utterance(self, u):
        """(samples, pcm, maximum) of utterance u of the resident batch."""
        b = self.batch
        n = int(b.numberSamples[u])
        ch = 2 if (b._ip[u].channels if isinstance(b._ip, C.Array) else b._ip.channels) == 2 else 1
        smp = np.zeros(max(n, 1), b.sample_dtype)
        pcm = np.zeros(max(n * ch, 1), np.int16)
        mx = C.c_double(0.0)
        check(N.lib().TRMResidentFetchUtterance(self._h, int(u), _ptr(smp), _ptr(pcm), C.byref(mx)), "TRMResidentFetchUtterance")
        return smp[:n], pcm[:n * ch], float(mx.value)

    def free(self):
        if getattr(self, "_h", None):
            try:
                N.lib().TRMResidentFree(self._h)
            except TypeError:   # interpreter shutdown
                pass
            self._h = None

    def __del__(self):
        self.free()


def sweep_synthesize(ip, n_frames, n, seed=1, first_index=0, precision=N.TRM_PRECISION_FP64, device=0, probes=()):
    """TRMSweepSynthesize: n utterances of walk2 tracks generated on the device.  Returns a dict with per-utterance
    `checksums` (uint64), `maxima`, `numberSamples`, `kernel_ms`, `launches` and, for the utterances in `probes`
    (indices relative to this call), their PCM as `probe_pcm[k]`."""
    probes = np.ascontiguousarray(sorted(int(p) for p in probes), dtype=np.int64)
    ns = C.c_int32(0)
    check(N.lib().TRMSweepSynthesize(C.byref(ip), int(n_frames), int(seed), int(first_index), 0, precision, device,
                                     _ptr(np.zeros(1, np.uint64)), None, 0, None, None, 0, C.byref(ns), None, None), "TRMSweepSynthesize")
    stride = int(ns.value) * (2 if ip.channels == 2 else 1)
    sums = np.zeros(max(int(n), 1), np.uint64)
    mx = np.zeros(max(int(n), 1), np.float64)
    ppcm = np.zeros((max(len(probes), 1), max(stride, 1)), np.int16)
    launches, ms = C.c_int64(0), C.c_double(0.0)
    check(N.lib().TRMSweepSynthesize(C.byref(ip), int(n_frames), int(seed), int(first_index), int(n), precision, device, _ptr(sums),
                                     _ptr(mx), len(probes), _ptr(probes) if len(probes) else None, _ptr(ppcm), stride, C.byref(ns),
                                     C.byref(launches), C.byref(ms)), "TRMSweepSynthesize")
    return dict(checksums=sums[:n], maxima=mx[:n], numberSamples=int(ns.value), kernel_ms=float(ms.value), launches=int(launches.value),
                probes=probes, probe_pcm=ppcm[:len(probes)])


def pcm_checksum(pcm):
    """The sweep's per-utterance checksum of a PCM16 array: sum(pcm[i] * (2 i + 1)) mod 2^64."""
    p = np.asarray(pcm).astype(np.int64).astype(np.uint64)
    w = (2 * np.arange(p.shape[0], dtype=np.uint64) + np.uint64(1))
    with np.errstate(over="ignore"):
        return np.uint64((p * w).sum(dtype=np.uint64))
