/*
 * trm.h -- C API of the B200-native Tube Resonance Model (TRM) synthesizer.
 *
 * Drop-in boundary for the reference's Tube.framework public classes
 * (/root/reference/Frameworks/Tube/Tube.h:7-10):
 *
 *   TRMInputParameters   <- TRMInputParameters.h:24-56   (utterance-rate "voice" parameters)
 *   TRMParameters        <- TRMParameters.h:7-19         (one 250 Hz control frame)
 *   TRMDataList          <- TRMDataList.h:8-18           (parameters + growing frame list, file parser)
 *   TRMTubeModel         <- TRMTubeModel.h:29-40         (-initWithInputData:, -synthesize,
 *                                                         -generateWAVData, -saveOutputToFile:error:)
 *
 * plus a batched entry point (TRMBatch*) that the reference does not have: many independent
 * utterances in one call, sharded over the GPUs of one box.
 *
 * All synthesis runs on the GPU through libtrm_cuda (include/trm_cuda.h).  There is NO CPU
 * fallback: if CUDA is unavailable every synthesize call returns TRM_ERR_CUDA.
 *
 * Host code is C99.  Nothing in these signatures is a torch or C++ type.
 */
#ifndef TRM_H
#define TRM_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Oropharynx regions / nasal sections (TRMTubeModel.h:7-25) */
#define TRM_TOTAL_REGIONS          8
#define TRM_TOTAL_NASAL_SECTIONS   6

/* TRMInputParameters.h:7-21 */
enum { TRMSoundFileFormat_AU = 0, TRMSoundFileFormat_AIFF = 1, TRMSoundFileFormat_WAVE = 2 };
enum { TRMWaveFormType_Pulse = 0, TRMWaveFormType_Sine = 1 };

/* Error codes.  The reference returns nil / NO and prints to stderr (TRMTubeModel.m:204-207,
 * TRMFIRFilter.m:49-51, TRMDataList.m:45-57) or asserts (TRMTubeModel.m:417,511). */
enum {
    TRM_OK               = 0,
    TRM_ERR_TUBE_LENGTH  = -1,   /* length <= 0                     (TRMTubeModel.m:204-207)            */
    TRM_ERR_FIR          = -2,   /* FIR design failure              (TRMFIRFilter.m:49-51)              */
    TRM_ERR_NOMEM        = -3,   /* allocation failure              (TRMWavetable.m:65-68)              */
    TRM_ERR_PARAM        = -4,   /* parameters outside what the path defines (see DESIGN.md "deviations")*/
    TRM_ERR_CUDA         = -5,   /* no usable CUDA device / CUDA runtime error; trm_cuda_last_error()   */
    TRM_ERR_IO           = -6,   /* file open / read / write failure (TRMDataList.m:45-49)              */
    TRM_ERR_STATE        = -7,   /* call order: pull before synthesize, synthesize twice (single-use)   */
    TRM_ERR_SILENT       = -8    /* maximumSampleValue == 0: reference asserts (TRMTubeModel.m:511)     */
};

/* Arithmetic mode of the GPU path (BASELINE.json north_star). */
enum {
    TRM_PRECISION_FP64 = 0,        /* conformance: every value double, within 1e-9 relative of the reference      */
    TRM_PRECISION_FP32 = 1,        /* fast: FP32 state/signal, FP64 pitch->f0->phase, integer noise; >= 80 dB SNR  */
    TRM_PRECISION_FP64_STRICT = 2  /* the reference's operations in the reference's order, no FMA contraction: the
                                      bit-faithful twin the conformance mode is checked against (about 2x slower)  */
};

/* TRMInputParameters.h:26-54.  Field order follows the reference declaration. */
typedef struct TRMInputParameters {
    int32_t outputFileFormat;          /* TRMSoundFileFormat_*                                          */
    float   outputRate;                /* output sample rate (22050, 44100 Hz)                          */
    float   controlRate;               /* 1.0-1000.0 input tables/second (Hz)                           */
    double  volume;                    /* master volume (0 - 60 dB)                                     */
    int32_t channels;                  /* # of sound output channels (1, 2)                             */
    double  balance;                   /* stereo balance (-1 to +1)                                     */
    int32_t waveform;                  /* TRMWaveFormType_*                                             */
    double  tp;                        /* % glottal pulse rise time                                     */
    double  tnMin;                     /* % glottal pulse fall time minimum                             */
    double  tnMax;                     /* % glottal pulse fall time maximum                             */
    double  breathiness;               /* % glottal source breathiness                                  */
    double  length;                    /* nominal tube length (10 - 20 cm)                              */
    double  temperature;               /* tube temperature (25 - 40 C)                                  */
    double  lossFactor;                /* junction loss factor in (0 - 5 %)                             */
    double  apScale;                   /* aperture scl. radius (3.05 - 12 cm)                           */
    double  mouthCoef;                 /* mouth aperture coefficient                                    */
    double  noseCoef;                  /* nose aperture coefficient                                     */
    double  noseRadius[TRM_TOTAL_NASAL_SECTIONS]; /* fixed nose radii (0 - 3 cm); [0] is never read     */
    double  throatCutoff;              /* throat lp cutoff (50 - nyquist Hz)                            */
    double  throatVol;                 /* throat volume (0 - 48 dB)                                     */
    int32_t usesModulation;            /* pulse mod. of noise                                           */
    double  mixOffset;                 /* noise crossmix offset (30 - 60 dB)                            */
} TRMInputParameters;

/* TRMParameters.h:9-17 -- 16 doubles, 128 bytes, the unit the GPU stages with bulk copies. */
typedef struct TRMParameters {
    double glottalPitch;
    double glottalVolume;
    double aspirationVolume;
    double fricationVolume;
    double fricationPosition;
    double fricationCenterFrequency;
    double fricationBandwidth;
    double radius[TRM_TOTAL_REGIONS];
    double velum;
} TRMParameters;

/* Male-voice defaults of Monet (MMSynthesisParameters.m:160-191), mono, `outputRate` as given. */
void TRMInputParametersSetDefaults(TRMInputParameters *ip, float outputRate);

/* Values derived in -initWithInputData: (TRMTubeModel.m:196-203) and the SRC set-up
 * (TRMSampleRateConverter.m:69-106), available without running anything. */
typedef struct TRMDerivedValues {
    int32_t  controlPeriod;
    int32_t  sampleRate;
    double   actualTubeLength;
    int32_t  padSize;
    uint32_t timeRegisterIncrement;
    int64_t  tubeSamples;        /* (n_frames-1)*controlPeriod                                          */
    int32_t  numberSamples;      /* output-rate frames the converter will emit for n_frames frames      */
} TRMDerivedValues;
int TRMDeriveValues(const TRMInputParameters *ip, size_t n_frames, TRMDerivedValues *out);
/* 1 if the REFERENCE would hit its converter flush bug for an utterance of n_frames frames with these parameters
 * (TRMSampleRateConverter.m:160-168: when down-sampling, a final drain that finds fewer new inputs than the previous pass
 * overshot by runs over a whole ring of stale data and appends ~1024 x ratio spurious samples; exact rule in trm_host.c).
 * This implementation produces the converter's defined output; the flag tells a caller that the reference's sample
 * count and tail differ for that utterance. */
int TRMReferenceFlushBug(const TRMInputParameters *ip, size_t n_frames);

/* ---------------------------------------------------------------------------------------------
 * TRMDataList  (TRMDataList.h:8-18; TRMSynthesizer.m:98-106 for add/removeAll)
 * ------------------------------------------------------------------------------------------- */
typedef struct TRMDataList TRMDataList;

TRMDataList *TRMDataListCreate(void);                                  /* -init                          */
TRMDataList *TRMDataListCreateWithContentsOfFile(const char *path, int *err); /* -initWithContentsOfFile: */
void         TRMDataListFree(TRMDataList *list);
TRMInputParameters *TRMDataListInputParameters(TRMDataList *list);     /* .inputParameters               */
int          TRMDataListAddParameters(TRMDataList *list, const TRMParameters *frame); /* [values addObject:] */
int          TRMDataListAddParametersArray(TRMDataList *list, const TRMParameters *frames, size_t n);
void         TRMDataListRemoveAllParameters(TRMDataList *list);        /* [values removeAllObjects]      */
size_t       TRMDataListCount(const TRMDataList *list);
const TRMParameters *TRMDataListValues(const TRMDataList *list);
/* Writes the list in the reference's text input format (MMSynthesisParameters.m:278-310,
 * TRMParameters.m:26-45) -- what Monet dumps to /tmp/Monet.parameters. */
int          TRMDataListWriteToFile(const TRMDataList *list, const char *path);

/* ---------------------------------------------------------------------------------------------
 * Utterance-rate ("voice") parameters as Monet keeps them: MMSynthesisParameters
 * (Frameworks/GnuSpeech/MonetModel/MMSynthesisParameters.h:22-52).  Field for field the reference's properties;
 * the defaults are the registered NSUserDefaults of MMSynthesisParameters.m:160-190.
 * ------------------------------------------------------------------------------------------- */
typedef struct TRMSynthesisParameters {
    double  masterVolume;        /* dB, 0..60   */
    double  vocalTractLength;    /* cm          */
    double  temperature;         /* deg C       */
    double  balance;             /* -1..+1      */
    double  breathiness;         /* % of GS amplitude */
    double  lossFactor;          /* % of unity gain   */
    double  pitch;               /* semitones, added to every frame's glottal pitch by the frame generator
                                    (EventList.m:985); NOT part of the TRM header */
    double  throatCutoff, throatVolume, apertureScaling, mouthCoef, noseCoef, mixOffset;
    double  n1, n2, n3, n4, n5;
    double  tp, tnMin, tnMax;
    int32_t glottalPulseShape;        /* 0 pulse, 1 sine  (MMGlottalPulseShape)                 */
    int32_t shouldUseNoiseModulation;
    int32_t samplingRate;             /* 0 = 22050 Hz, 1 = 44100 Hz  (MMSamplingRate)          */
    int32_t outputChannels;           /* 0 = mono, 1 = stereo        (MMChannels)              */
} TRMSynthesisParameters;

/* +initialize / -restoreDefaultValues (MMSynthesisParameters.m:160-225): the male voice. */
void TRMSynthesisParametersRestoreDefaults(TRMSynthesisParameters *sp);
/* The five voice types of the TextToSpeech kit (Other/voices.config:15-48): "Male", "Female", "LgChild", "SmChild",
 * "Baby" (case-insensitive): defaults with that voice's tract length, glottal pulse rise / fall times (the file gives
 * them as fractions of the period, the header wants per cent) and base pitch.  TRM_ERR_PARAM for an unknown name. */
int  TRMSynthesisParametersForVoice(const char *name, TRMSynthesisParameters *sp);
/* -[TRMSynthesizer setupSynthesisParameters:] (TRMSynthesizer.m:38-65): the TRM header of an utterance.
 * controlRate = 250, channels = outputChannels + 1, noseRadius[0] = 0, outputFileFormat keeps `fileFormat`. */
void TRMInputParametersFromSynthesisParameters(const TRMSynthesisParameters *sp, int32_t fileFormat, TRMInputParameters *ip);
/* -parameterString (MMSynthesisParameters.m:278-310): the 26 header lines of a TRM input file, byte for byte the
 * reference's printf formats.  Returns a malloc'ed string (TRMFree). */
char *TRMSynthesisParametersString(const TRMSynthesisParameters *sp);

/* ---------------------------------------------------------------------------------------------
 * TRMTubeModel  (TRMTubeModel.h:29-40).  Single-use like the reference (TRMSynthesizer.m:120).
 * ------------------------------------------------------------------------------------------- */
typedef struct TRMTubeModel TRMTubeModel;

/* -initWithInputData: (TRMTubeModel.m:186-260).  Copies parameters and frames.  NULL on error, *err set. */
TRMTubeModel *TRMTubeModelCreate(const TRMDataList *inputData, int *err);
void          TRMTubeModelFree(TRMTubeModel *model);
int           TRMTubeModelSetPrecision(TRMTubeModel *model, int precision);   /* default TRM_PRECISION_FP64 */
int           TRMTubeModelSetDevice(TRMTubeModel *model, int device);         /* default 0                  */

/* -synthesize (TRMTubeModel.m:272-361): whole utterance, blocking. */
int           TRMTubeModelSynthesize(TRMTubeModel *model);

/* sampleRateConverter.numberSamples / .maximumSampleValue / .resampledData (TRMSampleRateConverter.h:13-17) */
int32_t       TRMTubeModelNumberSamples(const TRMTubeModel *model);
int32_t       TRMTubeModelChannels(const TRMTubeModel *model);          /* 1 or 2: int16 elements per frame of PullPCM16 */
int           TRMTubeModelHitsReferenceFlushBug(const TRMTubeModel *model);
double        TRMTubeModelMaximumSampleValue(const TRMTubeModel *model);
const double *TRMTubeModelResampledData(const TRMTubeModel *model);
/* tube-rate signal before the converter (what -synthesize hands to dataFill:, TRMTubeModel.m:346) */
const double *TRMTubeModelTubeSignal(const TRMTubeModel *model, int64_t *count);
void          TRMTubeModelGetDerivedValues(const TRMTubeModel *model, TRMDerivedValues *out);

/* Scaled 16-bit PCM, host endian; channels interleaved (TRMTubeModel.m:515-557 scaling = the WAV variant;
 * file_variant != 0 selects the x2 stereo scaling of -saveOutputToFile:, TRMTubeModel.m:382-383).
 * Returns the number of sample frames written or a negative error. */
int64_t       TRMTubeModelPullPCM16(const TRMTubeModel *model, int16_t *dst, size_t max_frames, int file_variant);

/* -generateWAVData (TRMTubeModel.m:509-593): malloc'ed RIFF/WAVE bytes (18-byte fmt chunk as the reference
 * writes it); free with TRMFree. */
uint8_t      *TRMTubeModelGenerateWAVData(const TRMTubeModel *model, size_t *length, int *err);
/* -saveOutputToFile:error: (TRMTubeModel.m:365-490): AU / AIFF (big-endian) or WAVE by outputFileFormat. */
int           TRMTubeModelSaveOutputToFile(const TRMTubeModel *model, const char *path);
void          TRMFree(void *p);

/* ---------------------------------------------------------------------------------------------
 * Batched entry point (new).  n independent utterances; utterance u uses ip[u] (or ip[0] when
 * shared_parameters != 0) and frames[frame_offset[u] .. frame_offset[u]+n_frames[u]).
 * ------------------------------------------------------------------------------------------- */
typedef struct TRMBatch TRMBatch;

typedef struct TRMBatchLayout {
    int64_t total_frames;        /* frames consumed from the input array                                */
    int64_t total_pcm_samples;   /* int16 elements needed in the PCM output buffer                      */
    int64_t total_out_samples;   /* elements needed in the optional float/double output buffer          */
    double  audio_seconds;       /* sum over utterances of (n_frames-1)/controlRate                     */
    int64_t tube_samples;        /* sum of tube-rate samples                                            */
    int64_t out_samples;         /* sum of numberSamples                                                */
} TRMBatchLayout;

/* Plans the batch: validates parameters, derives per-utterance constants, sizes and offsets. */
TRMBatch *TRMBatchCreate(int n_utterances, const TRMInputParameters *ip, int shared_parameters,
                         const int64_t *frame_offset, const int32_t *n_frames, int precision, int *err);
void      TRMBatchFree(TRMBatch *batch);
void      TRMBatchGetLayout(const TRMBatch *batch, TRMBatchLayout *layout);
/* How the `frames` argument of TRMBatchSynthesize / TRMBatchSynthesizeAsync is read: TRMParameters rows (16 doubles,
 * the default) or rows of 16 floats in the same order.  Monet's frame generator holds its table in float
 * (EventList.m:968-1002) and TRMParameters only widens it, so float rows carry the same information in half the
 * bytes across PCIe; the waveguide kernel widens them when it reads them and the results are bit-identical. */
enum { TRM_FRAMES_F64 = 0, TRM_FRAMES_F32 = 1 };
int       TRMBatchSetFrameFormat(TRMBatch *batch, int format);
/* per-utterance results / placement; valid after TRMBatchCreate (offsets, counts) and after synthesis (max) */
const int32_t *TRMBatchNumberSamples(const TRMBatch *batch);       /* [n] output frames                   */
const int64_t *TRMBatchPCMOffsets(const TRMBatch *batch);          /* [n] element offset into pcm_out     */
const int64_t *TRMBatchOutOffsets(const TRMBatch *batch);          /* [n] element offset into samples_out */
const double  *TRMBatchMaximumSampleValues(const TRMBatch *batch); /* [n]                                 */
const uint8_t *TRMBatchReferenceFlushBugFlags(const TRMBatch *batch); /* [n] TRMReferenceFlushBug per utterance  */

/* Synthesizes the whole batch on `n_devices` GPUs (devices[] lists CUDA ordinals; NULL = 0..n-1), host
 * buffers in and out.  frames: TRMParameters array in host memory (pinned memory from TRMHostAlloc makes
 * the copies asynchronous).  pcm_out: int16, TRMBatchLayout.total_pcm_samples elements, may be NULL.
 * samples_out: unscaled output-rate samples, double (FP64 mode) or float (FP32 mode),
 * total_out_samples elements, may be NULL.  Blocking. */
int TRMBatchSynthesize(TRMBatch *batch, const TRMParameters *frames, int16_t *pcm_out, void *samples_out,
                       const int *devices, int n_devices);

/* Asynchronous form for callers with a stream of batches: returns at once with a ticket; TRMBatchWait blocks until the
 * outputs are in the host buffers, frees the ticket and returns the call's status.  Every device keeps up to three calls in
 * flight (three context lanes, each with its own streams and scratch), so the PCM of call k is copied out while call
 * k+1 computes and call k+2 uploads its frames.  One ticket per TRMBatch object at a time (the batch holds the call's maxima); inputs and outputs
 * must stay valid until TRMBatchWait returns.  (The reference has no counterpart: -synthesize is synchronous.) */
typedef struct TRMBatchTicket TRMBatchTicket;
TRMBatchTicket *TRMBatchSynthesizeAsync(TRMBatch *batch, const TRMParameters *frames, int16_t *pcm_out, void *samples_out,
                                        const int *devices, int n_devices, int *err);
int TRMBatchWait(TRMBatchTicket *ticket);

/* ---------------------------------------------------------------------------------------------
 * Control frames from event lists (SURVEY.md 8(f) rank 1): the step before the tube model in Monet,
 * -[EventList generateOutputInTimeRange:forSynthesizer:parameterLogger:] (Frameworks/GnuSpeech/MonetModel/
 * EventList.m:883-1061, full time range) with MMDriftGenerator (MMDriftGenerator.m:41-78), run on the GPU so that a
 * batch needs only its sparse event lists uploaded.
 * ------------------------------------------------------------------------------------------- */
#define TRM_EVENT_VALUES 36
/* Event (MonetModel/Event.h): time in ms; value[0..15] the 16 TRM parameters, [16..31] the "special" offsets added to
 * them, [32] macro intonation (semitones), [33..35] smooth-intonation slopes; NaN = no value at this event. */
typedef struct TRMEvent { int64_t time; double value[TRM_EVENT_VALUES]; } TRMEvent;
/* What the generator takes from MMIntonation (MMIntonation.m:74-80) and the model (EventList.m:983). */
typedef struct TRMFrameGeneration {
    int32_t useMacroIntonation, useMicroIntonation, useSmoothIntonation, useDrift;   /* defaults: all 1 */
    double  driftDeviation, driftCutoff;     /* defaults 1.0, 4 */
    double  pitch;                           /* synthesisParameters.pitch, added to every frame's glottal pitch */
    float   driftSeed;                       /* drift generator state at entry; 0.7892347 for a fresh generator */
    int32_t reserved;
} TRMFrameGeneration;
void    TRMFrameGenerationSetDefaults(TRMFrameGeneration *fg);
/* Number of 4 ms frames the generator emits for an event list (what n_frames of TRMBatchCreate must be). */
int64_t TRMEventListFrameCount(const TRMEvent *events, int64_t n_events);
/* Runs the generator for every utterance of the batch on `device` and returns the frames in frames_out
 * (TRMBatchLayout.total_frames entries, utterance u at the frame_offset given to TRMBatchCreate).  Utterance u reads
 * events[event_offset[u] .. +n_events[u]); fg has one entry per utterance, or one for all if shared_fg != 0.
 * drift_seed_out (n floats, may be NULL) receives each generator's seed at exit. */
int TRMBatchGenerateFrames(TRMBatch *batch, const TRMEvent *events, const int64_t *event_offset, const int32_t *n_events,
                           const TRMFrameGeneration *fg, int shared_fg, TRMParameters *frames_out, float *drift_seed_out,
                           int device);
/* Event lists in, PCM out: generator and tube model back to back on the device; the frames never exist on the host. */
int TRMBatchSynthesizeEvents(TRMBatch *batch, const TRMEvent *events, const int64_t *event_offset, const int32_t *n_events,
                             const TRMFrameGeneration *fg, int shared_fg, int16_t *pcm_out, void *samples_out, int device);

/* ---------------------------------------------------------------------------------------------
 * Streaming synthesis (SURVEY.md 8(f) rank 3): TRAcT's mode of use (Applications/TRAcT/tube.c:1096-1191) -- audio as
 * it is produced, parameters arriving while it plays, no normalisation to a global maximum -- for many voices at once.
 * n_streams independent streams with the same voice are advanced together: every push appends m control frames per
 * stream and returns the un-normalised output-rate samples that became computable (what .resampledData holds for a
 * whole utterance; double in FP64 mode, float in FP32 mode).  The state of every recurrence is carried on the device:
 * the pushes, concatenated, are bit-identical to synthesizing the whole utterance at once.
 * A stream owns its device buffers and wavetable copy; it does not hold a context lane between calls.
 * ------------------------------------------------------------------------------------------- */
typedef struct TRMStream TRMStream;
TRMStream *TRMStreamCreate(int n_streams, const TRMInputParameters *voice, int precision, int max_frames_per_push,
                           int device, int *err);
/* samples per stream one push can return = row stride (in samples) of samples_out */
int64_t TRMStreamCapacity(const TRMStream *stream);
/* frames: [stream][m] TRMParameters; samples_out: [stream][TRMStreamCapacity()] ; *n_samples = samples returned per
 * stream by this push.  flush != 0 ends the streams (the converter's tail, as at the end of -synthesize). */
int TRMStreamPush(TRMStream *stream, const TRMParameters *frames, int m, int flush, void *samples_out, int64_t *n_samples);
/* TRMStreamPoolSetVoice (below) for all n streams at once: every stream continues with `voice`.  The streams are in
 * lockstep, so one *tube_sample / *output_sample (either may be NULL) holds for all of them.  After the flush:
 * TRM_ERR_STATE. */
int TRMStreamSetVoice(TRMStream *stream, const TRMInputParameters *voice, int64_t *tube_sample, int64_t *output_sample);
void TRMStreamFree(TRMStream *stream);

/* ---------------------------------------------------------------------------------------------
 * Stream pool: serving many streams that start, advance and end independently, each with its own voice (tract length,
 * so control period, tube rate and converter signature; glottal pulse; output rate).  A slot is opened with a voice;
 * each push advances any subset of the open slots, each by its own number of frames, and all of them are synthesized by
 * one waveguide launch and one resampler launch.  A slot ends with its own flush (or is abandoned with Close) and can
 * then be opened again.  The contract of TRMStream holds per slot: its pushes, concatenated, are bit-identical to the
 * one-shot TRMBatch synthesis of that utterance with that voice, whatever the other slots do.
 * A pool owns its device buffers and one 512-entry wavetable row per slot (written when the slot opens); it holds no
 * context lane between calls.  A pool is used by one thread at a time.  No CPU fallback: without a device
 * TRMStreamPoolCreate fails with TRM_ERR_CUDA.
 * ------------------------------------------------------------------------------------------- */
typedef struct TRMStreamPool TRMStreamPool;
/* capacity slots on one device, one arithmetic mode for all of them. */
TRMStreamPool *TRMStreamPoolCreate(int capacity, int precision, int max_frames_per_push, int device, int *err);
/* Opens a free slot with this voice (validated exactly as TRMBatchCreate validates a voice); returns the slot >= 0 or a
 * negative TRM_ERR_*.  Pool full: TRM_ERR_STATE. */
int TRMStreamPoolOpen(TRMStreamPool *pool, const TRMInputParameters *voice);
/* Opens a free slot with `voice` whose control frames come from an event list (TRMEvent, as TRMBatchGenerateFrames
 * takes it) and frame-generation settings `fg`.  The list is validated as check_event_lists validates a batch's lists
 * and copied to the device; *n_frames_out (may be NULL) = TRMEventListFrameCount(events, n_events).
 * The voice is validated as TRMStreamPoolOpen validates it; a list the batch path refuses is refused with the same code
 * (TRM_ERR_PARAM); pool full: TRM_ERR_STATE.  Returns the slot >= 0 or a negative TRM_ERR_*.
 * Such a slot is an event slot until it ends:
 *   Push.  In TRMStreamPoolPush / TRMStreamPoolPushPCM16, n_frames[i] of an event slot's entry is the number of frames to
 *     generate for it, continuing where its previous push stopped; it takes nothing from `frames`, which frame-fed entries
 *     consume back to back as always (one push may mix both; `frames` may be NULL when no frame-fed entry has frames).
 *     An entry that would take the slot past its list's frame count is refused (TRM_ERR_PARAM) with the push's other
 *     refusals, before any device work.
 *   Continuation.  Advanced to the end of its list and flushed, a slot's pushes, concatenated, equal what
 *     TRMBatchSynthesizeEvents returns for a one-utterance batch with the same voice, events and fg, bit for bit: samples
 *     in every precision; PCM16 and the per-push maxima when the peak given is that utterance's maximumSampleValue --
 *     for any split of the frames over pushes, whatever the other slots do.
 *   Early end.  A flush before the end of the list ends the slot as a frame-fed flush does: its output equals the
 *     one-shot synthesis of the k frames generated so far (the first k of TRMBatchGenerateFrames' frames for the list).
 *   Close and flush free the slot as for any slot; it may be reopened either way.  TRMStreamPoolSave refuses event slots
 *     (TRM_ERR_STATE); TRMStreamPoolSaveAny saves them (format version 2, below). */
int TRMStreamPoolOpenEvents(TRMStreamPool *pool, const TRMInputParameters *voice, const TRMEvent *events,
                            int64_t n_events, const TRMFrameGeneration *fg, int64_t *n_frames_out);
/* Abandons an open slot without its tail (client went away); the slot becomes free. */
int TRMStreamPoolClose(TRMStreamPool *pool, int slot);
/* Samples one slot can return from one push (row bound for samples_out).  Sized at creation for the default voice; it
 * grows when a slot opens with a voice that produces more samples per control frame than any before, so read it after
 * opening slots. */
int64_t TRMStreamPoolSlotCapacity(const TRMStreamPool *pool);
/* Advances n distinct open slots: slot[i] gets n_frames[i] (0..max) frames, taken back to back from `frames`; flush[i] != 0
 * (flush may be NULL: no flush) ends slot[i] (converter tail, as at the end of -synthesize) and frees it.  Samples (double,
 * or float in FP32 mode) are packed: entry i's are samples_out[out_offset[i] .. out_offset[i+1]); samples_out holds
 * n * SlotCapacity elements.  An unopened slot (TRM_ERR_STATE), a slot named twice or too many frames (TRM_ERR_PARAM)
 * fail the whole push before any work: the pool is left exactly as it was.  So does any other error returned before the
 * push's first launch (out of device memory, say): every slot is as it was.  After a CUDA error during the push's device
 * work (TRM_ERR_CUDA) the pool's contents are undefined: free it. */
int TRMStreamPoolPush(TRMStreamPool *pool, int n, const int32_t *slot, const int32_t *n_frames, const TRMParameters *frames,
                      const uint8_t *flush, void *samples_out, int64_t *out_offset /* [n + 1] */);
/* As TRMStreamPoolPush, but entry i's new output comes back as 16-bit PCM, host endian, channels interleaved as the
 * slot's voice says (1 or 2):
 *   scale = (32767 / peak[i]) * amplitude(volume);  mono: rint(y * scale);
 *   stereo: rint(y * leftGain * scale), rint(y * rightGain * scale)   (the WAV variant, TRMTubeModel.m:515-559),
 *   saturated to [-32768, 32767].
 * With peak[i] equal to the utterance's maximumSampleValue, a slot's PCM pushes, concatenated, equal TRMBatch's pcm_out
 * for that utterance bit for bit.  Entry i's PCM is pcm_out[pcm_offset[i] .. pcm_offset[i+1]) (int16 elements; frames =
 * elements / channels); pcm_out holds 2 * n * TRMStreamPoolSlotCapacity elements.  max_out[i] (may be NULL): max |y| over
 * the samples entry i produced in this push, 0.0 if none (NaN never wins, as in maximumSampleValue); the maximum over a
 * slot's pushes equals TRMBatch's maximumSampleValue.  peak[i] must be finite and > 0 (TRM_ERR_PARAM).  All refusals of
 * TRMStreamPoolPush apply, and are checked, with peak, before any device work: a refused push leaves the pool unchanged.
 * Other errors leave the pool as they do for TRMStreamPoolPush.  A slot may be advanced by TRMStreamPoolPush and
 * TRMStreamPoolPushPCM16 in any order. */
int TRMStreamPoolPushPCM16(TRMStreamPool *pool, int n, const int32_t *slot, const int32_t *n_frames,
                           const TRMParameters *frames, const uint8_t *flush, const double *peak,
                           int16_t *pcm_out, int64_t *pcm_offset /* [n + 1] */, double *max_out);
/* Changes the voice of n distinct open slots (frame-fed or event-fed), effective from the next push: TRAcT's sliders on
 * a stream that keeps playing.  Slot slot[i] continues with voice[i]; every piece of carried state (oscillator, noise,
 * filter memories, tube waves, converter, pending frames) is kept, so the stream does not restart from silence.
 *   What may change.  Any field, as long as the new voice derives the same rate constants as the slot's current voice:
 *     control period, tube sample rate, converter increment and pad, channels (what a snapshot stores as "derived").  So
 *     outputRate, controlRate, temperature, channels and the tract length stay (a length or temperature that rounds to
 *     the same control period is accepted); changing the tract length is a new stream.  Everything else may change:
 *     volume, balance, waveform, tp / tnMin / tnMax, breathiness, lossFactor, apScale, mouthCoef, noseCoef,
 *     noseRadius[1..5], throatCutoff, throatVol, usesModulation, mixOffset.
 *   Where it takes effect.  The tube model uses the new voice from tube-rate sample tube_sample[i] on: the first sample
 *     the slot has not synthesized, floor16((frames pushed - 1) * controlPeriod) after two frames or more, else 0.  Frames
 *     already pushed whose samples lie at or after it are synthesized with the new voice.  volume and balance apply to the
 *     PCM16 of every output a later TRMStreamPoolPushPCM16 returns, from output sample output_sample[i] on; float samples
 *     are unscaled, so they do not depend on them.  tube_sample and output_sample may be NULL.
 *   Continuation.  A slot's pushes, concatenated, equal the synthesis of its frames with the voice schedule "opening voice
 *     from sample 0, each new voice from its tube_sample", within the tolerance of the slot's TRM_PRECISION_* mode, and
 *     the pushes after a change are bit-identical for any split of the frames over pushes.  One exception in FP32: that
 *     mode carries the mouth and nose reflection memories multiplied by the damping factor, so across a change of
 *     lossFactor they continue for one sample with the previous factor.  Measured against the exact schedule: about
 *     80 dB SNR for 0.5 -> 5 % alone on 0.4 s at control period 63, 71-75 dB for random changes that include it, down
 *     to 44-49 dB for a short stream (800 samples) at control period 8.  The FP64 modes have no such exception.
 *     TRMStreamPoolSave / SaveAny store the current voice (TRMStreamPoolSnapshotInfo reports it) and a restore continues
 *     with it, bit for bit; the snapshot format does not change.
 *   Refusals.  All n entries are checked before anything changes, and a refused call leaves the pool exactly as it was:
 *     an unopened slot (TRM_ERR_STATE); a slot named twice or a voice whose rate constants differ (TRM_ERR_PARAM); a voice
 *     TRMBatchCreate refuses (its code).  A CUDA error while the glottal table rows go up (TRM_ERR_CUDA) leaves the pool's
 *     contents undefined, as for a push. */
int TRMStreamPoolSetVoice(TRMStreamPool *pool, int n, const int32_t *slot, const TRMInputParameters *voice /* [n] */,
                          int64_t *tube_sample /* [n] or NULL */, int64_t *output_sample /* [n] or NULL */);
void TRMStreamPoolFree(TRMStreamPool *pool);

/* Snapshots: a live slot as a self-contained byte string that continues in any pool of the same precision, on any device,
 * in any process.  Moving streams off a GPU (save, close, restore elsewhere), growing a pool, surviving a restart and
 * branching a stream (restore while the saved slot keeps going) all use these three calls.
 *
 * Continuation.  A slot restored from a snapshot behaves as the saved slot would have from that point, whatever either
 * pool does: its later Push / PushPCM16 outputs, appended to what the saved slot had returned before the save, equal the
 * one-shot TRMBatch synthesis bit for bit (samples, PCM at a given peak, per-push maxima).  Saving does not change the
 * saved slot; closing it after the save is a migration, letting it continue is a fork.  The PCM peak is not part of the
 * state: it is passed with every push, as before.
 * What it depends on.  A snapshot holds no device pointers, slot numbers, device ordinals or pool sizes, and
 * save(restore(b)) == b byte for byte.  It restores into a pool with another capacity, max_frames_per_push, slot index or
 * device, but only into the same precision code (FP64 conformance and FP64 strict carry different states).
 * Format (little-endian, written field by field; libtrm owns it):
 *   header    8 bytes "TRMSNAP\0", u32 version (1), u32 precision, u64 total bytes, u64 FNV-1a 64 of every byte after it
 *   voice     TRMInputParameters field by field, no padding (192 bytes)
 *   derived   u32 controlPeriod, sampleRate, timeRegisterIncrement, padSize, channels, element size (4 or 8)
 *   counters  i64 frames pushed, tube-rate samples synthesized, output samples returned, first tube-rate sample kept,
 *             first pending frame; i32 pending frames, fresh (1 while the waveguide has not run)
 *   data      pending frames [n][16] f64; the carried waveguide state (32 + 96 x element size bytes) unless fresh; the
 *             kept tube-rate history [synthesized - first kept] of the precision's element type
 * Restore derives the glottal table and every derived constant again from the voice, as TRMStreamPoolOpen does, and checks
 * the counters against each other and the voice: a corrupt snapshot can give wrong audio but never an access outside
 * the slot's own buffers.
 *
 * Event slots (TRMStreamPoolOpenEvents) are saved by TRMStreamPoolSaveAny as format version 2, which carries the event list
 * and the frame generator's state with the stream.  A restored version-2 slot is an event slot: pushes give it frame
 * counts, it may flush early and it may be saved again.  Its continuation contract is the event slot's: advanced to the
 * end of its list and flushed, its outputs, appended to what the saved slot returned before the save, equal
 * TRMBatchSynthesizeEvents for that voice, list and fg bit for bit (samples; PCM16 and per-push maxima at the utterance's
 * peak); flushed earlier, they equal the one-shot synthesis of the frames generated so far.  Saving does not change the
 * slot, migration and fork both work, and save(restore(b)) == b.
 * Format version 2: header (version 2), voice, derived and counters as version 1 (frames pushed = frames generated), then
 *   events    (at byte 296, 72 bytes) i64 n_events, list_frames (TRMEventListFrameCount of the list); fg field by field:
 *             i32 useMacroIntonation, useMicroIntonation, useSmoothIntonation, useDrift, f64 driftDeviation, driftCutoff,
 *             pitch, f32 driftSeed, i32 reserved (0); u32 generator (1 exactly when frames generated > 0), u32 reserved (0)
 *   data      the version-1 data part (the pending frames are the generated ones the slot still needs); then, if generator
 *             is 1, the generator state: f64 cv[32], cd[32], cv32, cd32, cd33, cd34, cd35; i64 i; u64 now, next; f32 seed,
 *             prev, pitchDeviation, pitchOffset, a0, b1 (600 bytes); then the whole list, n_events x (i64 time, 36 f64)
 * Restore checks a version-2 snapshot as a version-1 one and further: the length against n_events and generator, the list
 * as TRMStreamPoolOpenEvents checks it, list_frames against the list, frames generated <= list_frames, the generator flag,
 * the generator's event index and clock (i, now, next) against the frames generated, and that the pending frames plus a
 * push of max_frames_per_push fit the destination's pending-frame rows (TRM_ERR_PARAM).  The tracks' values and deltas and
 * the drift state are not checked: they can give wrong audio, never an access outside the slot (only i and n_events index
 * the list, and the checks pin i to [1, n_events]). */
typedef struct TRMStreamSnapshotInfo {
    int32_t precision;               /* TRM_PRECISION_* the snapshot restores into                                 */
    int32_t channels;                /* int16 elements per PCM frame of the stream                                  */
    TRMInputParameters voice;
    int64_t frames_pushed;           /* control frames the stream has received                                      */
    int64_t samples_returned;        /* output-rate samples (PCM frames) it has returned                            */
    int64_t bytes;                   /* size of the snapshot                                                        */
} TRMStreamSnapshotInfo;
/* Snapshots of n distinct open slots, packed: slot[i]'s bytes are blob[offset[i] .. offset[i+1]).  blob == NULL: only
 * fills offset (sizes from host bookkeeping, no device work).  Refused before anything is written: an unopened slot or a
 * slot opened with TRMStreamPoolOpenEvents (TRM_ERR_STATE), a slot named twice or blob_capacity < offset[n]
 * (TRM_ERR_PARAM).  Writes version 1 only, so a caller that stores snapshots for a version-1 reader never gets another. */
int TRMStreamPoolSave(TRMStreamPool *pool, int n, const int32_t *slot, void *blob, int64_t blob_capacity,
                      int64_t *offset /* [n + 1] */);
/* TRMStreamPoolSave for slots of either kind: an event slot is saved as version 2 instead of being refused; a frame-fed
 * slot's snapshot is byte for byte what TRMStreamPoolSave writes.  One call may mix both kinds (draining a GPU is one
 * save).  Arguments, packing, blob == NULL sizing and the other refusals are TRMStreamPoolSave's. */
int TRMStreamPoolSaveAny(TRMStreamPool *pool, int n, const int32_t *slot, void *blob, int64_t blob_capacity,
                         int64_t *offset /* [n + 1] */);
/* Opens n free slots from n snapshots of version 1 or 2 (the same packing); slot_out[i] is the slot that continues
 * snapshot i.  All n are checked before anything changes, and a refused call leaves the pool as it was: bad magic,
 * version, length or checksum, another precision, derived constants that differ from the voice's (e.g. a snapshot from
 * another library build), counters that disagree, or a version-2 event part that fails its checks (TRM_ERR_PARAM); a
 * voice TRMBatchCreate refuses (its code); kept history and pending frames that would not fit this pool's next push of
 * max_frames_per_push frames (TRM_ERR_PARAM); fewer than n free slots (TRM_ERR_STATE).  SlotCapacity may grow, as with
 * Open. */
int TRMStreamPoolRestore(TRMStreamPool *pool, int n, const void *blob, const int64_t *offset /* [n + 1] */, int32_t *slot_out);
/* Host only (no device needed): validates one snapshot as Restore does, apart from the destination pool, and reports
 * what it holds.  Lets a router pick a pool before restoring. */
int TRMStreamPoolSnapshotInfo(const void *blob, int64_t bytes, TRMStreamSnapshotInfo *info);
/* What a version-2 snapshot holds about its event list.  A router schedules a restored event slot's pushes with
 * list_frames - frames_generated: a push past the end of the list is refused. */
typedef struct TRMStreamSnapshotEventInfo {
    int32_t from_events;             /* 1 for version 2 (an event slot); 0 for version 1, every other field 0           */
    int64_t n_events;                /* events of the list                                                          */
    int64_t list_frames;             /* TRMEventListFrameCount of the list                                          */
    int64_t frames_generated;        /* frames generated (and pushed) so far                                        */
    TRMFrameGeneration fg;
} TRMStreamSnapshotEventInfo;
/* Host only: checks the snapshot as TRMStreamPoolSnapshotInfo does and reports its event part. */
int TRMStreamPoolSnapshotEventInfo(const void *blob, int64_t bytes, TRMStreamSnapshotEventInfo *info);

/* ---------------------------------------------------------------------------------------------
 * Sweeps (BASELINE configs[4]: 10^6 synthetic 2 s utterances): n utterances of one voice whose control tracks are the walk2
 * workload of include/trm_workload.h, generated on the device (utterance k = index first_index + k of stream `seed`) --
 * 64 GB of frames per million utterances never cross PCIe.  The audio stays on the device as well: per utterance an
 * 8-byte checksum of its PCM16, sum(pcm[i] * (2 i + 1)) mod 2^64, and its maximumSampleValue come back (checksums equal
 * across any sharding of the index range); the PCM of the utterances listed in probe_utt (sorted, relative to this call)
 * is copied to probe_pcm (rows of probe_stride int16) for comparison with the reference.  *numberSamples: output frames per
 * utterance; *kernel_ms: device time of all chunks.
 * ------------------------------------------------------------------------------------------- */
int TRMSweepSynthesize(const TRMInputParameters *ip, int32_t n_frames, uint64_t seed, uint64_t first_index, int64_t n,
                       int precision, int device, uint64_t *checksums, double *maxima, int64_t n_probe, const int64_t *probe_utt,
                       int16_t *probe_pcm, int64_t probe_stride, int32_t *numberSamples, int64_t *launches, double *kernel_ms);

/* Debug / conformance variant on one device: additionally returns the tube-rate signal (what -synthesize
 * hands to dataFill:, TRMTubeModel.m:346) in the batch's arithmetic type; TRMBatchTubeElements() elements,
 * utterance u at TRMBatchTubeOffsets()[u]. */
int TRMBatchSynthesizeDebug(TRMBatch *batch, const TRMParameters *frames, int16_t *pcm_out, void *samples_out,
                            void *tube_out, int device);
int64_t        TRMBatchTubeElements(const TRMBatch *batch);
const int64_t *TRMBatchTubeOffsets(const TRMBatch *batch);
int64_t        TRMBatchKernelLaunches(const TRMBatch *batch);      /* kernels launched by the last synthesize */

/* Device-resident batch: frames uploaded once, each stage (TRM_STAGE_* of trm_cuda.h: 0 waveguide,
 * 1 resampler, 2 PCM) launched on the caller's CUDA stream (cudaStream_t as void*, NULL = default stream)
 * with no host<->device traffic, so the caller can bracket stages with CUDA events on that stream. */
typedef struct TRMResident TRMResident;
TRMResident *TRMBatchMakeResident(TRMBatch *batch, const TRMParameters *frames, int device, int *err);
int  TRMResidentRunStage(TRMResident *r, int stage, void *cuda_stream);
int  TRMResidentRun(TRMResident *r, void *cuda_stream);
int  TRMResidentFetch(TRMResident *r, int16_t *pcm_out, void *samples_out, double *maxima, void *tube_out);
/* one utterance of the resident batch: numberSamples output-rate samples, its PCM, its maximum (any may be NULL) */
int  TRMResidentFetchUtterance(TRMResident *r, int utterance, void *samples_out, int16_t *pcm_out, double *maximum);
void TRMResidentFree(TRMResident *r);

/* Copy-only probe (measurement aid): h2d_bytes from host_in to the device and d2h_bytes from the device to host_out at the
 * same time, `reps` times, no kernels; *ms = average time of one repetition.  With a step's byte counts this is the ceiling
 * the host / PCIe path sets for the end-to-end throughput of that step (bench.py e2e.ceiling, tools/pcie_ceiling.py). */
int TRMCopyProbe(int device, const void *host_in, size_t h2d_bytes, void *host_out, size_t d2h_bytes, int reps, double *ms);

/* Pinned host memory for the batch buffers. */
void *TRMHostAlloc(size_t bytes);
void  TRMHostFree(void *p);

/* Text of the last error of the calling thread's most recent failing call. */
const char *TRMLastErrorMessage(void);

#ifdef __cplusplus
}
#endif
#endif /* TRM_H */
