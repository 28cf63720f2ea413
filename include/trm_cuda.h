/*
 * trm_cuda.h -- thin C-ABI shim between the C host library (libtrm) and the sm_100a kernels
 * (libtrm_cuda).  Plain pointers and sizes only.
 *
 * What each entry point replaces in the reference (all under /root/reference/Frameworks/Tube/):
 *   trm_cuda_stage TRM_STAGE_TUBE  -> the sample-rate loop of -[TRMTubeModel synthesize]
 *                                     TRMTubeModel.m:292-354 (+611-688, 712-853), TRMWavetable.m:117-195,
 *                                     TRMFIRFilter.m:116-146, TRMFilters.m:9-86, TRMUtility.m:26-47,71-85
 *   trm_cuda_stage TRM_STAGE_SRC   -> -[TRMSampleRateConverter processDataFromRingBuffer:]
 *                                     TRMSampleRateConverter.m:155-298 + TRMRingBuffer.m:47-93 (stateless form)
 *   trm_cuda_stage TRM_STAGE_PCM   -> the scaling loops of -saveOutputToFile: / -generateWAVData
 *                                     TRMTubeModel.m:370-383,420-484 / 515-559
 * The derived constants in trm_cuda_utterance are computed by the host library exactly as
 * -initWithInputData: does (TRMTubeModel.m:196-241).
 */
#ifndef TRM_CUDA_H
#define TRM_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TRM_FIR_MAX_TAPS     64
#define TRM_SRC_FILTER_LEN   3328      /* 13 zero crossings x 256 phases (TRMSampleRateConverter.m:11-21) */
#define TRM_TABLE_LENGTH     512       /* TRMWavetable.m:22 */
#define TRM_NOISE_JUMP       16        /* noise powers 377^0..377^16 mod 2^44 */
#define TRM_ALIGN_ELEMS      32        /* every per-utterance buffer offset is a multiple of this */
#define TRM_SRC_ROWS         128       /* tube-rate samples per utterance the converter kernel stages for one work item;
                                          bounds the rate ratios libtrm accepts (an item needs 2*(padSize+1)+3 rows of
                                          halo plus its outputs' span) */

enum { TRM_STAGE_TUBE = 0, TRM_STAGE_SRC = 1, TRM_STAGE_PCM = 2, TRM_STAGE_COUNT = 3 };

/* One utterance as the kernels see it.  Offsets are element offsets into the job's buffers. */
typedef struct trm_cuda_utterance {
    int64_t  frame_offset;      /* first control frame (unit: frames of 16 doubles)                     */
    int64_t  tube_offset;       /* first tube-rate sample                                              */
    int64_t  out_offset;        /* first output-rate sample (also PCM frame offset)                     */
    int64_t  pcm_offset;        /* first int16 element of this utterance in the PCM buffer             */
    int64_t  n_tube;            /* (n_frames-1)*controlPeriod                                          */
    int64_t  n_out;             /* numberSamples                                                       */
    int32_t  n_frames;
    int32_t  controlPeriod;
    int32_t  waveform;          /* 0 pulse, 1 sine                                                     */
    int32_t  usesModulation;
    int32_t  voice;             /* row of the wavetable array                                          */
    int32_t  padSize;
    int32_t  upsample;          /* sampleRateRatio >= 1                                                */
    int32_t  channels;
    int32_t  div1, div2;        /* tableDiv1 / tableDiv2 (TRMWavetable.m:71-72)                        */
    uint32_t tri;               /* timeRegisterIncrement                                               */
    uint32_t phaseIncrement;
    double   sampleRate;        /* (double)_sampleRate                                                 */
    double   sampleRateRatio;
    double   dampingFactor;
    double   breathinessFactor;
    double   crossmixFactor;
    double   basicIncrement;
    double   tnDelta;
    double   mouth[5];          /* a10 b11 a20 a21 b21 (TRMFilters.m:34-45)                            */
    double   nose[5];
    double   nasal_coeff[5];    /* NC2..NC6 (TRMTubeModel.m:692-707)                                   */
    double   nr1sq;             /* noseRadius[1]^2 (TRMTubeModel.m:741)                                */
    double   apScale2;          /* apScale^2 (TRMTubeModel.m:724)                                      */
    double   ta0, tb1;          /* throat low-pass (TRMFilters.m:64-68)                                */
    double   throatGain;
    double   volumeAmp;         /* amplitude(volume)                                                   */
    double   leftGain, rightGain; /* stereo factors applied on top of scale (TRMTubeModel.m:532-533)   */
    /* stream pool (trm_cuda_pool_*), time split: a call continues an utterance.  All zero for whole utterances.   */
    int64_t  out_start;         /* first output-rate sample this call produces (earlier ones exist already)       */
    int64_t  in_start;          /* first tube-rate sample still in memory (multiple of 4; earlier ones are gone)  */
    int32_t  jc0;               /* tube samples already produced inside the first control interval of `frames`    */
    int32_t  reserved;
} trm_cuda_utterance;

/* Constant tables shared by all utterances; computed on the host by libtrm. */
typedef struct trm_cuda_tables {
    int32_t  fir_taps;
    double   fir_coef[TRM_FIR_MAX_TAPS];
    double   src_h[TRM_SRC_FILTER_LEN];
    double   src_dh[TRM_SRC_FILTER_LEN];
    uint64_t noise_pow[TRM_NOISE_JUMP + 1];   /* 377^i mod 2^44                                        */
    uint64_t noise_k0;                         /* state before the first draw: k1 * 377^-1 mod 2^44     */
} trm_cuda_tables;

/* Control-frame generator inputs (EventList.m:883-1061; include/trm.h TRMEvent / TRMFrameGeneration have the same layout) */
#define TRM_EVENT_VALUES 36
typedef struct trm_cuda_event { int64_t time; double value[TRM_EVENT_VALUES]; } trm_cuda_event;
typedef struct trm_cuda_framegen {
    int32_t useMacroIntonation, useMicroIntonation, useSmoothIntonation, useDrift;
    double  driftDeviation, driftCutoff, pitch;
    float   driftSeed;
    int32_t reserved;
} trm_cuda_framegen;

typedef struct trm_cuda_ctx trm_cuda_ctx;
typedef struct trm_cuda_resident trm_cuda_resident;

int         trm_cuda_device_count(void);
const char *trm_cuda_last_error(void);
void       *trm_cuda_host_alloc(size_t bytes);      /* pinned */
void        trm_cuda_host_free(void *p);

/* One context per (process, device): uploads the tables, owns streams and scratch. */
int  trm_cuda_ctx_create(int device, const trm_cuda_tables *tables, trm_cuda_ctx **ctx);
void trm_cuda_ctx_destroy(trm_cuda_ctx *ctx);
/* Glottal wavetables as built at init time (TRMWavetable.m:78-102), n_voices x 512 doubles; utterances pick a
 * row with trm_cuda_utterance.voice.  Replaces the previous set (blocking). */
int  trm_cuda_set_wavetables(trm_cuda_ctx *ctx, const double *tables, int n_voices);

/*
 * Host-buffer path (what TRMTubeModelSynthesize / TRMBatchSynthesize call): copies the frames of the
 * n utterances described by desc[] (offsets relative to the host arrays) to the device in chunks,
 * runs the three stages, copies PCM / samples / max back.  Chunks are double-buffered over CUDA
 * streams so copies overlap kernels.  Blocking.
 *   frame_format 0 = TRMParameters rows of 16 doubles (128 bytes), 1 = rows of 16 floats (64 bytes; what Monet's
 *                generator holds, EventList.m:968-1002), staged as they are and widened by the waveguide kernel when a
 *                parameter lane reads its value -- half the upload, identical results
 *   pcm_host     int16 [..]  or NULL      samples_host  double/float [..] or NULL
 *   max_host     double[n]   or NULL      tube_host     double/float tube-rate signal or NULL
 *   launches     receives the number of kernel launches issued (may be NULL)
 *   enqueued     (may be NULL) `enqueued(arg)` is invoked once, from the calling thread, as soon as the first chunk's
 *                copies and kernels are in the device queues -- libtrm's asynchronous tickets use it to start
 *                concurrent calls in submission order (the queues are shared per device, so the order of arrival
 *                there is the order of execution)
 */
int trm_cuda_synthesize_host(trm_cuda_ctx *ctx, int precision, int frame_format, int n, const trm_cuda_utterance *desc,
                             const void *frames_host, int16_t *pcm_host, void *samples_host,
                             double *max_host, void *tube_host, int64_t *launches,
                             void (*enqueued)(void *), void *arg);

/*
 * Device-resident path (bench `value`, roofline timing): inputs uploaded once, stages launched on the
 * caller's stream (a cudaStream_t passed as void*, NULL = the legacy default stream) without any
 * host<->device copy, so they can be bracketed by CUDA events on that stream.
 */
int  trm_cuda_resident_create(trm_cuda_ctx *ctx, int precision, int n, const trm_cuda_utterance *desc,
                              const double *frames_host, trm_cuda_resident **res);
void trm_cuda_resident_destroy(trm_cuda_resident *res);
int  trm_cuda_resident_stage(trm_cuda_resident *res, int stage, void *stream);   /* one kernel stage      */
int  trm_cuda_resident_run(trm_cuda_resident *res, void *stream);                /* all stages, in order  */
int  trm_cuda_resident_fetch(trm_cuda_resident *res, int16_t *pcm_host, void *samples_host,
                             double *max_host, void *tube_host);                 /* blocking D2H          */
int  trm_cuda_resident_fetch_utterance(trm_cuda_resident *res, int u, void *samples_host, int16_t *pcm_host,
                                       double *max_host);                        /* one utterance, blocking */
/* Sweep (BASELINE configs[4]): n utterances of one voice x n_frames frames, control tracks = the walk2 workload
 * (include/trm_workload.h) generated on the device (utterance k: index first_index + k of stream seed), synthesized in
 * chunks of one full wave; per utterance an 8-byte PCM checksum sum(pcm[i] * (2 i + 1)) mod 2^64 and the maximum come back,
 * plus the PCM of the utterances listed in probe_utt (sorted; rows of probe_stride int16).  kernel_ms: device time of
 * all chunks (CUDA events around generator + 3 stages + checksum). */
int  trm_cuda_sweep(trm_cuda_ctx *ctx, int precision, const trm_cuda_utterance *voice, int32_t n_frames, uint64_t seed,
                    uint64_t first_index, int64_t n, uint64_t *checksums_host, double *max_host, int64_t n_probe,
                    const int64_t *probe_utt, int16_t *probe_pcm, int64_t probe_stride, int64_t *launches, double *kernel_ms);
/* Copy-only probe: h2d_bytes up and d2h_bytes down concurrently, `reps` times; *ms = average per repetition. */
int  trm_cuda_copy_probe(int device, const void *host_in, size_t h2d_bytes, void *host_out, size_t d2h_bytes, int reps,
                         double *ms);

/*
 * Stream pool: `capacity` streaming slots that open, advance and end independently, each with its own voice (its own
 * template: control period, converter signature, glottal table).  A push advances any subset of open slots, each by its
 * own number of frames; all of them are synthesized by one waveguide launch and one resampler launch.  Each slot's pushes,
 * concatenated, are bit-identical to synthesizing its utterance at once.  Used by one thread at a time.
 * Return codes: 0, -4 (bad argument), -7 (call order: slot not open, pool full), -5 (CUDA error; trm_cuda_last_error()).
 * Arguments are checked before any device work: a call that returns -4 or -7 leaves the pool as it was.
 */
typedef struct trm_cuda_pool trm_cuda_pool;
int  trm_cuda_pool_create(trm_cuda_ctx *ctx, int precision, int capacity, int max_frames_per_push, trm_cuda_pool **out);
/* sizes the per-slot buffers for this voice (grows them if needed; SlotCapacity may grow) without opening a slot */
int  trm_cuda_pool_reserve(trm_cuda_pool *p, const trm_cuda_utterance *voice);
/* voice.voice is ignored: `wavetable` (512 doubles) becomes the slot's own glottal table.  *slot receives the slot. */
int  trm_cuda_pool_open(trm_cuda_pool *p, const trm_cuda_utterance *voice, const double *wavetable, int *slot);
/* The same, for a slot whose frames are generated on the device from an event list (libtrm has checked it: n_frames =
 * its frame count, every parameter track has a value after the first event) with settings fg, as
 * trm_cuda_generate_frames generates them.  The list is copied to the slot's device storage (grow-only, kept for later
 * opens of the slot). */
int  trm_cuda_pool_open_events(trm_cuda_pool *p, const trm_cuda_utterance *voice, const double *wavetable,
                               const trm_cuda_event *events, int64_t n_events, int64_t n_frames, const trm_cuda_framegen *fg,
                               int *slot);
int  trm_cuda_pool_close(trm_cuda_pool *p, int slot);
/* New voices for n distinct open slots (frame-fed or event-fed), effective from the next push: voice[i] replaces slot[i]'s
 * descriptor template (voice[i].voice is ignored) and wavetables[i] (512 doubles) its glottal table row; the carried
 * state, counters and pending frames are kept.  voice[i] must have the slot's rate constants (controlPeriod, sampleRate,
 * tri, padSize, channels; else -4: the slot's buffers and counters are laid out for them).  tube_sample[i] /
 * output_sample[i] (either may be NULL) receive the slot's first tube-rate sample and first output sample not yet
 * synthesized: where the new voice starts.  The rows go up in one copy and are scattered on the device; the slots change
 * only once that has finished. */
int  trm_cuda_pool_set_voice(trm_cuda_pool *p, int n, const int32_t *slot, const trm_cuda_utterance *voice,
                             const double *wavetables, int64_t *tube_sample, int64_t *output_sample);
int64_t trm_cuda_pool_slot_capacity(const trm_cuda_pool *p);     /* samples one slot can return from one push */
/* entry i: slot[i] gets n_frames[i] frames (taken back to back from frames_host, rows of 16 doubles; for a slot opened
 * with trm_cuda_pool_open_events, generated from its list instead -- -4 past the list's end); flush[i] != 0 ends
 * the slot and frees it.  out_offset[i+1] - out_offset[i] samples are entry i's.  out_stride == 0: samples_host receives
 * them packed (entry i: [out_offset[i], out_offset[i+1])); out_stride >= SlotCapacity (else -4): in rows, entry i's
 * from samples_host[i * out_stride] on (what follows them in the row is undefined).  A push changes its slots only once
 * its device work has finished: an error returned before its first launch (a refusal, an internal capacity failure, an
 * allocation or the upload failing) leaves every slot as it was; after a CUDA error during its device work the pool's
 * contents are undefined and the pool is to be destroyed. */
int  trm_cuda_pool_push(trm_cuda_pool *p, int n, const int32_t *slot, const int32_t *n_frames, const double *frames_host,
                        const uint8_t *flush, void *samples_host, int64_t out_stride, int64_t *out_offset);
/* the same push, returning PCM16 scaled against peak[i] (finite, > 0), saturated: entry i's int16 elements are
 * pcm_host[pcm_offset[i], pcm_offset[i+1]), channels interleaved; max_host[i] (may be NULL) receives max |y| over the
 * samples entry i produced (0.0 if none).  pcm_kernel's arithmetic (TRMTubeModel.m:515-559) and include/trm.h's contract. */
int  trm_cuda_pool_push_pcm16(trm_cuda_pool *p, int n, const int32_t *slot, const int32_t *n_frames, const double *frames_host,
                              const uint8_t *flush, const double *peak, int16_t *pcm_host, int64_t *pcm_offset, double *max_host);
/* Snapshots (include/trm.h TRMStreamPoolSave): what a slot carries from one push to the next apart from its voice.  The
 * counters are the slot's stream positions: frames received, tube-rate samples synthesized (a multiple of 16), output
 * samples returned, first tube-rate sample still kept, first pending frame; pending frames [pend_first, frames_seen) and
 * fresh = 1 while the waveguide has not run (no carried state exists yet). */
typedef struct trm_cuda_pool_slot_state {
    int64_t frames_seen, s_done, out_done, in_start, pend_first;
    int32_t pend_frames, fresh;
} trm_cuda_pool_slot_state;
/* Host only: 0 if a slot with this voice can hold these counters, -4 if not.  A slot restored with counters that pass
 * reads and writes only inside its own history row, state and pending frames. */
int  trm_cuda_pool_check_state(const trm_cuda_utterance *voice, const trm_cuda_pool_slot_state *st);
/* Bytes of a slot's data part: pend_frames x 16 doubles, the carried state unless fresh (trm::tube_state_bytes), then the
 * kept history s_done - in_start elements of the precision's type. */
int64_t trm_cuda_pool_slot_bytes(int precision, const trm_cuda_pool_slot_state *st);
/* What an event-fed slot (trm_cuda_pool_open_events) carries besides the counters.  Its data part is the frame-fed one
 * (its pending frames come from the slot's device row) followed by the generator state after frames_seen frames --
 * TRM_FRAMEGEN_STATE_BYTES, only when frames_seen > 0: f64 cv[32], cd[32], cv32, cd32, cd33, cd34, cd35; i64 i;
 * u64 now, next; f32 seed, prev, pitchDeviation, pitchOffset, a0, b1 -- then the whole list, n_events trm_cuda_event. */
#define TRM_FRAMEGEN_STATE_BYTES 600
typedef struct trm_cuda_pool_event_state {
    int32_t events;             /* 1: the slot is event-fed; 0: frame-fed, every other field 0 */
    int32_t reserved;
    int64_t n_events;           /* events of its list */
    int64_t ev_frames;          /* frames the list expands to (TRMEventListFrameCount) */
    trm_cuda_framegen fg;
} trm_cuda_pool_event_state;
/* Bytes of the event part that follows trm_cuda_pool_slot_bytes in an event-fed slot's data part (0 for frame-fed). */
int64_t trm_cuda_pool_event_bytes(const trm_cuda_pool_slot_state *st, const trm_cuda_pool_event_state *ev);
/* st[i] receives the counters of n distinct open slots; with dst (may be NULL: counters only, no device work), dst[i]
 * receives slot[i]'s data part (trm_cuda_pool_slot_bytes, plus trm_cuda_pool_event_bytes for an event-fed slot).  The
 * slots are not changed.  ev == NULL: a slot opened with trm_cuda_pool_open_events is refused (-7); otherwise ev[i]
 * describes slot[i].  -7: a slot is not open. */
int  trm_cuda_pool_save(trm_cuda_pool *p, int n, const int32_t *slot, trm_cuda_pool_slot_state *st,
                        trm_cuda_pool_event_state *ev, void *const *dst);
/* Opens n free slots continuing n saved ones: voice[i] (voice.voice ignored) with its glottal table wavetables[i][512],
 * counters st[i], event part ev[i] (ev may be NULL: all frame-fed) and data part src[i].  libtrm has checked an event
 * part's list and generator position against the counters.  Refused before any change: counters that fail
 * trm_cuda_pool_check_state or whose next full push would not fit this pool's rows or pending-frame rows (-4), fewer
 * than n free slots (-7).  Every allocation precedes the first slot opened.  slot_out[i] is entry i's slot. */
int  trm_cuda_pool_restore(trm_cuda_pool *p, int n, const trm_cuda_utterance *voice, const double *wavetables,
                           const trm_cuda_pool_slot_state *st, const trm_cuda_pool_event_state *ev, const void *const *src,
                           int32_t *slot_out);
void trm_cuda_pool_destroy(trm_cuda_pool *p);
/*
 * Control frames on the device (replaces -[EventList generateOutputInTimeRange:...], EventList.m:883-1061): uploads
 * the event lists of the n utterances (utterance u: events[ev_offset[u] .. +ev_count[u]); fg: one entry per
 * utterance, or one for all if shared_fg), runs the generator kernel and leaves the frames -- desc[u].n_frames of
 * them at frame desc[u].frame_offset -- in a device buffer owned by the context.  *frames_dev receives that buffer
 * (valid until the next call on this context; usable as the `frames_host` argument of trm_cuda_synthesize_host,
 * which copies with cudaMemcpyDefault).  frames_host / seed_host, if not NULL, receive copies.  Blocking.
 */
int  trm_cuda_generate_frames(trm_cuda_ctx *ctx, int n, const trm_cuda_utterance *desc, const trm_cuda_event *events,
                              const int64_t *ev_offset, const int32_t *ev_count, const trm_cuda_framegen *fg, int shared_fg,
                              const double **frames_dev, double *frames_host, float *seed_host);
/* Measures the device's FMA peak (TFLOP/s, 2 flops per FMA) with a register-resident FMA chain:
 * precision 0 = FP64, 1 = FP32.  The waveguide kernel's roofline denominator. */
int  trm_cuda_fp_peak(int device, int precision, int reps, double *tflops);

#ifdef __cplusplus
}
#endif
#endif /* TRM_CUDA_H */
