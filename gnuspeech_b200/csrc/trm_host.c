/*
 * trm_host.c -- C host library behind include/trm.h (libtrm.so).
 *
 * Mirrors the host-side half of the reference's Tube.framework:
 *   derived constants      -[TRMTubeModel initWithInputData:]        TRMTubeModel.m:186-260
 *   wavetable set-up       -[TRMWavetable initWithWaveform:...]      TRMWavetable.m:56-106
 *   FIR design             TRMFIRFilter.m:37-98, 161-310
 *   SRC set-up / filter    TRMSampleRateConverter.m:69-131, TRMUtility.m:50-66
 *   data list + parser     TRMDataList.m:22-247, TRMSynthesizer.m:98-106
 *   output containers      TRMTubeModel.m:365-593, NSData-STExtensions.m:7-38
 * Everything per-sample runs on the GPU through the libtrm_cuda shim; there is no CPU synthesis here.
 */
#include "trm.h"
#include "trm_cuda.h"

#include <math.h>
#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include <strings.h>

/* ------------------------------------------------------------------------------------------------
 * errors
 * ---------------------------------------------------------------------------------------------- */
static __thread char g_errmsg[512];

static int set_err(int code, const char *fmt, const char *detail)
{
    snprintf(g_errmsg, sizeof g_errmsg, fmt, detail ? detail : "");
    return code;
}
const char *TRMLastErrorMessage(void) { return g_errmsg; }
static int cuda_err(void) { return set_err(TRM_ERR_CUDA, "CUDA: %s", trm_cuda_last_error()); }

/* ------------------------------------------------------------------------------------------------
 * scalar conversions (TRMUtility.m:20-47)
 * ---------------------------------------------------------------------------------------------- */
static double sound_speed(double celsius) { return 331.4 + (0.6 * celsius); }

static double db_to_amplitude(double db)
{
    db -= 60.0;                       /* 0..60 dB -> -60..0 dB */
    if (db <= -60.0) return 0.0;
    if (db >= 0.0) return 1.0;
    return pow(10.0, db / 20.0);
}

/* ------------------------------------------------------------------------------------------------
 * shared tables: FIR coefficients, SRC filter, noise jump multipliers
 * ---------------------------------------------------------------------------------------------- */
#define FIR_LIMIT 200

/* best rational approximation p/q of x with q in [*order, 2*order] (TRMFIRFilter.m:265-310) */
static void best_rational(double x, int *order, int *num, int *den)
{
    if (*order <= 0) { *num = *den = 0; *order = -1; return; }
    const double frac = fabs(x - (int)x);
    int q_max = 2 * (*order);
    if (q_max > FIR_LIMIT) q_max = FIR_LIMIT;
    int best_p = 0;
    double best_err = 1.0;
    for (int q = *order; q <= q_max; q++) {
        const double scaled = q * frac;
        const int p = (int)(scaled + 0.5);
        const double err = fabs((scaled - (double)p) / (double)q);
        if (err < best_err) { best_err = err; best_p = p; *den = q; }
    }
    *num = (int)fabs(x) * (*den) + best_p;
    if (x < 0) *num = -*num;
    *order = *den - 1;
    if (*num == *den) { *den = q_max; *order = *num = *den - 1; }
}

/* maximally flat low-pass: one-sided coefficients w[1..*np] (TRMFIRFilter.m:161-233) */
static int flat_lowpass(double beta, double gamma, int *np, double *w)
{
    double mag[FIR_LIMIT + 1], cs[FIR_LIMIT + 1];
    *np = 0;
    if (beta <= 0.0 || beta >= 0.5) return 1;
    const double lim = ((2.0 * beta) < (1.0 - 2.0 * beta)) ? (2.0 * beta) : (1.0 - 2.0 * beta);
    if (gamma <= 0.0 || gamma >= lim) return 2;
    int nt = (int)(1.0 / (4.0 * gamma * gamma));
    if (nt > 160) return 3;
    const double ac = (1.0 + cos((2.0 * M_PI) * beta)) / 2.0;
    int k;
    best_rational(ac, &nt, &k, np);
    const int n = (2 * (*np)) - 1;
    if (k == 0) k = 1;
    cs[1] = mag[1] = 1.0;
    const int span = nt - k;
    for (int i = 2; i <= *np; i++) {
        double acc = 1.0;
        cs[i] = cos((2.0 * M_PI) * ((double)(i - 1) / (double)n));
        const double x = (1.0 - cs[i]) / 2.0;
        double y = x;
        if (k == nt) continue;
        for (int j = 1; j <= span; j++) {
            double z = y;
            if (k != 1)
                for (int jj = 1; jj <= (k - 1); jj++) z *= 1.0 + ((double)j / (double)jj);
            y *= x;
            acc += z;
        }
        mag[i] = acc * pow((1.0 - x), k);
    }
    for (int i = 1; i <= *np; i++) {       /* n-point inverse DFT of the sampled magnitude */
        w[i] = mag[1] / 2.0;
        for (int j = 2; j <= *np; j++) {
            int m = ((i - 1) * (j - 1)) % n;
            if (m > nt) m = n - m;
            w[i] += cs[m + 1] * mag[j];
        }
        w[i] *= 2.0 / (double)n;
    }
    return 0;
}

/* tap layout of -[TRMFIRFilter initWithBeta:gamma:cutoff:] (TRMFIRFilter.m:37-98; trim :236-244) */
static int design_fir(double *taps, int *n_taps)
{
    double w[FIR_LIMIT + 1];
    int nc;
    memset(w, 0, sizeof w);
    if (flat_lowpass(.2, .1, &nc, w) != 0) return TRM_ERR_FIR;     /* TRMFIRFilter.h:7-9 */
    for (int i = nc; i > 0; i--)
        if (fabs(w[i]) >= fabs(.00000001)) { nc = i; break; }
    *n_taps = (nc * 2) - 1;
    if (*n_taps > TRM_FIR_MAX_TAPS) return TRM_ERR_FIR;
    int step = -1, at = nc;
    for (int i = 0; i < *n_taps; i++) {
        taps[i] = w[at];
        at += step;
        if (at <= 0) { at = 2; step = 1; }
    }
    return TRM_OK;
}

/* modified Bessel I0 (TRMUtility.m:50-66) */
static double bessel_i0(double x)
{
    double sum = 1, term = 1, n = 1;
    const double half = x / 2.0;
    do {
        double t = half / n;
        n += 1;
        t *= t;
        term *= t;
        sum += term;
    } while (term >= (1E-21 * sum));
    return sum;
}

/* Kaiser-windowed sinc and its first difference (TRMSampleRateConverter.m:110-131) */
static void design_src_filter(double *h, double *dh)
{
    const double cutoff = 11.0 / 13.0, kaiser_beta = 5.658;
    h[0] = cutoff;
    const double step = M_PI / 256.0;
    for (int i = 1; i < TRM_SRC_FILTER_LEN; i++) {
        const double y = (double)i * step;
        h[i] = sin(y * cutoff) / y;
    }
    const double inv_i0 = 1.0 / bessel_i0(kaiser_beta);
    for (int i = 0; i < TRM_SRC_FILTER_LEN; i++) {
        const double t = (double)i / TRM_SRC_FILTER_LEN;
        h[i] *= bessel_i0(kaiser_beta * sqrt(1.0 - (t * t))) * inv_i0;
    }
    for (int i = 0; i < TRM_SRC_FILTER_LEN - 1; i++) dh[i] = h[i + 1] - h[i];
    dh[TRM_SRC_FILTER_LEN - 1] = 0.0 - h[TRM_SRC_FILTER_LEN - 1];
}

static trm_cuda_tables g_tables;
static int g_tables_rc = TRM_OK;
static pthread_once_t g_tables_once = PTHREAD_ONCE_INIT;

static void build_tables(void)
{
    memset(&g_tables, 0, sizeof g_tables);
    int taps = 0;
    g_tables_rc = design_fir(g_tables.fir_coef, &taps);
    g_tables.fir_taps = taps;
    design_src_filter(g_tables.src_h, g_tables.src_dh);
    /* The noise generator seed <- frac(seed*377), seed0 = 0.7892347 (TRMUtility.m:71-85) is, from the first
     * draw on, the multiplicative congruential generator k <- 377 k mod 2^44 on k = seed * 2^44: the first
     * product lies in [256,512) where doubles are spaced 2^-44, and 377 k < 2^53 keeps every later product exact. */
    const uint64_t mask = (1ull << 44) - 1ull;
    const double s0 = 0.7892347;
    const double prod = s0 * 377.0;
    const double s1 = prod - (int)prod;
    const uint64_t k1 = (uint64_t)ldexp(s1, 44);
    uint64_t inv = 377;                                  /* Newton iteration for 377^-1 mod 2^64 */
    for (int i = 0; i < 6; i++) inv *= 2ull - 377ull * inv;
    g_tables.noise_k0 = (k1 * inv) & mask;
    uint64_t p = 1;
    for (int i = 0; i <= TRM_NOISE_JUMP; i++) { g_tables.noise_pow[i] = p; p = (p * 377ull) & mask; }
}

static const trm_cuda_tables *tables(int *rc)
{
    pthread_once(&g_tables_once, build_tables);
    if (rc) *rc = g_tables_rc;
    return &g_tables;
}

/* ------------------------------------------------------------------------------------------------
 * defaults and derived values
 * ---------------------------------------------------------------------------------------------- */
void TRMInputParametersSetDefaults(TRMInputParameters *ip, float outputRate)
{
    /* MMSynthesisParameters.m:163-187; control rate TRMSynthesizer.m:41; mono */
    memset(ip, 0, sizeof *ip);
    ip->outputFileFormat = TRMSoundFileFormat_AU;
    ip->outputRate = outputRate;
    ip->controlRate = 250;
    ip->volume = 60;
    ip->channels = 1;
    ip->balance = 0;
    ip->waveform = TRMWaveFormType_Pulse;
    ip->tp = 40; ip->tnMin = 16; ip->tnMax = 32;
    ip->breathiness = 1;
    ip->length = 17.5; ip->temperature = 25; ip->lossFactor = 0.5;
    ip->apScale = 3.05; ip->mouthCoef = 5000; ip->noseCoef = 5000;
    ip->noseRadius[0] = 0; ip->noseRadius[1] = 1.35; ip->noseRadius[2] = 1.96;
    ip->noseRadius[3] = 1.91; ip->noseRadius[4] = 1.3; ip->noseRadius[5] = 0.73;
    ip->throatCutoff = 1500; ip->throatVol = 6;
    ip->usesModulation = 1;
    ip->mixOffset = 54;
}

typedef struct {
    int32_t controlPeriod, sampleRate, padSize, upsample;
    double actualTubeLength, ratio;
    uint32_t tri, phaseIncrement;
} rates_t;

static int derive_rates(const TRMInputParameters *ip, rates_t *r)
{
    if (!(ip->length > 0.0)) return set_err(TRM_ERR_TUBE_LENGTH, "Illegal tube length%s", "");
    if (!(ip->controlRate > 0.0f) || !(ip->outputRate > 0.0f))
        return set_err(TRM_ERR_PARAM, "controlRate and outputRate must be positive%s", "");
    /* TRMTubeModel.m:197-203 */
    const double c = sound_speed(ip->temperature);
    r->controlPeriod = rint((c * 10 * 100.0) / (ip->length * ip->controlRate));
    r->sampleRate = ip->controlRate * r->controlPeriod;
    /* the waveguide kernel stages 2 frames per bulk copy and consumes 16 samples per block: at most one
     * staging-buffer switch per block needs controlPeriod >= 8 (the reference's range gives >= 17) */
    if (r->controlPeriod < 8 || r->sampleRate < 1) return set_err(TRM_ERR_PARAM, "control period < 8 samples%s", "");
    r->actualTubeLength = (c * 10 * 100.0) / r->sampleRate;
    /* TRMSampleRateConverter.m:80-96 */
    r->ratio = (double)ip->outputRate / (double)r->sampleRate;
    r->tri = (int)rint(pow(2.0, 16) / r->ratio);
    if (r->tri == 0) return set_err(TRM_ERR_PARAM, "sample-rate ratio too large%s", "");
    const double rounded = pow(2.0, 16) / (double)r->tri;
    r->upsample = r->ratio >= 1.0;
    r->phaseIncrement = r->upsample ? 0u : (uint32_t)rint(r->ratio * 65536.0);
    r->padSize = r->upsample ? 13 : (int32_t)((float)13 / rounded) + 1;
    return TRM_OK;
}

static int64_t src_output_count(const rates_t *r, int64_t n_in)
{
    /* the converter emits one sample per time-register step until the read position reaches
     * n_in + 2*pad (TRMSampleRateConverter.m:171,221-232; TRMRingBuffer.m:85-93) */
    const int64_t total = n_in + 2 * (int64_t)r->padSize;
    return (total * 65536 + (int64_t)r->tri - 1) / (int64_t)r->tri;
}

/* The reference's streaming converter mis-handles its final drain when down-sampling (TRMSampleRateConverter.m:160-168,
 * TRMRingBuffer.m:55-59,85-93; SURVEY.md 0.11 / A.16b).  Its read pointer advances 1..3 input positions per output, so a
 * pass over the ring may stop o = 1..2 positions PAST the end pointer.  The next pass repairs "end < read" by adding the
 * ring size -- correct when the ring wrapped, wrong when the pass simply has fewer than o new inputs: it then runs over a
 * whole ring of stale data and appends ~1024 x ratio spurious samples.  Passes triggered by the fill counter always bring
 * fillSize new inputs; only the final pass of -flush can be short.  With total = N_in + 2 pad inputs, K = total / fillSize
 * counter-triggered passes and r = total % fillSize inputs left for the final one, the last counter-triggered pass ends
 * after n* = ceil(K fillSize 2^16 / tri) outputs at read position P = (n* tri) >> 16: the bug fires iff K >= 1 and
 * r < P - K fillSize.  (Checked against the oracle's restatement of the streaming converter over 6 voices x 498 lengths,
 * tests/test_host.py.)  This implementation computes the converter's defined output (the stateless form) and reports
 * the condition instead. */
static int flush_bug(const rates_t *r, int64_t n_in)
{
    if (r->upsample) return 0;
    const int64_t fill = 1024 - 2 * (int64_t)r->padSize, total = n_in + 2 * (int64_t)r->padSize;
    if (fill <= 0 || total < fill) return 0;
    const int64_t K = total / fill, rest = total - K * fill, tri = (int64_t)r->tri;
    const int64_t n_star = (K * fill * 65536 + tri - 1) / tri;
    const int64_t over = ((n_star * tri) >> 16) - K * fill;
    return rest < over;
}

int TRMReferenceFlushBug(const TRMInputParameters *ip, size_t n_frames)
{
    rates_t r;
    if (!ip || n_frames == 0 || derive_rates(ip, &r) != TRM_OK) return 0;
    return flush_bug(&r, (int64_t)(n_frames - 1) * r.controlPeriod);
}

int TRMDeriveValues(const TRMInputParameters *ip, size_t n_frames, TRMDerivedValues *out)
{
    rates_t r;
    int rc = derive_rates(ip, &r);
    if (rc) return rc;
    memset(out, 0, sizeof *out);
    out->controlPeriod = r.controlPeriod;
    out->sampleRate = r.sampleRate;
    out->actualTubeLength = r.actualTubeLength;
    out->padSize = r.padSize;
    out->timeRegisterIncrement = r.tri;
    out->tubeSamples = n_frames ? (int64_t)(n_frames - 1) * r.controlPeriod : 0;
    out->numberSamples = n_frames ? (int32_t)src_output_count(&r, out->tubeSamples) : 0;   /* TRMTubeModel.m:274-277 */
    return TRM_OK;
}

/* ------------------------------------------------------------------------------------------------
 * voices: the init-time glottal table (TRMWavetable.m:56-106), deduplicated per batch
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
    int32_t waveform, div1, div2;
    double tp, tnMin, tnMax, tnDelta;
} voice_key;

typedef struct {
    voice_key *keys;
    double *tables;          /* n x 512 */
    int n, cap;
} voice_set;

static void voice_set_free(voice_set *vs) { free(vs->keys); free(vs->tables); memset(vs, 0, sizeof *vs); }

static int voice_lookup(voice_set *vs, const TRMInputParameters *ip, voice_key *out_key)
{
    voice_key k;
    memset(&k, 0, sizeof k);
    k.waveform = ip->waveform; k.tp = ip->tp; k.tnMin = ip->tnMin; k.tnMax = ip->tnMax;
    for (int i = 0; i < vs->n; i++)
        if (vs->keys[i].waveform == k.waveform && vs->keys[i].tp == k.tp && vs->keys[i].tnMin == k.tnMin &&
            vs->keys[i].tnMax == k.tnMax) { *out_key = vs->keys[i]; return i; }
    /* TRMWavetable.m:71-74 */
    k.div1 = rint(TRM_TABLE_LENGTH * (ip->tp / 100.0));
    k.div2 = rint(TRM_TABLE_LENGTH * ((ip->tp + ip->tnMax) / 100.0));
    const double tnLength = k.div2 - k.div1;
    k.tnDelta = rint(TRM_TABLE_LENGTH * ((ip->tnMax - ip->tnMin) / 100.0));
    if (ip->waveform != TRMWaveFormType_Pulse && ip->waveform != TRMWaveFormType_Sine)
        return set_err(TRM_ERR_PARAM, "unknown glottal waveform type%s", "");
    if (ip->waveform == TRMWaveFormType_Pulse &&
        !(k.div1 > 0 && k.div1 < k.div2 && k.div2 <= TRM_TABLE_LENGTH && k.tnDelta >= 0.0 && k.tnDelta < tnLength))
        return set_err(TRM_ERR_PARAM, "glottal pulse shape (tp/tnMin/tnMax) outside 0 < tp, tnMin > 0, tp+tnMax <= 100%s", "");
    if (vs->n == vs->cap) {
        int cap = vs->cap ? vs->cap * 2 : 4;
        voice_key *nk = realloc(vs->keys, (size_t)cap * sizeof *nk);
        if (!nk) return set_err(TRM_ERR_NOMEM, "out of memory%s", "");
        vs->keys = nk;
        double *nt = realloc(vs->tables, (size_t)cap * TRM_TABLE_LENGTH * sizeof *nt);
        if (!nt) return set_err(TRM_ERR_NOMEM, "out of memory%s", "");
        vs->tables = nt;
        vs->cap = cap;
    }
    double *t = vs->tables + (size_t)vs->n * TRM_TABLE_LENGTH;
    if (ip->waveform == TRMWaveFormType_Pulse) {
        /* TRMWavetable.m:78-96 */
        for (int i = 0; i < k.div1; i++) {
            const double x = (double)i / (double)k.div1;
            const double x2 = x * x, x3 = x2 * x;
            t[i] = (3.0 * x2) - (2.0 * x3);
        }
        for (int i = k.div1, j = 0; i < k.div2; i++, j++) {
            const double x = (double)j / tnLength;
            t[i] = 1.0 - (x * x);
        }
        for (int i = k.div2; i < TRM_TABLE_LENGTH; i++) t[i] = 0.0;
    } else {
        /* TRMWavetable.m:99-101 */
        for (int i = 0; i < TRM_TABLE_LENGTH; i++) t[i] = sin(((double)i / (double)TRM_TABLE_LENGTH) * 2.0 * M_PI);
    }
    vs->keys[vs->n] = k;
    *out_key = k;
    return vs->n++;
}

/* ------------------------------------------------------------------------------------------------
 * per-utterance descriptor: -initWithInputData: (TRMTubeModel.m:196-241)
 * ---------------------------------------------------------------------------------------------- */

static void radrefl_coefficients(double coeff, double *f)
{
    /* TRMFilters.m:34-45: a10 b11 a20 a21 b21 */
    f[1] = -coeff;
    f[0] = 1.0 - fabs(f[1]);
    f[2] = coeff;
    f[3] = f[4] = -(f[2]);
}

static int describe(const TRMInputParameters *ip, int32_t n_frames, voice_set *vs, trm_cuda_utterance *d, rates_t *rates_out)
{
    rates_t r;
    int rc = derive_rates(ip, &r);
    if (rc) return rc;
    if (n_frames < 0) return set_err(TRM_ERR_PARAM, "negative frame count%s", "");
    if (ip->channels != 1 && ip->channels != 2) return set_err(TRM_ERR_PARAM, "channels must be 1 or 2%s", "");
    /* the resampler stages a bounded input window per output tile */
    /* (an item's outputs span (rows - halo) * ratio of them; the kernels need at least 8 when down-sampling and one
     * 8-output run per warp, up to 12 warps, when up-sampling) */
    if ((double)(TRM_SRC_ROWS - 3 - 2 * (r.padSize + 1)) * r.ratio < (r.upsample ? 96.0 : 8.0))
        return set_err(TRM_ERR_PARAM, "outputRate / tube sample rate below the supported ratio%s", "");
    voice_key vk;
    const int voice = voice_lookup(vs, ip, &vk);
    if (voice < 0) return voice;

    memset(d, 0, sizeof *d);
    d->n_frames = n_frames;
    d->controlPeriod = r.controlPeriod;
    d->n_tube = n_frames > 0 ? (int64_t)(n_frames - 1) * r.controlPeriod : 0;
    d->n_out = n_frames > 0 ? src_output_count(&r, d->n_tube) : 0;
    d->waveform = ip->waveform;
    d->usesModulation = ip->usesModulation != 0;
    d->voice = voice;
    d->padSize = r.padSize;
    d->upsample = r.upsample;
    d->channels = ip->channels;
    d->div1 = vk.div1;
    d->div2 = vk.div2;
    d->tri = r.tri;
    d->phaseIncrement = r.phaseIncrement;
    d->sampleRate = (double)r.sampleRate;
    d->sampleRateRatio = r.ratio;
    const double nyquist = (double)r.sampleRate / 2.0;
    d->dampingFactor = (1.0 - (ip->lossFactor / 100.0));                       /* m:216 */
    d->breathinessFactor = ip->breathiness / 100.0;                            /* m:210 */
    d->crossmixFactor = 1.0 / db_to_amplitude(ip->mixOffset);                  /* m:213 */
    d->basicIncrement = (double)TRM_TABLE_LENGTH / (double)r.sampleRate;       /* TRMWavetable.m:75 */
    d->tnDelta = vk.tnDelta;
    radrefl_coefficients((nyquist - ip->mouthCoef) / nyquist, d->mouth);       /* m:222 */
    radrefl_coefficients((nyquist - ip->noseCoef) / nyquist, d->nose);         /* m:225 */
    for (int i = 1; i < 5; i++) {                                              /* m:695-699: NC2..NC5 */
        const double a2 = ip->noseRadius[i] * ip->noseRadius[i];
        const double b2 = ip->noseRadius[i + 1] * ip->noseRadius[i + 1];
        d->nasal_coeff[i - 1] = (a2 - b2) / (a2 + b2);
    }
    {
        const double a2 = ip->noseRadius[5] * ip->noseRadius[5];               /* m:703-705: NC6 */
        const double b2 = ip->apScale * ip->apScale;
        d->nasal_coeff[4] = (a2 - b2) / (a2 + b2);
        d->apScale2 = b2;
    }
    d->nr1sq = ip->noseRadius[1] * ip->noseRadius[1];                          /* m:741 */
    d->ta0 = (ip->throatCutoff * 2.0) / r.sampleRate;                          /* TRMFilters.m:66-67 */
    d->tb1 = 1.0 - d->ta0;
    d->throatGain = db_to_amplitude(ip->throatVol);                            /* m:239 */
    d->volumeAmp = db_to_amplitude(ip->volume);                                /* m:515 */
    d->leftGain = -((ip->balance / 2.0) - 0.5);                                /* m:532 */
    d->rightGain = ((ip->balance / 2.0) + 0.5);                                /* m:533 */
    if (rates_out) *rates_out = r;
    return TRM_OK;
}

/* ------------------------------------------------------------------------------------------------
 * CUDA contexts: one per device, created on first use
 * ---------------------------------------------------------------------------------------------- */
#define MAX_DEVICES 64
/* Three context lanes per device (one call uploading, one computing, one downloading): each lane owns its streams, device arenas and pinned staging, so several calls can be
 * in flight on one GPU (TRMBatchSynthesizeAsync): the PCM of call k leaves for the host while call k+1 computes. */
#define CTX_LANES 3
static trm_cuda_ctx *g_ctx[MAX_DEVICES][CTX_LANES];
static int g_lane_busy[MAX_DEVICES][CTX_LANES];
static pthread_mutex_t g_lane_mu = PTHREAD_MUTEX_INITIALIZER;     /* covers g_lane_busy and context creation */
static pthread_cond_t g_lane_cv = PTHREAD_COND_INITIALIZER;

/* A context lane serves one call at a time.  A caller takes the first free lane of the device and, when all are busy,
 * waits on the condition variable until ANY of them is released (no lane is special; nothing is ever held across calls:
 * streams and device-resident batches own copies of what they need from the context). */
static int acquire_ctx(int device, trm_cuda_ctx **out, int *lane_out)
{
    int rc;
    const trm_cuda_tables *t = tables(&rc);
    if (rc) return set_err(rc, "FIR design failed%s", "");
    if (device < 0 || device >= MAX_DEVICES) return set_err(TRM_ERR_CUDA, "bad device ordinal%s", "");
    pthread_mutex_lock(&g_lane_mu);
    int lane = -1;
    for (;;) {
        for (int l = 0; l < CTX_LANES && lane < 0; l++)
            if (!g_lane_busy[device][l]) lane = l;
        if (lane >= 0) break;
        pthread_cond_wait(&g_lane_cv, &g_lane_mu);
    }
    g_lane_busy[device][lane] = 1;
    int failed = 0;
    if (!g_ctx[device][lane]) failed = trm_cuda_ctx_create(device, t, &g_ctx[device][lane]) != 0;
    if (failed) {
        g_lane_busy[device][lane] = 0;
        pthread_cond_broadcast(&g_lane_cv);
    }
    pthread_mutex_unlock(&g_lane_mu);
    if (failed) return cuda_err();
    *out = g_ctx[device][lane];
    *lane_out = lane;
    return TRM_OK;
}
static void release_ctx(int device, int lane)
{
    pthread_mutex_lock(&g_lane_mu);
    g_lane_busy[device][lane] = 0;
    pthread_cond_broadcast(&g_lane_cv);
    pthread_mutex_unlock(&g_lane_mu);
}

void *TRMHostAlloc(size_t bytes)
{
    void *p = trm_cuda_host_alloc(bytes);
    if (!p) cuda_err();
    return p;
}
void TRMHostFree(void *p) { trm_cuda_host_free(p); }
void TRMFree(void *p) { free(p); }

/* ------------------------------------------------------------------------------------------------
 * TRMDataList
 * ---------------------------------------------------------------------------------------------- */
struct TRMDataList {
    TRMInputParameters ip;
    TRMParameters *values;
    size_t count, cap;
};

TRMDataList *TRMDataListCreate(void) { return calloc(1, sizeof(TRMDataList)); }

void TRMDataListFree(TRMDataList *l)
{
    if (!l) return;
    free(l->values);
    free(l);
}

TRMInputParameters *TRMDataListInputParameters(TRMDataList *l) { return &l->ip; }
size_t TRMDataListCount(const TRMDataList *l) { return l->count; }
const TRMParameters *TRMDataListValues(const TRMDataList *l) { return l->values; }
void TRMDataListRemoveAllParameters(TRMDataList *l) { l->count = 0; }

int TRMDataListAddParametersArray(TRMDataList *l, const TRMParameters *f, size_t n)
{
    if (l->count + n > l->cap) {
        size_t cap = l->cap ? l->cap : 256;
        while (cap < l->count + n) cap *= 2;
        TRMParameters *nv = realloc(l->values, cap * sizeof *nv);
        if (!nv) return set_err(TRM_ERR_NOMEM, "out of memory%s", "");
        l->values = nv;
        l->cap = cap;
    }
    memcpy(l->values + l->count, f, n * sizeof *f);
    l->count += n;
    return TRM_OK;
}
int TRMDataListAddParameters(TRMDataList *l, const TRMParameters *f) { return TRMDataListAddParametersArray(l, f, 1); }

/* positional text format: 26 header lines (value first, comment ignored), then 16 numbers per line
 * (TRMDataList.m:43-247).  Lines are read in 128-byte pieces like the reference's fgets(line, 128, fp). */
TRMDataList *TRMDataListCreateWithContentsOfFile(const char *path, int *err)
{
    int dummy;
    if (!err) err = &dummy;
    FILE *fp = fopen(path, "r");
    if (!fp) { *err = set_err(TRM_ERR_IO, "Can't open input file \"%s\".", path); return NULL; }
    TRMDataList *l = TRMDataListCreate();
    if (!l) { fclose(fp); *err = set_err(TRM_ERR_NOMEM, "out of memory%s", ""); return NULL; }
    char line[128];
    TRMInputParameters *ip = &l->ip;
    double hv[26];
    static const char *what[26] = {
        "output file format", "output sample rate", "input control rate", "master volume",
        "number of sound output channels", "stereo balance", "glottal source waveform type",
        "glottal pulse rise time (tp)", "glottal pulse fall time minimum (tnMin)", "glottal pulse fall time maximum (tnMax)",
        "glottal source breathiness", "nominal tube length", "tube temperature", "junction loss factor",
        "aperture scaling radius", "mouth aperture coefficient", "nose aperture coefficient",
        "nose radius 1", "nose radius 2", "nose radius 3", "nose radius 4", "nose radius 5",
        "throat lowpass filter cutoff", "throat volume", "pulse modulation of noise flag", "noise crossmix offset"};
    static const int is_int[26] = {1, 0, 0, 0, 1, 0, 1, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 1, 0};
    for (int i = 0; i < 26; i++) {
        if (!fgets(line, sizeof line, fp)) {
            *err = set_err(TRM_ERR_IO, "Can't read %s.", what[i]);
            fclose(fp);
            TRMDataListFree(l);
            return NULL;
        }
        hv[i] = is_int[i] ? (double)strtol(line, NULL, 10) : strtod(line, NULL);
    }
    ip->outputFileFormat = (int32_t)hv[0]; ip->outputRate = hv[1]; ip->controlRate = hv[2]; ip->volume = hv[3];
    ip->channels = (int32_t)hv[4]; ip->balance = hv[5]; ip->waveform = (int32_t)hv[6]; ip->tp = hv[7];
    ip->tnMin = hv[8]; ip->tnMax = hv[9]; ip->breathiness = hv[10]; ip->length = hv[11]; ip->temperature = hv[12];
    ip->lossFactor = hv[13]; ip->apScale = hv[14]; ip->mouthCoef = hv[15]; ip->noseCoef = hv[16];
    for (int i = 1; i < TRM_TOTAL_NASAL_SECTIONS; i++) ip->noseRadius[i] = hv[16 + i];
    ip->throatCutoff = hv[22]; ip->throatVol = hv[23]; ip->usesModulation = (hv[24] != 0); ip->mixOffset = hv[25];

    while (fgets(line, sizeof line, fp)) {
        TRMParameters f;
        char *at = line;
        double *v = (double *)&f;
        for (int q = 0; q < 16; q++) v[q] = strtod(at, &at);
        if ((*err = TRMDataListAddParameters(l, &f)) != TRM_OK) { fclose(fp); TRMDataListFree(l); return NULL; }
    }
    if (l->count > 0) {               /* the parser doubles the last table (TRMDataList.m:239-241) */
        TRMParameters last = l->values[l->count - 1];
        if ((*err = TRMDataListAddParameters(l, &last)) != TRM_OK) { fclose(fp); TRMDataListFree(l); return NULL; }
    }
    fclose(fp);
    *err = TRM_OK;
    return l;
}

int TRMDataListWriteToFile(const TRMDataList *l, const char *path)
{
    FILE *fp = fopen(path, "w");
    if (!fp) return set_err(TRM_ERR_IO, "Can't open output file \"%s\".", path);
    const TRMInputParameters *ip = &l->ip;
    fprintf(fp, "%d\t\t; output file format (0 = AU, 1 = AIFF, 2 = WAVE)\n", ip->outputFileFormat);
    fprintf(fp, "%f\t; output sample rate (22050.0, 44100.0)\n", ip->outputRate);
    fprintf(fp, "%d\t\t; input control rate (1 - 1000 Hz)\n", (int)ip->controlRate);
    fprintf(fp, "%f\t; master volume (0 - 60 dB)\n", ip->volume);
    fprintf(fp, "%d\t\t; number of sound output channels (1 or 2)\n", ip->channels);
    fprintf(fp, "%f\t; stereo balance (-1 to +1)\n", ip->balance);
    fprintf(fp, "%d\t\t; glottal source waveform type (0 = pulse, 1 = sine)\n", ip->waveform);
    fprintf(fp, "%f\t; glottal pulse rise time (5 - 50 %% of GP period)\n", ip->tp);
    fprintf(fp, "%f\t; glottal pulse fall time minimum (5 - 50 %% of GP period)\n", ip->tnMin);
    fprintf(fp, "%f\t; glottal pulse fall time maximum (5 - 50 %% of GP period)\n", ip->tnMax);
    fprintf(fp, "%f\t; glottal source breathiness (0 - 10 %% of GS amplitude)\n", ip->breathiness);
    fprintf(fp, "%f\t; nominal tube length (10 - 20 cm)\n", ip->length);
    fprintf(fp, "%f\t; tube temperature (25 - 40 degrees celsius)\n", ip->temperature);
    fprintf(fp, "%f\t; junction loss factor (0 - 5 %% of unity gain)\n", ip->lossFactor);
    fprintf(fp, "%f\t; aperture scaling radius (3.05 - 12 cm)\n", ip->apScale);
    fprintf(fp, "%f\t; mouth aperture coefficient (0 - 0.99)\n", ip->mouthCoef);
    fprintf(fp, "%f\t; nose aperture coefficient (0 - 0.99)\n", ip->noseCoef);
    for (int i = 1; i < TRM_TOTAL_NASAL_SECTIONS; i++)
        fprintf(fp, "%f\t; radius of nose section %d (0 - 3 cm)\n", ip->noseRadius[i], i);
    fprintf(fp, "%f\t; throat lowpass frequency cutoff (50 - nyquist Hz)\n", ip->throatCutoff);
    fprintf(fp, "%f\t; throat volume (0 - 48 dB)\n", ip->throatVol);
    fprintf(fp, "%d\t\t; pulse modulation of noise (0 = off, 1 = on)\n", ip->usesModulation ? 1 : 0);
    fprintf(fp, "%f\t; noise crossmix offset (30 - 60 db)\n", ip->mixOffset);
    for (size_t i = 0; i < l->count; i++) {
        const double *v = (const double *)&l->values[i];
        for (int q = 0; q < 16; q++) fprintf(fp, q ? " %.3f" : "%.3f", v[q]);
        fputc('\n', fp);
    }
    if (fclose(fp) != 0) return set_err(TRM_ERR_IO, "write error on \"%s\"", path);
    return TRM_OK;
}

/* ------------------------------------------------------------------------------------------------
 * Voice parameters (MMSynthesisParameters.m:160-310, Other/voices.config:15-48, TRMSynthesizer.m:38-65)
 * ---------------------------------------------------------------------------------------------- */
void TRMSynthesisParametersRestoreDefaults(TRMSynthesisParameters *sp)
{
    memset(sp, 0, sizeof *sp);
    sp->masterVolume = 60;      sp->vocalTractLength = 17.5; sp->temperature = 25;  sp->balance = 0;
    sp->breathiness = 1;        sp->lossFactor = 0.5;        sp->pitch = -12;
    sp->throatCutoff = 1500;    sp->throatVolume = 6;        sp->apertureScaling = 3.05;
    sp->mouthCoef = 5000;       sp->noseCoef = 5000;         sp->mixOffset = 54;
    sp->n1 = 1.35; sp->n2 = 1.96; sp->n3 = 1.91; sp->n4 = 1.3; sp->n5 = 0.73;
    sp->tp = 40; sp->tnMin = 16; sp->tnMax = 32;
    sp->glottalPulseShape = 0;  sp->shouldUseNoiseModulation = 1;
    sp->samplingRate = 1;       /* 44100 */
    sp->outputChannels = 1;     /* stereo */
}

int TRMSynthesisParametersForVoice(const char *name, TRMSynthesisParameters *sp)
{
    static const struct { const char *name; double length, tp, tnMin, tnMax, pitch; } voices[] = {
        {"Male", 17.5, 0.40, 0.24, 0.24, -12.0}, {"Female", 15.0, 0.40, 0.32, 0.32, 0.0}, {"LgChild", 12.5, 0.40, 0.24, 0.24, 2.5},
        {"SmChild", 10.0, 0.40, 0.24, 0.24, 5.0}, {"Baby", 7.5, 0.40, 0.24, 0.24, 7.5},
    };
    if (!name || !sp) return set_err(TRM_ERR_PARAM, "null argument%s", "");
    for (size_t i = 0; i < sizeof voices / sizeof voices[0]; i++) {
        if (strcasecmp(name, voices[i].name) == 0) {
            TRMSynthesisParametersRestoreDefaults(sp);
            sp->vocalTractLength = voices[i].length;
            sp->tp = voices[i].tp * 100.0;
            sp->tnMin = voices[i].tnMin * 100.0;
            sp->tnMax = voices[i].tnMax * 100.0;
            sp->pitch = voices[i].pitch;
            return TRM_OK;
        }
    }
    return set_err(TRM_ERR_PARAM, "unknown voice \"%s\"", name);
}

void TRMInputParametersFromSynthesisParameters(const TRMSynthesisParameters *sp, int32_t fileFormat, TRMInputParameters *ip)
{
    memset(ip, 0, sizeof *ip);
    ip->outputFileFormat = fileFormat;
    ip->outputRate = sp->samplingRate == 0 ? 22050.0f : 44100.0f;
    ip->controlRate = 250;
    ip->volume = sp->masterVolume;
    ip->channels = sp->outputChannels + 1;
    ip->balance = sp->balance;
    ip->waveform = sp->glottalPulseShape;
    ip->tp = sp->tp; ip->tnMin = sp->tnMin; ip->tnMax = sp->tnMax;
    ip->breathiness = sp->breathiness;
    ip->length = sp->vocalTractLength;
    ip->temperature = sp->temperature;
    ip->lossFactor = sp->lossFactor;
    ip->apScale = sp->apertureScaling;
    ip->mouthCoef = sp->mouthCoef;
    ip->noseCoef = sp->noseCoef;
    ip->noseRadius[0] = 0;
    ip->noseRadius[1] = sp->n1; ip->noseRadius[2] = sp->n2; ip->noseRadius[3] = sp->n3;
    ip->noseRadius[4] = sp->n4; ip->noseRadius[5] = sp->n5;
    ip->throatCutoff = sp->throatCutoff;
    ip->throatVol = sp->throatVolume;
    ip->usesModulation = sp->shouldUseNoiseModulation;
    ip->mixOffset = sp->mixOffset;
}

char *TRMSynthesisParametersString(const TRMSynthesisParameters *sp)
{
    char *buf = malloc(4096);
    if (!buf) { set_err(TRM_ERR_NOMEM, "out of memory%s", ""); return NULL; }
    int n = 0;
#define LINE(fmt, v, text) n += snprintf(buf + n, 4096 - (size_t)n, fmt, v, text)
    LINE("%u\t\t; %s\n", 0u, "output file format (0 = AU, 1 = AIFF, 2 = WAVE)");
    LINE("%g\t\t; %s\n", sp->samplingRate == 0 ? 22050.0 : 44100.0, "output sample rate (22050.0, 44100.0)");
    LINE("%u\t\t; %s\n", 250u, "input control rate (1 - 1000 Hz)");
    LINE("%f\t; %s\n", sp->masterVolume, "master volume (0 - 60 dB)");
    LINE("%lu\t\t; %s\n", (unsigned long)(sp->outputChannels + 1), "number of sound output channels (1 or 2)");
    LINE("%f\t; %s\n", sp->balance, "stereo balance (-1 to +1)");
    LINE("%lu\t\t; %s\n", (unsigned long)sp->glottalPulseShape, "glottal source waveform type (0 = pulse, 1 = sine)");
    LINE("%f\t; %s\n", sp->tp, "glottal pulse rise time (5 - 50 % of GP period)");
    LINE("%f\t; %s\n", sp->tnMin, "glottal pulse fall time minimum (5 - 50 % of GP period)");
    LINE("%f\t; %s\n", sp->tnMax, "glottal pulse fall time maximum (5 - 50 % of GP period)");
    LINE("%f\t; %s\n", sp->breathiness, "glottal source breathiness (0 - 10 % of GS amplitude)");
    LINE("%f\t; %s\n", sp->vocalTractLength, "nominal tube length (10 - 20 cm)");
    LINE("%f\t; %s\n", sp->temperature, "tube temperature (25 - 40 degrees celsius)");
    LINE("%f\t; %s\n", sp->lossFactor, "junction loss factor (0 - 5 % of unity gain)");
    LINE("%f\t; %s\n", sp->apertureScaling, "aperture scaling radius (3.05 - 12 cm)");
    LINE("%f\t; %s\n", sp->mouthCoef, "mouth aperture coefficient (0 - 0.99)");
    LINE("%f\t; %s\n", sp->noseCoef, "nose aperture coefficient (0 - 0.99)");
    LINE("%f\t; %s\n", sp->n1, "radius of nose section 1 (0 - 3 cm)");
    LINE("%f\t; %s\n", sp->n2, "radius of nose section 2 (0 - 3 cm)");
    LINE("%f\t; %s\n", sp->n3, "radius of nose section 3 (0 - 3 cm)");
    LINE("%f\t; %s\n", sp->n4, "radius of nose section 4 (0 - 3 cm)");
    LINE("%f\t; %s\n", sp->n5, "radius of nose section 5 (0 - 3 cm)");
    LINE("%f\t; %s\n", sp->throatCutoff, "throat lowpass frequency cutoff (50 - nyquist Hz)");
    LINE("%f\t; %s\n", sp->throatVolume, "throat volume (0 - 48 dB)");
    LINE("%d\t\t; %s\n", (int)sp->shouldUseNoiseModulation, "pulse modulation of noise (0 = off, 1 = on)");
    LINE("%f\t; %s", sp->mixOffset, "noise crossmix offset (30 - 60 db)");
#undef LINE
    return buf;
}

/* ------------------------------------------------------------------------------------------------
 * TRMBatch
 * ---------------------------------------------------------------------------------------------- */
struct TRMBatch {
    int n, precision;
    trm_cuda_utterance *desc;      /* offsets relative to the caller's arrays */
    voice_set voices;
    int32_t *numberSamples;
    int64_t *pcm_offsets, *out_offsets, *tube_offsets;
    double *maxima;
    uint8_t *flush_bug;            /* per utterance: the reference would hit its converter flush bug (TRMReferenceFlushBug) */
    int frame_format;              /* TRM_FRAMES_F64 / TRM_FRAMES_F32: how the `frames` argument of the synthesize calls is read */
    TRMBatchLayout layout;
    int64_t total_tube_elems;
    int64_t launches;
};

static int precision_ok(int p) { return p == TRM_PRECISION_FP64 || p == TRM_PRECISION_FP32 || p == TRM_PRECISION_FP64_STRICT; }
static int64_t round_up_elems(int64_t v) { return (v + TRM_ALIGN_ELEMS - 1) / TRM_ALIGN_ELEMS * TRM_ALIGN_ELEMS; }

void TRMBatchFree(TRMBatch *b)
{
    if (!b) return;
    free(b->desc); free(b->numberSamples); free(b->pcm_offsets); free(b->out_offsets); free(b->tube_offsets); free(b->maxima); free(b->flush_bug);
    voice_set_free(&b->voices);
    free(b);
}

TRMBatch *TRMBatchCreate(int n, const TRMInputParameters *ip, int shared, const int64_t *frame_offset,
                         const int32_t *n_frames, int precision, int *err)
{
    int dummy;
    if (!err) err = &dummy;
    if (n < 0 || !precision_ok(precision)) {
        *err = set_err(TRM_ERR_PARAM, "bad batch size or precision%s", "");
        return NULL;
    }
    int rc;
    tables(&rc);
    if (rc) { *err = set_err(rc, "FIR design failed%s", ""); return NULL; }
    TRMBatch *b = calloc(1, sizeof *b);
    if (!b) { *err = set_err(TRM_ERR_NOMEM, "out of memory%s", ""); return NULL; }
    b->n = n;
    b->precision = precision;
    const size_t nn = (size_t)(n > 0 ? n : 1);
    b->desc = calloc(nn, sizeof *b->desc);
    b->numberSamples = calloc(nn, sizeof *b->numberSamples);
    b->pcm_offsets = calloc(nn, sizeof *b->pcm_offsets);
    b->out_offsets = calloc(nn, sizeof *b->out_offsets);
    b->tube_offsets = calloc(nn, sizeof *b->tube_offsets);
    b->maxima = calloc(nn, sizeof *b->maxima);
    b->flush_bug = calloc(nn, 1);
    if (!b->flush_bug || !b->numberSamples || !b->pcm_offsets || !b->out_offsets || !b->tube_offsets || !b->maxima) {
        TRMBatchFree(b);
        *err = set_err(TRM_ERR_NOMEM, "out of memory%s", "");
        return NULL;
    }
    int64_t pcm_at = 0, out_at = 0, tube_at = 0, frames_hi = 0;
    trm_cuda_utterance shared_desc;
    rates_t shared_rates;
    int32_t shared_nf = -1;
    for (int u = 0; u < n; u++) {
        const TRMInputParameters *p = shared ? ip : ip + u;
        trm_cuda_utterance *d = &b->desc[u];
        rates_t r;
        if (shared && shared_nf >= 0) {
            /* same voice: only the counts depend on the number of frames */
            *d = shared_desc;
            r = shared_rates;
            if (n_frames[u] < 0) { rc = set_err(TRM_ERR_PARAM, "negative frame count%s", ""); goto bad; }
            d->n_frames = n_frames[u];
            d->n_tube = n_frames[u] > 0 ? (int64_t)(n_frames[u] - 1) * r.controlPeriod : 0;
            d->n_out = n_frames[u] > 0 ? src_output_count(&r, d->n_tube) : 0;
        } else {
            rc = describe(p, n_frames[u], &b->voices, d, &r);
            if (rc) goto bad;
            if (shared) { shared_desc = *d; shared_rates = r; shared_nf = n_frames[u]; }
        }
        if (d->n_out > INT32_MAX) { rc = set_err(TRM_ERR_PARAM, "utterance too long (numberSamples is int32 in the reference)%s", ""); goto bad; }
        d->frame_offset = frame_offset[u];
        d->tube_offset = tube_at;
        d->out_offset = out_at;
        d->pcm_offset = pcm_at;
        b->numberSamples[u] = (int32_t)d->n_out;
        b->flush_bug[u] = n_frames[u] > 0 && flush_bug(&r, d->n_tube);
        b->tube_offsets[u] = tube_at;
        b->out_offsets[u] = out_at;
        b->pcm_offsets[u] = pcm_at;
        tube_at += round_up_elems(d->n_tube);
        out_at += round_up_elems(d->n_out);
        pcm_at += round_up_elems(d->n_out * d->channels);
        if (frame_offset[u] + n_frames[u] > frames_hi) frames_hi = frame_offset[u] + n_frames[u];
        b->layout.audio_seconds += n_frames[u] > 0 ? (double)(n_frames[u] - 1) / (double)p->controlRate : 0.0;
        b->layout.tube_samples += d->n_tube;
        b->layout.out_samples += d->n_out;
    }
    b->layout.total_frames = frames_hi;
    b->layout.total_pcm_samples = pcm_at;
    b->layout.total_out_samples = out_at;
    b->total_tube_elems = tube_at;
    *err = TRM_OK;
    return b;
bad:
    TRMBatchFree(b);
    *err = rc;
    return NULL;
}

void TRMBatchGetLayout(const TRMBatch *b, TRMBatchLayout *l) { *l = b->layout; }
int TRMBatchSetFrameFormat(TRMBatch *b, int format)
{
    if (format != TRM_FRAMES_F64 && format != TRM_FRAMES_F32) return set_err(TRM_ERR_PARAM, "unknown frame format%s", "");
    b->frame_format = format;
    return TRM_OK;
}
const int32_t *TRMBatchNumberSamples(const TRMBatch *b) { return b->numberSamples; }
const int64_t *TRMBatchPCMOffsets(const TRMBatch *b) { return b->pcm_offsets; }
const int64_t *TRMBatchOutOffsets(const TRMBatch *b) { return b->out_offsets; }
const double *TRMBatchMaximumSampleValues(const TRMBatch *b) { return b->maxima; }
const uint8_t *TRMBatchReferenceFlushBugFlags(const TRMBatch *b) { return b->flush_bug; }
int64_t TRMBatchTubeElements(const TRMBatch *b) { return b->total_tube_elems; }
const int64_t *TRMBatchTubeOffsets(const TRMBatch *b) { return b->tube_offsets; }
int64_t TRMBatchKernelLaunches(const TRMBatch *b) { return b->launches; }

typedef struct {
    TRMBatch *b;
    const TRMParameters *frames;
    int16_t *pcm;
    void *samples, *tube;
    int device, u0, u1, rc;
    int64_t launches;
    char msg[512];
    void (*enqueued)(void *);      /* asynchronous tickets: called when the shard's first chunk is in the device queues */
    void *enqueued_arg;
} shard_job;

static void *shard_main(void *arg)
{
    shard_job *j = arg;
    trm_cuda_ctx *ctx;
    int lane = 0;
    j->rc = acquire_ctx(j->device, &ctx, &lane);
    if (j->rc == TRM_OK) {
        if (trm_cuda_set_wavetables(ctx, j->b->voices.tables, j->b->voices.n) != 0 ||
            trm_cuda_synthesize_host(ctx, j->b->precision, j->b->frame_format, j->u1 - j->u0, j->b->desc + j->u0, j->frames,
                                     j->pcm, j->samples, j->b->maxima + j->u0, j->tube, &j->launches, j->enqueued,
                                     j->enqueued_arg) != 0)
            j->rc = cuda_err();
        release_ctx(j->device, lane);
    }
    if (j->rc) snprintf(j->msg, sizeof j->msg, "%s", g_errmsg);
    return NULL;
}

/* Asynchronous tickets start in submission order: ticket k's shards put their first chunk into the device queues before
 * ticket k+1 is let in.  (The copy-in and compute queues are shared per device, so without this the order in which the
 * host threads happen to be scheduled decides which call runs first, and a caller waiting for its oldest ticket can
 * find it executed last.) */
static pthread_mutex_t g_order_mu = PTHREAD_MUTEX_INITIALIZER;
static pthread_cond_t g_order_cv = PTHREAD_COND_INITIALIZER;
static unsigned long long g_order_next = 0, g_order_turn = 0;
typedef struct { unsigned long long seq; int pending, passed; } order_gate;

static void gate_pass(order_gate *g)
{
    pthread_mutex_lock(&g_order_mu);
    if (!g->passed) {
        g->passed = 1;
        g_order_turn = g->seq + 1;
        pthread_cond_broadcast(&g_order_cv);
    }
    pthread_mutex_unlock(&g_order_mu);
}
static void gate_shard_enqueued(void *arg)
{
    order_gate *g = arg;
    pthread_mutex_lock(&g_order_mu);
    const int last = --g->pending <= 0;
    pthread_mutex_unlock(&g_order_mu);
    if (last) gate_pass(g);
}

static int batch_run(TRMBatch *b, const TRMParameters *frames, int16_t *pcm, void *samples, void *tube,
                     const int *devices, int n_devices, order_gate *gate)
{
    if (b->n == 0) return TRM_OK;
    if (n_devices < 1) n_devices = 1;
    if (n_devices > b->n) n_devices = b->n;
    if (n_devices > MAX_DEVICES) n_devices = MAX_DEVICES;
    if (gate) gate->pending = n_devices;
    shard_job jobs[MAX_DEVICES];
    pthread_t th[MAX_DEVICES];
    /* contiguous shards with equal shares of the tube-rate work; no data crosses devices */
    const double per = (double)b->layout.tube_samples / n_devices;
    int u = 0;
    double acc = 0;
    for (int k = 0; k < n_devices; k++) {
        memset(&jobs[k], 0, sizeof jobs[k]);
        jobs[k].b = b; jobs[k].frames = frames; jobs[k].pcm = pcm; jobs[k].samples = samples; jobs[k].tube = tube;
        jobs[k].device = devices ? devices[k] : k;
        if (gate) { jobs[k].enqueued = gate_shard_enqueued; jobs[k].enqueued_arg = gate; }
        jobs[k].u0 = u;
        if (k == n_devices - 1) u = b->n;
        else {
            const int remaining_devices = n_devices - 1 - k;
            while (u < b->n - remaining_devices && (u == jobs[k].u0 || acc + (double)b->desc[u].n_tube <= per * (k + 1))) {
                acc += (double)b->desc[u].n_tube;
                u++;
            }
        }
        jobs[k].u1 = u;
    }
    if (n_devices == 1) shard_main(&jobs[0]);
    else {
        for (int k = 0; k < n_devices; k++)
            if (pthread_create(&th[k], NULL, shard_main, &jobs[k]) != 0) { jobs[k].rc = TRM_ERR_NOMEM; th[k] = 0; shard_main(&jobs[k]); }
        for (int k = 0; k < n_devices; k++)
            if (th[k]) pthread_join(th[k], NULL);
    }
    b->launches = 0;
    for (int k = 0; k < n_devices; k++) {
        b->launches += jobs[k].launches;
        if (jobs[k].rc) { snprintf(g_errmsg, sizeof g_errmsg, "%s", jobs[k].msg); return jobs[k].rc; }
    }
    return TRM_OK;
}

int TRMBatchSynthesize(TRMBatch *b, const TRMParameters *frames, int16_t *pcm_out, void *samples_out,
                       const int *devices, int n_devices)
{
    return batch_run(b, frames, pcm_out, samples_out, NULL, devices, n_devices, NULL);
}

/* ---- sweeps over device-generated tracks (BASELINE configs[4]) ---- */
int TRMSweepSynthesize(const TRMInputParameters *ip, int32_t n_frames, uint64_t seed, uint64_t first_index, int64_t n,
                       int precision, int device, uint64_t *checksums, double *maxima, int64_t n_probe, const int64_t *probe_utt,
                       int16_t *probe_pcm, int64_t probe_stride, int32_t *numberSamples, int64_t *launches, double *kernel_ms)
{
    if (!ip || n < 0 || n_frames < 0 || !precision_ok(precision) || !checksums) return set_err(TRM_ERR_PARAM, "bad sweep arguments%s", "");
    voice_set vs;
    memset(&vs, 0, sizeof vs);
    trm_cuda_utterance d;
    int rc = describe(ip, n_frames, &vs, &d, NULL);
    if (rc) { voice_set_free(&vs); return rc; }
    if (numberSamples) *numberSamples = (int32_t)d.n_out;
    if (n == 0) { voice_set_free(&vs); return TRM_OK; }
    trm_cuda_ctx *ctx;
    int lane = 0;
    if ((rc = acquire_ctx(device, &ctx, &lane)) != TRM_OK) { voice_set_free(&vs); return rc; }
    if (trm_cuda_set_wavetables(ctx, vs.tables, vs.n) != 0 ||
        trm_cuda_sweep(ctx, precision, &d, n_frames, seed, first_index, n, checksums, maxima, n_probe, probe_utt, probe_pcm,
                       probe_stride, launches, kernel_ms) != 0)
        rc = cuda_err();
    release_ctx(device, lane);
    voice_set_free(&vs);
    return rc;
}

/* ---- control frames from event lists (EventList.m:883-1061) ---- */
void TRMFrameGenerationSetDefaults(TRMFrameGeneration *fg)
{
    memset(fg, 0, sizeof *fg);
    fg->useMacroIntonation = fg->useMicroIntonation = fg->useSmoothIntonation = fg->useDrift = 1;   /* MMIntonation.m:74-80 */
    fg->driftDeviation = 1.0;
    fg->driftCutoff = 4;
    fg->pitch = -12;                 /* MMSynthesisParameters default */
    fg->driftSeed = 0.7892347f;      /* MMDriftGenerator.m:6 */
}

/* The time loop of -generateOutputInTimeRange: without the values (planning: how many frames will there be?).
 * The reference emits one frame per 4 ms step while events remain, and after each step moves on to the next event
 * once the clock has reached the current one's time -- at most one event per step (m:973-1030).  So event i is
 * "current" for max(1, ceil((time_i - now) / 4)) steps, where now is the clock when it became current: O(events)
 * instead of O(frames).  (tests/test_oracle.py checks this against the oracle's literal loop.) */
int64_t TRMEventListFrameCount(const TRMEvent *ev, int64_t count)
{
    if (!ev || count < 2) return 0;
    int64_t emitted = 0;
    uint64_t now = 0;
    for (int64_t i = 1; i < count; i++) {
        const uint64_t next = (uint64_t)ev[i].time;
        uint64_t steps = next > now ? (next - now + 3) / 4 : 1;
        if (steps < 1) steps = 1;
        emitted += (int64_t)steps;
        now += 4 * steps;
    }
    return emitted;
}

/* One event list the generator runs on: n_frames must be its TRMEventListFrameCount. */
static int check_event_list(const TRMEvent *ev, int64_t n_events, int64_t n_frames)
{
    const int64_t want = n_events >= 0 ? TRMEventListFrameCount(ev, n_events) : -1;
    if (want != n_frames)
        return set_err(TRM_ERR_PARAM, "utterance frame count differs from TRMEventListFrameCount of its event list%s", "");
    /* every TRM parameter track needs a value after the first event: the reference's set-up loop (EventList.m:919-930)
     * scans forward for one without a bound and reads past the array otherwise */
    for (int j = 0; j < 16 && n_events >= 2; j++) {
        int found = 0;
        for (int64_t k = 1; k < n_events && !found; k++) found = !isnan(ev[k].value[j]);
        if (!found) return set_err(TRM_ERR_PARAM, "event list: a parameter track has no value after the first event%s", "");
    }
    return TRM_OK;
}

static int check_event_lists(const TRMBatch *b, const TRMEvent *events, const int64_t *event_offset, const int32_t *n_events)
{
    if (!events || !event_offset || !n_events) return set_err(TRM_ERR_PARAM, "null event arguments%s", "");
    for (int u = 0; u < b->n; u++) {
        const int rc = check_event_list(events + event_offset[u], n_events[u], b->desc[u].n_frames);
        if (rc != TRM_OK) return rc;
    }
    return TRM_OK;
}

int TRMBatchGenerateFrames(TRMBatch *b, const TRMEvent *events, const int64_t *event_offset, const int32_t *n_events,
                           const TRMFrameGeneration *fg, int shared_fg, TRMParameters *frames_out, float *drift_seed_out,
                           int device)
{
    int rc = check_event_lists(b, events, event_offset, n_events);
    if (rc) return rc;
    if (b->n == 0) return TRM_OK;
    trm_cuda_ctx *ctx;
    int lane = 0;
    if ((rc = acquire_ctx(device, &ctx, &lane)) != TRM_OK) return rc;
    if (trm_cuda_generate_frames(ctx, b->n, b->desc, (const trm_cuda_event *)events, event_offset, n_events,
                                 (const trm_cuda_framegen *)fg, shared_fg, NULL, (double *)frames_out, drift_seed_out) != 0)
        rc = cuda_err();
    release_ctx(device, lane);
    return rc;
}

int TRMBatchSynthesizeEvents(TRMBatch *b, const TRMEvent *events, const int64_t *event_offset, const int32_t *n_events,
                             const TRMFrameGeneration *fg, int shared_fg, int16_t *pcm_out, void *samples_out, int device)
{
    int rc = check_event_lists(b, events, event_offset, n_events);
    if (rc) return rc;
    if (b->n == 0) return TRM_OK;
    trm_cuda_ctx *ctx;
    int lane = 0;
    if ((rc = acquire_ctx(device, &ctx, &lane)) != TRM_OK) return rc;
    const double *frames_dev = NULL;
    if (trm_cuda_set_wavetables(ctx, b->voices.tables, b->voices.n) != 0 ||
        trm_cuda_generate_frames(ctx, b->n, b->desc, (const trm_cuda_event *)events, event_offset, n_events,
                                 (const trm_cuda_framegen *)fg, shared_fg, &frames_dev, NULL, NULL) != 0 ||
        trm_cuda_synthesize_host(ctx, b->precision, 0, b->n, b->desc, frames_dev, pcm_out, samples_out, b->maxima, NULL,
                                 &b->launches, NULL, NULL) != 0)
        rc = cuda_err();
    else
        b->launches += 1;
    release_ctx(device, lane);
    return rc;
}

/* ---- streaming (TRAcT-style): many voices advanced together, state carried on the device ---- */
/* The lockstep use of the stream pool: slot i is stream i, every push advances all of them by the same frames. */
struct TRMStream {
    trm_cuda_pool *p;
    int n, max_m, flushed;
    TRMInputParameters voice;       /* every stream's voice (TRMStreamSetVoice changes it) */
    int32_t *slot, *n_frames;       /* [n] the entries of every push: stream i's slot, m frames each */
    uint8_t *flush;                 /* [n] */
    int64_t *offset;                /* [n+1] packed offsets the pool returns (every stream gets the same count) */
};

TRMStream *TRMStreamCreate(int n_streams, const TRMInputParameters *voice, int precision, int max_frames_per_push,
                           int device, int *err)
{
    int dummy;
    if (!err) err = &dummy;
    if (n_streams <= 0 || max_frames_per_push <= 0 || !voice || !precision_ok(precision)) {
        *err = set_err(TRM_ERR_PARAM, "bad stream arguments%s", "");
        return NULL;
    }
    TRMStream *t = calloc(1, sizeof *t);
    if (t) {
        t->slot = calloc((size_t)n_streams, sizeof *t->slot);
        t->n_frames = calloc((size_t)n_streams, sizeof *t->n_frames);
        t->flush = calloc((size_t)n_streams, sizeof *t->flush);
        t->offset = calloc((size_t)n_streams + 1, sizeof *t->offset);
    }
    if (!t || !t->slot || !t->n_frames || !t->flush || !t->offset) {
        TRMStreamFree(t);
        *err = set_err(TRM_ERR_NOMEM, "out of memory%s", "");
        return NULL;
    }
    t->n = n_streams;
    t->max_m = max_frames_per_push;
    t->voice = *voice;
    voice_set vs;
    trm_cuda_utterance d;
    memset(&vs, 0, sizeof vs);
    if ((*err = describe(voice, 2, &vs, &d, NULL)) != TRM_OK) { voice_set_free(&vs); TRMStreamFree(t); return NULL; }
    trm_cuda_ctx *ctx;
    int lane;
    if ((*err = acquire_ctx(device, &ctx, &lane)) != TRM_OK) { voice_set_free(&vs); TRMStreamFree(t); return NULL; }
    int rc = trm_cuda_pool_create(ctx, precision, n_streams, max_frames_per_push, &t->p);
    release_ctx(device, lane);      /* the pool owns its buffers, wavetables, stream and scratch: no lane is held */
    /* sized for this voice alone, so that the capacity is what one stream of it needs */
    if (rc == 0) rc = trm_cuda_pool_reserve(t->p, &d);
    for (int i = 0; i < n_streams && rc == 0; i++)
        rc = trm_cuda_pool_open(t->p, &d, vs.tables + (size_t)d.voice * TRM_TABLE_LENGTH, &t->slot[i]);
    voice_set_free(&vs);
    if (rc != 0) {
        *err = cuda_err();
        TRMStreamFree(t);
        return NULL;
    }
    *err = TRM_OK;
    return t;
}

int64_t TRMStreamCapacity(const TRMStream *t) { return t ? trm_cuda_pool_slot_capacity(t->p) : 0; }

int TRMStreamPush(TRMStream *t, const TRMParameters *frames, int m, int flush, void *samples_out, int64_t *n_samples)
{
    if (!t) return set_err(TRM_ERR_PARAM, "null stream%s", "");
    if (n_samples) *n_samples = 0;
    if (t->flushed) return set_err(TRM_ERR_CUDA, "CUDA: %s", "trm_cuda_stream_push: the streams were flushed");
    if (m < 0 || m > t->max_m)
        return set_err(TRM_ERR_CUDA, "CUDA: %s", "trm_cuda_stream_push: more frames than the stream was created for");
    for (int i = 0; i < t->n; i++) {
        t->n_frames[i] = m;
        t->flush[i] = flush ? 1 : 0;
    }
    /* [stream][m][16] is the pool's back-to-back frame layout; samples come back in rows of the capacity */
    if (trm_cuda_pool_push(t->p, t->n, t->slot, t->n_frames, (const double *)frames, t->flush, samples_out,
                           trm_cuda_pool_slot_capacity(t->p), t->offset) != 0)
        return cuda_err();
    if (flush) t->flushed = 1;      /* the pool has freed the slots */
    if (n_samples) *n_samples = t->offset[1] - t->offset[0];
    return TRM_OK;
}

void TRMStreamFree(TRMStream *t)
{
    if (!t) return;
    trm_cuda_pool_destroy(t->p);
    free(t->slot);
    free(t->n_frames);
    free(t->flush);
    free(t->offset);
    free(t);
}

/* ---- stream pool: independent streaming slots, each with its own voice ---- */
struct TRMStreamPool {
    trm_cuda_pool *p;
    int capacity, precision;
    TRMInputParameters *voice;      /* [capacity]: the voice each open slot was opened or restored with (snapshots) */
};

/* shim codes: -4 / -7 are argument / call-order refusals (message set by the shim), anything else is CUDA */
static int pool_rc(int rc)
{
    if (rc == TRM_ERR_PARAM || rc == TRM_ERR_STATE) return set_err(rc, "%s", trm_cuda_last_error());
    return cuda_err();
}

TRMStreamPool *TRMStreamPoolCreate(int capacity, int precision, int max_frames_per_push, int device, int *err)
{
    int dummy;
    if (!err) err = &dummy;
    if (capacity <= 0 || max_frames_per_push <= 0 || !precision_ok(precision)) {
        *err = set_err(TRM_ERR_PARAM, "bad stream pool arguments%s", "");
        return NULL;
    }
    TRMStreamPool *t = calloc(1, sizeof *t);
    if (t) t->voice = calloc((size_t)capacity, sizeof *t->voice);
    if (!t || !t->voice) { free(t); *err = set_err(TRM_ERR_NOMEM, "out of memory%s", ""); return NULL; }
    t->capacity = capacity;
    t->precision = precision;
    trm_cuda_ctx *ctx;
    int lane;
    if ((*err = acquire_ctx(device, &ctx, &lane)) != TRM_OK) { free(t->voice); free(t); return NULL; }
    int rc = trm_cuda_pool_create(ctx, precision, capacity, max_frames_per_push, &t->p);
    release_ctx(device, lane);      /* the pool owns its buffers, wavetables, stream and scratch: no lane is held */
    if (rc == 0) {
        /* initial sizes: the default voice (TRMInputParametersSetDefaults at 44.1 kHz) */
        TRMInputParameters ip;
        voice_set vs;
        trm_cuda_utterance d;
        memset(&vs, 0, sizeof vs);
        TRMInputParametersSetDefaults(&ip, 44100.0f);
        if (describe(&ip, 2, &vs, &d, NULL) == TRM_OK) rc = trm_cuda_pool_reserve(t->p, &d);
        voice_set_free(&vs);
    }
    if (rc != 0) {
        *err = pool_rc(rc);
        trm_cuda_pool_destroy(t->p);
        free(t->voice);
        free(t);
        return NULL;
    }
    *err = TRM_OK;
    return t;
}

/* Opens a free slot with this voice, fed with frames or, when event_fed, from an event list (*n_frames receives its frame
 * count).  Returns the slot or a TRM_ERR_*. */
static int pool_open(TRMStreamPool *t, const TRMInputParameters *voice, int event_fed, const TRMEvent *events, int64_t n_events,
                     const TRMFrameGeneration *fg, int64_t *n_frames)
{
    if (!t || !voice) return set_err(TRM_ERR_PARAM, "null stream pool or voice%s", "");
    voice_set vs;
    trm_cuda_utterance d;
    memset(&vs, 0, sizeof vs);
    int rc = describe(voice, 2, &vs, &d, NULL);
    if (rc == TRM_OK && event_fed) {
        if (!events || !fg) {
            rc = set_err(TRM_ERR_PARAM, "null event arguments%s", "");
        } else {
            *n_frames = n_events >= 0 ? TRMEventListFrameCount(events, n_events) : 0;
            rc = check_event_list(events, n_events, *n_frames);
        }
    }
    if (rc != TRM_OK) { voice_set_free(&vs); return rc; }
    const double *wavetable = vs.tables + (size_t)d.voice * TRM_TABLE_LENGTH;
    int slot = -1;
    rc = event_fed ? trm_cuda_pool_open_events(t->p, &d, wavetable, (const trm_cuda_event *)events, n_events, *n_frames,
                                               (const trm_cuda_framegen *)fg, &slot)
                   : trm_cuda_pool_open(t->p, &d, wavetable, &slot);
    voice_set_free(&vs);
    if (rc != 0) return pool_rc(rc);
    t->voice[slot] = *voice;
    return slot;
}

int TRMStreamPoolOpen(TRMStreamPool *t, const TRMInputParameters *voice)
{
    return pool_open(t, voice, 0, NULL, 0, NULL, NULL);
}

int TRMStreamPoolOpenEvents(TRMStreamPool *t, const TRMInputParameters *voice, const TRMEvent *events, int64_t n_events,
                            const TRMFrameGeneration *fg, int64_t *n_frames_out)
{
    int64_t n_frames = 0;
    const int slot = pool_open(t, voice, 1, events, n_events, fg, &n_frames);
    if (slot >= 0 && n_frames_out) *n_frames_out = n_frames;
    return slot;
}

int TRMStreamPoolClose(TRMStreamPool *t, int slot)
{
    if (!t) return set_err(TRM_ERR_PARAM, "null stream pool%s", "");
    const int rc = trm_cuda_pool_close(t->p, slot);
    if (rc != 0) return pool_rc(rc);
    memset(&t->voice[slot], 0, sizeof t->voice[slot]);
    return TRM_OK;
}

/* a push succeeded: the slots it flushed are free again */
static void pool_forget_flushed(TRMStreamPool *t, int n, const int32_t *slot, const uint8_t *flush)
{
    for (int i = 0; flush && i < n; i++)
        if (flush[i]) memset(&t->voice[slot[i]], 0, sizeof t->voice[slot[i]]);
}

int64_t TRMStreamPoolSlotCapacity(const TRMStreamPool *t) { return t ? trm_cuda_pool_slot_capacity(t->p) : 0; }

int TRMStreamPoolPush(TRMStreamPool *t, int n, const int32_t *slot, const int32_t *n_frames, const TRMParameters *frames,
                      const uint8_t *flush, void *samples_out, int64_t *out_offset)
{
    if (!t) return set_err(TRM_ERR_PARAM, "null stream pool%s", "");
    const int rc = trm_cuda_pool_push(t->p, n, slot, n_frames, (const double *)frames, flush, samples_out, 0, out_offset);
    if (rc != 0) return pool_rc(rc);
    pool_forget_flushed(t, n, slot, flush);
    return TRM_OK;
}

int TRMStreamPoolPushPCM16(TRMStreamPool *t, int n, const int32_t *slot, const int32_t *n_frames, const TRMParameters *frames,
                           const uint8_t *flush, const double *peak, int16_t *pcm_out, int64_t *pcm_offset, double *max_out)
{
    if (!t) return set_err(TRM_ERR_PARAM, "null stream pool%s", "");
    const int rc = trm_cuda_pool_push_pcm16(t->p, n, slot, n_frames, (const double *)frames, flush, peak, pcm_out, pcm_offset,
                                            max_out);
    if (rc != 0) return pool_rc(rc);
    pool_forget_flushed(t, n, slot, flush);
    return TRM_OK;
}

void TRMStreamPoolFree(TRMStreamPool *t)
{
    if (!t) return;
    trm_cuda_pool_destroy(t->p);
    free(t->voice);
    free(t);
}

/* ---- stream pool snapshots (include/trm.h): header, voice and derived constants here, the slot part in the shim ---- */
#if defined(__BYTE_ORDER__) && __BYTE_ORDER__ != __ORDER_LITTLE_ENDIAN__
#error "snapshot data parts are copied as they lie in memory: little-endian hosts only"
#endif
#define SNAP_VERSION   1u                 /* frame-fed slots */
#define SNAP_VERSION_EVENTS 2u            /* event-fed slots: the event header, generator state and list follow */
#define SNAP_HEADER    32                 /* magic, version, precision, total bytes, checksum */
#define SNAP_VOICE     192
#define SNAP_DERIVED   24
#define SNAP_COUNTERS  48
#define SNAP_FIXED     (SNAP_HEADER + SNAP_VOICE + SNAP_DERIVED + SNAP_COUNTERS)
#define SNAP_EVHEADER  72                 /* n_events, list_frames, fg (48 bytes), generator flag, reserved */
static const unsigned char snap_magic[8] = {'T', 'R', 'M', 'S', 'N', 'A', 'P', 0};

static uint64_t fnv1a64(const unsigned char *p, size_t n)
{
    uint64_t h = 0xcbf29ce484222325ull;
    for (size_t i = 0; i < n; i++) h = (h ^ p[i]) * 0x100000001b3ull;
    return h;
}

/* little-endian writers / readers, one field at a time */
static unsigned char *put_u32(unsigned char *o, uint32_t v) { for (int i = 0; i < 4; i++) o[i] = (unsigned char)(v >> (8 * i)); return o + 4; }
static unsigned char *put_u64(unsigned char *o, uint64_t v) { for (int i = 0; i < 8; i++) o[i] = (unsigned char)(v >> (8 * i)); return o + 8; }
static unsigned char *put_f32(unsigned char *o, float v) { uint32_t b; memcpy(&b, &v, 4); return put_u32(o, b); }
static unsigned char *put_f64(unsigned char *o, double v) { uint64_t b; memcpy(&b, &v, 8); return put_u64(o, b); }
static uint32_t get_u32(const unsigned char **q) { uint32_t v = 0; for (int i = 0; i < 4; i++) v |= (uint32_t)(*q)[i] << (8 * i); *q += 4; return v; }
static uint64_t get_u64(const unsigned char **q) { uint64_t v = 0; for (int i = 0; i < 8; i++) v |= (uint64_t)(*q)[i] << (8 * i); *q += 8; return v; }
static float get_f32(const unsigned char **q) { uint32_t b = get_u32(q); float v; memcpy(&v, &b, 4); return v; }
static double get_f64(const unsigned char **q) { uint64_t b = get_u64(q); double v; memcpy(&v, &b, 8); return v; }

static unsigned char *put_voice(unsigned char *o, const TRMInputParameters *ip)
{
    o = put_u32(o, (uint32_t)ip->outputFileFormat); o = put_f32(o, ip->outputRate); o = put_f32(o, ip->controlRate);
    o = put_f64(o, ip->volume); o = put_u32(o, (uint32_t)ip->channels); o = put_f64(o, ip->balance);
    o = put_u32(o, (uint32_t)ip->waveform);
    o = put_f64(o, ip->tp); o = put_f64(o, ip->tnMin); o = put_f64(o, ip->tnMax); o = put_f64(o, ip->breathiness);
    o = put_f64(o, ip->length); o = put_f64(o, ip->temperature); o = put_f64(o, ip->lossFactor); o = put_f64(o, ip->apScale);
    o = put_f64(o, ip->mouthCoef); o = put_f64(o, ip->noseCoef);
    for (int i = 0; i < TRM_TOTAL_NASAL_SECTIONS; i++) o = put_f64(o, ip->noseRadius[i]);
    o = put_f64(o, ip->throatCutoff); o = put_f64(o, ip->throatVol); o = put_u32(o, (uint32_t)ip->usesModulation);
    return put_f64(o, ip->mixOffset);
}

static void get_voice(const unsigned char **q, TRMInputParameters *ip)
{
    memset(ip, 0, sizeof *ip);
    ip->outputFileFormat = (int32_t)get_u32(q); ip->outputRate = get_f32(q); ip->controlRate = get_f32(q);
    ip->volume = get_f64(q); ip->channels = (int32_t)get_u32(q); ip->balance = get_f64(q);
    ip->waveform = (int32_t)get_u32(q);
    ip->tp = get_f64(q); ip->tnMin = get_f64(q); ip->tnMax = get_f64(q); ip->breathiness = get_f64(q);
    ip->length = get_f64(q); ip->temperature = get_f64(q); ip->lossFactor = get_f64(q); ip->apScale = get_f64(q);
    ip->mouthCoef = get_f64(q); ip->noseCoef = get_f64(q);
    for (int i = 0; i < TRM_TOTAL_NASAL_SECTIONS; i++) ip->noseRadius[i] = get_f64(q);
    ip->throatCutoff = get_f64(q); ip->throatVol = get_f64(q); ip->usesModulation = (int32_t)get_u32(q);
    ip->mixOffset = get_f64(q);
}

/* the event header of a version-2 snapshot (the generator flag is 1 exactly when frames were generated) */
static unsigned char *put_event_header(unsigned char *o, const trm_cuda_pool_event_state *ev, int64_t frames_generated)
{
    o = put_u64(o, (uint64_t)ev->n_events); o = put_u64(o, (uint64_t)ev->ev_frames);
    o = put_u32(o, (uint32_t)ev->fg.useMacroIntonation); o = put_u32(o, (uint32_t)ev->fg.useMicroIntonation);
    o = put_u32(o, (uint32_t)ev->fg.useSmoothIntonation); o = put_u32(o, (uint32_t)ev->fg.useDrift);
    o = put_f64(o, ev->fg.driftDeviation); o = put_f64(o, ev->fg.driftCutoff); o = put_f64(o, ev->fg.pitch);
    o = put_f32(o, ev->fg.driftSeed); o = put_u32(o, 0u);   /* reserved */
    o = put_u32(o, frames_generated > 0 ? 1u : 0u);
    return put_u32(o, 0u);
}

/* the derived constants a snapshot stores, from the voice's descriptor */
static void snap_derived(const trm_cuda_utterance *d, int precision, uint32_t out[6])
{
    out[0] = (uint32_t)d->controlPeriod; out[1] = (uint32_t)d->sampleRate; out[2] = d->tri;
    out[3] = (uint32_t)d->padSize; out[4] = (uint32_t)d->channels; out[5] = precision == TRM_PRECISION_FP32 ? 4u : 8u;
}

/* framegen_step's current event, clock and time of the current event after k frames of a list that expands to at least
 * k (k >= 1): the walk of TRMEventListFrameCount stopped after k steps.  (framegen_step leaves `next` as it is once the
 * last event is passed.) */
static void framegen_position(const TRMEvent *ev, int64_t count, int64_t k, int64_t *i, uint64_t *now, uint64_t *next)
{
    int64_t j = 1;
    uint64_t t = 0, nx = (uint64_t)ev[1].time;
    while (k > 0) {
        const uint64_t steps = nx > t ? (nx - t + 3) / 4 : 1;
        if ((uint64_t)k < steps) { t += 4 * (uint64_t)k; break; }
        t += 4 * steps;
        k -= (int64_t)steps;
        if (++j == count) break;
        nx = (uint64_t)ev[j].time;
    }
    *i = j; *now = t; *next = nx;
}

/* A version-2 snapshot's event header at *q (moved past it), checked with the rest of the snapshot up to `end` against
 * the counters: the length, the generator flag, the list as TRMStreamPoolOpenEvents checks it, its frame count and the
 * generator's position.  The track values, deltas and drift state are not checked: they only ever reach the audio. */
static int snap_parse_events(const unsigned char **q, const unsigned char *end, const trm_cuda_pool_slot_state *st,
                             int precision, trm_cuda_pool_event_state *ev)
{
    const unsigned char *h = *q;
    ev->events = 1;
    ev->n_events = (int64_t)get_u64(&h); ev->ev_frames = (int64_t)get_u64(&h);
    ev->fg.useMacroIntonation = (int32_t)get_u32(&h); ev->fg.useMicroIntonation = (int32_t)get_u32(&h);
    ev->fg.useSmoothIntonation = (int32_t)get_u32(&h); ev->fg.useDrift = (int32_t)get_u32(&h);
    ev->fg.driftDeviation = get_f64(&h); ev->fg.driftCutoff = get_f64(&h); ev->fg.pitch = get_f64(&h);
    ev->fg.driftSeed = get_f32(&h); ev->fg.reserved = (int32_t)get_u32(&h);
    const uint32_t generator = get_u32(&h), reserved = get_u32(&h);
    if (ev->fg.reserved != 0 || reserved != 0) return set_err(TRM_ERR_PARAM, "snapshot: reserved event header fields are not 0%s", "");
    if (generator != (st->frames_seen > 0 ? 1u : 0u))
        return set_err(TRM_ERR_PARAM, "snapshot: the generator flag does not agree with the frames generated%s", "");
    const int64_t fixed = trm_cuda_pool_slot_bytes(precision, st), gen = generator ? TRM_FRAMEGEN_STATE_BYTES : 0;
    const int64_t list_bytes = (int64_t)(end - h) - fixed - gen;
    if (ev->n_events < 0 || list_bytes < 0 || list_bytes % (int64_t)sizeof(TRMEvent) != 0 ||
        list_bytes / (int64_t)sizeof(TRMEvent) != ev->n_events)
        return set_err(TRM_ERR_PARAM, "snapshot: length does not match its counters and events%s", "");
    if (ev->ev_frames < 0 || st->frames_seen > ev->ev_frames)
        return set_err(TRM_ERR_PARAM, "snapshot: more frames generated than the event list has%s", "");
    /* the list, aligned for reading (the blob may sit at any offset) */
    TRMEvent *list = malloc((size_t)ev->n_events * sizeof *list + 1);
    if (!list) return set_err(TRM_ERR_NOMEM, "out of memory%s", "");
    memcpy(list, h + fixed + gen, (size_t)ev->n_events * sizeof *list);
    int rc = check_event_list(list, ev->n_events, ev->ev_frames);
    if (rc == TRM_OK && generator) {
        const unsigned char *g = h + fixed + 552;          /* i, now, next after cv[32], cd[32] and tracks 32..35 */
        const int64_t gi = (int64_t)get_u64(&g);
        const uint64_t gnow = get_u64(&g), gnext = get_u64(&g);
        int64_t wi;
        uint64_t wnow, wnext;
        framegen_position(list, ev->n_events, st->frames_seen, &wi, &wnow, &wnext);
        if (gi != wi || gnow != wnow || gnext != wnext)
            rc = set_err(TRM_ERR_PARAM, "snapshot: the generator's position does not agree with the frames generated%s", "");
    }
    free(list);
    *q = h;
    return rc;
}

/* One snapshot, checked as far as it can be without a pool: on success *ip, *d (descriptor, n_frames = 2 as Open builds
 * it), the glottal table row in vs (row d->voice), the counters, the event part (ev->events = 0 for version 1) and a
 * pointer to the data part. */
static int snap_parse(const unsigned char *b, int64_t bytes, voice_set *vs, int *precision, TRMInputParameters *ip,
                      trm_cuda_utterance *d, trm_cuda_pool_slot_state *st, trm_cuda_pool_event_state *ev,
                      const unsigned char **data)
{
    memset(ev, 0, sizeof *ev);
    if (!b || bytes < SNAP_HEADER) return set_err(TRM_ERR_PARAM, "snapshot: shorter than its header%s", "");
    const unsigned char *q = b + 8;
    if (memcmp(b, snap_magic, 8) != 0) return set_err(TRM_ERR_PARAM, "snapshot: not a stream pool snapshot%s", "");
    const uint32_t version = get_u32(&q);
    if (version != SNAP_VERSION && version != SNAP_VERSION_EVENTS) return set_err(TRM_ERR_PARAM, "snapshot: unknown format version%s", "");
    const int64_t fixed = SNAP_FIXED + (version == SNAP_VERSION_EVENTS ? SNAP_EVHEADER : 0);
    const uint32_t prec = get_u32(&q);
    const uint64_t total = get_u64(&q), sum = get_u64(&q);
    if (total != (uint64_t)bytes || bytes < fixed) return set_err(TRM_ERR_PARAM, "snapshot: length does not match%s", "");
    if (fnv1a64(b + SNAP_HEADER, (size_t)bytes - SNAP_HEADER) != sum) return set_err(TRM_ERR_PARAM, "snapshot: checksum mismatch%s", "");
    if (prec > 2u || !precision_ok((int)prec)) return set_err(TRM_ERR_PARAM, "snapshot: unknown precision%s", "");
    *precision = (int)prec;
    get_voice(&q, ip);
    int rc = describe(ip, 2, vs, d, NULL);
    if (rc != TRM_OK) return rc;
    uint32_t want[6];
    snap_derived(d, *precision, want);
    for (int i = 0; i < 6; i++)
        if (get_u32(&q) != want[i])
            return set_err(TRM_ERR_PARAM, "snapshot: derived constants differ from the voice's (another library build?)%s", "");
    st->frames_seen = (int64_t)get_u64(&q); st->s_done = (int64_t)get_u64(&q); st->out_done = (int64_t)get_u64(&q);
    st->in_start = (int64_t)get_u64(&q); st->pend_first = (int64_t)get_u64(&q);
    st->pend_frames = (int32_t)get_u32(&q); st->fresh = (int32_t)get_u32(&q);
    if (trm_cuda_pool_check_state(d, st) != 0) return set_err(TRM_ERR_PARAM, "%s", trm_cuda_last_error());
    if (version == SNAP_VERSION_EVENTS) {
        if ((rc = snap_parse_events(&q, b + bytes, st, *precision, ev)) != TRM_OK) return rc;
    } else if (bytes != SNAP_FIXED + trm_cuda_pool_slot_bytes(*precision, st)) {
        return set_err(TRM_ERR_PARAM, "snapshot: length does not match its counters%s", "");
    }
    *data = q;
    return TRM_OK;
}

/* TRMStreamPoolSave (any_kind = 0: event slots refused) and TRMStreamPoolSaveAny (= 1: they are saved as version 2) */
static int pool_save(TRMStreamPool *t, int n, const int32_t *slot, void *blob, int64_t blob_capacity, int64_t *offset,
                     int any_kind)
{
    if (!t) return set_err(TRM_ERR_PARAM, "null stream pool%s", "");
    if (n < 0 || !offset || (n > 0 && !slot)) return set_err(TRM_ERR_PARAM, "bad snapshot arguments%s", "");
    trm_cuda_pool_slot_state *st = calloc((size_t)n + 1, sizeof *st);
    trm_cuda_pool_event_state *ev = any_kind ? calloc((size_t)n + 1, sizeof *ev) : NULL;
    void **dst = calloc((size_t)n + 1, sizeof *dst);
    voice_set vs;
    memset(&vs, 0, sizeof vs);
    int rc = TRM_OK;
    if (!st || !dst || (any_kind && !ev)) { rc = set_err(TRM_ERR_NOMEM, "out of memory%s", ""); goto done; }
    if ((rc = trm_cuda_pool_save(t->p, n, slot, st, ev, NULL)) != 0) { rc = pool_rc(rc); goto done; }   /* checks the slots */
    offset[0] = 0;
    for (int i = 0; i < n; i++) {
        const int64_t head = SNAP_FIXED + (ev && ev[i].events ? SNAP_EVHEADER + trm_cuda_pool_event_bytes(&st[i], &ev[i]) : 0);
        offset[i + 1] = offset[i] + head + trm_cuda_pool_slot_bytes(t->precision, &st[i]);
    }
    if (!blob) goto done;
    if (blob_capacity < offset[n]) { rc = set_err(TRM_ERR_PARAM, "snapshot buffer too small%s", ""); goto done; }
    unsigned char *base = blob;
    for (int i = 0; i < n; i++) dst[i] = base + offset[i] + SNAP_FIXED + (ev && ev[i].events ? SNAP_EVHEADER : 0);
    if ((rc = trm_cuda_pool_save(t->p, n, slot, st, ev, dst)) != 0) { rc = pool_rc(rc); goto done; }
    for (int i = 0; i < n; i++) {
        const TRMInputParameters *ip = &t->voice[slot[i]];
        trm_cuda_utterance d;
        if ((rc = describe(ip, 2, &vs, &d, NULL)) != TRM_OK) goto done;
        uint32_t dv[6];
        snap_derived(&d, t->precision, dv);
        const int events = ev && ev[i].events;
        unsigned char *b = base + offset[i], *o = b;
        memcpy(o, snap_magic, 8);
        o = put_u32(o + 8, events ? SNAP_VERSION_EVENTS : SNAP_VERSION);
        o = put_u32(o, (uint32_t)t->precision);
        o = put_u64(o, (uint64_t)(offset[i + 1] - offset[i]));
        unsigned char *sum_at = o;
        o = put_voice(o + 8, ip);
        for (int k = 0; k < 6; k++) o = put_u32(o, dv[k]);
        o = put_u64(o, (uint64_t)st[i].frames_seen); o = put_u64(o, (uint64_t)st[i].s_done);
        o = put_u64(o, (uint64_t)st[i].out_done); o = put_u64(o, (uint64_t)st[i].in_start);
        o = put_u64(o, (uint64_t)st[i].pend_first);
        o = put_u32(o, (uint32_t)st[i].pend_frames); o = put_u32(o, (uint32_t)st[i].fresh);
        if (events) put_event_header(o, &ev[i], st[i].frames_seen);
        put_u64(sum_at, fnv1a64(b + SNAP_HEADER, (size_t)(offset[i + 1] - offset[i]) - SNAP_HEADER));
    }
done:
    voice_set_free(&vs);
    free(st);
    free(ev);
    free(dst);
    return rc;
}

int TRMStreamPoolSave(TRMStreamPool *t, int n, const int32_t *slot, void *blob, int64_t blob_capacity, int64_t *offset)
{
    return pool_save(t, n, slot, blob, blob_capacity, offset, 0);
}

int TRMStreamPoolSaveAny(TRMStreamPool *t, int n, const int32_t *slot, void *blob, int64_t blob_capacity, int64_t *offset)
{
    return pool_save(t, n, slot, blob, blob_capacity, offset, 1);
}

int TRMStreamPoolRestore(TRMStreamPool *t, int n, const void *blob, const int64_t *offset, int32_t *slot_out)
{
    if (!t) return set_err(TRM_ERR_PARAM, "null stream pool%s", "");
    if (n < 0 || (n > 0 && (!blob || !offset || !slot_out))) return set_err(TRM_ERR_PARAM, "bad snapshot arguments%s", "");
    if (n == 0) return TRM_OK;
    trm_cuda_pool_slot_state *st = calloc((size_t)n, sizeof *st);
    trm_cuda_pool_event_state *ev = calloc((size_t)n, sizeof *ev);
    trm_cuda_utterance *d = calloc((size_t)n, sizeof *d);
    TRMInputParameters *ip = calloc((size_t)n, sizeof *ip);
    double *tables = malloc((size_t)n * TRM_TABLE_LENGTH * sizeof *tables);
    const void **src = calloc((size_t)n, sizeof *src);
    voice_set vs;
    memset(&vs, 0, sizeof vs);
    int rc = TRM_OK;
    if (!st || !ev || !d || !ip || !tables || !src) { rc = set_err(TRM_ERR_NOMEM, "out of memory%s", ""); goto done; }
    for (int i = 0; i < n; i++) {
        if (offset[i] < 0 || offset[i + 1] < offset[i]) { rc = set_err(TRM_ERR_PARAM, "snapshot offsets are not ascending%s", ""); goto done; }
        int prec;
        const unsigned char *data;
        if ((rc = snap_parse((const unsigned char *)blob + offset[i], offset[i + 1] - offset[i], &vs, &prec, &ip[i], &d[i], &st[i],
                             &ev[i], &data)) != TRM_OK)
            goto done;
        if (prec != t->precision) { rc = set_err(TRM_ERR_PARAM, "snapshot of another precision%s", ""); goto done; }
        src[i] = data;
    }
    /* the table rows are final only now (vs may have grown while parsing) */
    for (int i = 0; i < n; i++)
        memcpy(tables + (size_t)i * TRM_TABLE_LENGTH, vs.tables + (size_t)d[i].voice * TRM_TABLE_LENGTH, TRM_TABLE_LENGTH * sizeof *tables);
    if ((rc = trm_cuda_pool_restore(t->p, n, d, tables, st, ev, (const void *const *)src, slot_out)) != 0) { rc = pool_rc(rc); goto done; }
    for (int i = 0; i < n; i++) t->voice[slot_out[i]] = ip[i];
done:
    voice_set_free(&vs);
    free(st); free(ev); free(d); free(ip); free(tables); free(src);
    return rc;
}

/* a snapshot parsed as Restore parses it, no pool needed */
static int snap_read(const void *blob, int64_t bytes, int *prec, TRMInputParameters *ip, trm_cuda_utterance *d,
                     trm_cuda_pool_slot_state *st, trm_cuda_pool_event_state *ev)
{
    voice_set vs;
    memset(&vs, 0, sizeof vs);
    const unsigned char *data;
    const int rc = snap_parse(blob, bytes, &vs, prec, ip, d, st, ev, &data);
    voice_set_free(&vs);
    return rc;
}

int TRMStreamPoolSnapshotInfo(const void *blob, int64_t bytes, TRMStreamSnapshotInfo *info)
{
    if (!blob || !info) return set_err(TRM_ERR_PARAM, "null snapshot or info%s", "");
    int prec;
    TRMInputParameters ip;
    trm_cuda_utterance d;
    trm_cuda_pool_slot_state st;
    trm_cuda_pool_event_state ev;
    const int rc = snap_read(blob, bytes, &prec, &ip, &d, &st, &ev);
    if (rc != TRM_OK) return rc;
    memset(info, 0, sizeof *info);
    info->precision = prec;
    info->channels = d.channels;
    info->voice = ip;
    info->frames_pushed = st.frames_seen;
    info->samples_returned = st.out_done;
    info->bytes = bytes;
    return TRM_OK;
}

int TRMStreamPoolSnapshotEventInfo(const void *blob, int64_t bytes, TRMStreamSnapshotEventInfo *info)
{
    if (!blob || !info) return set_err(TRM_ERR_PARAM, "null snapshot or info%s", "");
    int prec;
    TRMInputParameters ip;
    trm_cuda_utterance d;
    trm_cuda_pool_slot_state st;
    trm_cuda_pool_event_state ev;
    const int rc = snap_read(blob, bytes, &prec, &ip, &d, &st, &ev);
    if (rc != TRM_OK) return rc;
    memset(info, 0, sizeof *info);
    if (!ev.events) return TRM_OK;
    info->from_events = 1;
    info->n_events = ev.n_events;
    info->list_frames = ev.ev_frames;
    info->frames_generated = st.frames_seen;
    memcpy(&info->fg, &ev.fg, sizeof info->fg);
    return TRM_OK;
}

/* ---- voice changes (TRMStreamPoolSetVoice, TRMStreamSetVoice) ---- */
/* Entry i moves slot[i] of pool p from the voice *cur[i] to voice[shared ? 0 : i].  cur[i] is NULL for a slot number
 * outside the pool (the shim refuses it).  Only on success does *cur[i] become the new voice. */
static int pool_set_voice(trm_cuda_pool *p, int n, const int32_t *slot, TRMInputParameters *const *cur,
                          const TRMInputParameters *voice, int shared, int64_t *tube_sample, int64_t *output_sample)
{
    trm_cuda_utterance *d = calloc((size_t)n + 1, sizeof *d);
    double *tables = malloc(((size_t)n + 1) * TRM_TABLE_LENGTH * sizeof *tables);
    voice_set vs;
    memset(&vs, 0, sizeof vs);
    int rc = TRM_OK;
    if (!d || !tables) { rc = set_err(TRM_ERR_NOMEM, "out of memory%s", ""); goto done; }
    for (int i = 0; i < n; i++) {
        if ((rc = describe(&voice[shared ? 0 : i], 2, &vs, &d[i], NULL)) != TRM_OK) goto done;
        /* an open slot's voice always describes (it was checked when the slot opened); an unopened slot's does not, and
         * the shim refuses the slot */
        trm_cuda_utterance now;
        if (cur[i] && describe(cur[i], 2, &vs, &now, NULL) == TRM_OK) {
            uint32_t want[6], got[6];
            snap_derived(&now, TRM_PRECISION_FP64, want);
            snap_derived(&d[i], TRM_PRECISION_FP64, got);
            if (memcmp(want, got, sizeof want) != 0) {
                rc = set_err(TRM_ERR_PARAM, "the new voice's rate constants (control period, sample rate, converter, channels) "
                                            "differ from the stream's: a new tract length, temperature or rate is a new stream%s", "");
                goto done;
            }
        }
    }
    /* the table rows are final only now (vs may have grown while describing) */
    for (int i = 0; i < n; i++)
        memcpy(tables + (size_t)i * TRM_TABLE_LENGTH, vs.tables + (size_t)d[i].voice * TRM_TABLE_LENGTH, TRM_TABLE_LENGTH * sizeof *tables);
    if ((rc = trm_cuda_pool_set_voice(p, n, slot, d, tables, tube_sample, output_sample)) != 0) { rc = pool_rc(rc); goto done; }
    for (int i = 0; i < n; i++) *cur[i] = voice[shared ? 0 : i];
done:
    voice_set_free(&vs);
    free(d);
    free(tables);
    return rc;
}

int TRMStreamPoolSetVoice(TRMStreamPool *t, int n, const int32_t *slot, const TRMInputParameters *voice, int64_t *tube_sample,
                          int64_t *output_sample)
{
    if (!t) return set_err(TRM_ERR_PARAM, "null stream pool%s", "");
    if (n < 0 || n > t->capacity || (n > 0 && (!slot || !voice))) return set_err(TRM_ERR_PARAM, "bad voice change arguments%s", "");
    TRMInputParameters **cur = calloc((size_t)n + 1, sizeof *cur);
    if (!cur) return set_err(TRM_ERR_NOMEM, "out of memory%s", "");
    for (int i = 0; i < n; i++) cur[i] = slot[i] >= 0 && slot[i] < t->capacity ? &t->voice[slot[i]] : NULL;
    const int rc = pool_set_voice(t->p, n, slot, cur, voice, 0, tube_sample, output_sample);
    free(cur);
    return rc;
}

int TRMStreamSetVoice(TRMStream *t, const TRMInputParameters *voice, int64_t *tube_sample, int64_t *output_sample)
{
    if (!t || !voice) return set_err(TRM_ERR_PARAM, "null stream or voice%s", "");
    if (t->flushed) return set_err(TRM_ERR_STATE, "the streams were flushed%s", "");
    TRMInputParameters **cur = calloc((size_t)t->n, sizeof *cur);
    int64_t *ts = calloc((size_t)t->n, sizeof *ts), *os = calloc((size_t)t->n, sizeof *os);
    int rc = TRM_OK;
    if (!cur || !ts || !os) rc = set_err(TRM_ERR_NOMEM, "out of memory%s", "");
    for (int i = 0; rc == TRM_OK && i < t->n; i++) cur[i] = &t->voice;
    if (rc == TRM_OK) rc = pool_set_voice(t->p, t->n, t->slot, cur, voice, 1, ts, os);
    /* the streams advance in lockstep: every one is at the same sample */
    if (rc == TRM_OK && tube_sample) *tube_sample = ts[0];
    if (rc == TRM_OK && output_sample) *output_sample = os[0];
    free(cur); free(ts); free(os);
    return rc;
}

/* ---- asynchronous calls: one host thread per ticket; two tickets per device overlap (context lanes) ---- */
struct TRMBatchTicket {
    pthread_t th;
    TRMBatch *b;
    const TRMParameters *frames;
    int16_t *pcm;
    void *samples;
    int devices[MAX_DEVICES], n_devices, has_devices;
    int rc;
    char msg[512];
    order_gate gate;
    int inline_run;
};

static double host_ms(void)
{
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return 1e3 * (double)ts.tv_sec + 1e-6 * (double)ts.tv_nsec;
}

static void *ticket_main(void *arg)
{
    TRMBatchTicket *t = arg;
    pthread_mutex_lock(&g_order_mu);
    while (g_order_turn != t->gate.seq) pthread_cond_wait(&g_order_cv, &g_order_mu);
    pthread_mutex_unlock(&g_order_mu);
    t->rc = batch_run(t->b, t->frames, t->pcm, t->samples, NULL, t->has_devices ? t->devices : NULL, t->n_devices, &t->gate);
    gate_pass(&t->gate);          /* (empty batches and error paths never reached the queues) */
    if (t->rc) snprintf(t->msg, sizeof t->msg, "%s", g_errmsg);
    if (getenv("TRM_TRACE")) fprintf(stderr, "[trm trace] ticket %p: thread returns at %.2f (CLOCK_MONOTONIC ms)\n", (void *)t, host_ms());
    return NULL;
}

TRMBatchTicket *TRMBatchSynthesizeAsync(TRMBatch *b, const TRMParameters *frames, int16_t *pcm_out, void *samples_out,
                                        const int *devices, int n_devices, int *err)
{
    int dummy;
    if (!err) err = &dummy;
    TRMBatchTicket *t = calloc(1, sizeof *t);
    if (!t) { *err = set_err(TRM_ERR_NOMEM, "out of memory%s", ""); return NULL; }
    t->b = b; t->frames = frames; t->pcm = pcm_out; t->samples = samples_out;
    t->n_devices = n_devices > MAX_DEVICES ? MAX_DEVICES : n_devices;
    t->has_devices = devices != NULL;
    for (int k = 0; devices && k < t->n_devices; k++) t->devices[k] = devices[k];
    pthread_mutex_lock(&g_order_mu);
    t->gate.seq = g_order_next++;
    pthread_mutex_unlock(&g_order_mu);
    if (pthread_create(&t->th, NULL, ticket_main, t) != 0) {
        t->inline_run = 1;        /* no thread: the call runs here, in its turn, and the ticket is complete on return */
        ticket_main(t);
    }
    *err = TRM_OK;
    return t;
}

int TRMBatchWait(TRMBatchTicket *t)
{
    if (!t) return set_err(TRM_ERR_PARAM, "null ticket%s", "");
    const double t0 = getenv("TRM_TRACE") ? host_ms() : 0.0;
    if (!t->inline_run) pthread_join(t->th, NULL);
    if (getenv("TRM_TRACE")) fprintf(stderr, "[trm trace] ticket %p: wait entered %.2f, joined %.2f\n", (void *)t, t0, host_ms());
    const int rc = t->rc;
    if (rc) snprintf(g_errmsg, sizeof g_errmsg, "%s", t->msg);
    free(t);
    return rc;
}

/* like TRMBatchSynthesize, additionally returning the tube-rate signal (TRMBatchTubeElements() elements) */
int TRMBatchSynthesizeDebug(TRMBatch *b, const TRMParameters *frames, int16_t *pcm_out, void *samples_out,
                            void *tube_out, int device)
{
    return batch_run(b, frames, pcm_out, samples_out, tube_out, &device, 1, NULL);
}

/* ---- device-resident batches (bench `value`, per-stage timing) ---- */
typedef struct TRMResident {
    trm_cuda_resident *res;
    int device;
} TRMResident;

TRMResident *TRMBatchMakeResident(TRMBatch *b, const TRMParameters *frames, int device, int *err)
{
    int dummy;
    if (!err) err = &dummy;
    trm_cuda_ctx *ctx;
    int lane = 0;
    if ((*err = acquire_ctx(device, &ctx, &lane)) != TRM_OK) return NULL;
    TRMResident *r = calloc(1, sizeof *r);
    if (!r) { release_ctx(device, lane); *err = set_err(TRM_ERR_NOMEM, "out of memory%s", ""); return NULL; }
    r->device = device;
    if (trm_cuda_set_wavetables(ctx, b->voices.tables, b->voices.n) != 0 ||
        trm_cuda_resident_create(ctx, b->precision, b->n, b->desc, (const double *)frames, &r->res) != 0) {
        *err = cuda_err();
        free(r);
        r = NULL;
    } else
        *err = TRM_OK;
    release_ctx(device, lane);
    return r;
}
int TRMResidentRunStage(TRMResident *r, int stage, void *cuda_stream)
{
    return trm_cuda_resident_stage(r->res, stage, cuda_stream) ? cuda_err() : TRM_OK;
}
int TRMResidentRun(TRMResident *r, void *cuda_stream) { return trm_cuda_resident_run(r->res, cuda_stream) ? cuda_err() : TRM_OK; }
int TRMResidentFetchUtterance(TRMResident *r, int u, void *samples, int16_t *pcm, double *maximum)
{
    return trm_cuda_resident_fetch_utterance(r->res, u, samples, pcm, maximum) ? cuda_err() : TRM_OK;
}
int TRMCopyProbe(int device, const void *host_in, size_t h2d_bytes, void *host_out, size_t d2h_bytes, int reps, double *ms)
{
    return trm_cuda_copy_probe(device, host_in, h2d_bytes, host_out, d2h_bytes, reps, ms) ? cuda_err() : TRM_OK;
}
int TRMResidentFetch(TRMResident *r, int16_t *pcm, void *samples, double *maxima, void *tube)
{
    return trm_cuda_resident_fetch(r->res, pcm, samples, maxima, tube) ? cuda_err() : TRM_OK;
}
void TRMResidentFree(TRMResident *r)
{
    if (!r) return;
    trm_cuda_resident_destroy(r->res);
    free(r);
}

/* ------------------------------------------------------------------------------------------------
 * TRMTubeModel
 * ---------------------------------------------------------------------------------------------- */
struct TRMTubeModel {
    TRMInputParameters ip;
    TRMParameters *frames;
    size_t n_frames;
    int precision, device, done;
    TRMDerivedValues derived;
    double *resampled, *tube;
    int16_t *pcm;             /* device-scaled PCM (WAV variant) */
    int32_t numberSamples;
    double maximum;
};

TRMTubeModel *TRMTubeModelCreate(const TRMDataList *in, int *err)
{
    int dummy;
    if (!err) err = &dummy;
    TRMDerivedValues dv;
    if ((*err = TRMDeriveValues(&in->ip, in->count, &dv)) != TRM_OK) {
        if (*err == TRM_ERR_TUBE_LENGTH) fprintf(stderr, "Illegal tube length: %g\n", in->ip.length);   /* m:205 */
        return NULL;
    }
    /* validate everything else now, as -initWithInputData: builds the wavetable / filters up front */
    voice_set vs;
    memset(&vs, 0, sizeof vs);
    trm_cuda_utterance d;
    *err = describe(&in->ip, (int32_t)in->count, &vs, &d, NULL);
    voice_set_free(&vs);
    if (*err) return NULL;
    TRMTubeModel *m = calloc(1, sizeof *m);
    if (!m) { *err = set_err(TRM_ERR_NOMEM, "out of memory%s", ""); return NULL; }
    m->ip = in->ip;
    m->n_frames = in->count;
    m->derived = dv;
    if (in->count) {
        m->frames = malloc(in->count * sizeof *m->frames);
        if (!m->frames) { free(m); *err = set_err(TRM_ERR_NOMEM, "out of memory%s", ""); return NULL; }
        memcpy(m->frames, in->values, in->count * sizeof *m->frames);
    }
    *err = TRM_OK;
    return m;
}

void TRMTubeModelFree(TRMTubeModel *m)
{
    if (!m) return;
    free(m->frames); free(m->resampled); free(m->tube); free(m->pcm);
    free(m);
}

int TRMTubeModelSetPrecision(TRMTubeModel *m, int precision)
{
    if (!precision_ok(precision)) return set_err(TRM_ERR_PARAM, "bad precision%s", "");
    m->precision = precision;
    return TRM_OK;
}
int TRMTubeModelSetDevice(TRMTubeModel *m, int device) { m->device = device; return TRM_OK; }
void TRMTubeModelGetDerivedValues(const TRMTubeModel *m, TRMDerivedValues *out) { *out = m->derived; }

int TRMTubeModelSynthesize(TRMTubeModel *m)
{
    if (m->done) return set_err(TRM_ERR_STATE, "a TRMTubeModel is single-use%s", "");
    m->done = 1;
    if (m->n_frames == 0) return TRM_OK;                 /* no data: returns without flushing (m:274-277) */
    int err;
    const int64_t off = 0;
    const int32_t nf = (int32_t)m->n_frames;
    TRMBatch *b = TRMBatchCreate(1, &m->ip, 1, &off, &nf, m->precision, &err);
    if (!b) return err;
    const size_t n_out = (size_t)b->layout.total_out_samples, n_pcm = (size_t)b->layout.total_pcm_samples;
    const size_t n_tube = (size_t)b->total_tube_elems;
    const size_t esz = m->precision != TRM_PRECISION_FP32 ? sizeof(double) : sizeof(float);
    void *samples = malloc((n_out ? n_out : 1) * esz), *tube = malloc((n_tube ? n_tube : 1) * esz);
    m->pcm = malloc((n_pcm ? n_pcm : 1) * sizeof(int16_t));
    m->resampled = malloc((n_out ? n_out : 1) * sizeof(double));
    m->tube = malloc((n_tube ? n_tube : 1) * sizeof(double));
    if (!samples || !tube || !m->pcm || !m->resampled || !m->tube) {
        free(samples); free(tube); TRMBatchFree(b);
        return set_err(TRM_ERR_NOMEM, "out of memory%s", "");
    }
    err = TRMBatchSynthesizeDebug(b, m->frames, m->pcm, samples, tube, m->device);
    if (err == TRM_OK) {
        m->numberSamples = b->numberSamples[0];
        m->maximum = b->maxima[0];
        if (m->precision != TRM_PRECISION_FP32) {
            memcpy(m->resampled, samples, (size_t)m->numberSamples * sizeof(double));
            memcpy(m->tube, tube, (size_t)b->desc[0].n_tube * sizeof(double));
        } else {
            for (int32_t i = 0; i < m->numberSamples; i++) m->resampled[i] = ((float *)samples)[i];
            for (int64_t i = 0; i < b->desc[0].n_tube; i++) m->tube[i] = ((float *)tube)[i];
        }
    }
    free(samples); free(tube);
    TRMBatchFree(b);
    return err;
}

int32_t TRMTubeModelNumberSamples(const TRMTubeModel *m) { return m->numberSamples; }
int32_t TRMTubeModelChannels(const TRMTubeModel *m) { return m->ip.channels == 2 ? 2 : 1; }
int TRMTubeModelHitsReferenceFlushBug(const TRMTubeModel *m) { return TRMReferenceFlushBug(&m->ip, m->n_frames); }
double TRMTubeModelMaximumSampleValue(const TRMTubeModel *m) { return m->maximum; }
const double *TRMTubeModelResampledData(const TRMTubeModel *m) { return m->resampled; }
const double *TRMTubeModelTubeSignal(const TRMTubeModel *m, int64_t *count)
{
    if (count) *count = m->done ? m->derived.tubeSamples : 0;
    return m->tube;
}

int64_t TRMTubeModelPullPCM16(const TRMTubeModel *m, int16_t *dst, size_t max_frames, int file_variant)
{
    if (!m->done) return set_err(TRM_ERR_STATE, "pull before synthesize%s", "");
    size_t n = (size_t)m->numberSamples;
    if (n > max_frames) n = max_frames;
    const int ch = m->ip.channels == 2 ? 2 : 1;
    if (!(file_variant && ch == 2)) {
        if (n) memcpy(dst, m->pcm, n * ch * sizeof(int16_t));          /* scaled on the GPU (m:515-557) */
        return (int64_t)n;
    }
    /* -saveOutputToFile: stereo scaling carries an extra factor 2 (m:382-383) */
    const double scale = (32767.0 / m->maximum) * db_to_amplitude(m->ip.volume);
    const double ls = -((m->ip.balance / 2.0) - 0.5) * scale * 2.0, rs = ((m->ip.balance / 2.0) + 0.5) * scale * 2.0;
    for (size_t i = 0; i < n; i++) {
        dst[2 * i] = (int16_t)rint(m->resampled[i] * ls);
        dst[2 * i + 1] = (int16_t)rint(m->resampled[i] * rs);
    }
    return (int64_t)n;
}

static void wr_le16(uint8_t **p, uint16_t v) { (*p)[0] = (uint8_t)v; (*p)[1] = (uint8_t)(v >> 8); *p += 2; }
static void wr_le32(uint8_t **p, uint32_t v) { wr_le16(p, (uint16_t)v); wr_le16(p, (uint16_t)(v >> 16)); }
static void wr_be16(uint8_t **p, uint16_t v) { (*p)[0] = (uint8_t)(v >> 8); (*p)[1] = (uint8_t)v; *p += 2; }
static void wr_be32(uint8_t **p, uint32_t v) { wr_be16(p, (uint16_t)(v >> 16)); wr_be16(p, (uint16_t)v); }

uint8_t *TRMTubeModelGenerateWAVData(const TRMTubeModel *m, size_t *length, int *err)
{
    int dummy;
    if (!err) err = &dummy;
    if (!m->done) { *err = set_err(TRM_ERR_STATE, "generateWAVData before synthesize%s", ""); return NULL; }
    if (m->maximum == 0) { *err = set_err(TRM_ERR_SILENT, "maximumSampleValue is 0%s", ""); return NULL; }   /* m:511 */
    const int ch = m->ip.channels == 2 ? 2 : 1;
    const size_t data_bytes = (size_t)m->numberSamples * ch * 2;
    uint8_t *buf = malloc(46 + data_bytes), *p = buf;
    if (!buf) { *err = set_err(TRM_ERR_NOMEM, "out of memory%s", ""); return NULL; }
    /* m:562-590: RIFF / WAVE / "fmt " with an 18-byte chunk (extra cbSize = 0) / data */
    const int frameSize = (int)ceil(m->ip.channels * ((double)16 / 8));
    const int bytesPerSecond = (int)ceil(m->ip.outputRate * frameSize);
    wr_be32(&p, 0x52494646u); wr_le32(&p, (uint32_t)(4 + (8 + 18) + (8 + data_bytes))); wr_be32(&p, 0x57415645u);
    wr_be32(&p, 0x666d7420u); wr_le32(&p, 18); wr_le16(&p, 1); wr_le16(&p, (uint16_t)m->ip.channels);
    wr_le32(&p, (uint32_t)m->ip.outputRate); wr_le32(&p, (uint32_t)bytesPerSecond);
    wr_le16(&p, (uint16_t)frameSize); wr_le16(&p, 16); wr_le16(&p, 0);
    wr_be32(&p, 0x64617461u); wr_le32(&p, (uint32_t)data_bytes);
    for (size_t i = 0; i < data_bytes / 2; i++) wr_le16(&p, (uint16_t)m->pcm[i]);
    *length = 46 + data_bytes;
    *err = TRM_OK;
    return buf;
}

/* 80-bit IEEE extended for the AIFF COMM chunk */
static void wr_ext80(uint8_t **p, double v)
{
    int e;
    double f = frexp(v, &e);                 /* v = f * 2^e, f in [0.5,1) */
    uint64_t mant = (uint64_t)ldexp(f, 64);
    wr_be16(p, (uint16_t)(e - 1 + 16383));
    wr_be32(p, (uint32_t)(mant >> 32));
    wr_be32(p, (uint32_t)mant);
}

int TRMTubeModelSaveOutputToFile(const TRMTubeModel *m, const char *path)
{
    if (!m->done) return set_err(TRM_ERR_STATE, "saveOutputToFile before synthesize%s", "");
    const int ch = m->ip.channels == 2 ? 2 : 1;
    const size_t n = (size_t)m->numberSamples, data_bytes = n * ch * 2;
    int16_t *pcm = malloc(data_bytes ? data_bytes : 2);
    if (!pcm) return set_err(TRM_ERR_NOMEM, "out of memory%s", "");
    TRMTubeModelPullPCM16(m, pcm, n, 1);
    uint8_t hdr[64], *p = hdr;
    const int fmt = m->ip.outputFileFormat;
    const uint32_t rate = (uint32_t)m->ip.outputRate;
    if (fmt == TRMSoundFileFormat_WAVE) {
        wr_be32(&p, 0x52494646u); wr_le32(&p, (uint32_t)(36 + data_bytes)); wr_be32(&p, 0x57415645u);
        wr_be32(&p, 0x666d7420u); wr_le32(&p, 16); wr_le16(&p, 1); wr_le16(&p, (uint16_t)ch);
        wr_le32(&p, rate); wr_le32(&p, rate * 2u * ch); wr_le16(&p, (uint16_t)(2 * ch)); wr_le16(&p, 16);
        wr_be32(&p, 0x64617461u); wr_le32(&p, (uint32_t)data_bytes);
    } else if (fmt == TRMSoundFileFormat_AIFF) {
        wr_be32(&p, 0x464f524du); wr_be32(&p, (uint32_t)(4 + 26 + 16 + data_bytes)); wr_be32(&p, 0x41494646u);
        wr_be32(&p, 0x434f4d4du); wr_be32(&p, 18); wr_be16(&p, (uint16_t)ch); wr_be32(&p, (uint32_t)n); wr_be16(&p, 16);
        wr_ext80(&p, (double)m->ip.outputRate);
        wr_be32(&p, 0x53534e44u); wr_be32(&p, (uint32_t)(8 + data_bytes)); wr_be32(&p, 0); wr_be32(&p, 0);
    } else if (fmt == TRMSoundFileFormat_AU) {
        wr_be32(&p, 0x2e736e64u); wr_be32(&p, 24); wr_be32(&p, (uint32_t)data_bytes); wr_be32(&p, 3);
        wr_be32(&p, rate); wr_be32(&p, (uint32_t)ch);
    } else {
        free(pcm);
        return set_err(TRM_ERR_PARAM, "unknown output file format%s", "");
    }
    FILE *fp = fopen(path, "wb");
    if (!fp) { free(pcm); return set_err(TRM_ERR_IO, "Can't open output file \"%s\".", path); }
    int ok = fwrite(hdr, 1, (size_t)(p - hdr), fp) == (size_t)(p - hdr);
    if (fmt != TRMSoundFileFormat_WAVE) {             /* AU / AIFF are big-endian (m:410-412) */
        uint8_t *b = (uint8_t *)pcm;
        for (size_t i = 0; i < data_bytes; i += 2) { uint8_t t = b[i]; b[i] = b[i + 1]; b[i + 1] = t; }
    }
    ok = ok && fwrite(pcm, 1, data_bytes, fp) == data_bytes;
    ok = (fclose(fp) == 0) && ok;
    free(pcm);
    return ok ? TRM_OK : set_err(TRM_ERR_IO, "write error on \"%s\"", path);
}
