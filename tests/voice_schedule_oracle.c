/*
 * voice_schedule_oracle.c -- TEST INFRASTRUCTURE: the CPU oracle (oracle/trm_oracle.c) with a voice schedule, the
 * checker of TRMStreamPoolSetVoice / TRMStreamSetVoice (a stream whose voice changes while it plays).
 *
 * The oracle is included as it stands and extended here, in its own translation unit and library (built by
 * tests/voice_schedule.py into a temporary directory), so that the oracle itself is not changed: its static helpers are
 * reused and oracle_synthesize's loop is restated with one addition, the voice change.
 */
#include "trm_oracle.c"

int oracle_synthesize_voices(const oracle_input_parameters *ip, int n_voices, const int64_t *from_sample,
                             const oracle_frame *frames, size_t n_frames, int flags, double *tube_out, double **out,
                             oracle_result_info *info);

/* A voice change between two tube-rate samples: everything tube_init derives from the voice is derived again from `ip`,
 * which has the same rate constants; every state variable is kept (oscillator position and FIR history, noise,
 * band-pass, reflection / radiation and throat memories, waves, parameter interpolation, converter). */
static void tube_revoice(tube_t *t, const oracle_input_parameters *ip)
{
    t->ip = ip;
    const double nyquist = (double)t->sampleRate / 2.0;
    t->breathinessFactor = ip->breathiness / 100.0;
    t->crossmixFactor = 1.0 / oracle_amplitude(ip->mixOffset);
    t->dampingFactor = (1.0 - (ip->lossFactor / 100.0));
    /* the glottal table and its shape; wavetable_init also resets the position and the FIR filter, which are kept
     * (the FIR design it repeats depends on nothing of the voice) */
    const fir_t fir = t->wt.fir;
    const double position = t->wt.position;
    wavetable_init(&t->wt, ip->waveform, ip->tp, ip->tnMin, ip->tnMax, t->sampleRate, t->wt.analytic);
    t->wt.fir = fir;
    t->wt.position = position;
    /* radiation / reflection coefficients; radrefl_init also zeroes the memories, which are kept */
    const radrefl_t mouth = t->mouth, nose = t->nasalPair;
    radrefl_init(&t->mouth, (nyquist - ip->mouthCoef) / nyquist);
    radrefl_init(&t->nasalPair, (nyquist - ip->noseCoef) / nyquist);
    t->mouth.reflY = mouth.reflY; t->mouth.radX = mouth.radX; t->mouth.radY = mouth.radY;
    t->nasalPair.reflY = nose.reflY; t->nasalPair.radX = nose.radX; t->nasalPair.radY = nose.radY;
    initialize_nasal_cavity(t);
    t->ta0 = (ip->throatCutoff * 2.0) / t->sampleRate;
    t->tb1 = 1.0 - t->ta0;
    t->throatGain = oracle_amplitude(ip->throatVol);
}

/* tube_synthesize (TRMTubeModel.m:272-361) with voice k of ip[0 .. n_voices) from tube-rate sample from_sample[k] on
 * (voice 0 is the one tube_init was given): the same statements, and the change before the sample is computed. */
static void tube_synthesize_voices(tube_t *t, const oracle_input_parameters *ip, int n_voices, const int64_t *from_sample,
                                   const oracle_frame *frames, size_t n_frames, int flags, double *tube_out, int64_t *n_tube)
{
    int next_voice = 1;
    *n_tube = 0;
    if (n_frames == 0) return;
    const int stateless = (flags & ORACLE_SRC_STATELESS) != 0;
    double *xs = NULL;
    int64_t total = (int64_t)(n_frames - 1) * t->controlPeriod;
    if (stateless) xs = (double *)malloc((size_t)(total > 0 ? total : 1) * sizeof(double));

    for (size_t fi = 1; fi < n_frames; fi++) {
        const double *prev = frames[fi - 1].v, *next = frames[fi].v;
        for (int q = 0; q < 16; q++) {
            t->current[q] = prev[q];
            t->delta[q] = (next[q] - t->current[q]) / (double)t->controlPeriod;
        }
        for (int32_t j = 0; j < t->controlPeriod; j++) {
            while (next_voice < n_voices && from_sample[next_voice] == *n_tube) tube_revoice(t, &ip[next_voice++]);
            double f0 = oracle_frequency(t->current[P_PITCH]);
            double ax = oracle_amplitude(t->current[P_GLOTVOL]);
            double ah1 = oracle_amplitude(t->current[P_ASPVOL]);
            calculate_tube_coefficients(t);
            set_frication_taps(t);
            bandpass_coefficients(&t->bp, t->sampleRate, t->current[P_FRICCF], t->current[P_FRICBW]);

            double nz = noise_next(&t->noiseSeed);
            double lp_noise = nz + t->noiseFilterX;
            t->noiseFilterX = nz;

            if (t->ip->waveform == 0) wavetable_update(&t->wt, ax);
            double pulse = wavetable_oscillator(&t->wt, f0);
            double pulsed_noise = lp_noise * pulse;
            pulse = ax * ((pulse * (1.0 - t->breathinessFactor)) + (pulsed_noise * t->breathinessFactor));
            double signal;
            if (t->ip->usesModulation) {
                double crossmix = ax * t->crossmixFactor;
                crossmix = (crossmix < 1.0) ? crossmix : 1.0;
                signal = (pulsed_noise * crossmix) + (lp_noise * (1.0 - crossmix));
            } else
                signal = lp_noise;

            signal = update_vocal_tract(t, ((pulse + (ah1 * signal)) * VT_SCALE), bandpass_filter(&t->bp, signal));

            t->throatY = (t->ta0 * (pulse * VT_SCALE)) + (t->tb1 * t->throatY);
            signal += t->throatY * t->throatGain;

            if (tube_out) tube_out[*n_tube] = signal;
            if (stateless) xs[*n_tube] = signal;
            else src_data_fill(&t->src, signal);
            (*n_tube)++;

            for (int q = 0; q < 16; q++) t->current[q] += t->delta[q];
        }
    }
    if (stateless) {
        src_stateless(&t->src, xs, *n_tube);
        free(xs);
    } else
        src_flush(&t->src);
}

/* oracle_synthesize with a voice schedule: voice ip[k] applies from tube-rate sample from_sample[k] on
 * (from_sample[0] == 0, non-decreasing).  -4 for a bad schedule or voices whose rate constants (control period, sample
 * rate, converter increment and pad, channels) differ; n_voices == 1 gives oracle_synthesize's results bit for bit. */
int oracle_synthesize_voices(const oracle_input_parameters *ip, int n_voices, const int64_t *from_sample,
                             const oracle_frame *frames, size_t n_frames, int flags, double *tube_out, double **out,
                             oracle_result_info *info)
{
    if (n_voices < 1 || from_sample[0] != 0) return -4;
    for (int k = 1; k < n_voices; k++) {
        if (from_sample[k] < from_sample[k - 1]) return -4;
        oracle_result_info a, b;
        int rc = oracle_derive(&ip[0], 0, &a);
        if (rc == 0) rc = oracle_derive(&ip[k], 0, &b);
        if (rc) return rc;
        if (a.controlPeriod != b.controlPeriod || a.sampleRate != b.sampleRate || a.padSize != b.padSize ||
            a.timeRegisterIncrement != b.timeRegisterIncrement || ip[0].channels != ip[k].channels)
            return -4;
    }
    tube_t *t = (tube_t *)malloc(sizeof(tube_t));
    if (!t) return -3;
    int rc = tube_init(t, ip, flags);
    if (rc) { free(t->src.out); free(t); return rc; }
    int64_t n_tube = 0;
    tube_synthesize_voices(t, ip, n_voices, from_sample, frames, n_frames, flags, tube_out, &n_tube);
    if (t->src.oom) { free(t->src.out); free(t); return -3; }
    if (info) {
        memset(info, 0, sizeof(*info));
        info->controlPeriod = t->controlPeriod;
        info->sampleRate = t->sampleRate;
        info->actualTubeLength = t->actualTubeLength;
        info->numberTaps = t->wt.fir.taps;
        info->padSize = t->src.padSize;
        info->timeRegisterIncrement = t->src.timeRegisterIncrement;
        info->numberSamples = t->src.numberSamples;
        info->maximumSampleValue = t->src.maximumSampleValue;
        info->finalNoiseSeed = t->noiseSeed;
        info->tubeSamples = n_tube;
    }
    if (out) *out = t->src.out;
    else free(t->src.out);
    free(t);
    return 0;
}
