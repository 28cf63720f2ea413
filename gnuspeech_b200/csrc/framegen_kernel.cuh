// framegen_kernel.cuh -- control-frame generator on the device (SURVEY.md 8(f) rank 1).
//
// Replaces -[EventList generateOutputInTimeRange:forSynthesizer:parameterLogger:]
// (/root/reference/Frameworks/GnuSpeech/MonetModel/EventList.m:883-1061, full time range) and MMDriftGenerator
// (MMDriftGenerator.m:41-78): piece-wise linear interpolation of the 33 event tracks to 4 ms frames by repeated
// adds, micro / macro / smooth intonation sums, float rounding of the output table, drift (float MCG x 377 + one-pole
// low-pass).  The frames are written where the waveguide kernel reads them: a batch then needs only its sparse event
// lists uploaded (a few hundred bytes per event) instead of 128 B per 4 ms frame.
//
// One warp per utterance, lane j = event-track index j (0..31); tracks 32..35 (macro / smooth intonation) are
// carried redundantly by every lane.  The loop over frames is sequential, as in the reference; all control flow is
// warp-uniform except the per-track searches for the next non-NaN event value.  Arithmetic in the reference's
// order and types (double tracks, float table and drift; this TU is compiled with -fmad=false).
//
// The generator is a state (FrameGen) with a set-up (framegen_setup, m:919-961) and a step that emits one frame and
// advances (framegen_step, m:973-1057).  framegen_kernel runs set-up and every step of whole utterances;
// framegen_pool_kernel runs a stream pool slot's steps a push at a time, its state kept in memory between pushes.
#pragma once

#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "kernel_args.h"
#include "trm_cuda.h"

namespace trm {

// One warp's generator.  cv / cd are lane j's track j (0..15 the parameters, 16..31 the "special" offsets, which change
// at event boundaries); everything else is the same in every lane.
struct FrameGen {
    double cv, cd;                                  // currentValues[lane], currentDeltas[lane]
    double cv32, cd32, cd33, cd34, cd35;            // tracks 32..35
    long long i;                                    // current event
    unsigned long long now, next;                   // clock (ms) and the time of event i
    float seed, prev;                               // drift generator: MCG state, low-pass memory
    float pitchDeviation, pitchOffset, a0, b1;      // drift constants
};

// first values and deltas, drift constants (m:919-961; MMDriftGenerator.m:41-58).  count >= 2.
__device__ __forceinline__ void framegen_setup(FrameGen &g, const trm_cuda_event *__restrict__ ev, long long count,
                                               const trm_cuda_framegen &fg, int lane)
{
    const double ms = 1000.0 / 250.0;
    g.seed = fg.driftSeed;
    g.pitchDeviation = 0.0f; g.pitchOffset = 0.0f; g.a0 = 0.0f; g.b1 = 0.0f; g.prev = 0.0f;
    if (fg.useDrift) {
        const float deviation = (float)fg.driftDeviation, sampleRate = (float)(1000 / 4);
        float cutoff = (float)fg.driftCutoff;
        g.pitchDeviation = (float)((double)deviation * 2.0);
        g.pitchOffset = deviation;
        if ((double)cutoff < 0.0) cutoff = 0.0f;
        else if ((double)cutoff > ((double)sampleRate / 2.0)) cutoff = (float)((double)sampleRate / 2.0);
        g.a0 = (float)(((double)cutoff * 2.0) / (double)sampleRate);
        g.b1 = (float)(1.0 - (double)g.a0);
    }
    // tracks 0..31: this lane's current value and delta (m:919-930)
    g.cv = 0.0; g.cd = 0.0;
    if (lane < 16) {
        long long j = 1;
        double temp;
        // (bounded: the reference walks past the end of the array when a track has no later value; libtrm refuses such
        //  lists -- check_event_list -- and the kernel never reads outside this utterance's events)
        while (isnan(temp = ev[j].value[lane]) && j < count - 1) j++;
        g.cv = ev[0].value[lane];
        g.cd = isnan(temp) ? 0.0 : ((temp - g.cv) / (double)ev[j].time) * ms;
    }
    // tracks 32..35 (m:932-961)
    g.cd33 = 0.0; g.cd34 = 0.0; g.cd35 = 0.0;
    {
        double temp;
        if (fg.useSmoothIntonation) {
            long long j = 0;
            while (isnan(temp = ev[j].value[32])) {
                j++;
                if (j >= count) break;
            }
            g.cv32 = j < count ? ev[j].value[32] : __longlong_as_double(0x7ff8000000000000ll);
            g.cd32 = 0.0;
        } else {
            long long j = 1;
            while (isnan(temp = ev[j].value[32])) {
                j++;
                if (j >= count) break;
            }
            g.cv32 = ev[0].value[32];
            if (j < count) g.cd32 = ((temp - g.cv32) / (double)ev[j].time) * ms;
            else g.cd32 = 0.0;
            g.cv32 = -20.0;
        }
    }
    g.i = 1;
    g.now = 0ull;
    g.next = (unsigned long long)ev[1].time;
}

// One frame (m:973-1057): returns the table value of track `lane` (meaningful in lanes 0..15) at the current clock, then
// advances the tracks and the clock and moves to the next event once the clock reaches it.  Call while g.i < count.
__device__ __forceinline__ float framegen_step(FrameGen &g, const trm_cuda_event *__restrict__ ev, long long count,
                                               const trm_cuda_framegen &fg, int lane)
{
    const double ms = 1000.0 / 250.0;
    // table[j] = (float)currentValues[j] + (float)currentValues[j+16]  (m:974-976)
    const double hi = __shfl_down_sync(0xFFFFFFFFu, g.cv, 16);
    float t = __fadd_rn((float)g.cv, (float)hi);
    if (lane == 0) {
        if (!fg.useMicroIntonation) t = 0.0f;
    }
    {
        // drift (MMDriftGenerator.m:65-78): every lane keeps the generator, lane 0 uses it
        float d = 0.0f;
        if (fg.useDrift) {
            float temp = __fmul_rn(g.seed, 377.0f);
            g.seed = __fsub_rn(temp, (float)(int)temp);
            temp = __fsub_rn(__fmul_rn(g.seed, g.pitchDeviation), g.pitchOffset);
            g.prev = __fadd_rn(__fmul_rn(g.a0, temp), __fmul_rn(g.b1, g.prev));
            d = g.prev;
        }
        if (lane == 0) {
            if (fg.useDrift) t = __fadd_rn(t, d);
            if (fg.useMacroIntonation) t = (float)((double)t + g.cv32);
            t = (float)((double)t + fg.pitch);
        }
    }
    if (g.cd != 0.0) g.cv += g.cd;                                   // m:1007-1010 (tracks 0..31)
    if (fg.useSmoothIntonation) {                                    // m:1011-1018
        g.cd34 += g.cd35;
        g.cd33 += g.cd34;
        g.cv32 += g.cd33;
    } else {
        if (g.cd32 != 0.0) g.cv32 += g.cd32;
    }
    g.now = (unsigned long long)((double)g.now + ms);

    if (g.now >= g.next) {                                           // m:1025
        g.i++;
        if (g.i == count) return t;
        const long long i = g.i;
        g.next = (unsigned long long)ev[i].time;
        // new deltas for every track whose previous event carried a value (m:1031-1047): lane j < 32 its own
        // track, then track 32 by everybody
        for (int pass = 0; pass < 2; ++pass) {
            const int j = pass == 0 ? lane : 32;
            if (!isnan(ev[i - 1].value[j])) {
                long long k = i;
                double temp;
                bool zeroed = false;
                while (isnan(temp = ev[k].value[j])) {
                    if (k >= count - 1) { zeroed = true; break; }
                    k++;
                }
                const double cur = pass == 0 ? g.cv : g.cv32;
                double nd = 0.0;
                bool set = false;
                if (zeroed) { nd = 0.0; set = true; }
                if (!isnan(temp)) {
                    nd = (temp - cur) / (double)((unsigned long long)ev[k].time - g.now) * ms;
                    set = true;
                }
                if (set) { if (pass == 0) g.cd = nd; else g.cd32 = nd; }
            }
        }
        if (fg.useSmoothIntonation) {                                // m:1049-1057
            if (!isnan(ev[i - 1].value[33])) {
                g.cv32 = ev[i - 1].value[32];
                g.cd32 = 0.0;
                g.cd33 = ev[i - 1].value[33];
                g.cd34 = ev[i - 1].value[34];
                g.cd35 = ev[i - 1].value[35];
            }
        }
    }
    return t;
}

__global__ void __launch_bounds__(128) framegen_kernel(FrameGenArgs a)
{
    const int lane = threadIdx.x & 31;
    const int u = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (u >= a.n_utt) return;
    const trm_cuda_event *__restrict__ ev = a.events + a.ev_offset[u];
    const long long count = a.ev_count[u];
    const trm_cuda_framegen fg = a.fg[a.shared_fg ? 0 : u];
    const long long n_frames = a.desc[u].n_frames;
    double *__restrict__ out = a.frames + a.desc[u].frame_offset * 16;
    if (count < 2) {
        if (a.seed_out && lane == 0) a.seed_out[u] = fg.driftSeed;
        return;
    }
    FrameGen g;
    framegen_setup(g, ev, count, fg, lane);
    long long f = 0;
    while (g.i < count) {                                            // m:973
        const float t = framegen_step(g, ev, count, fg, lane);
        if (lane < 16 && f < n_frames) out[f * 16 + lane] = (double)t;      // 128 B per frame, coalesced
        ++f;
    }
    if (a.seed_out && lane == 0) a.seed_out[u] = g.seed;
}

// Stream pool (trm_cuda_pool_push): one warp per event-fed entry of a push.  The slot's generator is set up on its first
// frames or loaded whole from state[slot]; entry.m frames go to entry.out, then the state is stored back.
__global__ void __launch_bounds__(128) framegen_pool_kernel(FrameGenPoolArgs a)
{
    const int lane = threadIdx.x & 31;
    const int e = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (e >= a.n) return;
    const FrameGenPoolEntry en = a.ent[e];
    FrameGenPoolState *__restrict__ ps = a.state + en.slot;
    const trm_cuda_event *__restrict__ ev = reinterpret_cast<const trm_cuda_event *>(en.events);
    const trm_cuda_framegen fg = ps->fg;
    FrameGen g;
    if (en.setup) {
        framegen_setup(g, ev, en.count, fg, lane);
    } else {
        g.cv = ps->cv[lane]; g.cd = ps->cd[lane];
        g.cv32 = ps->cv32; g.cd32 = ps->cd32; g.cd33 = ps->cd33; g.cd34 = ps->cd34; g.cd35 = ps->cd35;
        g.i = ps->i; g.now = ps->now; g.next = ps->next;
        g.seed = ps->seed; g.prev = ps->prev;
        g.pitchDeviation = ps->pitchDeviation; g.pitchOffset = ps->pitchOffset; g.a0 = ps->a0; g.b1 = ps->b1;
    }
    double *__restrict__ out = reinterpret_cast<double *>(en.out);
    for (int f = 0; f < en.m && g.i < en.count; ++f) {
        const float t = framegen_step(g, ev, en.count, fg, lane);
        if (lane < 16) out[f * 16 + lane] = (double)t;
    }
    ps->cv[lane] = g.cv; ps->cd[lane] = g.cd;
    if (lane == 0) {
        ps->cv32 = g.cv32; ps->cd32 = g.cd32; ps->cd33 = g.cd33; ps->cd34 = g.cd34; ps->cd35 = g.cd35;
        ps->i = g.i; ps->now = g.now; ps->next = g.next;
        ps->seed = g.seed; ps->prev = g.prev;
        ps->pitchDeviation = g.pitchDeviation; ps->pitchOffset = g.pitchOffset; ps->a0 = g.a0; ps->b1 = g.b1;
    }
}

}  // namespace trm
