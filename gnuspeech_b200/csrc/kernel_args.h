// kernel_args.h -- plain structs and tile constants shared by the kernels (device) and the shim (host).
#pragma once

#include <stdint.h>

#include "trm_cuda.h"

// Every kernels_*.cu translation unit instantiates the kernel templates under its own compiler flags (FMA contraction
// on / off), so each one puts them into its own namespace: identical template instantiations from two TUs would otherwise
// be merged by the linker.  TRM_STRICT = 1 selects the reference-order FP64 arithmetic (tube_wide.cuh).
#ifndef TRM_KERNEL_NS
#define TRM_KERNEL_NS trm_kernels
#endif
#ifndef TRM_STRICT
#define TRM_STRICT 0
#endif

namespace trm {

constexpr int TB = 16;           // samples per block == lanes per utterance
constexpr int FIR_TAPS = 49;     // TRMFIRFilter.h:7-9 fixed design -> 49 taps (checked on the host)
constexpr int FIR_HIST = 24;     // (FIR_TAPS-1)/2 previous even / odd oscillator values
constexpr int FRAME_CHUNK = 2;   // control frames per bulk copy (256 B)


constexpr int SRC_ROWS = TRM_SRC_ROWS; // staged input rows per work item (include/trm_cuda.h: the host checks rate ratios against it)
constexpr int SRC_CHUNK = 8;         // consecutive outputs a warp finishes before the transposed write-back
constexpr int SRC_ZC = 13;           // zero crossings -> 13 taps per wing when up-sampling
constexpr int SRC_TAPS = 2 * SRC_ZC; // coefficients per output
constexpr int SRC_CLD = 28;          // row stride of the coefficient table (16-byte aligned rows in both precisions)
constexpr int PCM_THREADS = 256;
constexpr int PCM_PER_THREAD = 8;

// Carried state of one utterance for streaming synthesis (tube_wide.cuh): 4 eight-byte header words
// {oscillator position (double), the same in 2^-55 table entries (fast mode), noise generator state, "no sample
// produced yet" flag} followed by STATE_R values of the arithmetic type: oscillator history even / odd (24 + 24),
// band-pass input x[n-1], x[n-2], then the 41 recurrence values (waves, reflection / radiation memories, band-pass
// and throat outputs).
constexpr int STATE_HDR = 4;
constexpr int STATE_R = 96;
constexpr int STATE_HE = 0, STATE_HO = 24, STATE_XM = 48, STATE_SER = 50;
inline size_t tube_state_bytes(size_t esz) { return STATE_HDR * 8 + STATE_R * esz; }

struct TubeArgs {
    void *state;                 // streaming: carried states indexed like desc (loaded at the start, stored after each
                                 // utterance's last block), else null
    const trm_cuda_utterance *desc;
    const int *order;            // slot -> utterance (longest first), may be null
    int n_utt;
    const void *frames;          // [frame][16] doubles, or floats when frames_f32
    int frames_f32;
    void *tube;                  // Real[...]
    const double *wavetables;    // [voice][512]
    uint64_t noise_k0;
};

template <typename R> struct alignas(2 * sizeof(R)) HD { R h, dh; };   // one vector load per entry

struct SrcArgs {
    const trm_cuda_utterance *desc;
    int n_utt;
    const void *tube;                // Real[]
    void *out;                       // Real[]
    unsigned long long *maxbits;     // [n_utt] bit pattern of the running max |y| as double
    const void *table;               // HD<Real>[256][13]: filter index l + 256 k at [l][k]
    const void *ctab;                // Real[65536][SRC_CLD]: interpolated coefficients per time-register fraction
    // work decomposition: tiles of <= 32 utterances that share the converter signature
    const int *tile_utt;             // [n_tiles][tile width] utterance index or -1 (width: KernelInfo.src[shape].tile)
    const int *tile_nt;              // [n_tiles] outputs per work item of that tile (window fits SRC_ROWS)
    const long long *tile_max_out;   // [n_tiles] longest utterance of the tile
    const long long *tile_first_out; // [n_tiles] first output of the tile's first work item (0 unless streaming)
    const long long *item_base;      // [n_tiles+1] prefix sum of work items
    int n_tiles;
    long long total_items;
    long long item_begin, item_end;  // work items this launch processes ([0, total_items) when item_end == 0)
};

// Resampler of a stream pool (src_pool_kernel): entries are slots at independent positions.  desc[e] is the resampler view
// of entry e: outputs [out_start, n_out) of its stream are produced and written to out[out_offset + (n - out_start)]
// (packed, entry after entry); input sample q of the stream is tube[tube_offset + q], valid for q in [in_start, n_tube).
struct SrcPoolArgs {
    const trm_cuda_utterance *desc;
    int n;
    const long long *item_base;      // [n+1] prefix sum of work items (runs of 32 consecutive outputs of one entry)
    long long total_items;
    const void *tube;                // Real[]
    void *out;                       // Real[]
    const void *table;               // HD<Real>[256][13] (down-sampling phase walk)
    const void *ctab;                // Real[65536][SRC_CLD] (up-sampling coefficient rows)
};

// PCM16 of a stream pool push (pcm_pool_kernel): the same entries and work items as SrcPoolArgs, read from the packed
// outputs.  Entry e's PCM goes to pcm[desc[e].pcm_offset + channels * (n - out_start)] (packed, entry after entry),
// scaled against peak[e]; maxbits[e] (zero on entry) receives the bit pattern of max |y| over its outputs, as double.
struct PcmPoolArgs {
    const trm_cuda_utterance *desc;
    int n;
    const long long *item_base;      // [n+1] prefix sum of work items (runs of 32 consecutive outputs of one entry)
    long long total_items;
    const void *out;                 // Real[]
    const double *peak;              // [n]
    int16_t *pcm;
    unsigned long long *maxbits;     // [n]
};

// Per-push bookkeeping kernels of a stream pool (kernels_aux.cu)
struct PoolPrepArgs {
    const trm_cuda_utterance *src;   // [n] waveguide descriptors of this push
    const int *slot;                 // [n] slot of each
    const int *reset;                // [n] != 0: the slot was opened since its last launch, its carried state starts fresh
    trm_cuda_utterance *dst;         // [capacity] descriptor array the waveguide indexes by slot
    void *state;                     // [capacity] carried states
    unsigned long long state_bytes;
    unsigned long long noise_k0;
    int n;
};
// Ragged device-to-device copies (segment_copy_kernel): a push's history moves, a snapshot's gather and scatter
struct CopySeg {
    unsigned long long src, dst;     // device addresses
    unsigned long long bytes;        // a multiple of 4
};
struct SegCopyArgs {
    const CopySeg *seg;              // [n], no two overlapping
    int n;
};

struct PcmArgs {
    const trm_cuda_utterance *desc;
    int n_utt;
    const void *out;                 // Real[]
    const unsigned long long *maxbits;
    int16_t *pcm;
    int u_begin;                     // utterances [u_begin, n_utt) are scaled by this launch
};

// control-frame generator (framegen_kernel.cuh)
struct FrameGenArgs {
    const trm_cuda_utterance *desc;       // frame_offset / n_frames of every utterance
    int n_utt;
    const trm_cuda_event *events;         // all utterances back to back
    const long long *ev_offset;           // [n_utt] first event of utterance u
    const int *ev_count;                  // [n_utt]
    const trm_cuda_framegen *fg;          // [n_utt] or [1] if shared
    int shared_fg;
    double *frames;                       // [frame][16]
    float *seed_out;                      // [n_utt] drift seed at exit, may be null
};

// A stream pool slot's generator between pushes (framegen_pool_kernel): the whole FrameGen of its warp -- cv / cd of all
// 32 lanes, the rest as every lane holds it -- and the slot's settings, written when the slot opens.
struct FrameGenPoolState {
    double cv[32], cd[32];
    double cv32, cd32, cd33, cd34, cd35;
    long long i;
    unsigned long long now, next;
    float seed, prev, pitchDeviation, pitchOffset, a0, b1;
    trm_cuda_framegen fg;
};
struct FrameGenPoolEntry {
    unsigned long long events;            // device address of the slot's event list
    long long count;                      // its events
    unsigned long long out;               // device address of the first new frame (rows of 16 doubles)
    int slot;                             // index into FrameGenPoolArgs::state
    int m;                                // frames to generate (the list has at least that many left)
    int setup;                            // != 0: the slot's first frames, the state is set up from fg instead of loaded
    int reserved;
};
struct FrameGenPoolArgs {
    const FrameGenPoolEntry *ent;         // [n]
    int n;
    FrameGenPoolState *state;             // [capacity]
};

struct KernelInfo {
    // resampler shapes (src_kernel.cuh SrcCfg): [0] handles every converter signature, [1] (if n_src_shapes == 2) is
    // the faster shape for up-sampling signatures whose work-item window fits its smaller staging buffer
    struct SrcShape {
        int smem_bytes, threads, ctas_per_sm, regs;
        int tile;                  // utterances per tile (32 x utterances per lane)
        int rows;                  // tube-rate samples per utterance staged for one work item
        int nt_max;                // outputs per work item, at most
    } src[2];
    int n_src_shapes;
    int pcm_regs;
    int wide_smem_bytes, wide_threads, wide_max_utt, wide_regs;   // batch-throughput waveguide mapping (tube_wide.cuh)
};

}  // namespace trm
