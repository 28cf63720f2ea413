// src_kernel.cuh -- batch-wide sample-rate converter and PCM scaling kernels for sm_100a.
//
// src_kernel replaces -[TRMSampleRateConverter processDataFromRingBuffer:]
// (/root/reference/Frameworks/Tube/TRMSampleRateConverter.m:155-298) together with the ring buffer that
// feeds it (TRMRingBuffer.m:27-105).  The streaming converter is equivalent to a stateless gather
// (SURVEY.md 8(a) row 16, checked on the CPU by tests/test_oracle.py): with xb[p] = x[p - pad]
// (zero outside [0, n_in)), output n has time register T = n*TRI, P = T>>16, F = T&0xFFFF and
//   up-sampling  : y = sum_{k=0..12} xb[P-k]  *(h[l +256k] + dH[l +256k]*m /256)        (l ,m ) = (F>>8, F&255)
//                    + sum_{k=0..12} xb[P+1+k]*(h[l'+256k] + dH[l'+256k]*m'/256)        (l',m') from (~F)&0xFFFF
//   down-sampling: phase walks of TRMSampleRateConverter.m:246-270.
// Accumulation order (left wing first, from 0.0) is the reference's.  Also produces the per-utterance
// maximumSampleValue (m:206-208) with an order-independent integer atomicMax on the bit pattern.
//
// pcm_kernel replaces the scaling loops of -generateWAVData (TRMTubeModel.m:515-559):
//   scale = (32767 / max) * amplitude(volume);  int16 = rint(sample * scale)  (mono)
//   stereo: left = rint(sample * leftGain*scale), right = rint(sample * rightGain*scale), interleaved.
//
// Persistent CTAs: input windows are staged per work item with coalesced loads, the item's interpolated filter
// coefficients are computed once into shared memory; outputs are written as full sectors.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

#include "kernel_args.h"
#include "trm_cuda.h"
#include "tube_common.cuh"   // mbarrier / TMA bulk-copy helpers

namespace TRM_KERNEL_NS {
using namespace trm;

// 16 bytes of R through the native vector type (keeps the elements in registers)
template <typename R> struct Vec16;
template <> struct Vec16<float> {
    float e[4];
    __device__ __forceinline__ void load(const float *p) { const float4 v = *reinterpret_cast<const float4 *>(p); e[0] = v.x; e[1] = v.y; e[2] = v.z; e[3] = v.w; }
    __device__ __forceinline__ void store(float *p) const { *reinterpret_cast<float4 *>(p) = make_float4(e[0], e[1], e[2], e[3]); }
};
template <> struct Vec16<double> {
    double e[2];
    __device__ __forceinline__ void load(const double *p) { const double2 v = *reinterpret_cast<const double2 *>(p); e[0] = v.x; e[1] = v.y; }
    __device__ __forceinline__ void store(double *p) const { *reinterpret_cast<double2 *>(p) = make_double2(e[0], e[1]); }
};

// Shapes of the resampler.  U = utterances per lane: a coefficient read from shared memory (a broadcast 16-byte load
// returns 512 bytes to the warp's registers, and the SM delivers 128 bytes per clock) serves U multiply-adds; with U = 1
// that return path, not the arithmetic, bounded both precisions.
//   shape 0 handles every converter signature (both directions, windows up to TRM_SRC_ROWS rows).  FP32: U = 2.  FP64:
//           U = 1 -- the register window is 52 registers per utterance.
//   A second shape can be added per precision (SrcShapes<R>::N = 2; the launcher picks shape 1 for chunks whose
//   utterances all up-sample with a window that fits it, trm_cuda.cu plan_chunk()).  Measured and not kept: FP64 with
//   U = 2 -- 166 registers, so either one 12-warp CTA per SM (14.1 ms on 4096 x 10 s) or two 6-warp CTAs with work items
//   half as long (<= 96 outputs, 76 staged rows: 12.0 ms), against 11.6 ms for shape 0.
// WINDOWS = 2 prefetches the next work item's window into a second buffer (measured: no gain, the copy latency was
// already hidden by the SM's other CTA).  CBUFS = 2 does the same for the coefficient rows (gain in FP32).
// XLD: elements per utterance row of the staged windows (rows + alignment slack).  Rows start on 16-byte boundaries
// (bulk-copy destinations), so the lanes of a warp reading the same element of their rows always collide somewhat;
// strides of 4 banks mod 32 keep that to 4 (FP32) / 2 (FP64) lanes per bank.
template <typename R, int SHAPE> struct SrcCfg;
template <> struct SrcCfg<float, 0> {
    static constexpr int U = 2, WINDOWS = 1, CBUFS = 2, THREADS = 256, MIN_CTAS = 2;
    static constexpr int ROWS = SRC_ROWS, XLD = 132, NT_MAX = 192;
};
template <> struct SrcCfg<double, 0> {
    static constexpr int U = 1, WINDOWS = 1, CBUFS = 1, THREADS = 256, MIN_CTAS = 2;
    static constexpr int ROWS = SRC_ROWS, XLD = 130, NT_MAX = 192;
};
template <typename R> struct SrcShapes { static constexpr int N = 1; };

template <typename R> __device__ __forceinline__ R r_abs(R x);
template <> __device__ __forceinline__ double r_abs<double>(double x) { return fabs(x); }
template <> __device__ __forceinline__ float r_abs<float>(float x) { return fabsf(x); }
// max(a, b) that returns a when b is NaN (a is never NaN here): the (b > a) ? b : a of the reference's running maximum
template <typename R> __device__ __forceinline__ R r_max(R a, R b);
template <> __device__ __forceinline__ double r_max<double>(double a, double b) { return (b > a) ? b : a; }
template <> __device__ __forceinline__ float r_max<float>(float a, float b) { return fmaxf(a, b); }

// One work item = one tile of 32 utterances with the same converter signature (time-register increment, pad,
// direction, phase increment) x one run of `nt` consecutive output samples.  Lane = utterance: every lane of a
// warp computes the SAME output index n, so the time register, the filter phase and all 26 interpolated
// coefficients are warp-uniform.
//
// Up-sampling (the common case: tube rate < output rate) is bound by shared-memory bandwidth unless both operands of
// the multiply-add are reused, so
//   * the 26 coefficients of every output of the item are computed ONCE per CTA into a shared table C[n][26]
//     (left wing k = 0..12, then right wing; same two operations per coefficient as the reference) and read back
//     with broadcast vector loads -- they serve 32 utterances;
//   * each warp walks a run of consecutive outputs and keeps the 26 input samples under the filter in REGISTERS:
//     when the time register's integer part advances the window slides by one (register moves + one shared-memory
//     load) instead of 26 loads per output;
//   * the input windows (one contiguous span per utterance) are staged by TMA bulk copies (cp.async.bulk + mbarrier)
//     issued by 32 lanes: no thread touches the data on its way in.  Spans are widened to 16-byte boundaries;
//     positions before the first / after the last sample of an utterance are zero-filled afterwards (first and last
//     items of an utterance only).
// Accumulation order (left wing first, newest -> oldest, from 0.0) is the reference's; one multiply and one add per
// tap.  Outputs go back through a small per-warp transpose tile and leave as 128-bit stores.
template <typename R, int SHAPE>
__global__ void __launch_bounds__(SrcCfg<R, SHAPE>::THREADS, SrcCfg<R, SHAPE>::MIN_CTAS) src_kernel(SrcArgs args)
{
    using Cfg = SrcCfg<R, SHAPE>;
    constexpr int A = 16 / (int)sizeof(R);                               // elements per 16 bytes
    constexpr int YLD = SRC_CHUNK + 1;
    constexpr int U = Cfg::U, TW = 32 * Cfg::U;
    constexpr int NBUF = Cfg::WINDOWS, SRC_NT_MAX = Cfg::NT_MAX;
    constexpr unsigned FULL = 0xFFFFFFFFu;
    constexpr int SRC_THREADS = Cfg::THREADS, SRC_XLD = Cfg::XLD;
    static_assert(SRC_THREADS >= SRC_NT_MAX, "one coefficient row per thread");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    R *xU0 = reinterpret_cast<R *>(smem_raw);                            // [NBUF][TW][SRC_XLD] input windows, utterance-major
    R *Cf0 = xU0 + NBUF * TW * SRC_XLD;                                  // [CBUFS][SRC_NT_MAX][SRC_CLD] coefficient rows
    R *yT = Cf0 + Cfg::CBUFS * SRC_NT_MAX * SRC_CLD;                              // [warps][TW][YLD]
    __shared__ long long s_tube_off[TW], s_out_off[TW], s_n_in[TW], s_n_out[TW], s_out_start[TW], s_in_start[TW];
    __shared__ int s_tile;
    __shared__ unsigned long long s_bar[2], s_cbar[2];
    __shared__ unsigned char s_flag[SRC_NT_MAX];

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const HD<R> *__restrict__ tab = reinterpret_cast<const HD<R> *>(args.table);
    if (threadIdx.x == 0) {
        mbar_init(&s_bar[0], U);                                         // one arrival per requesting warp
        mbar_init(&s_bar[1], U);
        mbar_init(&s_cbar[0], 1);
        mbar_init(&s_cbar[1], 1);
        mbar_fence_init();
    }
    uint32_t bar_phase = 0;                                              // bit b: parity to wait for on s_bar[b]
    int buf = 0;                                                         // window buffer of the current item
    bool in_flight = false;                                              // its window was requested during the previous item
    uint32_t cbar_phase = 0;
    int cb = 0;                                                          // coefficient buffer of the current item
    bool c_in_flight = false;                                            // its coefficient rows were requested during the previous item

    // every CTA takes a contiguous range of work items: consecutive items belong to the same tile, whose descriptors
    // are read from global memory once and kept in shared memory
    const long long range_lo = args.item_begin, range_hi = args.item_end > 0 ? args.item_end : args.total_items;
    const long long per_cta = (range_hi - range_lo + gridDim.x - 1) / gridDim.x;
    const long long item_lo = range_lo + (long long)blockIdx.x * per_cta;
    const long long item_hi = (item_lo + per_cta < range_hi) ? item_lo + per_cta : range_hi;
    long long tile_first = 0, tile_end = 0;                              // items [tile_first, tile_end) belong to `tile`
    int tile = 0;
    unsigned tri = 0, phaseIncrement = 0;
    int pad = 0, reach = 0, nt = 0;
    bool up = true;
    double ratio = 1.0;
    long long tile_max = 0, tile_out0 = 0;
    // lane l owns the utterances in rows l, l + 32, .. of the tile
    R local_max[U];
#pragma unroll
    for (int k = 0; k < U; ++k) local_max[k] = (R)0;
    auto flush_max = [&]() {
        // per-utterance maximum: integer atomicMax on the bit pattern (order independent for non-negative doubles)
#pragma unroll
        for (int k = 0; k < U; ++k) {
            if (local_max[k] > (R)0) {
                const int u = args.tile_utt[tile * TW + lane + 32 * k];
                if (u >= 0) atomicMax(args.maxbits + u, (unsigned long long)__double_as_longlong((double)local_max[k]));
            }
            local_max[k] = (R)0;
        }
    };

    for (long long item = item_lo; item < item_hi; ++item) {
        __syncthreads();                       // previous item's window / descriptors no longer read
        if (item >= tile_end) {                // CTA-uniform: first item, or the range crosses into the next tile
            if (item > item_lo) flush_max();
            if (threadIdx.x == 0) {
                int lo = 0, hi = args.n_tiles; // largest tile with item_base[tile] <= item
                while (hi - lo > 1) {
                    const int mid = (lo + hi) >> 1;
                    if (args.item_base[mid] <= item) lo = mid; else hi = mid;
                }
                s_tile = lo;
            }
            __syncthreads();
            tile = s_tile;
            if (warp < U) {
                const int row = warp * 32 + lane;
                const int u = args.tile_utt[tile * TW + row];
                const trm_cuda_utterance *D = args.desc + (u >= 0 ? u : 0);
                s_tube_off[row] = D->tube_offset;
                s_out_off[row] = D->out_offset;
                s_n_in[row] = u >= 0 ? D->n_tube : -1;
                s_n_out[row] = u >= 0 ? D->n_out : 0;
                s_out_start[row] = u >= 0 ? D->out_start : 0;       // streaming: earlier outputs exist already,
                s_in_start[row] = u >= 0 ? D->in_start : 0;         // earlier inputs are no longer in memory
            }
            // signature of the tile (row 0 is always a real utterance)
            const trm_cuda_utterance *__restrict__ D0 = args.desc + args.tile_utt[tile * TW];
            tri = D0->tri;
            pad = D0->padSize; reach = pad + 1;
            up = D0->upsample != 0;
            ratio = D0->sampleRateRatio;
            phaseIncrement = D0->phaseIncrement;
            nt = args.tile_nt[tile];
            tile_first = args.item_base[tile];
            tile_end = args.item_base[tile + 1];
            tile_max = args.tile_max_out[tile];
            tile_out0 = args.tile_first_out[tile];
            __syncthreads();
        }
        // geometry of a work item of the current tile: its outputs and the window of input samples under them
        struct Geo { long long n_s, P0, q0, qb; int n_item, off, span; unsigned frac0; };
        auto geometry = [&](long long it) {
            Geo g;
            g.n_s = tile_out0 + (it - tile_first) * nt;
            g.n_item = (int)((g.n_s + nt < tile_max) ? nt : tile_max - g.n_s);         // outputs of this item
            const unsigned long long T0 = (unsigned long long)g.n_s * tri;
            g.P0 = (long long)(T0 >> 16);
            g.frac0 = (unsigned)(T0 & 0xFFFFull);
            const int rows = (int)((((unsigned long long)g.frac0 + (unsigned long long)(g.n_item - 1) * tri) >> 16)) + 2 * reach + 2;
            // window of utterance r: elements q0 .. q0+rows-1 of its tube-rate signal, q = p - pad (xb[p] = x[p - pad])
            g.q0 = g.P0 - reach - pad;
            g.qb = (g.q0 >= 0) ? g.q0 / A * A : -((-g.q0 + A - 1) / A * A);            // 16-byte aligned start (floor)
            g.off = (int)(g.q0 - g.qb);                                                // window element i sits at xU[r][off + i]
            g.span = (g.off + rows + A - 1) / A * A;
            return g;
        };
        // warps 0..U-1: bulk copies of [lo, hi) of every utterance (clipped to its 16-byte-padded extent) into window buffer b
        auto request_window = [&](const Geo &g, int b) {
            const int row = warp * 32 + lane;
            const long long n_in = s_n_in[row];
            const long long n_al = (n_in + A - 1) / A * A;
            long long lo = g.qb > 0 ? g.qb : 0;
            if (lo < s_in_start[row]) lo = s_in_start[row];              // (a multiple of A; only discarded outputs look below it)
            const long long hi = (g.qb + g.span < n_al) ? g.qb + g.span : n_al;
            const unsigned bytes = (hi > lo) ? (unsigned)(hi - lo) * (unsigned)sizeof(R) : 0u;
            unsigned total = bytes;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) total += __shfl_xor_sync(FULL, total, o);
            if (lane == 0) mbar_expect_tx(&s_bar[b], total);
            __syncwarp();
            if (bytes)
                tma_bulk_g2s(xU0 + (b * TW + row) * SRC_XLD + (int)(lo - g.qb), reinterpret_cast<const R *>(args.tube) + s_tube_off[row] + lo,
                             bytes, &s_bar[b]);
        };
        const Geo geo = geometry(item);
        const long long n_s = geo.n_s, P0 = geo.P0, q0 = geo.q0, qb = geo.qb;
        const int n_item = geo.n_item, off = geo.off, span = geo.span;
        const unsigned frac0 = geo.frac0;
        const unsigned long long T0 = (unsigned long long)n_s * tri;
        R *const xU = xU0 + buf * TW * SRC_XLD;
        if (warp < U && !in_flight) request_window(geo, buf);
        const int run = nt / (SRC_THREADS / 32);                         // consecutive outputs per warp (multiple of SRC_CHUNK)
        // Coefficient rows of an item: output n has C[n][t] = h[l + 256 k] + dH[l + 256 k] * (m / 256), (l, m) from the
        // fraction F of its time register for the left wing (t = k) and from ~F for the right wing (t = 13 + k)
        // (m:179-203) -- a function of F alone, so the rows come from the context's table of all 65,536 fractions
        // (src_ctab_kernel below; a few MB that stay in L2), one bulk copy per row, one row per thread.  The rows of the
        // NEXT item are requested before this one is computed and land in the other buffer meanwhile.
        constexpr unsigned ROWB = SRC_CLD * (unsigned)sizeof(R);
        const R *__restrict__ ct = reinterpret_cast<const R *>(args.ctab);
        auto request_rows = [&](const Geo &g, int b) {
            if (threadIdx.x == 0) mbar_expect_tx(&s_cbar[b], (unsigned)g.n_item * ROWB);
            if ((int)threadIdx.x < g.n_item) {
                const unsigned f = g.frac0 + threadIdx.x * tri;
                tma_bulk_g2s(Cf0 + (b * SRC_NT_MAX + (int)threadIdx.x) * SRC_CLD, ct + (size_t)(f & 0xFFFFu) * SRC_CLD, ROWB, &s_cbar[b]);
            }
        };
        const bool more = item + 1 < item_hi && item + 1 < tile_end;     // the next item belongs to this tile too
        const R *const Cf = Cf0 + cb * SRC_NT_MAX * SRC_CLD;
        if (up) {
            if (!c_in_flight) request_rows(geo, cb);
            if (Cfg::CBUFS == 2 && more) request_rows(geometry(item + 1), cb ^ 1);
            // what follows output n for the warp that walks it: 0 = same input position, 1 = the integer part of the time
            // register advances (slide the window), 2 = last output of the warp's run
            if ((int)threadIdx.x < n_item) {
                const int nr = threadIdx.x;
                const unsigned f = frac0 + (unsigned)nr * tri;
                const bool last = (nr + 1 == n_item) || ((nr + 1) % run == 0);
                s_flag[nr] = last ? 2 : ((((f + tri) >> 16) != (f >> 16)) ? 1 : 0);
            }
        }
        __syncthreads();                                                 // descriptors + coefficients visible
        // (WINDOWS = 2) the next item's window is requested now and lands while this item is computed; its buffer was last
        // read by the item before this one, which every warp has left
        const bool prefetch = NBUF == 2 && item + 1 < item_hi && item + 1 < tile_end;
        if (prefetch && warp < U) request_window(geometry(item + 1), buf ^ 1);
        mbar_wait(&s_bar[buf], (bar_phase >> buf) & 1u);
        bar_phase ^= 1u << buf;
        if (up) {
            mbar_wait(&s_cbar[cb], (cbar_phase >> cb) & 1u);
            cbar_phase ^= 1u << cb;
        }
        {
            // zero-fill outside [0, n_in): only the first / last items of an utterance have such positions
            bool mine = false;
#pragma unroll
            for (int k = 0; k < U; ++k) mine = mine || (q0 < 0) || (qb + span > s_n_in[lane + 32 * k]);
            if (__any_sync(FULL, mine)) {
                for (int r = warp; r < TW; r += SRC_THREADS / 32) {
                    const long long nin = s_n_in[r];
                    if (qb >= 0 && qb + span <= nin) continue;
                    for (int i = lane; i < span; i += 32) {
                        const long long q = qb + i;
                        if (q < 0 || q >= nin) xU[r * SRC_XLD + i] = (R)0;
                    }
                }
                __syncthreads();
            }
        }

        // this lane's utterances: outputs [my_lo, my_out) of the item are theirs to produce
        int my_out[U], my_lo[U];
        bool all_mine = true;
#pragma unroll
        for (int k = 0; k < U; ++k) {
            const long long no = s_n_out[lane + 32 * k] - n_s, os = s_out_start[lane + 32 * k] - n_s;
            my_out[k] = (int)((no < (long long)n_item) ? (no > 0 ? no : 0) : n_item);
            my_lo[k] = (int)((os > 0) ? ((os < (long long)n_item) ? os : n_item) : 0);
            all_mine = all_mine && my_lo[k] == 0 && my_out[k] == n_item;
        }
        R *yw = yT + warp * (TW * YLD);
        const R *xl = xU + lane * SRC_XLD + off;                         // xl[32 k SRC_XLD + i] = window element i of utterance k
        if (up) {
            const int nr_first = warp * run;
            // every utterance of the tile has all outputs of this item and none of them exists already (streaming):
            // no per-output or per-piece range checks
            const bool interior = __all_sync(FULL, all_mine);
            // Register window of the 26 input samples under the filter.  Logical element i (= xb[P - 12 + i]; left wing
            // xb[P-k] is i = 12-k, right wing xb[P+1+k] is i = 13+k) lives in register W[(i + ph) % 26] where ph is the
            // window phase.  When the integer part P of the time register advances, the oldest sample's register
            // receives the new one and ph increases: the loop below is unrolled over the 26 phases, so every register
            // index is a compile-time constant and sliding the window costs one shared-memory load and no moves.
            // xb[P0 + Prel + d] is window element reach + Prel + d.
            R W[U][SRC_TAPS];
            int nr = nr_first;
            const int Pc0 = (int)((frac0 + (unsigned)(nr_first < n_item ? nr_first : 0) * tri) >> 16);
#pragma unroll
            for (int k = 0; k < U; ++k) {
                const R *xp = xl + 32 * k * SRC_XLD + (reach - (SRC_ZC - 1)) + Pc0;
#pragma unroll
                for (int i = 0; i < SRC_TAPS; ++i) W[k][i] = xp[i];
            }
            const R *xn = xl + reach + SRC_ZC + Pc0;                     // newest window element; the next one enters on a slide
            const R *crow = Cf + nr_first * SRC_CLD;
            const unsigned char *fl = s_flag + nr_first;
            R *const ys = yw + lane * YLD;                               // utterance k: row lane + 32 k of the warp's tile
            int c0 = nr_first, j = 0;                                    // start of the current write-back chunk, outputs in it
            constexpr int PIECES = SRC_CHUNK / A;                        // 16-byte pieces per utterance and chunk
            constexpr int NP = U * PIECES;                               // pieces per lane and chunk
            // piece i of this lane: tile row (32 / PIECES) * i + lane / PIECES, elements A * (lane % PIECES) ..
            R *dstp[NP];
#pragma unroll
            for (int i = 0; i < NP; ++i)
                dstp[i] = reinterpret_cast<R *>(args.out) + s_out_off[(32 / PIECES) * i + lane / PIECES] + n_s + nr_first + A * (lane % PIECES);
            auto write_back = [&](bool fast) {
                __syncwarp();
                if (fast) {
#pragma unroll
                    for (int i = 0; i < NP; ++i) {
                        const R *src = yw + ((32 / PIECES) * i + lane / PIECES) * YLD + A * (lane % PIECES);
                        Vec16<R> v;
#pragma unroll
                        for (int e = 0; e < A; ++e) v.e[e] = src[e];
                        v.store(dstp[i]);
                    }
                } else {
#pragma unroll
                    for (int i = 0; i < NP; ++i) {
                        const int r = (32 / PIECES) * i + lane / PIECES, part = lane % PIECES;
                        const long long left = s_n_out[r] - (n_s + c0) - A * part;        // valid samples from this piece on
                        const long long skip = s_out_start[r] - (n_s + c0) - A * part;   // leading samples that exist already
                        if (left > 0 && A * part < j && skip < A) {
                            R *dst = dstp[i];
                            const R *src = yw + r * YLD + A * part;
                            if (left >= A && A * part + A <= j && skip <= 0) {
                                Vec16<R> v;
#pragma unroll
                                for (int e = 0; e < A; ++e) v.e[e] = src[e];
                                v.store(dst);
                            } else {
                                for (int e = 0; e < A && e < left && A * part + e < j; ++e)
                                    if (e >= skip) dst[e] = src[e];
                            }
                        }
                    }
                }
                __syncwarp();
#pragma unroll
                for (int i = 0; i < NP; ++i) dstp[i] += j;
                c0 += j;
                j = 0;
            };
            auto walk = [&](auto tag) {
                constexpr bool INTERIOR = decltype(tag)::value;
                for (;;) {
#pragma unroll
                    for (int ph = 0; ph < SRC_TAPS; ++ph) {
                        int flag;
                        do {
                            // coefficient row: broadcast 128-bit loads, consumed as they arrive (tap t: t < 13 is the left
                            // wing, logical element 12-t; else the right wing, logical element t); every coefficient
                            // serves the lane's U utterances
                            R acc[U];
#pragma unroll
                            for (int k = 0; k < U; ++k) acc[k] = (R)0;
                            flag = *fl++;
#pragma unroll
                            for (int q = 0; q < (SRC_TAPS + A - 1) / A; ++q) {
                                Vec16<R> cq;
                                cq.load(crow + A * q);
#pragma unroll
                                for (int e = 0; e < A; ++e) {
                                    const int t = A * q + e;
#pragma unroll
                                    for (int k = 0; k < U; ++k) {
                                        if (t < SRC_ZC) acc[k] += W[k][(SRC_ZC - 1 - t + ph) % SRC_TAPS] * cq.e[e];
                                        else if (t < SRC_TAPS) acc[k] += W[k][(t + ph) % SRC_TAPS] * cq.e[e];
                                    }
                                }
                            }
#pragma unroll
                            for (int k = 0; k < U; ++k) {
                                ys[32 * k * YLD + j] = acc[k];
                                if constexpr (INTERIOR) {
                                    local_max[k] = r_max<R>(local_max[k], r_abs<R>(acc[k]));   // NaN never wins, like the reference
                                } else {
                                    const R av = (nr < my_out[k] && nr >= my_lo[k]) ? r_abs<R>(acc[k]) : (R)0;
                                    local_max[k] = (av > local_max[k]) ? av : local_max[k];
                                }
                            }
                            if constexpr (!INTERIOR) ++nr;
                            crow += SRC_CLD;
                            if (++j == SRC_CHUNK) write_back(INTERIOR);
                        } while (flag == 0);
                        if (flag == 2) return;
                        // slide: logical element 0 (register ph) leaves, xb[P + 14] enters as logical element 25 of phase ph+1
                        ++xn;
#pragma unroll
                        for (int k = 0; k < U; ++k) W[k][ph] = xn[32 * k * SRC_XLD];
                    }
                }
            };
            if (nr_first < n_item) {
                if (interior) walk(std::true_type{}); else walk(std::false_type{});
                if (j > 0) write_back(false);
            }
        } else {
            // down-sampling (short tubes): chunks are dealt round-robin to the warps, taps walk the filter phase
            for (int c0 = warp * SRC_CHUNK; c0 < n_item; c0 += (SRC_THREADS / 32) * SRC_CHUNK) {
                const int jn = (n_item - c0 < SRC_CHUNK) ? n_item - c0 : SRC_CHUNK;
                for (int j = 0; j < jn; ++j) {
                    const unsigned long long T = T0 + (unsigned long long)(c0 + j) * tri;
                    const int base = (int)((long long)(T >> 16) - P0) + reach;
                    const unsigned F = (unsigned)(T & 0xFFFFull);
#pragma unroll
                    for (int k = 0; k < U; ++k) {
                        R acc = (R)0;
                        unsigned ph = (unsigned)rint((double)F * ratio), ii;
                        const R *xq = xl + 32 * k * SRC_XLD + base;
                        while ((ii = (ph >> 8)) < (unsigned)TRM_SRC_FILTER_LEN) {
                            const HD<R> c = tab[(ii & 255u) * SRC_ZC + (ii >> 8)];
                            const R impulse = c.h + (c.dh * ((R)(ph & 255u) / (R)256));
                            acc += (*xq * impulse);
                            xq -= 1;
                            ph += phaseIncrement;
                        }
                        ph = (unsigned)rint((double)((~F) & 0xFFFFu) * ratio);
                        xq = xl + 32 * k * SRC_XLD + base + 1;
                        while ((ii = (ph >> 8)) < (unsigned)TRM_SRC_FILTER_LEN) {
                            const HD<R> c = tab[(ii & 255u) * SRC_ZC + (ii >> 8)];
                            const R impulse = c.h + (c.dh * ((R)(ph & 255u) / (R)256));
                            acc += (*xq * impulse);
                            xq += 1;
                            ph += phaseIncrement;
                        }
                        yw[(lane + 32 * k) * YLD + j] = acc;
                        const R av = (c0 + j < my_out[k] && c0 + j >= my_lo[k]) ? r_abs<R>(acc) : (R)0;
                        local_max[k] = (av > local_max[k]) ? av : local_max[k];
                    }
                }
                __syncwarp();
#pragma unroll
                for (int i = 0; i < U * SRC_CHUNK; ++i) {
                    const int r = (32 / SRC_CHUNK) * i + lane / SRC_CHUNK, cc = lane % SRC_CHUNK;
                    if (n_s + c0 + cc < s_n_out[r] && n_s + c0 + cc >= s_out_start[r])
                        (reinterpret_cast<R *>(args.out) + s_out_off[r])[n_s + c0 + cc] = yw[r * YLD + cc];
                }
                __syncwarp();
            }
        }
        in_flight = prefetch;
        buf = (NBUF == 2) ? buf ^ 1 : 0;
        c_in_flight = Cfg::CBUFS == 2 && up && more;
        cb = (Cfg::CBUFS == 2) ? cb ^ 1 : 0;
    }
    if (item_hi > item_lo) flush_max();
}

// Resampler of a stream pool (trm_cuda_pool_push): the entries are streams at unrelated positions with their own voices,
// so src_kernel's tiles (lane = utterance, one output index per warp) do not apply -- a tile spans from the earliest
// missing output of its utterances to the latest, and the coefficients are not warp-uniform across signatures.  Here a
// work item is a run of 32 consecutive outputs of ONE entry and lane = output.  Each lane reads its coefficient row
// ctab[F] (the context's table, L2-resident) and its inputs directly.  The values and their order are src_kernel's: the
// same coefficients, the taps left wing newest -> oldest from 0.0 then right wing, the same `acc += x * c` expression in
// the same translation unit (so FMA contraction treats both kernels alike), and the same phase walk when
// down-sampling -- the pool's output is bit-identical to the batch path's.
template <typename R>
__global__ void __launch_bounds__(256) src_pool_kernel(SrcPoolArgs args)
{
    constexpr int A = 16 / (int)sizeof(R);
    const int lane = threadIdx.x & 31;
    const long long n_warps = (long long)gridDim.x * (blockDim.x >> 5);
    const R *__restrict__ X = reinterpret_cast<const R *>(args.tube);
    const HD<R> *__restrict__ tab = reinterpret_cast<const HD<R> *>(args.table);
    const R *__restrict__ ct = reinterpret_cast<const R *>(args.ctab);
    for (long long item = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); item < args.total_items; item += n_warps) {
        int lo = 0, hi = args.n;                                         // entry: largest e with item_base[e] <= item
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (args.item_base[mid] <= item) lo = mid; else hi = mid;
        }
        const trm_cuda_utterance *__restrict__ D = args.desc + lo;
        const long long n = D->out_start + (item - args.item_base[lo]) * 32 + lane;   // output index in the stream
        if (n >= D->n_out) continue;
        const long long base = D->tube_offset, q_lo = D->in_start, q_hi = D->n_tube;
        const int pad = D->padSize;
        // xb[p] = x[p - pad]; zero before the first sample and after the last one (a flush: the converter's tail)
        auto x = [&](long long q) -> R { return (q >= q_lo && q < q_hi) ? X[base + q] : (R)0; };
        const unsigned long long T = (unsigned long long)n * D->tri;
        const long long P = (long long)(T >> 16);
        const unsigned F = (unsigned)(T & 0xFFFFull);
        R acc = (R)0;
        if (D->upsample) {
            R xv[SRC_TAPS];
#pragma unroll
            for (int t = 0; t < SRC_ZC; ++t) {
                xv[t] = x(P - t - pad);                                  // left wing xb[P - t]
                xv[SRC_ZC + t] = x(P + 1 + t - pad);                     // right wing xb[P + 1 + t]
            }
            const R *crow = ct + (size_t)F * SRC_CLD;
#pragma unroll
            for (int q = 0; q < (SRC_TAPS + A - 1) / A; ++q) {
                Vec16<R> cq;
                cq.load(crow + A * q);
#pragma unroll
                for (int e = 0; e < A; ++e) {
                    const int t = A * q + e;
                    if (t < SRC_TAPS) acc += xv[t] * cq.e[e];
                }
            }
        } else {
            const double ratio = D->sampleRateRatio;
            const unsigned phaseIncrement = D->phaseIncrement;
            unsigned ph = (unsigned)rint((double)F * ratio), ii;
            long long q = P - pad;
            while ((ii = (ph >> 8)) < (unsigned)TRM_SRC_FILTER_LEN) {
                const HD<R> c = tab[(ii & 255u) * SRC_ZC + (ii >> 8)];
                const R impulse = c.h + (c.dh * ((R)(ph & 255u) / (R)256));
                acc += (x(q) * impulse);
                q -= 1;
                ph += phaseIncrement;
            }
            ph = (unsigned)rint((double)((~F) & 0xFFFFu) * ratio);
            q = P + 1 - pad;
            while ((ii = (ph >> 8)) < (unsigned)TRM_SRC_FILTER_LEN) {
                const HD<R> c = tab[(ii & 255u) * SRC_ZC + (ii >> 8)];
                const R impulse = c.h + (c.dh * ((R)(ph & 255u) / (R)256));
                acc += (x(q) * impulse);
                q += 1;
                ph += phaseIncrement;
            }
        }
        reinterpret_cast<R *>(args.out)[D->out_offset + (n - D->out_start)] = acc;
    }
}

// PCM16 of a stream pool push (trm_cuda_pool_push_pcm16), run after src_pool_kernel on its packed outputs with the same
// work items (32 consecutive outputs of one entry, lane = output).  The scaling is pcm_kernel's, expression for
// expression, with the caller's peak in place of the utterance's maximum; the result is then saturated to the int16
// range, which never triggers when the peak is the true maximum (|y * scale| <= 32767 * amplitude <= 32767).  Entry
// offsets are not 16-byte aligned (packed), so loads and stores are scalar; a stereo entry's PCM may start at an odd
// element (after a mono entry with an odd count), so its two channels are two int16 stores.  max |y| per warp, then
// one integer atomicMax on the double's bit pattern per work item (order independent for non-negative doubles); NaN
// never wins, as in src_kernel.
__device__ __forceinline__ int16_t pcm_sat(double v)
{
    const int q = __double2int_rn(v);
    return (int16_t)(q < -32768 ? -32768 : (q > 32767 ? 32767 : q));
}

template <typename R>
__global__ void __launch_bounds__(256) pcm_pool_kernel(PcmPoolArgs args)
{
    const int lane = threadIdx.x & 31;
    const long long n_warps = (long long)gridDim.x * (blockDim.x >> 5);
    const R *__restrict__ Y = reinterpret_cast<const R *>(args.out);
    for (long long item = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); item < args.total_items; item += n_warps) {
        int lo = 0, hi = args.n;                                         // entry: largest e with item_base[e] <= item
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (args.item_base[mid] <= item) lo = mid; else hi = mid;
        }
        const trm_cuda_utterance *__restrict__ D = args.desc + lo;
        const long long k = (item - args.item_base[lo]) * 32 + lane;   // output of this push, relative to out_start
        double m = 0.0;
        if (D->out_start + k < D->n_out) {
            const R v = Y[D->out_offset + k];
            const double scale = (32767.0 / args.peak[lo]) * D->volumeAmp;          // TRMTubeModel.m:515
            if (D->channels == 2) {
                const double ls = D->leftGain * scale, rs = D->rightGain * scale;  // TRMTubeModel.m:532-533
                int16_t *p = args.pcm + D->pcm_offset + 2 * k;
                p[0] = pcm_sat((double)v * ls);
                p[1] = pcm_sat((double)v * rs);
            } else {
                args.pcm[D->pcm_offset + k] = pcm_sat((double)v * scale);
            }
            const double av = fabs((double)v);
            m = av > m ? av : m;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double t = __shfl_xor_sync(0xffffffffu, m, o);
            m = t > m ? t : m;
        }
        if (lane == 0 && m > 0.0) atomicMax(args.maxbits + lo, (unsigned long long)__double_as_longlong(m));
    }
}

// All interpolated filter coefficients of the up-sampling converter: row F (the 16-bit fraction of the time register)
// holds the 13 left-wing and 13 right-wing coefficients of an output with that fraction, computed with the reference's two
// operations per coefficient (TRMSampleRateConverter.m:179-203).  Built once per context.
template <typename R>
__global__ void src_ctab_kernel(const HD<R> *__restrict__ tab, R *__restrict__ ctab)
{
    const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned row = i / SRC_CLD, t = i - row * SRC_CLD;
    if (row >= 65536u) return;
    R c = (R)0;
    if (t < (unsigned)SRC_TAPS) {
        const bool right = t >= (unsigned)SRC_ZC;
        const unsigned F = right ? ((~row) & 0xFFFFu) : row;
        const HD<R> a = tab[(F >> 8) * SRC_ZC + (right ? t - SRC_ZC : t)];
        c = a.h + a.dh * ((R)(F & 255u) / (R)256);
    }
    ctab[i] = c;
}

template <typename R>
__global__ void __launch_bounds__(PCM_THREADS) pcm_kernel(PcmArgs args)
{
  // blockIdx.y strides over the utterances (gridDim.y is capped at 65,535; larger batches loop)
  for (int u = args.u_begin + blockIdx.y; u < args.n_utt; u += gridDim.y) {
    const trm_cuda_utterance *__restrict__ D = args.desc + u;
    const long long n_out = D->n_out;
    const long long n0 = ((long long)blockIdx.x * PCM_THREADS + threadIdx.x) * PCM_PER_THREAD;
    if (n0 >= n_out) continue;
    const double mx = __longlong_as_double((long long)args.maxbits[u]);
    const double scale = (32767.0 / mx) * D->volumeAmp;                  // TRMTubeModel.m:515
    const R *__restrict__ z = reinterpret_cast<const R *>(args.out) + D->out_offset + n0;
    alignas(16) R v[PCM_PER_THREAD];
    const bool full = n0 + PCM_PER_THREAD <= n_out;
    if (full) {
        // out_offset and n0 are multiples of 8 elements: 128-bit loads
        constexpr int NV = (int)(PCM_PER_THREAD * sizeof(R) / 16);
        const float4 *zv = reinterpret_cast<const float4 *>(z);
        float4 *vv = reinterpret_cast<float4 *>(v);
#pragma unroll
        for (int i = 0; i < NV; ++i) vv[i] = zv[i];
    } else {
        for (int i = 0; i < PCM_PER_THREAD; ++i) v[i] = (n0 + i < n_out) ? z[i] : (R)0;
    }
    if (D->channels == 2) {
        const double ls = D->leftGain * scale, rs = D->rightGain * scale;  // TRMTubeModel.m:532-533
        int16_t *p = args.pcm + D->pcm_offset + 2 * n0;
        alignas(16) short2 q[PCM_PER_THREAD];
#pragma unroll
        for (int i = 0; i < PCM_PER_THREAD; ++i) {
            q[i].x = (short)__double2int_rn((double)v[i] * ls);
            q[i].y = (short)__double2int_rn((double)v[i] * rs);
        }
        if (full) {
            int4 *pv = reinterpret_cast<int4 *>(p);
            const int4 *qv = reinterpret_cast<const int4 *>(q);
            pv[0] = qv[0];
            pv[1] = qv[1];
        } else {
            for (int i = 0; i < PCM_PER_THREAD && n0 + i < n_out; ++i) reinterpret_cast<short2 *>(p)[i] = q[i];
        }
    } else {
        int16_t *p = args.pcm + D->pcm_offset + n0;
        alignas(16) short q[PCM_PER_THREAD];
#pragma unroll
        for (int i = 0; i < PCM_PER_THREAD; ++i) q[i] = (short)__double2int_rn((double)v[i] * scale);
        if (full) {
            *reinterpret_cast<int4 *>(p) = *reinterpret_cast<const int4 *>(q);
        } else {
            for (int i = 0; i < PCM_PER_THREAD && n0 + i < n_out; ++i) p[i] = q[i];
        }
    }
  }
}

}  // namespace TRM_KERNEL_NS
