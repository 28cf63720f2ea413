// tube_wide.cuh -- the TRM waveguide kernel for sm_100a.
//
// Replaces the sample-rate loop of -[TRMTubeModel synthesize] (/root/reference/Frameworks/Tube/TRMTubeModel.m:292-354) and
// everything it calls: parameter interpolation (m:611-688), frequency()/amplitude() (TRMUtility.m:26-47), tube and
// frication coefficients (m:712-773), band-pass coefficients/filter (TRMFilters.m:9-29), noise + one-zero low-pass
// (TRMUtility.m:71-85, TRMFilters.m:81-86), glottal wavetable + 2x oversampling oscillator + 49-tap FIR
// (TRMWavetable.m:117-195, TRMFIRFilter.m:116-146), source mixing (m:305-337), Kelly-Lochbaum ladder with the velum
// 3-way junction and nasal branch (m:778-853), mouth/nose reflection + radiation filters (TRMFilters.m:34-60) and the
// throat low-pass (TRMFilters.m:64-77).  The work is split by KIND, not by utterance:
//
//   feed-forward warps (one per utterance pair; lane = parameter in the interpolation phase S0, lane = sample t of a
//       16-sample block in the phases A1 / S1 / A2): parameter interpolation, conversions, junction / tap / band-pass
//       coefficients, jump-ahead noise, oscillator position, glottal table, 49-tap FIR, source mixing.  Nothing here
//       depends on the tube state.  Results go to a shared-memory ring of per-sample coefficient records.
//   ONE recurrence warp per CTA (lane = utterance): the strictly sequential part only -- Kelly-Lochbaum ladder,
//       velum 3-way junction, nasal branch, mouth / nose reflection + radiation filters, frication band-pass
//       and throat low-pass recursions (TRMTubeModel.m:778-853, TRMFilters.m:19-29,47-77).  All 32 waves and
//       9 filter memories of an utterance live in that lane's registers; the 16 junctions of one sample are
//       independent of each other (they read the previous time slice only), so the lane has 16-wide ILP and
//       there is NO cross-lane traffic: no shuffles, no role blends.
//
// One CTA per SM, up to 28 utterances per CTA; the ring is double-buffered so the feed-forward warps work on block b+1
// while the recurrence warp consumes block b (mbarrier full / empty pairs).  Control frames are staged by TMA bulk copies
// (cp.async.bulk + mbarrier, FRAME_CHUNK frames ahead of the sample loop).  Tube-rate output is transposed through shared
// memory and stored with 128-bit coalesced stores.
//
// Real = double : FP64 conformance mode (this file's cheaper forms, FMA contraction) or, with TRM_STRICT, the reference's
//                 operations in the reference's order (that TU is compiled with -fmad=false).
// Real = float  : FP32 fast mode: state/signal/coefficients FP32; parameter interpolation, pitch -> increment -> table
//                 position, the glottal-closure decision rint(ax*tnDelta) and the noise MCG stay FP64 / integer
//                 (SURVEY.md Appendix E).
#pragma once

#include <stdio.h>

#include "tube_common.cuh"

namespace TRM_KERNEL_NS {
using namespace trm;

// Arithmetic of this translation unit's double instantiation (kernel_args.h):
//   STRICT (kernels_f64s.cu, -fmad=false): the reference's operations in the reference's order -- sequential oscillator
//       chain, IEEE divisions, library exp2 / exp10 / tan / cos every sample, one-chain FIR sum, ladder as written in
//       TRMTubeModel.m:778-853.
//   conformance (kernels_f64.cu): the same values to <= 1e-9 (measured ~1e-12) from cheaper forms --
//       * every transcendental on the path is a function of a parameter that is LINEAR inside a control interval, so
//         2^(a + j b), 10^(a + j b), cos / sin(a + j b) are geometric sequences: the parameter lanes seed a complex value
//         and its per-sample ratio at each control frame (two exp2 or two sincos per frame, not per sample) and step it
//         with one complex multiplication per sample next to the interpolation add;
//       * oscillator phase in 64-bit fixed point with a warp scan (as the FP32 mode) instead of a 32-step dependent chain
//         walked by every lane;
//       * reflection coefficients from a Newton-refined hardware reciprocal; damping folded into them (k d), so that a
//         two-port junction of the ladder is 4 operations (e = a - b, x = kd e, fma(a, d, x), fma(b, d, x)) instead of 7;
//       * FIR as four partial sums of fused multiply-adds.
//     The discontinuous decisions of the path (glottal closure point rint(ax tnDelta), amplitude() clamps, frication
//     tap position, table indices) are taken on exactly interpolated parameters; the closure point is re-evaluated with
//     a directly computed amplitude whenever the product comes within 1e-6 of a rounding boundary.
constexpr bool STRICT = TRM_STRICT != 0;

template <typename R> struct Wide;
template <> struct Wide<float> {
    using Unit = float4;
    static constexpr int MAX_PAIRS = 14;
    static constexpr int NF = 11;                    // 16-byte units per utterance-sample
    static constexpr int UP = 2 * MAX_PAIRS + 1;     // padded utterance dimension: odd -> conflict-free writers
    static constexpr int THREADS = 32 * (2 + MAX_PAIRS);   // recurrence warp + feed-forward warps + one idle warp
    static constexpr int OUT_LD = 20;                // 16-byte aligned rows of the output transpose tile
    static constexpr int REGS_HI = 0, REGS_DONOR = 0;   // no register redistribution
};
template <> struct Wide<double> {
    using Unit = double2;
    static constexpr int MAX_PAIRS = 14;
    static constexpr int NF = STRICT ? 12 : 10;      // conformance: the frication taps travel as two values and a mask
    static constexpr int UP = 2 * MAX_PAIRS + 1;
    static constexpr int OUT_LD = 18;
    // Register redistribution (conformance mode): the CTA is launched with one extra warpgroup, which caps every thread
    // at 65536 / 640 -> 96 registers; the extra warpgroup gives its registers back at once (setmaxnreg.dec 24) and
    // exits, and warpgroup 0 -- the recurrence warp, which carries 41 FP64 state values per lane and needs its per-sample
    // record in flight to cover load and FP64 latencies -- takes them (setmaxnreg.inc): 96 + 72 = 168.
#ifndef TRM_DONOR_WARPS
#define TRM_DONOR_WARPS 4
#endif
    static constexpr int DONORS = STRICT ? 0 : TRM_DONOR_WARPS;
    static constexpr int THREADS = 32 * (2 + MAX_PAIRS) + 32 * DONORS;
    static constexpr int REGS_BASE = (65536 / THREADS) / 8 * 8;                      // what __launch_bounds__ gives every thread
    static constexpr int REGS_DONOR = 24;
    static constexpr int REGS_HI = DONORS ? (REGS_BASE + (DONORS * 32 * (REGS_BASE - REGS_DONOR) / 128) / 8 * 8) : 0;
};
constexpr int WIDE_SLOTS = 2;
// Warp w is scheduled by SM sub-partition w % 4, and the recurrence warp (warp 0) alone keeps its partition's FP64
// pipe busy for ~2.6 feed-forward warps' worth of a block.  Warp WIDE_IDLE_WARP (same partition) therefore exits at
// once and its pair moves to warp 15: partitions carry {recurrence + 2, 4, 4, 4} feed-forward warps instead of
// {recurrence + 3, 4, 4, 3}.
constexpr int WIDE_IDLE_WARP = 12;

// Oscillator history (even / odd 2x-rate samples) that the 49-tap FIR of a block reads: FIR_HIST old values, then the
// block's TB new ones.  FP64 conformance mode keeps a circular buffer of FIR_RING values whose first FIR_HIST entries are
// repeated past its end: the window of block b starts at TB * (b % 3) and is always contiguous, and a block only writes
// its new values (a value that lands in the repeated part is written twice).  Nothing moves, which saves a slide's
// shared-memory traffic and a warp barrier per block.  The other modes keep the window at the start of the buffer and
// slide it down by one block after every block (strict mode's 12-unit ring leaves no room for the larger buffer, and
// in FP32 fast mode the circular form costs the stream-pool kernel spills).
template <typename R> constexpr bool HIST_RING = sizeof(R) == 8 && !STRICT;
constexpr int FIR_RING = 3 * TB;                     // a multiple of TB, >= FIR_HIST + TB
template <typename R> constexpr int HIST_LEN = HIST_RING<R> ? FIR_RING + FIR_HIST : FIR_HIST + TB;

// feed-forward state of one utterance that must be in shared memory
template <typename R>
struct alignas(16) FFHalf {
    double FR[2][FRAME_CHUNK][16];           // TMA destination, double-buffered
    unsigned long long mbar[2];
    double CST[12];                          // per-utterance constants of the feed-forward phases (global loads of the
                                             // descriptor inside the block loop sat on the warp's critical path)
    double INC[TB];                          // oscillator increments of the block (conformance mode: every lane walks them)
    R HE[HIST_LEN<R>], HO[HIST_LEN<R>];      // oscillator history, even / odd 2x-rate samples
    R pad[16 / sizeof(R)];                   // FP32: size = 64 mod 128 bytes, so the two utterances of a warp (adjacent
                                             // FFHalf's, 16 consecutive floats each) read disjoint bank halves
};
static_assert(sizeof(FFHalf<float>) % 128 == 64, "FFHalf<float> must offset its neighbour by 16 banks");

template <typename R>
struct WideSmem {
    typename Wide<R>::Unit ring[WIDE_SLOTS][Wide<R>::NF][TB][Wide<R>::UP];
    FFHalf<R> ff[2 * Wide<R>::MAX_PAIRS];
    alignas(16) R outb[32][Wide<R>::OUT_LD];
    unsigned long long full[WIDE_SLOTS], empty[WIDE_SLOTS];
    double kc[sizeof(R) == 8 ? 18 : 1][32];   // conformance mode: per-utterance constants of the recurrence warp
    long long n_tube[32];
    R *out_ptr[32];
    long long n_cta;
};
static_assert(sizeof(WideSmem<double>) <= 227 * 1024 && sizeof(WideSmem<float>) <= 227 * 1024, "one CTA per SM: 227 kB");

// Waiting on a ring barrier.  try_wait returns after a short hardware-defined time whether or not the phase completed,
// so a bare loop around it spins: measured (ncu, round 2), the 14 feed-forward warps of a CTA waiting for the recurrence
// warp issued 47 % of ALL warp instructions of the kernel in this loop, through the very issue slots and shared-memory
// port the recurrence warp needs.  BACKOFF_NS > 0 parks the warp between polls (the feed-forward warps have two blocks
// of slack); the recurrence warp, which is the critical path, polls without a pause.
#ifndef TRM_PROFILE_PHASES
#define TRM_PROFILE_PHASES 0
#endif
#ifndef TRM_WAIT_NS
#define TRM_WAIT_NS 400
#endif
#ifndef TRM_WAIT_FULL_NS
#define TRM_WAIT_FULL_NS 100
#endif
template <int BACKOFF_NS>
__device__ __forceinline__ void mbar_wait_sleep(void *bar, uint32_t parity)
{
    uint32_t ok = 0;
    for (uint32_t spin = 0; !ok; ++spin) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(smem_u32(bar)), "r"(parity), "r"(0x989680u)
            : "memory");
        if (!ok) {
            if (BACKOFF_NS > 0) __nanosleep(BACKOFF_NS);
            if (spin > (1u << 22)) __trap();
        }
    }
}

// predicated shared-memory store as ONE instruction (@p STS): written as a C++ `if`, three of them per interpolation
// step became a divergent branch region with a reconvergence barrier -- per step -- in the parameter phase
__device__ __forceinline__ void sts_f64_if(bool pred, double *p, double v)
{
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %2, 0;\n\t@q st.shared.f64 [%0], %1;\n\t}" ::"r"(smem_u32(p)), "d"(v), "r"((unsigned)pred) : "memory");
}

__device__ __forceinline__ void mbar_arrive(void *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// streaming state of utterance u (kernel_args.h): header words and the R-typed part
template <typename R> __device__ __forceinline__ unsigned long long *state_hdr(void *state, int u)
{
    return reinterpret_cast<unsigned long long *>(reinterpret_cast<unsigned char *>(state) + (size_t)u * (STATE_HDR * 8 + STATE_R * sizeof(R)));
}
template <typename R> __device__ __forceinline__ R *state_vals(void *state, int u)
{
    return reinterpret_cast<R *>(state_hdr<R>(state, u) + STATE_HDR);
}

// Streaming state capture.  PER_UTT = false (batch and time split: every utterance of a CTA gets the same number of
// samples, or there is no state): the state is stored when the CTA's loop ends.  PER_UTT = true (stream pool,
// trm_cuda_pool_push: the utterances of one CTA may have different sample counts, and the warps keep running past an
// utterance's end until the longest one of the CTA is done): each utterance's state is stored at the end of the block
// that holds its last sample.  Two instantiations, so that the paths without per-utterance capture keep their code.
__device__ __forceinline__ bool ends_in_block(long long n_tube, int blk)
{
    const long long left = n_tube - (long long)blk * TB;
    return left > 0 && left <= TB;
}

struct WideArgs {
    TubeArgs t;
    int n_groups;      // CTAs; group g holds utterances order[start(g) .. start(g+1))
};
// Profiling builds only (never in the shipped library): -DTRM_PROFILE_SKIP=1 makes the feed-forward warps skip their
// work, =2 the recurrence warp, to time the two halves of the kernel separately.
#ifndef TRM_PROFILE_SKIP
#define TRM_PROFILE_SKIP 0
#endif

__device__ __forceinline__ void wide_group(int n, int n_groups, int g, int &start, int &count)
{
    const int base = n / n_groups, rem = n % n_groups;
    start = g * base + (g < rem ? g : rem);
    count = base + (g < rem ? 1 : 0);
}

// =========================================================================================================
// recurrence warp (warp 0 of the CTA): lane = utterance
// =========================================================================================================
template <typename R, bool PER_UTT>
__device__ __forceinline__ void wide_recurrence_warp(WideSmem<R> &W, const WideArgs &wargs, int g_start, int g_count, int n_blocks, int lane)
{
    constexpr bool FAST = sizeof(R) == 4;                  // FP32 fast mode
    constexpr bool F64C = !FAST && !STRICT;                // FP64 conformance mode (cheaper forms, see the top of the file)
    (void)F64C;
    const TubeArgs &args = wargs.t;
        // =====================================================================================================
        // recurrence warp
        // =====================================================================================================
        const bool has = lane < g_count;
        const int u = args.order ? args.order[g_start + (has ? lane : 0)] : g_start + (has ? lane : 0);
        const trm_cuda_utterance *__restrict__ D = args.desc + u;
        const R d = (R)D->dampingFactor;
        R *const orow = &W.outb[lane][0];

        if constexpr (FAST) {
            const float tb1 = (float)D->tb1, gain = (float)D->throatGain;
            const float m_b11 = (float)D->mouth[1], m_a20 = (float)D->mouth[2], m_a21 = (float)D->mouth[3], m_b21 = (float)D->mouth[4];
            const float n_b11 = (float)D->nose[1], n_a20 = (float)D->nose[2], n_a21 = (float)D->nose[3], n_b21 = (float)D->nose[4];
            // constant junctions: nasal N2|N3 .. N5|N6 and the nose termination, folded like the variable ones
            float nA[4], nB[4], nC[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const double k = D->nasal_coeff[q];
                nA[q] = (float)(D->dampingFactor * (1.0 + k));
                nB[q] = (float)(D->dampingFactor * k);
                nC[q] = (float)(D->dampingFactor * (1.0 - k));
            }
            const float nose_rk = (float)(D->dampingFactor * D->nose[0] * D->nasal_coeff[4]);    // d a10 k
            const float nose_1k = (float)(1.0 + D->nasal_coeff[4]);
            const float m_nb11 = -m_b11, n_nb11 = -n_b11;
            // waves: t[j] / bt[j] = top / bottom of oropharynx section Sj+1, nt / nb nasal
            float t[10], bt[10], nt[6], nb[6];
#pragma unroll
            for (int q = 0; q < 10; ++q) { t[q] = 0.0f; bt[q] = 0.0f; }
#pragma unroll
            for (int q = 0; q < 6; ++q) { nt[q] = 0.0f; nb[q] = 0.0f; }
            float m_ry = 0.0f, m_rx = 0.0f, m_rY = 0.0f, n_ry = 0.0f, n_rx = 0.0f, n_rY = 0.0f;
            float y1 = 0.0f, y2 = 0.0f, thy = 0.0f;
            float *const sv = (args.state && has) ? state_vals<float>(args.state, u) + STATE_SER : nullptr;
            if (sv) {                                      // streaming: continue where the previous call stopped
#pragma unroll
                for (int q = 0; q < 10; ++q) { t[q] = sv[q]; bt[q] = sv[10 + q]; }
#pragma unroll
                for (int q = 0; q < 6; ++q) { nt[q] = sv[20 + q]; nb[q] = sv[26 + q]; }
                m_ry = sv[32]; m_rx = sv[33]; m_rY = sv[34]; n_ry = sv[35]; n_rx = sv[36]; n_rY = sv[37];
                y1 = sv[38]; y2 = sv[39]; thy = sv[40];
            }

            for (int blk = 0; blk < n_blocks; ++blk) {
                const int slot = blk & 1;
                mbar_wait_sleep<TRM_WAIT_FULL_NS>(&W.full[slot], (uint32_t)((blk >> 1) & 1));
#pragma unroll 1
                for (int s0 = 0; s0 < ((TRM_PROFILE_SKIP & 2) ? 0 : TB); s0 += 4) {
                  float yo[4];
#pragma unroll
                  for (int si = 0; si < 4; ++si) {
                    const int s = s0 + si;
                    const float4 j0 = W.ring[slot][0][s][lane], j1 = W.ring[slot][1][s][lane], j2 = W.ring[slot][2][s][lane];
                    const float4 w3 = W.ring[slot][3][s][lane], j4 = W.ring[slot][4][s][lane], j6 = W.ring[slot][5][s][lane];
                    const float4 j7 = W.ring[slot][6][s][lane], j8 = W.ring[slot][7][s][lane], mo = W.ring[slot][8][s][lane];
                    const float4 j10 = W.ring[slot][9][s][lane], sc = W.ring[slot][10][s][lane];
                    // frication band-pass (TRMFilters.m:19-29; factor 2 folded into the coefficients) and throat low-pass
                    const float fr = (sc.y + (mo.w * y1)) - (j10.w * y2);
                    y2 = y1; y1 = fr;
                    const float th = sc.z + (tb1 * thy);
                    thy = th;
                    // glottis end (m:792) and S1|S2 (m:796-798)
                    const float t0n = (bt[0] * d) + sc.x;
                    const float t1n = (j0.x * t[0]) - (j0.y * bt[1]);
                    const float b0n = (j0.y * t[0]) + (j0.z * bt[1]);
                    // S2|S3, S3|S4 (m:803-807)
                    const float t2n = ((j1.x * t[1]) - (j1.y * bt[2])) + (j1.w * fr);
                    const float b1n = (j1.y * t[1]) + (j1.z * bt[2]);
                    const float t3n = ((j2.x * t[2]) - (j2.y * bt[3])) + (j2.w * fr);
                    const float b2n = (j2.y * t[2]) + (j2.z * bt[3]);
                    // velum 3-way junction (m:810-813): {d aL, d(aL-1), d aU, d(aU-1)}
                    const float uc = w3.z * nb[0];
                    const float b3n = ((w3.y * t[3]) + (w3.x * bt[4])) + uc;
                    const float t4n = (((w3.x * t[3]) + (w3.y * bt[4])) + uc) + (mo.z * fr);
                    const float nt0n = ((w3.x * t[3]) + (w3.x * bt[4])) + (w3.w * nb[0]);
                    // S5|S6 (m:816-818), S6|S7 pure delay (m:821-822)
                    const float t5n = ((j4.x * t[4]) - (j4.y * bt[5])) + (j4.w * fr);
                    const float b4n = (j4.y * t[4]) + (j4.z * bt[5]);
                    const float t6n = (t[5] * d) + (j0.w * fr);
                    const float b5n = bt[6] * d;
                    // S7|S8 .. S9|S10 (m:825-829)
                    const float t7n = ((j6.x * t[6]) - (j6.y * bt[7])) + (j6.w * fr);
                    const float b6n = (j6.y * t[6]) + (j6.z * bt[7]);
                    const float t8n = ((j7.x * t[7]) - (j7.y * bt[8])) + (j7.w * fr);
                    const float b7n = (j7.y * t[7]) + (j7.z * bt[8]);
                    const float t9n = ((j8.x * t[8]) - (j8.y * bt[9])) + (j8.w * fr);
                    const float b8n = (j8.y * t[8]) + (j8.z * bt[9]);
                    // mouth (m:832-835): bottom = d a10 k8 top - b11 bottom_prev ; radiation of (1+k8) top
                    const float b9n = (mo.x * t[9]) + (m_nb11 * m_ry);
                    m_ry = b9n;
                    const float xm = mo.y * t[9];
                    const float radm = ((m_a20 * xm) + (m_a21 * m_rx)) - (m_b21 * m_rY);
                    m_rx = xm; m_rY = radm;
                    // nasal branch (m:839-843): N1|N2 varies with the velum, the rest is constant
                    const float nt1n = (j10.x * nt[0]) - (j10.y * nb[1]);
                    const float nb0n = (j10.y * nt[0]) + (j10.z * nb[1]);
                    float ntn[6], nbn[6];
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        ntn[q + 2] = (nA[q] * nt[q + 1]) - (nB[q] * nb[q + 2]);
                        nbn[q + 1] = (nB[q] * nt[q + 1]) + (nC[q] * nb[q + 2]);
                    }
                    // nose (m:846-849)
                    const float nb5n = (nose_rk * nt[5]) + (n_nb11 * n_ry);
                    n_ry = nb5n;
                    const float xn = nose_1k * nt[5];
                    const float radn = ((n_a20 * xn) + (n_a21 * n_rx)) - (n_b21 * n_rY);
                    n_rx = xn; n_rY = radn;

                    t[0] = t0n; t[1] = t1n; t[2] = t2n; t[3] = t3n; t[4] = t4n; t[5] = t5n; t[6] = t6n; t[7] = t7n; t[8] = t8n; t[9] = t9n;
                    bt[0] = b0n; bt[1] = b1n; bt[2] = b2n; bt[3] = b3n; bt[4] = b4n; bt[5] = b5n; bt[6] = b6n; bt[7] = b7n; bt[8] = b8n;
                    bt[9] = b9n;
                    nt[0] = nt0n; nt[1] = nt1n; nb[0] = nb0n;
#pragma unroll
                    for (int q = 0; q < 4; ++q) { nt[q + 2] = ntn[q + 2]; nb[q + 1] = nbn[q + 1]; }
                    nb[5] = nb5n;
                    yo[si] = (radm + radn) + (th * gain);
                  }
                  *reinterpret_cast<float4 *>(&orow[s0]) = make_float4(yo[0], yo[1], yo[2], yo[3]);
                }
                __syncwarp(FULL);
                if (lane == 0) mbar_arrive(&W.empty[slot]);
                // transposed write-back: 4 lanes store the 16 samples of one utterance as 128-bit vectors
                {
                    const int64_t n0 = (int64_t)blk * TB;
#pragma unroll 1
                    for (int v0 = 0; v0 < g_count; v0 += 8) {
                        const int v = v0 + (lane >> 2), part = lane & 3;
                        if (v < g_count) {
                            const int64_t left = W.n_tube[v] - n0;
                            R *dst = W.out_ptr[v] + n0;
                            if (left >= TB) {
                                reinterpret_cast<float4 *>(dst)[part] = *reinterpret_cast<const float4 *>(&W.outb[v][4 * part]);
                            } else {
                                for (int i = 4 * part; i < 4 * part + 4; ++i)
                                    if (i < left) dst[i] = W.outb[v][i];
                            }
                        }
                    }
                }
                __syncwarp(FULL);
                if (PER_UTT && sv && ends_in_block(W.n_tube[lane], blk)) {
#pragma unroll
                    for (int q = 0; q < 10; ++q) { sv[q] = t[q]; sv[10 + q] = bt[q]; }
#pragma unroll
                    for (int q = 0; q < 6; ++q) { sv[20 + q] = nt[q]; sv[26 + q] = nb[q]; }
                    sv[32] = m_ry; sv[33] = m_rx; sv[34] = m_rY; sv[35] = n_ry; sv[36] = n_rx; sv[37] = n_rY;
                    sv[38] = y1; sv[39] = y2; sv[40] = thy;
                }
            }
            if (!PER_UTT && sv) {
#pragma unroll
                for (int q = 0; q < 10; ++q) { sv[q] = t[q]; sv[10 + q] = bt[q]; }
#pragma unroll
                for (int q = 0; q < 6; ++q) { sv[20 + q] = nt[q]; sv[26 + q] = nb[q]; }
                sv[32] = m_ry; sv[33] = m_rx; sv[34] = m_rY; sv[35] = n_ry; sv[36] = n_rx; sv[37] = n_rY;
                sv[38] = y1; sv[39] = y2; sv[40] = thy;
            }
        } else if constexpr (STRICT) {
            // ---- strict mode: the reference's operations in the reference's order -------------------------------
            // The 16 junctions of one sample are independent; the code is written stage by stage ACROSS the junctions
            // (all differences, then all k-products, ...) so that consecutive instructions are independent and the
            // FP64 pipe never waits on its own result.  Per-utterance constants other than the damping factor are read
            // from shared memory when needed: registers are for the 41 state values and the interleaving.
            enum { K_TB1, K_GAIN, K_MA10, K_MB11, K_MA20, K_MA21, K_MB21, K_NA10, K_NB11, K_NA20, K_NA21, K_NB21,
                   K_NK0, K_NK1, K_NK2, K_NK3, K_NK4 };
            {
                double (*kc)[32] = W.kc;
                kc[K_TB1][lane] = D->tb1; kc[K_GAIN][lane] = D->throatGain;
                kc[K_MA10][lane] = D->mouth[0]; kc[K_MB11][lane] = D->mouth[1]; kc[K_MA20][lane] = D->mouth[2];
                kc[K_MA21][lane] = D->mouth[3]; kc[K_MB21][lane] = D->mouth[4];
                kc[K_NA10][lane] = D->nose[0]; kc[K_NB11][lane] = D->nose[1]; kc[K_NA20][lane] = D->nose[2];
                kc[K_NA21][lane] = D->nose[3]; kc[K_NB21][lane] = D->nose[4];
#pragma unroll
                for (int q = 0; q < 5; ++q) kc[K_NK0 + q][lane] = D->nasal_coeff[q];
            }
            __syncwarp(FULL);
#define KC(i) (W.kc[i][lane])
            double t0 = 0, t1 = 0, t2 = 0, t3 = 0, t4 = 0, t5 = 0, t6 = 0, t7 = 0, t8 = 0, t9 = 0;
            double b0 = 0, b1 = 0, b2 = 0, b3 = 0, b4 = 0, b5 = 0, b6 = 0, b7 = 0, b8 = 0, b9 = 0;
            double nt0 = 0, nt1 = 0, nt2 = 0, nt3 = 0, nt4 = 0, nt5 = 0, nb0 = 0, nb1 = 0, nb2 = 0, nb3 = 0, nb4 = 0, nb5 = 0;
            double m_ry = 0.0, m_rx = 0.0, m_rY = 0.0, n_ry = 0.0, n_rx = 0.0, n_rY = 0.0;
            double y1 = 0.0, y2 = 0.0, thy = 0.0;
            double *const sv = (args.state && has) ? state_vals<double>(args.state, u) + STATE_SER : nullptr;
            if (sv) {                                      // streaming: continue where the previous call stopped
                t0 = sv[0]; t1 = sv[1]; t2 = sv[2]; t3 = sv[3]; t4 = sv[4]; t5 = sv[5]; t6 = sv[6]; t7 = sv[7]; t8 = sv[8]; t9 = sv[9];
                b0 = sv[10]; b1 = sv[11]; b2 = sv[12]; b3 = sv[13]; b4 = sv[14]; b5 = sv[15]; b6 = sv[16]; b7 = sv[17]; b8 = sv[18]; b9 = sv[19];
                nt0 = sv[20]; nt1 = sv[21]; nt2 = sv[22]; nt3 = sv[23]; nt4 = sv[24]; nt5 = sv[25];
                nb0 = sv[26]; nb1 = sv[27]; nb2 = sv[28]; nb3 = sv[29]; nb4 = sv[30]; nb5 = sv[31];
                m_ry = sv[32]; m_rx = sv[33]; m_rY = sv[34]; n_ry = sv[35]; n_rx = sv[36]; n_rY = sv[37];
                y1 = sv[38]; y2 = sv[39]; thy = sv[40];
            }

            for (int blk = 0; blk < n_blocks; ++blk) {
                const int slot = blk & 1;
                mbar_wait_sleep<TRM_WAIT_FULL_NS>(&W.full[slot], (uint32_t)((blk >> 1) & 1));
#pragma unroll 1
                for (int s0 = 0; s0 < ((TRM_PROFILE_SKIP & 2) ? 0 : TB); s0 += 2) {
                    double yo[2];
#pragma unroll
                    for (int si = 0; si < 2; ++si) {
                        const int s = s0 + si;
                        // record: {k0,k1} {k2,aL} {k4,k6} {k7,k8} {k9,k10} {aU,FC1} {FC2,FC3} {FC4,FC5} {FC6,FC7} {FC8,2g} {2b,in} {ff,thr}
                        const double2 q9 = W.ring[slot][9][s][lane], q10 = W.ring[slot][10][s][lane], q11 = W.ring[slot][11][s][lane];
                        const double2 q0 = W.ring[slot][0][s][lane], q1 = W.ring[slot][1][s][lane], q5 = W.ring[slot][5][s][lane];
                        const double2 q2 = W.ring[slot][2][s][lane], q3 = W.ring[slot][3][s][lane], q4 = W.ring[slot][4][s][lane];
                        // frication band-pass (TRMFilters.m:19-29, factor 2 folded in) and throat low-pass (TRMFilters.m:72-77)
                        const double fr = (q11.x + (q9.y * y1)) - (q10.x * y2);
                        y2 = y1; y1 = fr;
                        const double th = q11.y + (KC(K_TB1) * thy);
                        thy = th;
                        // ---- stage 1: differences / first products of every junction (m:792-849) ----
                        const double e0 = t0 - b1, e1 = t1 - b2, e2 = t2 - b3, e4 = t4 - b5, e6 = t6 - b7, e7 = t7 - b8, e8 = t8 - b9;
                        const double en0 = nt0 - nb1, en1 = nt1 - nb2, en2 = nt2 - nb3, en3 = nt3 - nb4, en4 = nt4 - nb5;
                        const double pa = q1.y * t3, pb = q1.y * b4, pc = q5.x * nb0;
                        const double g0 = b0 * d, g5 = t5 * d, h5 = b6 * d;
                        const double mk = q4.x * t9, mx1 = (1.0 + q4.x) * t9;
                        const double nkk = KC(K_NK4) * nt5, nx1 = (1.0 + KC(K_NK4)) * nt5;
                        // ---- stage 2: deltas ----
                        const double d0 = q0.x * e0, d1 = q0.y * e1, d2 = q1.x * e2, d4 = q2.x * e4, d6 = q2.y * e6, d7 = q3.x * e7, d8 = q3.y * e8;
                        const double dn0 = q4.y * en0, dn1 = KC(K_NK0) * en1, dn2 = KC(K_NK1) * en2, dn3 = KC(K_NK2) * en3, dn4 = KC(K_NK3) * en4;
                        const double jp = (pa + pb) + pc;
                        const double mr1 = KC(K_MA10) * mk, mr2 = KC(K_MB11) * m_ry;
                        const double nr1 = KC(K_NA10) * nkk, nr2 = KC(K_NB11) * n_ry;
                        const double ma = KC(K_MA20) * mx1, mb = KC(K_MA21) * m_rx, mc = KC(K_MB21) * m_rY;
                        const double na = KC(K_NA20) * nx1, nbb = KC(K_NA21) * n_rx, nc = KC(K_NB21) * n_rY;
                        // ---- stage 3: sums ----
                        const double u1 = t0 + d0, v0 = b1 + d0, u2 = t1 + d1, v1 = b2 + d1, u3 = t2 + d2, v2 = b3 + d2;
                        const double u5 = t4 + d4, v4 = b5 + d4, u7 = t6 + d6, v6 = b7 + d6, u8 = t7 + d7, v7 = b8 + d7, u9 = t8 + d8, v8 = b9 + d8;
                        const double w3 = jp - t3, w4 = jp - b4, wn = jp - nb0;
                        const double un1 = nt0 + dn0, vn0 = nb1 + dn0, un2 = nt1 + dn1, vn1 = nb2 + dn1, un3 = nt2 + dn2, vn2 = nb3 + dn2;
                        const double un4 = nt3 + dn3, vn3 = nb4 + dn3, un5 = nt4 + dn4, vn4 = nb5 + dn4;
                        const double refl = mr1 - mr2, refn = nr1 - nr2;
                        const double radm = (ma + mb) - mc, radn = (na + nbb) - nc;
                        const double f1 = q5.y * fr;
                        // the remaining taps are loaded late: their registers are free again by now
                        const double2 q6 = W.ring[slot][6][s][lane], q7 = W.ring[slot][7][s][lane], q8 = W.ring[slot][8][s][lane];
                        const double f2 = q6.x * fr, f3 = q6.y * fr, f4 = q7.x * fr, f5 = q7.y * fr, f6 = q8.x * fr, f7 = q8.y * fr, f8 = q9.x * fr;
                        // ---- stage 4: damping, stage 5: frication injection ----
                        m_ry = refl; m_rx = mx1; m_rY = radm;
                        n_ry = refn; n_rx = nx1; n_rY = radn;
                        const double nt0n = wn * d;
                        t0 = g0 + q10.y;
                        t1 = u1 * d;             b0 = v0 * d;
                        t2 = (u2 * d) + f1;      b1 = v1 * d;
                        t3 = (u3 * d) + f2;      b2 = v2 * d;
                        b3 = w3 * d;
                        const double t4n = (w4 * d) + f3;
                        t5 = (u5 * d) + f4;      b4 = v4 * d;
                        t6 = g5 + f5;            b5 = h5;
                        t7 = (u7 * d) + f6;      b6 = v6 * d;
                        t8 = (u8 * d) + f7;      b7 = v7 * d;
                        t9 = (u9 * d) + f8;      b8 = v8 * d;
                        b9 = d * refl;
                        t4 = t4n;
                        nt1 = un1 * d;           nb0 = vn0 * d;
                        nt2 = un2 * d;           nb1 = vn1 * d;
                        nt3 = un3 * d;           nb2 = vn2 * d;
                        nt4 = un4 * d;           nb3 = vn3 * d;
                        nt5 = un5 * d;           nb4 = vn4 * d;
                        nb5 = d * refn;
                        nt0 = nt0n;
                        yo[si] = (radm + radn) + (th * KC(K_GAIN));
                    }
                    *reinterpret_cast<double2 *>(&orow[s0]) = make_double2(yo[0], yo[1]);
                }
#undef KC
                __syncwarp(FULL);
                if (lane == 0) mbar_arrive(&W.empty[slot]);
                {
                    const int64_t n0 = (int64_t)blk * TB;
#pragma unroll 1
                    for (int v0 = 0; v0 < g_count; v0 += 4) {
                        const int v = v0 + (lane >> 3), part = lane & 7;
                        if (v < g_count) {
                            const int64_t left = W.n_tube[v] - n0;
                            R *dst = W.out_ptr[v] + n0;
                            if (left >= TB) {
                                reinterpret_cast<float4 *>(dst)[part] = *reinterpret_cast<const float4 *>(&W.outb[v][2 * part]);
                            } else {
                                for (int i = 2 * part; i < 2 * part + 2; ++i)
                                    if (i < left) dst[i] = W.outb[v][i];
                            }
                        }
                    }
                }
                __syncwarp(FULL);
                if (PER_UTT && sv && ends_in_block(W.n_tube[lane], blk)) {
                    sv[0] = t0; sv[1] = t1; sv[2] = t2; sv[3] = t3; sv[4] = t4; sv[5] = t5; sv[6] = t6; sv[7] = t7; sv[8] = t8; sv[9] = t9;
                    sv[10] = b0; sv[11] = b1; sv[12] = b2; sv[13] = b3; sv[14] = b4; sv[15] = b5; sv[16] = b6; sv[17] = b7; sv[18] = b8; sv[19] = b9;
                    sv[20] = nt0; sv[21] = nt1; sv[22] = nt2; sv[23] = nt3; sv[24] = nt4; sv[25] = nt5;
                    sv[26] = nb0; sv[27] = nb1; sv[28] = nb2; sv[29] = nb3; sv[30] = nb4; sv[31] = nb5;
                    sv[32] = m_ry; sv[33] = m_rx; sv[34] = m_rY; sv[35] = n_ry; sv[36] = n_rx; sv[37] = n_rY;
                    sv[38] = y1; sv[39] = y2; sv[40] = thy;
                }
            }
            if (!PER_UTT && sv) {
                sv[0] = t0; sv[1] = t1; sv[2] = t2; sv[3] = t3; sv[4] = t4; sv[5] = t5; sv[6] = t6; sv[7] = t7; sv[8] = t8; sv[9] = t9;
                sv[10] = b0; sv[11] = b1; sv[12] = b2; sv[13] = b3; sv[14] = b4; sv[15] = b5; sv[16] = b6; sv[17] = b7; sv[18] = b8; sv[19] = b9;
                sv[20] = nt0; sv[21] = nt1; sv[22] = nt2; sv[23] = nt3; sv[24] = nt4; sv[25] = nt5;
                sv[26] = nb0; sv[27] = nb1; sv[28] = nb2; sv[29] = nb3; sv[30] = nb4; sv[31] = nb5;
                sv[32] = m_ry; sv[33] = m_rx; sv[34] = m_rY; sv[35] = n_ry; sv[36] = n_rx; sv[37] = n_rY;
                sv[38] = y1; sv[39] = y2; sv[40] = thy;
            }
        } else {
            // ---- FP64 conformance mode: damping folded into the reflection coefficients, fused multiply-adds ----------
            // A two-port junction with incident waves a (from the left) and b (from the right), k d = kd:
            //     e = a - b;  x = kd e;  right-going = fma(a, d, x) (+ tap fr);  left-going = fma(b, d, x)
            // which is (a + k e) d and (b + k e) d of TRMTubeModel.m:796-829 with one rounding placed differently.
            // Record of one sample (feed-forward warps, below):
            //   {kd0,kd1} {kd2,aL d} {kd4,kd6} {kd7,kd8} {k9,kd10} {aU d,2g} {2b,tsel} {tE,tO} {in,ff} {thr,-}
            // Frication tap k (FC(k+1), injected into junction k) is tE / tO for an even / odd k if bit k of tsel is set,
            // else +0 -- the same value the reference's eight-tap array holds (at most two taps are non-zero), so every
            // junction still adds tap * fr with the same fused multiply-add and the same bits: selects replace the loads of
            // six zeros.
            // Per-utterance constants live in registers (the warp has 168 of them): the shared-memory pipe is this kernel's
            // bottleneck (ncu: 74 % of its wavefront rate), and 17 constant loads per sample were 11 % of the traffic.
            const double c_tb1 = D->tb1, c_gain = D->throatGain;
            const double c_ma10 = D->mouth[0], c_mb11 = D->mouth[1], c_ma20 = D->mouth[2];
            const double c_na10 = D->nose[0], c_nb11 = D->nose[1], c_na20 = D->nose[2];
            const double c_nk0 = D->nasal_coeff[0] * D->dampingFactor, c_nk1 = D->nasal_coeff[1] * D->dampingFactor;      // constant junctions: kd
            const double c_nk2 = D->nasal_coeff[2] * D->dampingFactor, c_nk3 = D->nasal_coeff[3] * D->dampingFactor;
            const double c_nk4 = D->nasal_coeff[4];
            double t[10], bt[10], nt[6], nb[6];
#pragma unroll
            for (int q = 0; q < 10; ++q) { t[q] = 0.0; bt[q] = 0.0; }
#pragma unroll
            for (int q = 0; q < 6; ++q) { nt[q] = 0.0; nb[q] = 0.0; }
            double m_ry = 0.0, m_rx = 0.0, m_rY = 0.0, n_ry = 0.0, n_rx = 0.0, n_rY = 0.0;
            double y1 = 0.0, y2 = 0.0, thy = 0.0;
            double *const sv = (args.state && has) ? state_vals<double>(args.state, u) + STATE_SER : nullptr;
            if (sv) {                                      // streaming: continue where the previous call stopped
#pragma unroll
                for (int q = 0; q < 10; ++q) { t[q] = sv[q]; bt[q] = sv[10 + q]; }
#pragma unroll
                for (int q = 0; q < 6; ++q) { nt[q] = sv[20 + q]; nb[q] = sv[26 + q]; }
                m_ry = sv[32]; m_rx = sv[33]; m_rY = sv[34]; n_ry = sv[35]; n_rx = sv[36]; n_rY = sv[37];
                y1 = sv[38]; y2 = sv[39]; thy = sv[40];
            }

            for (int blk = 0; blk < n_blocks; ++blk) {
                const int slot = blk & 1;
                mbar_wait_sleep<TRM_WAIT_FULL_NS>(&W.full[slot], (uint32_t)((blk >> 1) & 1));
#pragma unroll 1
                for (int s0 = 0; s0 < ((TRM_PROFILE_SKIP & 2) ? 0 : TB); s0 += 2) {
                    double yo[2];
#pragma unroll
                    for (int si = 0; si < 2; ++si) {
                        const int s = s0 + si;
                        // Written stage by stage ACROSS the junctions: the operations of one stage are mutually independent,
                        // so the FP64 pipe (one warp instruction per ~2.25 cycles, 8-cycle latency) always has a ready one.
                        const double2 q5 = W.ring[slot][5][s][lane], q6 = W.ring[slot][6][s][lane], q8 = W.ring[slot][8][s][lane];
                        const double2 q9 = W.ring[slot][9][s][lane], q0 = W.ring[slot][0][s][lane], q1 = W.ring[slot][1][s][lane];
                        const double2 q2 = W.ring[slot][2][s][lane], q3 = W.ring[slot][3][s][lane], q4 = W.ring[slot][4][s][lane];
                        const double2 q7 = W.ring[slot][7][s][lane];
                        const unsigned tsel = (unsigned)__double_as_longlong(q6.y);
                        auto tap = [&](int k) { return (tsel & (1u << k)) ? ((k & 1) ? q7.y : q7.x) : 0.0; };
                        // ---- stage 1: differences, first products ----
                        const double fr1 = fma(q5.y, y1, q8.y);                       // band-pass (TRMFilters.m:19-29, factor 2 folded in)
                        const double th = fma(c_tb1, thy, q9.x);                      // throat low-pass (TRMFilters.m:72-77)
                        const double e0 = t[0] - bt[1], e1 = t[1] - bt[2], e2 = t[2] - bt[3], e4 = t[4] - bt[5];
                        const double e6 = t[6] - bt[7], e7 = t[7] - bt[8], e8 = t[8] - bt[9];
                        const double en0 = nt[0] - nb[1], en1 = nt[1] - nb[2], en2 = nt[2] - nb[3], en3 = nt[3] - nb[4], en4 = nt[4] - nb[5];
                        const double pa = q1.y * t[3];                                // velum 3-way junction (m:810-813), d folded in
                        const double mk = q4.x * t[9], nkk = c_nk4 * nt[5];           // mouth / nose (m:832-835, 846-849)
                        const double m1 = c_mb11 * m_ry, n1 = c_nb11 * n_ry;
                        const double g0 = fma(bt[0], d, q8.x);                        // glottis end (m:792)
                        const double h5 = bt[6] * d;                                  // S6|S7: pure delay (m:821-822)
                        // ---- stage 2: kd-products ----
                        const double fr = fma(-q6.x, y2, fr1);
                        const double x0 = q0.x * e0, x1 = q0.y * e1, x2 = q1.x * e2, x4 = q2.x * e4, x6 = q2.y * e6, x7 = q3.x * e7, x8 = q3.y * e8;
                        const double xn0 = q4.y * en0, xn1 = c_nk0 * en1, xn2 = c_nk1 * en2, xn3 = c_nk2 * en3, xn4 = c_nk3 * en4;
                        const double pb = fma(q1.y, bt[4], pa);
                        const double refl = fma(c_ma10, mk, -m1), refn = fma(c_na10, nkk, -n1);
                        const double mx1 = t[9] + mk, nx1 = nt[5] + nkk;
                        y2 = y1; y1 = fr; thy = th;
                        // ---- stage 3: waves before injection, radiation filters ----
                        const double jp = fma(q5.x, nb[0], pb);
                        const double u1 = fma(t[0], d, x0), v0 = fma(bt[1], d, x0);
                        const double u2 = fma(t[1], d, x1), v1 = fma(bt[2], d, x1);
                        const double u3 = fma(t[2], d, x2), v2 = fma(bt[3], d, x2);
                        const double u5 = fma(t[4], d, x4), v4 = fma(bt[5], d, x4);
                        const double u7 = fma(t[6], d, x6), v6 = fma(bt[7], d, x6);
                        const double u8 = fma(t[7], d, x7), v7 = fma(bt[8], d, x7);
                        const double u9 = fma(t[8], d, x8), v8 = fma(bt[9], d, x8);
                        const double un1 = fma(nt[0], d, xn0), vn0 = fma(nb[1], d, xn0);
                        const double un2 = fma(nt[1], d, xn1), vn1 = fma(nb[2], d, xn1);
                        const double un3 = fma(nt[2], d, xn2), vn2 = fma(nb[3], d, xn2);
                        const double un4 = fma(nt[3], d, xn3), vn3 = fma(nb[4], d, xn3);
                        const double un5 = fma(nt[4], d, xn4), vn4 = fma(nb[5], d, xn4);
                        const double f5 = tap(4) * fr;
                        // radiation filter (TRMFilters.m:47-60): a21 = b21 = -a20 by construction (TRMFilters.m:34-45), so
                        // a20 x + a21 x[n-1] - b21 y[n-1] = a20 ((x - x[n-1]) + y[n-1])
                        const double ra = mx1 - m_rx, rb = nx1 - n_rx;
                        const double b9n = d * refl, nb5n = d * refn;
                        // ---- stage 4: frication injection (m:803-829), 3-way outputs ----
                        const double rc = ra + m_rY, rd = rb + n_rY;
                        const double b3n = fma(-d, t[3], jp), w4 = fma(-d, bt[4], jp), nt0n = fma(-d, nb[0], jp);
                        const double t6n = fma(t[5], d, f5);
                        t[0] = g0;
                        t[1] = u1;                    bt[0] = v0;
                        t[2] = fma(tap(0), fr, u2);   bt[1] = v1;
                        t[3] = fma(tap(1), fr, u3);   bt[2] = v2;
                        t[5] = fma(tap(3), fr, u5);   bt[4] = v4;
                        t[7] = fma(tap(5), fr, u7);   bt[6] = v6;
                        t[8] = fma(tap(6), fr, u8);   bt[7] = v7;
                        t[9] = fma(tap(7), fr, u9);   bt[8] = v8;
                        t[4] = fma(tap(2), fr, w4);   bt[3] = b3n;
                        t[6] = t6n;                   bt[5] = h5;
                        bt[9] = b9n;
                        nt[0] = nt0n;
                        nt[1] = un1; nb[0] = vn0; nt[2] = un2; nb[1] = vn1; nt[3] = un3; nb[2] = vn2;
                        nt[4] = un4; nb[3] = vn3; nt[5] = un5; nb[4] = vn4; nb[5] = nb5n;
                        const double radm = c_ma20 * rc, radn = c_na20 * rd;
                        m_ry = refl; m_rx = mx1; m_rY = radm;
                        n_ry = refn; n_rx = nx1; n_rY = radn;
                        yo[si] = fma(th, c_gain, radm + radn);
                    }
                    *reinterpret_cast<double2 *>(&orow[s0]) = make_double2(yo[0], yo[1]);
                }
                __syncwarp(FULL);
                if (lane == 0) mbar_arrive(&W.empty[slot]);
                {
                    const int64_t n0 = (int64_t)blk * TB;
#pragma unroll 1
                    for (int v0 = 0; v0 < g_count; v0 += 4) {
                        const int v = v0 + (lane >> 3), part = lane & 7;
                        if (v < g_count) {
                            const int64_t left = W.n_tube[v] - n0;
                            R *dst = W.out_ptr[v] + n0;
                            if (left >= TB) {
                                reinterpret_cast<float4 *>(dst)[part] = *reinterpret_cast<const float4 *>(&W.outb[v][2 * part]);
                            } else {
                                for (int i = 2 * part; i < 2 * part + 2; ++i)
                                    if (i < left) dst[i] = W.outb[v][i];
                            }
                        }
                    }
                }
                __syncwarp(FULL);
                if (PER_UTT && sv && ends_in_block(W.n_tube[lane], blk)) {
#pragma unroll
                    for (int q = 0; q < 10; ++q) { sv[q] = t[q]; sv[10 + q] = bt[q]; }
#pragma unroll
                    for (int q = 0; q < 6; ++q) { sv[20 + q] = nt[q]; sv[26 + q] = nb[q]; }
                    sv[32] = m_ry; sv[33] = m_rx; sv[34] = m_rY; sv[35] = n_ry; sv[36] = n_rx; sv[37] = n_rY;
                    sv[38] = y1; sv[39] = y2; sv[40] = thy;
                }
            }
            if (!PER_UTT && sv) {
#pragma unroll
                for (int q = 0; q < 10; ++q) { sv[q] = t[q]; sv[10 + q] = bt[q]; }
#pragma unroll
                for (int q = 0; q < 6; ++q) { sv[20 + q] = nt[q]; sv[26 + q] = nb[q]; }
                sv[32] = m_ry; sv[33] = m_rx; sv[34] = m_rY; sv[35] = n_ry; sv[36] = n_rx; sv[37] = n_rY;
                sv[38] = y1; sv[39] = y2; sv[40] = thy;
            }
        }
}

// =========================================================================================================
// feed-forward warp: utterances 2*pair and 2*pair+1 of the group, lane = sample of a 16-sample block
// (phases S0 / A1 / S1 / A2; the results go to the ring)
// =========================================================================================================
template <typename R, bool PER_UTT>
__device__ __forceinline__ void wide_feed_forward_warp(WideSmem<R> &W, const WideArgs &wargs, int g_start, int g_count, int n_blocks, int pair, int lane)
{
    constexpr bool FAST = sizeof(R) == 4;                  // FP32 fast mode
    constexpr bool F64C = !FAST && !STRICT;                // FP64 conformance mode (cheaper forms, see the top of the file)
    (void)F64C;
    const TubeArgs &args = wargs.t;
    const int half = lane >> 4, hl = lane & 15;
    const int ucol = 2 * pair + half;                     // column of this half's utterance in the ring
    FFHalf<R> &S = W.ff[ucol];
    const bool has_utt = ucol < g_count;
    const int u = args.order ? args.order[g_start + (has_utt ? ucol : 0)] : g_start + (has_utt ? ucol : 0);
    const trm_cuda_utterance *__restrict__ D = args.desc + u;
    // a half without an utterance (odd group size) recomputes the group's first utterance into a ring column nobody
    // reads: all-zero parameters would send every division and transcendental of that half down its slow path
    const int64_t n_tube = D->n_tube;
    const int n_frames = D->n_frames;
    const int cp = D->controlPeriod;
    // control frames: rows of 16 doubles (128 bytes) or, when the caller gave float32 rows, of 16 floats (64 bytes) --
    // staged as they are and widened when a parameter lane reads its value (exact)
    const uint32_t frow = args.frames_f32 ? 64u : 128u;
    const unsigned char *__restrict__ F = reinterpret_cast<const unsigned char *>(args.frames) + (size_t)D->frame_offset * frow;
    auto staged = [&](int buf, int row) -> double {
        return args.frames_f32 ? (double)reinterpret_cast<const float *>(&S.FR[buf][0][0])[row * 16 + hl] : S.FR[buf][row][hl];
    };
    const double *__restrict__ wt_base = args.wavetables + (size_t)D->voice * TRM_TABLE_LENGTH;
    const bool pulse_wave = D->waveform == 0;
    const bool modulation = D->usesModulation != 0;
    const int div1 = D->div1, div2 = D->div2;

    enum { C_BASICINC, C_TNDELTA, C_DAMP, C_SR, C_NR1SQ, C_APSCALE2, C_MOUTH0, C_BF, C_CMIX, C_TA0, C_RSR, C_INVDIV1 };
    if (hl == 0) {
        S.CST[C_BASICINC] = D->basicIncrement; S.CST[C_TNDELTA] = D->tnDelta; S.CST[C_DAMP] = D->dampingFactor;
        S.CST[C_SR] = D->sampleRate; S.CST[C_RSR] = 1.0 / D->sampleRate; S.CST[C_NR1SQ] = D->nr1sq; S.CST[C_APSCALE2] = D->apScale2; S.CST[C_MOUTH0] = D->mouth[0];
        S.CST[C_BF] = D->breathinessFactor; S.CST[C_CMIX] = D->crossmixFactor; S.CST[C_TA0] = D->ta0;
        S.CST[C_INVDIV1] = 1.0 / (double)D->div1;
    }
    const bool feeds = n_tube > 0;
    const int n_chunks = (n_frames + FRAME_CHUNK - 1) / FRAME_CHUNK;
    if (hl == 0 && feeds) {
        mbar_init(&S.mbar[0], 1);
        mbar_init(&S.mbar[1], 1);
        mbar_fence_init();
    }
    __syncwarp(FULL);
    if (hl == 0 && feeds) {
        for (int c = 0; c < 2 && c < n_chunks; ++c) {
            int cnt = min(FRAME_CHUNK, n_frames - c * FRAME_CHUNK);
            mbar_expect_tx(&S.mbar[c], (uint32_t)cnt * frow);
            tma_bulk_g2s(&S.FR[c][0][0], F + (size_t)c * FRAME_CHUNK * frow, (uint32_t)cnt * frow, &S.mbar[c]);
        }
    }
    if (feeds) mbar_wait(&S.mbar[0], 0);

    double p_cur = 0.0, p_delta = 0.0, p_next = feeds ? staged(0, 0) : 0.0;
    int f_idx = 0, jc = 0;
    double pos = 0.0;
    unsigned long long pos_fx = 0ull;
    unsigned long long kb = args.noise_k0;
    bool fresh = true;                     // no sample of this utterance exists yet (first-sample rule of the noise filter)
    unsigned long long *const st_h = (args.state && has_utt) ? state_hdr<R>(args.state, u) : nullptr;
    R *const st_v = st_h ? state_vals<R>(args.state, u) : nullptr;
    const unsigned long long MASK44 = (1ull << 44) - 1ull;
    const unsigned long long pw1 = c_noise_pow[hl + 1], pwB = c_noise_pow[TB];
    R xm1 = 0, xm2 = 0;
    int hs = 0;                                            // oscillator history: start of this block's FIR window
    const int pf = hl >> 1, pc = hl & 1;                   // parameter lane -> (unit, component) of the staged value
    if (st_h) {
        // streaming: oscillator position, noise generator, oscillator / band-pass input history of the previous call
        pos = __longlong_as_double((long long)st_h[0]);
        pos_fx = st_h[1];
        kb = st_h[2];
        fresh = st_h[3] != 0ull;
        xm1 = st_v[STATE_XM]; xm2 = st_v[STATE_XM + 1];
        for (int i = hl; i < FIR_HIST; i += TB) {
            const R e = st_v[STATE_HE + i], o = st_v[STATE_HO + i];
            S.HE[i] = e; S.HO[i] = o;
            if (HIST_RING<R>) { S.HE[FIR_RING + i] = e; S.HO[FIR_RING + i] = o; }
        }
    }
    // FP64 conformance mode: parameter lane p also carries function p of its parameter as a complex number (rc, rs) that
    // is multiplied by (dc, ds) every sample -- geometric for the exponentials (rs = ds = 0), a rotation for the angles:
    //   0 pitch    -> oscillator increment (220 * 2^((p+3)/12) / 2) * basicIncrement   (TRMUtility.m:44-47, TRMWavetable.m:165)
    //   1..3 dB    -> 10^((p-60)/20), unclamped (the clamps of amplitude() are applied per sample on the exact parameter)
    //   5 centre f -> cos(2 pi p / sr)        6 bandwidth -> cos, sin(pi p / sr)        (TRMFilters.m:9-17)
    double rc = 0.0, rs = 0.0, dc = 0.0, ds = 0.0;
    // (FP32 fast mode: only function 0 -- the oscillator increment, which that mode keeps in double -- is carried this way;
    //  its lane stages the increment in place of the pitch, which nothing else reads)
    constexpr bool GEO = F64C || FAST;                      // modes whose parameter lanes carry functions
    const bool fn_exp = F64C ? hl < 4 : hl == 0, fn_rot = F64C && ((hl == 5) | (hl == 6));
    const double fn_w = GEO ? (hl == 0 ? (1.0 / 12.0) : (hl < 4 ? 0.16609640474436813 : (hl == 5 ? 6.28318530717958647692 : 3.14159265358979323846) / D->sampleRate)) : 0.0;
    const double fn_off = hl == 0 ? 3.0 : -60.0, fn_scale = hl == 0 ? 110.0 * D->basicIncrement : 1.0;
    auto seed_functions = [&](double pc0, double pd0, double &c, double &sn, double &cd, double &sd) {
        // for a control interval that starts at pc0 and moves by pd0 per sample: two exp2 or two sincos per interval
        if (fn_exp) {
            c = fn_scale * exp2_inline((pc0 + fn_off) * fn_w);
            cd = exp2_inline(pd0 * fn_w);
            sn = 0.0; sd = 0.0;
        } else if (fn_rot) {
            sincos_inline(pc0 * fn_w, &sn, &c);
            sincos_inline(pd0 * fn_w, &sd, &cd);
        }
    };
    auto step_functions = [&]() {
        const double c2 = fma(-rs, ds, rc * dc);
        rs = fma(rc, ds, rs * dc);
        rc = c2;
    };
    if (feeds && D->jc0 > 0 && n_frames > 1) {
        // the call starts inside a control interval: redo its jc0 interpolation adds (exactly the reference's sequence)
        const double nxt = staged(0, 1);
        p_cur = p_next;
        p_delta = (nxt - p_cur) / (double)cp;
        p_next = nxt;
        if constexpr (GEO) seed_functions(p_cur, p_delta, rc, rs, dc, ds);
        for (int i = 0; i < D->jc0; ++i) {
            p_cur += p_delta;
            if constexpr (F64C) step_functions(); else if constexpr (FAST) rc *= dc;
        }
        jc = D->jc0;
    }
    // conformance-mode staging: where this parameter lane puts its value / its function inside the ring slot.  Unit
    // u (16 bytes) of sample t sits at ring[slot][u][(t + u) & 15][ucol]; the reader (lane = sample) takes units 0..9:
    //   {p1,p2} {p3,p4} {r1,r2} {r3,r4} {r5,r6} {r7,r8} {velum,sin6} {inc,c1} {c2,c3} {cos5,cos6}
    // Two stores per lane and step: store A carries the parameter (lane 6, whose parameter nobody reads, sends the sine
    // of its angle through it), store B the function value -- every store instruction of the parameter phase costs
    // shared-memory wavefronts, the resource that bounds this kernel.
    const int uA = F64C ? (hl == 6 ? 6 : (hl >= 7 ? (hl - 3) >> 1 : (hl - 1) >> 1)) : pf, cA = F64C ? (hl == 6 ? 1 : (hl >= 7 ? (hl - 3) & 1 : (hl - 1) & 1)) : pc;
    const bool wantA = !F64C || !(hl == 0 || hl == 5);
    const bool sendsFn = (F64C && hl == 6) || (FAST && hl == 0);      // lanes whose store A carries a function value
    auto fn_value = [&]() { return FAST ? rc : rs; };
    const int uB = hl <= 1 ? 7 : (hl <= 3 ? 8 : 9), cB = (hl == 1 || hl == 3 || hl == 6) ? 1 : 0;
    const bool wantB = F64C && (fn_exp || fn_rot);
    __syncwarp(FULL);

#if TRM_PROFILE_PHASES
    __shared__ unsigned tph[12];
    unsigned tph_t = (unsigned)clock();
    const bool tph_on = blockIdx.x == 0 && pair == 0 && lane == 0;
    if (tph_on) for (int i = 0; i < 12; ++i) tph[i] = 0u;
#define TPH(i) do { if (tph_on) { const unsigned _t = (unsigned)clock(); tph[i] += _t - tph_t; tph_t = _t; } } while (0)
    unsigned tphx_t = 0;      // sub-timers inside a phase: TPHX(0) starts, TPHX(i) adds the time since the previous TPHX to tph[i]
#define TPHX(i) do { if (tph_on) { const unsigned _t = (unsigned)clock(); if (i) tph[i] += _t - tphx_t; tphx_t = _t; } } while (0)
#else
#define TPH(i) do { } while (0)
#define TPHX(i) do { } while (0)
#endif
    for (int blk = 0; blk < n_blocks; ++blk) {
        const int slot = blk & 1;
        const int64_t n0 = (int64_t)blk * TB;
        const int64_t left = n_tube - n0;
        const int nb = left >= TB ? TB : (left > 0 ? (int)left : 0);
        const bool active = hl < nb;
        if (blk >= WIDE_SLOTS) mbar_wait_sleep<TRM_WAIT_NS>(&W.empty[slot], (uint32_t)(((blk >> 1) - 1) & 1));
        if (TRM_PROFILE_SKIP & 1) {
            __syncwarp(FULL);
            if (lane == 0) mbar_arrive(&W.full[slot]);
            continue;
        }

        TPH(0);
        // ---- S0: parameter interpolation, lane = parameter (m:611-688).  The 16 x 16 interpolated values are
        //      staged INSIDE this utterance's part of the ring slot (fields 0..7, sample position rotated by the
        //      field so that the stores of the 16 parameter lanes fall into different banks); phase A1 reads
        //      them back into registers before it writes any record.
        int refill = -1;
        constexpr int RS = (int)(Wide<R>::UP * sizeof(typename Wide<R>::Unit) / sizeof(double));   // doubles per sample row
        const int ib = (jc == 0) ? 0 : cp - jc;             // step of this block at which the next control interval starts
        if (ib + cp >= TB) {
            // At most one interval starts inside the block (always, for the reference's control periods >= 17): 16 straight-line
            // steps with constant store offsets.  The values of the new interval are prepared before the loop and swapped in
            // at step ib -- same operations on the same values as the reference's loop (m:611-688), no data-dependent loop.
            const int fb = f_idx + (jc == 0 ? 0 : 1);       // index of the interval that starts at step ib
            const bool starts = ib < TB && fb + 1 < n_frames && feeds;
            double np = p_cur, nd = p_delta, nrc = rc, nrs = rs, ndc = dc, nds = ds;
            if (starts) {
                TPHX(0);
                const int fn = fb + 1;
                const int ch = fn / FRAME_CHUNK;
                if ((fn % FRAME_CHUNK) == 0) {
                    refill = ch + 1;
                    mbar_wait(&S.mbar[ch & 1], (uint32_t)((ch >> 1) & 1));
                }
                TPHX(9);
                const double nxt = staged(ch & 1, fn % FRAME_CHUNK);
                np = p_next;
                nd = (nxt - np) / (double)cp;
                p_next = nxt;
                TPHX(10);
                if constexpr (GEO) seed_functions(np, nd, nrc, nrs, ndc, nds);
                TPHX(11);
            }
            double *const a0 = reinterpret_cast<double *>(&W.ring[slot][uA][uA][ucol]) + cA;   // row of step 0; steps TB-u .. wrap
            double *const b0 = reinterpret_cast<double *>(&W.ring[slot][uB][uB][ucol]) + cB;
            if (!starts) {
#pragma unroll
                for (int i = 0; i < TB; ++i) {
                    sts_f64_if(wantA, (i + uA < TB ? a0 : a0 - TB * RS) + i * RS, sendsFn ? fn_value() : p_cur);
                    if constexpr (F64C) {
                        sts_f64_if(wantB, (i + uB < TB ? b0 : b0 - TB * RS) + i * RS, rc);
                        step_functions();
                    } else if constexpr (FAST) {
                        rc *= dc;
                    }
                    p_cur += p_delta;
                }
            } else {
#pragma unroll
                for (int i = 0; i < TB; ++i) {
                    if (i == ib) {
                        p_cur = np; p_delta = nd;
                        if constexpr (F64C) { rc = nrc; rs = nrs; dc = ndc; ds = nds; }
                        else if constexpr (FAST) { rc = nrc; dc = ndc; }
                    }
                    sts_f64_if(wantA, (i + uA < TB ? a0 : a0 - TB * RS) + i * RS, sendsFn ? fn_value() : p_cur);
                    if constexpr (F64C) {
                        sts_f64_if(wantB, (i + uB < TB ? b0 : b0 - TB * RS) + i * RS, rc);
                        step_functions();
                    } else if constexpr (FAST) {
                        rc *= dc;
                    }
                    p_cur += p_delta;
                }
            }
            jc += TB;
            if (jc >= cp) { jc -= cp; ++f_idx; }
        } else {
            // control periods below 16 samples (outside the reference's range, accepted down to 8): run by run
            for (int s = 0; s < TB;) {
                if (jc == 0 && f_idx + 1 < n_frames && feeds) {
                    const int fn = f_idx + 1;
                    const int ch = fn / FRAME_CHUNK;
                    if ((fn % FRAME_CHUNK) == 0) {
                        refill = ch + 1;
                        mbar_wait(&S.mbar[ch & 1], (uint32_t)((ch >> 1) & 1));
                    }
                    const double nxt = staged(ch & 1, fn % FRAME_CHUNK);
                    p_cur = p_next;
                    p_delta = (nxt - p_cur) / (double)cp;
                    p_next = nxt;
                    if constexpr (GEO) seed_functions(p_cur, p_delta, rc, rs, dc, ds);
                }
                const int run = min(TB - s, cp - jc);
                for (int i = 0; i < run; ++i) {
                    sts_f64_if(wantA, reinterpret_cast<double *>(&W.ring[slot][uA][(s + i + uA) & (TB - 1)][ucol]) + cA, sendsFn ? fn_value() : p_cur);
                    if constexpr (F64C) {
                        sts_f64_if(wantB, reinterpret_cast<double *>(&W.ring[slot][uB][(s + i + uB) & (TB - 1)][ucol]) + cB, rc);
                        step_functions();
                    } else if constexpr (FAST) {
                        rc *= dc;
                    }
                    p_cur += p_delta;
                }
                s += run;
                jc += run;
                if (jc == cp) { jc = 0; ++f_idx; }
            }
        }
        __syncwarp(FULL);
        if (hl == 0 && refill >= 0 && refill < n_chunks) {
            const int cnt = min(FRAME_CHUNK, n_frames - refill * FRAME_CHUNK);
            mbar_expect_tx(&S.mbar[refill & 1], (uint32_t)cnt * frow);
            tma_bulk_g2s(&S.FR[refill & 1][0][0], F + (size_t)refill * FRAME_CHUNK * frow, (uint32_t)cnt * frow, &S.mbar[refill & 1]);
        }

        TPH(1);
        // ---- A1: lane = sample: conversions and coefficients (m:294-300, 712-773; TRMFilters.m:9-17) ---------
        // (conformance mode stages 10 units -- see the layout above --, the other modes the 16 parameters in 8 units)
        constexpr int N_STAGED = F64C ? 10 : 8;
        double prm[2 * N_STAGED];
#pragma unroll
        for (int f = 0; f < N_STAGED; ++f) {
            const double2 v = *reinterpret_cast<const double2 *>(&W.ring[slot][f][(hl + f) & (TB - 1)][ucol]);
            prm[2 * f] = v.x; prm[2 * f + 1] = v.y;
        }
        __syncwarp(FULL);                                   // every staged value is in registers: records may be written
        TPH(2);
        double inc_d;
        if constexpr (F64C) {
            inc_d = prm[14];
        } else if constexpr (FAST) {
            inc_d = prm[0];                                 // staged by parameter lane 0 in place of the pitch
        } else {
            const double f0 = 220.0 * exp2(div_known(prm[0] + 3.0, 12.0, 1.0 / 12.0));
            inc_d = (f0 / 2.0) * S.CST[C_BASICINC];
            if constexpr (!FAST) S.INC[hl] = inc_d;
        }
        double ax_d;
        R ax, ah1;
        R bp_alpha2;
        if constexpr (F64C) {
            // amplitude() (TRMUtility.m:26-41): clamps decided on the interpolated parameter (the reference's adds) with the
            // reference's bounds, 0 for dB <= 2^-48 and 1 for dB >= 60; value from the geometric sequence
            const double p1 = prm[0], p2 = prm[1], p3 = prm[2], fpos = prm[3];
            ax_d = (p1 <= AMP_ZERO_DB) ? 0.0 : ((p1 >= 60.0) ? 1.0 : prm[15]);
            {
                // glottal closure point rint(ax * tnDelta) (TRMWavetable.m:122): when the product is within 1e-6 of a
                // rounding boundary, decide with the amplitude computed directly from the parameter
                const double tq = ax_d * S.CST[C_TNDELTA];
                if (fabs(fabs(tq - rint(tq)) - 0.5) < 1e-6 && p1 > AMP_ZERO_DB && p1 < 60.0)
                    ax_d = exp2_inline((p1 - 60.0) * 0.16609640474436813);
            }
            ax = ax_d;
            ah1 = (p2 <= AMP_ZERO_DB) ? 0.0 : ((p2 >= 60.0) ? 1.0 : prm[16]);
            const double fa = (p3 <= AMP_ZERO_DB) ? 0.0 : ((p3 >= 60.0) ? 1.0 : prm[17]);
            const double dd = S.CST[C_DAMP];
            double r2[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) { const double r = prm[4 + q]; r2[q] = r * r; }
            // k d of the two-port junctions (m:716-741), reciprocals by Newton refinement
            auto kd = [&](double a2, double b2) { return ((a2 - b2) * dd) * rcp_fast(a2 + b2); };
            const double kd0 = kd(r2[0], r2[1]), kd1 = kd(r2[1], r2[2]), kd2 = kd(r2[2], r2[3]), kd4 = kd(r2[3], r2[4]);
            const double kd6 = kd(r2[4], r2[5]), kd7 = kd(r2[5], r2[6]), kd8 = kd(r2[6], r2[7]);
            const double ap2 = S.CST[C_APSCALE2];
            const double k9 = (r2[7] - ap2) * rcp_fast(r2[7] + ap2);
            const double vel = prm[12];
            const double v2 = vel * vel;
            const double sum = (2.0 * dd) * rcp_fast((r2[3] + r2[3]) + v2);
            const double aLd = sum * r2[3], aUd = sum * v2;
            const double kd10 = kd(v2, S.CST[C_NR1SQ]);
            // frication taps (m:760-773): (1 - c) amp at i = (int) position, c amp at i + 1 if that is a tap, 0 elsewhere.
            // Sent as the even junction's value, the odd junction's value and the set of junctions that take them.
            const int ipos = (int)fpos;
            const double comp = fpos - (double)ipos;
            const double t0 = (1.0 - comp) * fa, t1 = comp * fa;
            const bool even = (ipos & 1) == 0;
            const unsigned tsel = ((unsigned)ipos < 8u) ? (3u << ipos) & 0xFFu : 0u;
            // band-pass (TRMFilters.m:9-17): beta = (1 - tan u) / (2 (1 + tan u)) = (cos u - sin u) / (2 (cos u + sin u))
            const double cu = prm[19], su = prm[13], cosv = prm[18];
            const double beta2 = (cu - su) * rcp_fast(cu + su);
            const double gamma2 = (1.0 + beta2) * cosv;
            bp_alpha2 = 0.5 - 0.5 * beta2;
            W.ring[slot][0][hl][ucol] = make_double2(kd0, kd1);
            W.ring[slot][1][hl][ucol] = make_double2(kd2, aLd);
            W.ring[slot][2][hl][ucol] = make_double2(kd4, kd6);
            W.ring[slot][3][hl][ucol] = make_double2(kd7, kd8);
            W.ring[slot][4][hl][ucol] = make_double2(k9, kd10);
            W.ring[slot][5][hl][ucol] = make_double2(aUd, gamma2);
            W.ring[slot][6][hl][ucol] = make_double2(beta2, __longlong_as_double((long long)tsel));
            W.ring[slot][7][hl][ucol] = make_double2(even ? t0 : t1, even ? t1 : t0);
        } else if constexpr (FAST) {
            const float axf = amplitude_f(prm[1]);
            ax_d = (double)axf;
            {
                const float tq = axf * (float)S.CST[C_TNDELTA];
                const float fr = tq - floorf(tq);
                if (fabsf(fr - 0.5f) < 2e-3f) ax_d = amplitude_db(prm[1]);
            }
            ax = axf;
            ah1 = amplitude_f(prm[2]);
            const float fa = amplitude_f(prm[3]);
            const float dd = (float)S.CST[C_DAMP];
            float r2[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) { const float r = (float)prm[7 + q]; r2[q] = r * r; }
            float tap[8];
            {
                const double fpos = prm[4];
                const int ipos = (int)fpos;
                const float comp = (float)(fpos - (double)ipos);
                const float t0 = (1.0f - comp) * fa, t1 = comp * fa;
#pragma unroll
                for (int q = 0; q < 8; ++q) tap[q] = (q == ipos) ? t0 : ((ipos >= 0 && q == ipos + 1) ? t1 : 0.0f);
            }
            auto two_port = [&](float ra2, float rb2, float w) {
                const float inv = __fdividef(dd, ra2 + rb2);
                return make_float4(2.0f * ra2 * inv, (ra2 - rb2) * inv, 2.0f * rb2 * inv, w);
            };
            float beta2, gamma2;
            {
                const float sr = (float)S.CST[C_SR];
                const float pi = 3.14159265358979323846f;
                const float inv_sr = 1.0f / sr;
                float su, cu;
                __sincosf((pi * (float)prm[6]) * inv_sr, &su, &cu);
                const float cosv = __cosf(((2.0f * pi) * (float)prm[5]) * inv_sr);
                beta2 = __fdividef(cu - su, cu + su);
                gamma2 = (1.0f + beta2) * cosv;
                bp_alpha2 = 0.5f - 0.5f * beta2;
            }
            W.ring[slot][0][hl][ucol] = two_port(r2[0], r2[1], tap[4]);      // S1|S2; .w = FC5 (pure-delay junction S6|S7)
            W.ring[slot][1][hl][ucol] = two_port(r2[1], r2[2], tap[0]);
            W.ring[slot][2][hl][ucol] = two_port(r2[2], r2[3], tap[1]);
            W.ring[slot][4][hl][ucol] = two_port(r2[3], r2[4], tap[3]);
            W.ring[slot][5][hl][ucol] = two_port(r2[4], r2[5], tap[5]);
            W.ring[slot][6][hl][ucol] = two_port(r2[5], r2[6], tap[6]);
            W.ring[slot][7][hl][ucol] = two_port(r2[6], r2[7], tap[7]);
            {
                const float vel = (float)prm[15], v2 = vel * vel;
                const float inv = __fdividef(dd, (r2[3] + r2[3]) + v2);
                W.ring[slot][3][hl][ucol] = make_float4(2.0f * r2[3] * inv, -v2 * inv, 2.0f * v2 * inv, (v2 - (r2[3] + r2[3])) * inv);
                W.ring[slot][9][hl][ucol] = two_port(v2, (float)S.CST[C_NR1SQ], beta2);
            }
            {
                const float ap2 = (float)S.CST[C_APSCALE2];
                const float inv = __fdividef(1.0f, r2[7] + ap2);
                W.ring[slot][8][hl][ucol] = make_float4(dd * (float)S.CST[C_MOUTH0] * ((r2[7] - ap2) * inv), 2.0f * r2[7] * inv, tap[2], gamma2);
            }
        } else {
            ax_d = amplitude_db(prm[1]);
            ax = (R)ax_d;
            ah1 = (R)amplitude_db(prm[2]);
            double r2[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) { const double r = prm[7 + q]; r2[q] = r * r; }
            const double k0 = (r2[0] - r2[1]) / (r2[0] + r2[1]);
            const double k1 = (r2[1] - r2[2]) / (r2[1] + r2[2]);
            const double k2 = (r2[2] - r2[3]) / (r2[2] + r2[3]);
            const double k4 = (r2[3] - r2[4]) / (r2[3] + r2[4]);
            const double k6 = (r2[4] - r2[5]) / (r2[4] + r2[5]);
            const double k7 = (r2[5] - r2[6]) / (r2[5] + r2[6]);
            const double k8 = (r2[6] - r2[7]) / (r2[6] + r2[7]);
            const double ap2 = S.CST[C_APSCALE2];
            const double k9 = (r2[7] - ap2) / (r2[7] + ap2);
            const double vel = prm[15];
            const double v2 = vel * vel;
            const double sum = 2.0 / ((r2[3] + r2[3]) + v2);
            const double aL = sum * r2[3], aU = sum * v2;
            const double n2 = S.CST[C_NR1SQ];
            const double k10 = (v2 - n2) / (v2 + n2);
            double tap[8];
            {
                const double fa = amplitude_db(prm[3]);
                const double fpos = prm[4];
                const int ipos = (int)fpos;
                const double comp = fpos - (double)ipos;
                const double rem = 1.0 - comp;
                const double t0 = rem * fa, t1 = comp * fa;
#pragma unroll
                for (int q = 0; q < 8; ++q) tap[q] = (q == ipos) ? t0 : ((ipos >= 0 && q == ipos + 1) ? t1 : 0.0);
            }
            double beta2, gamma2;
            {
                const double sr = S.CST[C_SR];
                const double pi = 3.14159265358979323846;
                const double rsr = S.CST[C_RSR];                 // RN(1 / sr)
                const double tanv = tan(div_known(pi * prm[6], sr, rsr));
                const double cosv = cos(div_known((2.0 * pi) * prm[5], sr, rsr));
                const double beta = (1.0 - tanv) / (2.0 * (1.0 + tanv));
                beta2 = 2.0 * beta;
                gamma2 = 2.0 * ((0.5 + beta) * cosv);
                bp_alpha2 = (R)(2.0 * ((0.5 - beta) / 2.0));
            }
            W.ring[slot][0][hl][ucol] = make_double2(k0, k1);
            W.ring[slot][1][hl][ucol] = make_double2(k2, aL);
            W.ring[slot][2][hl][ucol] = make_double2(k4, k6);
            W.ring[slot][3][hl][ucol] = make_double2(k7, k8);
            W.ring[slot][4][hl][ucol] = make_double2(k9, k10);
            W.ring[slot][5][hl][ucol] = make_double2(aU, tap[0]);
            W.ring[slot][6][hl][ucol] = make_double2(tap[1], tap[2]);
            W.ring[slot][7][hl][ucol] = make_double2(tap[3], tap[4]);
            W.ring[slot][8][hl][ucol] = make_double2(tap[5], tap[6]);
            W.ring[slot][9][hl][ucol] = make_double2(tap[7], gamma2);
            reinterpret_cast<double *>(&W.ring[slot][10][hl][ucol])[0] = beta2;
        }
        TPH(3);
        // noise (TRMUtility.m:71-85 as the MCG mod 2^44) + one-zero low-pass (TRMFilters.m:81-86)
        R lp_noise;
        {
            // (a 44-bit integer becomes a double by placing it in the mantissa of 2^52 and subtracting 2^52 -- exact, like the
            //  conversion instruction, but two ALU operations and an add instead of a trip through the conversion unit)
            auto draw = [&](unsigned long long k) {
                const double kd_ = __hiloint2double((int)(0x43300000u | (unsigned)(k >> 32)), (int)(unsigned)k) - 4503599627370496.0;
                return kd_ * TWO_M44 - 0.5;
            };
            const unsigned long long kt = (kb * pw1) & MASK44;
            const double nz = draw(kt);
            // x[n-1]: the draw of the lane below; lane 0 takes the last draw of the previous block (the state kb itself)
            double nzp = __shfl_up_sync(FULL, nz, 1, 16);
            const double nz_prev = (fresh && n0 == 0) ? 0.0 : draw(kb);
            nzp = (hl == 0) ? nz_prev : nzp;
            lp_noise = (R)(nz + nzp);
            kb = (kb * pwB) & MASK44;
        }

        TPH(4);
        // ---- S1: oscillator position (TRMWavetable.m:165-168, 28-34) -------------------------------------------
        double p0, p1;
        if constexpr (FAST || F64C) {
            // 64-bit fixed point, 2^55 units per table entry: 512 entries are exactly 2^64, so the table wrap is the
            // integer overflow, addition is associative and the 32 positions of a block come from a 4-step warp scan
            // instead of a 32-step dependent chain.  (Resolution 2.8e-17 entries; the reference's own double
            // accumulator rounds to 5.7e-14.)  mod0 quirk: values in (511, 512) are reported as negative.
            const unsigned long long inc_fx = __double2ull_rn(inc_d * 36028797018963968.0);
            unsigned long long incl = inc_fx + inc_fx;
#pragma unroll
            for (int o = 1; o < TB; o <<= 1) {
                const unsigned long long up = __shfl_up_sync(FULL, incl, o, 16);
                if (hl >= o) incl += up;
            }
            unsigned long long ub = pos_fx + incl, ua = ub - inc_fx;
            const unsigned long long top = 511ull << 55;
            if constexpr (F64C) {
                // The reference accumulates the position in double: every addition rounds to the grid of the sum's binade
                // (2^-44 table entries for sums in [256, 512), 2^-43 just before a wrap, ...).  For a varying increment
                // these roundings average out (measured 8e-13 of peak after 30 s); for a CONSTANT one they are the same
                // every period and the reference drifts away from the exact phase by 5.6e-11 of peak per second -- past
                // the 1e-9 contract after 18 s of a static vowel.  So whenever a block's increment is constant, the scan
                // is repeated with every half-step's increment rounded as the reference's addition rounds it (binades
                // from the first pass; exact ties, which the reference resolves to even, keep the exact increment).
                const unsigned half_mask = (lane & 16) ? 0xFFFF0000u : 0x0000FFFFu;
                const bool same = inc_fx == __shfl_sync(FULL, inc_fx, lane & 16);
                const unsigned vote = __ballot_sync(FULL, same);
                const bool constant = (vote & half_mask) == half_mask;
                if (__any_sync(FULL, constant)) {
                    auto rounded = [&](unsigned long long before, unsigned long long after) {
                        // grid of the (unwrapped) sum: after a wrap the sum was in [512, 1024); values in (511, 512) are
                        // kept as negative numbers by mod0 (TRMWavetable.m:28-34)
                        const bool wrapped = after < before;
                        const unsigned long long mag = (after > top) ? (0ull - after) : after;
                        int sh = wrapped ? 12 : 11 - __clzll((long long)mag);
                        if (mag == 0ull || sh <= 0) return inc_fx;
                        const unsigned long long low = inc_fx & ((1ull << sh) - 1ull), halfg = 1ull << (sh - 1);
                        if (low == halfg) return inc_fx;
                        return (inc_fx - low) + (low > halfg ? (1ull << sh) : 0ull);
                    };
                    const unsigned long long prev = ua - inc_fx;           // position before this lane's first half-step
                    const unsigned long long ra = rounded(prev, ua), rb = rounded(ua, ub);
                    unsigned long long incl2 = ra + rb;
#pragma unroll
                    for (int o = 1; o < TB; o <<= 1) {
                        const unsigned long long up = __shfl_up_sync(FULL, incl2, o, 16);
                        if (hl >= o) incl2 += up;
                    }
                    if (constant) { ub = pos_fx + incl2; ua = ub - rb; incl = incl2; }
                }
            }
            pos_fx += __shfl_sync(FULL, incl, (lane & 16) | (TB - 1));
            p0 = (ua > top) ? -((double)(0ull - ua) * 2.77555756156289135e-17) : (double)ua * 2.77555756156289135e-17;
            p1 = (ub > top) ? -((double)(0ull - ub) * 2.77555756156289135e-17) : (double)ub * 2.77555756156289135e-17;
        } else {
            __syncwarp(FULL);                               // INC of the whole block is visible
            p0 = 0.0; p1 = 0.0;
#pragma unroll
            for (int s = 0; s < TB; ++s) {
                const double di = S.INC[s];
                pos = pos + di;
                pos = pos - ((pos > 511.0) ? 512.0 : 0.0);     // mod0: wraps only above 511 (TRMWavetable.m:28-34)
                const double pa = pos;
                pos = pos + di;
                pos = pos - ((pos > 511.0) ? 512.0 : 0.0);
                if (hl == s) { p0 = pa; p1 = pos; }
            }
        }

        TPH(5);
        // ---- A2: table look-ups, FIR, source mixing (TRMWavetable.m:174-195, m:305-337) --------------------------
        R *const he = &S.HE[hs + FIR_HIST + hl], *const ho = &S.HO[hs + FIR_HIST + hl];   // this lane's new value
        {
            R ev, ov;
            if (!active) { p0 = 0.0; p1 = 0.0; }
            const double newDiv2 = (double)div2 - rint(ax_d * S.CST[C_TNDELTA]);
            const double Ld = newDiv2 - (double)div1;
            int lo0 = ((int)p0) & (TRM_TABLE_LENGTH - 1), lo1 = ((int)p1) & (TRM_TABLE_LENGTH - 1);
            int hi0 = lo0 + 1, hi1 = lo1 + 1;
            if (hi0 > 511) hi0 -= 512;
            if (hi1 > 511) hi1 -= 512;
            if constexpr (FAST) {
                const float Lf = (float)Ld;
                const float scale = __fdividef(1.0f, Lf * Lf);
                const float inv_div1 = 1.0f / (float)div1;
                const float w00 = table_value_fast(wt_base, lo0, div1, inv_div1, newDiv2, scale, pulse_wave);
                const float w01 = table_value_fast(wt_base, hi0, div1, inv_div1, newDiv2, scale, pulse_wave);
                const float w10 = table_value_fast(wt_base, lo1, div1, inv_div1, newDiv2, scale, pulse_wave);
                const float w11 = table_value_fast(wt_base, hi1, div1, inv_div1, newDiv2, scale, pulse_wave);
                ev = w00 + ((float)(p0 - (double)lo0) * (w01 - w00));
                ov = w10 + ((float)(p1 - (double)lo1) * (w11 - w10));
            } else {
                const R scale = F64C ? (R)rcp_fast(Ld * Ld) : (R)(1.0 / (Ld * Ld));
                if (F64C && pulse_wave) {
                    // conformance mode, pulse waveform: the whole table is a function of the index -- rise 3x^2 - 2x^3 with
                    // x = i / div1 (TRMWavetable.m:78-87), fall 1 - j^2 / L^2 up to the closure point, 0 after it -- so it is
                    // evaluated without a memory access or a branch (the strict mode reads the rise from the init-time table)
                    const double inv_div1 = S.CST[C_INVDIV1];
                    auto value = [&](int i) {
                        const double di = (double)i, x = di * inv_div1, x2 = x * x;
                        const double rise = fma(-2.0 * x2, x, 3.0 * x2);
                        const double j = di - (double)div1;
                        const double fall = fma(-(j * j), scale, 1.0);
                        const double v = (i < div1) ? rise : fall;
                        return (di >= newDiv2) ? 0.0 : v;
                    };
                    const double w00 = value(lo0), w01 = value(hi0), w10 = value(lo1), w11 = value(hi1);
                    ev = fma(p0 - (double)lo0, w01 - w00, w00);
                    ov = fma(p1 - (double)lo1, w11 - w10, w10);
                } else {
                    R w0 = table_value<R>(wt_base, lo0, div1, div2, newDiv2, scale, pulse_wave);
                    R w1 = table_value<R>(wt_base, hi0, div1, div2, newDiv2, scale, pulse_wave);
                    ev = w0 + ((R)(p0 - (double)lo0) * (w1 - w0));
                    w0 = table_value<R>(wt_base, lo1, div1, div2, newDiv2, scale, pulse_wave);
                    w1 = table_value<R>(wt_base, hi1, div1, div2, newDiv2, scale, pulse_wave);
                    ov = w0 + ((R)(p1 - (double)lo1) * (w1 - w0));
                }
            }
            *he = ev; *ho = ov;
            if (HIST_RING<R> && hs + FIR_HIST + hl >= FIR_RING) { he[-FIR_RING] = ev; ho[-FIR_RING] = ov; }
        }
        __syncwarp(FULL);
        TPH(6);
        R sig;
        {
            R pulse0;
            // (Measured and not kept: two outputs per lane from 13 + 13 aligned 128-bit loads -- 52 shared-memory wavefronts
            //  per block instead of 98, but half the lanes idle and twice the FP64 instructions: 10.85 -> 11.19 ms.)
            if constexpr (FAST || F64C) {
                R s0 = (R)0, s1 = (R)0, s2 = (R)0, s3 = (R)0;
#pragma unroll
                for (int q = 0; q < FIR_HIST; q += 2) {
                    s0 += ho[-q] * FirCoef<R>::at(2 * q);
                    s1 += he[-q] * FirCoef<R>::at(2 * q + 1);
                    s2 += ho[-q - 1] * FirCoef<R>::at(2 * q + 2);
                    s3 += he[-q - 1] * FirCoef<R>::at(2 * q + 3);
                }
                s0 += ho[-FIR_HIST] * FirCoef<R>::at(2 * FIR_HIST);
                pulse0 = (s0 + s1) + (s2 + s3);
            } else {
                R acc = (R)0;
#pragma unroll
                for (int q = 0; q < FIR_HIST; ++q) {
                    acc += ho[-q] * FirCoef<R>::at(2 * q);
                    acc += he[-q] * FirCoef<R>::at(2 * q + 1);
                }
                acc += ho[-FIR_HIST] * FirCoef<R>::at(2 * FIR_HIST);
                pulse0 = acc;
            }
            const R bf = (R)S.CST[C_BF], one_minus_bf = (R)(1.0 - S.CST[C_BF]);
            const R pulsed_noise = lp_noise * pulse0;
            const R pulse = ax * ((pulse0 * one_minus_bf) + (pulsed_noise * bf));
            if (modulation) {
                R crossmix = ax * (R)S.CST[C_CMIX];
                crossmix = (crossmix < (R)1) ? crossmix : (R)1;
                sig = (pulsed_noise * crossmix) + (lp_noise * ((R)1 - crossmix));
            } else
                sig = lp_noise;
            const R tube_in = (pulse + (ah1 * sig)) * (R)0.125;
            const R thr_in = (R)S.CST[C_TA0] * (pulse * (R)0.125);
            // band-pass feed-forward part alpha*(x[n]-x[n-2]); x[n-2] comes from two lanes down or the carry
            R x2 = __shfl_sync(FULL, sig, (lane & 16) | ((hl - 2) & 15));
            if (hl == 0) x2 = xm2;
            if (hl == 1) x2 = xm1;
            const R bp_ff = bp_alpha2 * (sig - x2);
            const int last = nb > 0 ? nb - 1 : 0;
            const R l1 = __shfl_sync(FULL, sig, (lane & 16) | last);
            const R l2 = __shfl_sync(FULL, sig, (lane & 16) | (last > 0 ? last - 1 : 0));
            xm2 = (last > 0) ? l2 : xm1;
            xm1 = l1;
            if constexpr (FAST) {
                W.ring[slot][10][hl][ucol] = make_float4(tube_in, bp_ff, thr_in, 0.0f);
            } else if constexpr (F64C) {
                W.ring[slot][8][hl][ucol] = make_double2(tube_in, bp_ff);
                reinterpret_cast<double *>(&W.ring[slot][9][hl][ucol])[0] = thr_in;
            } else {
                reinterpret_cast<double *>(&W.ring[slot][10][hl][ucol])[1] = tube_in;
                W.ring[slot][11][hl][ucol] = make_double2(bp_ff, thr_in);
            }
        }
        __syncwarp(FULL);
        TPH(7);
        if (lane == 0) mbar_arrive(&W.full[slot]);
        if constexpr (HIST_RING<R>) {
            hs = (hs + TB == FIR_RING) ? 0 : hs + TB;
        } else {
            // slide the oscillator history down by one block (rows TB.. -> 0..)
            const R e0 = S.HE[TB + hl], o0 = S.HO[TB + hl];
            const R e1 = (hl < FIR_HIST - TB) ? S.HE[2 * TB + hl] : (R)0;
            const R o1 = (hl < FIR_HIST - TB) ? S.HO[2 * TB + hl] : (R)0;
            __syncwarp(FULL);
            S.HE[hl] = e0; S.HO[hl] = o0;
            if (hl < FIR_HIST - TB) { S.HE[TB + hl] = e1; S.HO[TB + hl] = o1; }
            __syncwarp(FULL);
        }
        if (PER_UTT && st_h && ends_in_block(n_tube, blk)) {
            // the utterance's last sample is in this block (a whole block except at the end of a stream): the state after it
            if (hl == 0) {
                st_h[0] = (unsigned long long)__double_as_longlong(pos);
                st_h[1] = pos_fx;
                st_h[2] = kb;
                st_h[3] = 0ull;
                st_v[STATE_XM] = xm1; st_v[STATE_XM + 1] = xm2;
            }
            for (int i = hl; i < FIR_HIST; i += TB) { st_v[STATE_HE + i] = S.HE[hs + i]; st_v[STATE_HO + i] = S.HO[hs + i]; }
        }
        TPH(8);
    }
#if TRM_PROFILE_PHASES
    if (tph_on)
        printf("[phases %s] cycles/block: wait %u S0 %u (of which per block: frame wait %u, delta %u, seeds %u) stage-read %u A1 %u noise %u S1 %u A2-table %u FIR+mix %u tail %u  (blocks %d)\n",
               FAST ? "f32" : (STRICT ? "f64s" : "f64"), tph[0] / n_blocks, tph[1] / n_blocks, tph[9] / n_blocks, tph[10] / n_blocks, tph[11] / n_blocks,
               tph[2] / n_blocks, tph[3] / n_blocks, tph[4] / n_blocks,
               tph[5] / n_blocks, tph[6] / n_blocks, tph[7] / n_blocks, tph[8] / n_blocks, n_blocks);
#endif
    if (!PER_UTT && st_h) {
        // lockstep calls cover whole 16-sample blocks of equally long utterances: the state after the last sample
        if (hl == 0) {
            st_h[0] = (unsigned long long)__double_as_longlong(pos);
            st_h[1] = pos_fx;
            st_h[2] = kb;
            st_h[3] = 0ull;
            st_v[STATE_XM] = xm1; st_v[STATE_XM + 1] = xm2;
        }
        for (int i = hl; i < FIR_HIST; i += TB) { st_v[STATE_HE + i] = S.HE[hs + i]; st_v[STATE_HO + i] = S.HO[hs + i]; }
    }
}

template <typename R, bool PER_UTT>
__global__ void __launch_bounds__(Wide<R>::THREADS, 1) tube_wide_kernel(WideArgs wargs)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    WideSmem<R> &W = *reinterpret_cast<WideSmem<R> *>(smem_raw);
    const TubeArgs &args = wargs.t;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int g_start, g_count;
    wide_group(args.n_utt, wargs.n_groups, blockIdx.x, g_start, g_count);
    const int n_pairs = (g_count + 1) >> 1;

    // ---- CTA init: zero the ring and histories, barriers, per-utterance pointers ---------------------------
    {
        uint32_t *w = reinterpret_cast<uint32_t *>(&W.ring[0][0][0][0]);
        constexpr int NW = (int)(sizeof(W.ring) / 4);
        for (int i = threadIdx.x; i < NW; i += blockDim.x) w[i] = 0u;
        for (int h = warp; h < 2 * Wide<R>::MAX_PAIRS; h += blockDim.x >> 5) {
            for (int i = lane; i < HIST_LEN<R>; i += 32) { W.ff[h].HE[i] = (R)0; W.ff[h].HO[i] = (R)0; }
            if (lane < TB) W.ff[h].INC[lane] = 0.0;
        }
        if (threadIdx.x == 0) {
            W.n_cta = 0;
            for (int s = 0; s < WIDE_SLOTS; ++s) { mbar_init(&W.full[s], (uint32_t)n_pairs); mbar_init(&W.empty[s], 1); }
            mbar_fence_init();
        }
    }
    __syncthreads();
    if (threadIdx.x < 32) {
        const bool has = lane < g_count;
        const int u = args.order ? args.order[g_start + (has ? lane : 0)] : g_start + (has ? lane : 0);
        const trm_cuda_utterance *D = args.desc + u;
        W.n_tube[lane] = has ? D->n_tube : 0;
        W.out_ptr[lane] = reinterpret_cast<R *>(args.tube) + D->tube_offset;
        if (has) atomicMax((unsigned long long *)&W.n_cta, (unsigned long long)D->n_tube);
    }
    __syncthreads();
    const int64_t n_cta = W.n_cta;
    const int pair = warp - 1 - (warp > WIDE_IDLE_WARP ? 1 : 0);
    const int n_blocks = (int)((n_cta + TB - 1) / TB);
    // Register redistribution (setmaxnreg, warpgroup granularity; see Wide<double>).  Every warp of a warpgroup executes
    // the instruction, before any of them exits; the donors release before the recurrence warpgroup's request can be met.
    if constexpr (Wide<R>::REGS_HI > 0) {
        if (warp >= 16) {
            asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(Wide<R>::REGS_DONOR));
            return;
        }
        if (warp < 4) {
            asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(Wide<R>::REGS_HI));
            if (n_cta <= 0 || pair >= n_pairs) return;
            if (warp == 0) wide_recurrence_warp<R, PER_UTT>(W, wargs, g_start, g_count, n_blocks, lane);
            else wide_feed_forward_warp<R, PER_UTT>(W, wargs, g_start, g_count, n_blocks, pair, lane);
        } else {
            if (n_cta <= 0 || warp == WIDE_IDLE_WARP || pair >= n_pairs) return;
            wide_feed_forward_warp<R, PER_UTT>(W, wargs, g_start, g_count, n_blocks, pair, lane);
        }
    } else {
        if (n_cta <= 0 || warp == WIDE_IDLE_WARP || pair >= n_pairs) return;
        if (warp == 0) wide_recurrence_warp<R, PER_UTT>(W, wargs, g_start, g_count, n_blocks, lane);
        else wide_feed_forward_warp<R, PER_UTT>(W, wargs, g_start, g_count, n_blocks, pair, lane);
    }
}

}  // namespace TRM_KERNEL_NS
