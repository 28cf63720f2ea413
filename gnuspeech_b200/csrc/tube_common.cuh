// tube_common.cuh -- what the TRM kernels for sm_100a share: per-TU constant tables, mbarrier / TMA bulk-copy helpers and
// the math helpers of the waveguide path (amplitude(), the glottal table as a function of the index, exact division by
// known divisors, and the cheaper forms of the FP64 conformance mode: Newton reciprocal, inline exp2 / sincos).
//
// Round 1 also had a second waveguide kernel here, the lane-per-section mapping BASELINE.json's north_star describes (one
// utterance per half-warp, lane = scattering junction, three __shfl_sync per sample, feed-forward and ladder phases
// alternating inside one warp).  It was slower than the lane-per-utterance mapping of tube_wide.cuh at every batch size in
// both rounds (4096 x 10 s: 123.7 vs 65.7 ms FP64; one utterance: 17.9 vs 9.9 ms), was never selected by default, and
// its ladder grafted behind the feed-forward warps of tube_wide.cuh (round 2, for CTAs with one or two utterances) was
// slower again (DESIGN.md 8) -- it is removed; the strict FP64 mode of tube_wide.cuh is the bit-faithful twin now.
#pragma once

#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>
#include <math.h>

#include "kernel_args.h"
#include "trm_cuda.h"

namespace TRM_KERNEL_NS {
using namespace trm;

constexpr double TWO_M44 = 5.684341886080801486968994140625e-14;   // 2^-44 exactly

// Per-TU constant tables (uploaded by the TU's upload function).
static __constant__ double c_fir_d[FIR_TAPS];
static __constant__ float c_fir_f[FIR_TAPS];
static __constant__ unsigned long long c_noise_pow[TRM_NOISE_JUMP + 1];

template <typename R> struct FirCoef;
template <> struct FirCoef<double> { static __device__ __forceinline__ double at(int i) { return c_fir_d[i]; } };
template <> struct FirCoef<float> { static __device__ __forceinline__ float at(int i) { return c_fir_f[i]; } };

// ---------------------------------------------------------------------------------------------
// PTX helpers: mbarrier + TMA bulk copy (global -> shared)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(void *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init()
{
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(void *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(void *bar, uint32_t parity)
{
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(void *bar, uint32_t parity)
{
    // try_wait suspends in hardware; the bound turns a lost copy into a trap instead of a hang
    for (uint32_t spin = 0; !mbar_try_wait(bar, parity); ++spin)
        if (spin > (1u << 24)) __trap();
}
__device__ __forceinline__ void tma_bulk_g2s(void *dst, const void *src, uint32_t bytes, void *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// ---------------------------------------------------------------------------------------------
// math helpers
// ---------------------------------------------------------------------------------------------
// amplitude(): TRMUtility.m:26-41.  Always evaluated in double (it is off the serial chain and the
// glottal-closure decision rint(ax*tnDelta) must not move).
// a / c for a divisor known in advance, rc = RN(1 / c): one multiply and two fused operations instead of the ~26
// instructions of a general IEEE division.  q' = RN(q + (a - c q) rc) with the residual exact is the correctly rounded
// quotient (Markstein's correction step; Brisebarre, Muller & Raina 2004): the value rounded last differs from a / c by
// <= 2^-105 |a / c|, closer than a quotient of two doubles comes to a rounding boundary except for isolated operand
// pairs.  Same result as `a / c`, so the conformance arithmetic is unchanged.
__device__ __forceinline__ double div_known(double a, double c, double rc)
{
    const double q = a * rc;
    const double r = fma(-c, q, a);
    return fma(r, rc, q);
}

__device__ __forceinline__ double amplitude_db(double dB)
{
    double x = dB - 60.0;
    if (x <= -60.0) return 0.0;
    if (x >= 0.0) return 1.0;
    return exp10(div_known(x, 20.0, 1.0 / 20.0));
}
// ---- helpers of the FP64 conformance mode's cheaper forms (tolerance 1e-9, BASELINE.json; none of them is used when
// TRM_STRICT = 1) -----------------------------------------------------------------------------------------------------
// 1 / s: hardware seed (MUFU.RCP64H, >= 16 good bits) refined by one cubic Newton step, x (1 + e + e^2) with
// e = 1 - s x: relative error <= 2^-48 in the worst case the seed allows, 5e-19 for its typical 2^-22.  No special
// cases: s = 0 gives inf * 0 = NaN in the correction, which is what the reference's 0 / 0 between two closed sections
// produces (TRMTubeModel.m:716-718) and must propagate.
__device__ __forceinline__ double rcp_fast(double s)
{
    double x;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(x) : "d"(s));
    const double e = fma(-s, x, 1.0);
    const double e2 = fma(e, e, e);
    return fma(x, e2, x);
}

// 2^x for |x| <= 1000: x = n + f, |f| <= 1/2, 2^f = exp(f ln 2) by its Taylor series to degree 13 (|f ln 2| <= 0.347:
// truncation 4e-18), exponent added as an integer.  Straight-line code; ~1 ulp.
__device__ __forceinline__ double exp2_inline(double x)
{
    x = fmin(fmax(x, -1000.0), 1000.0);
    const double n = rint(x);
    const double g = (x - n) * 0.693147180559945309417;
    double p = 1.6059043836821613e-10;                 // 1/13!
    p = fma(p, g, 2.08767569878681e-09);               // 1/12!
    p = fma(p, g, 2.505210838544172e-08);              // 1/11!
    p = fma(p, g, 2.755731922398589e-07);              // 1/10!
    p = fma(p, g, 2.7557319223985893e-06);             // 1/9!
    p = fma(p, g, 2.48015873015873e-05);               // 1/8!
    p = fma(p, g, 0.0001984126984126984);              // 1/7!
    p = fma(p, g, 0.001388888888888889);               // 1/6!
    p = fma(p, g, 0.008333333333333333);               // 1/5!
    p = fma(p, g, 0.041666666666666664);               // 1/4!
    p = fma(p, g, 0.16666666666666666);                // 1/3!
    p = fma(p, g, 0.5);
    p = fma(p, g, 1.0);
    p = fma(p, g, 1.0);
    return __hiloint2double(__double2hiint(p) + ((int)n << 20), __double2loint(p));
}

// sin and cos for |x| <= ~100 (the arguments here are below 2 pi): Cody-Waite reduction by pi/2 in two parts with
// fused multiply-adds, then the minimax kernels of fdlibm (k_sin.c / k_cos.c coefficients) on |r| <= pi/4; ~1 ulp.
__device__ __forceinline__ void sincos_inline(double x, double *sn, double *cs)
{
    const double n = rint(x * 0.63661977236758134308);
    double r = fma(-n, 1.5707963267948966, x);
    r = fma(-n, 6.123233995736766e-17, r);
    const int q = (int)n;
    const double z = r * r;
    double ps = 1.58969099521155010221e-10;
    ps = fma(ps, z, -2.50507602534068634195e-08);
    ps = fma(ps, z, 2.75573137070700676789e-06);
    ps = fma(ps, z, -1.98412698298579493134e-04);
    ps = fma(ps, z, 8.33333333332248946124e-03);
    ps = fma(ps, z, -1.66666666666666324348e-01);
    const double sr = fma(r * z, ps, r);
    double pc = -1.13596475577881948265e-11;
    pc = fma(pc, z, 2.08757232129817482790e-09);
    pc = fma(pc, z, -2.75573143513906633035e-07);
    pc = fma(pc, z, 2.48015872894767294178e-05);
    pc = fma(pc, z, -1.38888888888741095749e-03);
    pc = fma(pc, z, 4.16666666666666019037e-02);
    const double cr = fma(z * z, pc, fma(-0.5, z, 1.0));
    const double s0 = (q & 1) ? cr : sr, c0 = (q & 1) ? sr : cr;
    *sn = (q & 2) ? -s0 : s0;
    *cs = ((q + 1) & 2) ? -c0 : c0;
}

// Bit-wise select (one LOP3 per 32 bits): m = all ones -> x, m = 0 -> y.  Used instead of ?: in the junction
// loop so that the per-lane roles stay straight-line code (the compiler turns lane-dependent ternaries into
// divergent branch regions with reconvergence barriers and a divergence check before every shuffle).
__device__ __forceinline__ float blend(unsigned m, float x, float y)
{
    return __uint_as_float((__float_as_uint(x) & m) | (__float_as_uint(y) & ~m));
}
__device__ __forceinline__ double blend(unsigned m, double x, double y)
{
    const unsigned lo = ((unsigned)__double2loint(x) & m) | ((unsigned)__double2loint(y) & ~m);
    const unsigned hi = ((unsigned)__double2hiint(x) & m) | ((unsigned)__double2hiint(y) & ~m);
    return __hiloint2double((int)hi, (int)lo);
}

// amplitude()'s lower clamp (TRMUtility.m:26-41) as the reference decides it: `dB -= 60; if (dB <= -60) return 0` in double
// holds for every dB <= 2^-48 (half an ulp of 60 rounds to even, to -60), not only for dB <= 0
constexpr double AMP_ZERO_DB = 0x1p-48;

// fast-mode amplitude(): 10^((dB-60)/20) as 2^(..), FP32 (relative error ~5e-7, i.e. -126 dB on a linear gain).  The clamp
// to 0 is decided on the double parameter: (float)dB - 60 already rounds to -60 below 2^-19, where the reference gives 1e-3.
__device__ __forceinline__ float amplitude_f(double dB)
{
    const float x = (float)dB - 60.0f;
    const float v = exp2f(fminf(x, 0.0f) * 0.16609640474436813f);    // x >= 0 -> exactly 1
    return (dB <= AMP_ZERO_DB) ? 0.0f : v;
}

// fast-mode glottal table: rise 3x^2 - 2x^3 (x = i/div1), fall 1 - (j*j)/L^2, closed 0 -- evaluated, never loaded
// (TRMWavetable.m:78-96, 117-162).  The sine waveform (rare) still reads the 512-entry table.
__device__ __forceinline__ float table_value_fast(const double *__restrict__ base, int i, int div1, float inv_div1,
                                                  double newDiv2, float scale, bool pulse)
{
    if (!pulse) return (float)__ldg(base + i);
    const float x = (float)i * inv_div1;
    const float rise = (x * x) * (3.0f - 2.0f * x);
    const float j = (float)(i - div1);
    const float fall = 1.0f - ((j * j) * scale);
    const float v = (i < div1) ? rise : fall;
    return ((double)i >= newDiv2) ? 0.0f : v;
}

// Glottal table value at integer index i for the current closure point (TRMWavetable.m:78-102 init,
// :117-162 update, vDSP order 1 - (j*j)*(1/(L*L))).  The reference rewrites the table every sample; the
// table is a pure function of the current amplitude, so it is evaluated on look-up instead.
template <typename R>
__device__ __forceinline__ R table_value(const double *__restrict__ base, int i, int div1, int div2, double newDiv2,
                                         R scale, bool pulse)
{
    if (!pulse || i < div1 || i >= div2) return (R)__ldg(base + i);
    if ((double)i >= newDiv2) return (R)0;
    R j = (R)(i - div1);
    return (R)1 - ((j * j) * scale);
}

constexpr unsigned FULL = 0xFFFFFFFFu;

}  // namespace TRM_KERNEL_NS
