// kernels_aux.cu -- kernels that are the same in both precision modes (compiled with -fmad=false: the frame
// generator's float / double arithmetic follows the reference operation by operation).
#include "framegen_kernel.cuh"

extern "C" int trm_k_framegen(const trm::FrameGenArgs *a, cudaStream_t s)
{
    if (a->n_utt <= 0) return 0;
    const int warps = 4;
    trm::framegen_kernel<<<(a->n_utt + warps - 1) / warps, warps * 32, 0, s>>>(*a);
    return (int)cudaGetLastError();
}

extern "C" int trm_k_framegen_pool(const trm::FrameGenPoolArgs *a, cudaStream_t s)
{
    if (a->n <= 0) return 0;
    const int warps = 4;
    trm::framegen_pool_kernel<<<(a->n + warps - 1) / warps, warps * 32, 0, s>>>(*a);
    return (int)cudaGetLastError();
}

// ---- config 5: control tracks generated on the device (include/trm_workload.h TRMWorkloadWalk2, bit-identical) -----------
__device__ __forceinline__ unsigned long long w2_splitmix(unsigned long long &s)
{
    unsigned long long z = (s += 0x9E3779B97F4A7C15ull);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
__device__ __forceinline__ double w2_uniform(unsigned long long &s) { return __dmul_rn((double)(w2_splitmix(s) >> 11), 1.0 / 9007199254740992.0); }

__constant__ double c_w2_lo[16] = {-22, 0, 0, 0, 0, 864, 500, 0.8, 0.05, 0.05, 0.05, 0.05, 0.05, 0.05, 0.05, 0.1};
__constant__ double c_w2_hi[16] = {-2, 60, 10, 24, 7, 5500, 4500, 0.8, 2.61, 2.61, 2.61, 2.61, 2.61, 2.61, 2.61, 1.5};

// one thread per (utterance, parameter): 16 consecutive threads write one 128-byte frame row per step
__global__ void workload_walk2_kernel(unsigned long long seed, unsigned long long first_index, long long n_utt, int n_frames,
                                      double *__restrict__ frames)
{
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long u = t >> 4;
    const int q = (int)(t & 15);
    if (u >= n_utt) return;
    unsigned long long s = seed * 0xD1342543DE82EF95ull + (first_index + (unsigned long long)u) * 0x9E3779B97F4A7C15ull +
                           (unsigned long long)q * 0xC2B2AE3D27D4EB4Full + 0x632BE59BD9B4E019ull;
    w2_splitmix(s);
    const double lo = c_w2_lo[q], hi = c_w2_hi[q], range = __dsub_rn(hi, lo);
    const double step = __dmul_rn(__dmul_rn(range, 1.7320508075688772), 0.02);
    double x = __dadd_rn(lo, __dmul_rn(range, w2_uniform(s)));
    double *out = frames + (size_t)u * (size_t)n_frames * 16 + q;
    for (int i = 0; i < n_frames; ++i) {
        if (i > 0 && range > 0) {
            double g = w2_uniform(s);
            g = __dadd_rn(g, w2_uniform(s));
            g = __dadd_rn(g, w2_uniform(s));
            g = __dadd_rn(g, w2_uniform(s));
            g = __dsub_rn(g, 2.0);
            x = __dadd_rn(x, __dmul_rn(g, step));
            for (int it = 0; it < 4 && (x < lo || x > hi); ++it) {
                if (x < lo) x = __dsub_rn(__dmul_rn(2.0, lo), x);
                if (x > hi) x = __dsub_rn(__dmul_rn(2.0, hi), x);
            }
        }
        out[(size_t)i * 16] = (double)(float)x;
    }
}

extern "C" int trm_k_workload_walk2(unsigned long long seed, unsigned long long first_index, long long n_utt, int n_frames,
                                    double *frames, cudaStream_t s)
{
    if (n_utt <= 0 || n_frames <= 0) return 0;
    const int threads = 256;
    const long long total = n_utt * 16;
    workload_walk2_kernel<<<(unsigned)((total + threads - 1) / threads), threads, 0, s>>>(seed, first_index, n_utt, n_frames, frames);
    return (int)cudaGetLastError();
}

// Per-utterance checksum of the PCM (the sink of config 5: 10^6 utterances' audio stays on the device, 8 bytes per
// utterance come back): sum over samples of (int64)pcm[i] * (2 i + 1) mod 2^64 -- position dependent, order independent.
__global__ void pcm_checksum_kernel(const trm_cuda_utterance *__restrict__ desc, int n_utt, const int16_t *__restrict__ pcm,
                                    unsigned long long *__restrict__ sums)
{
    const int u = blockIdx.x;
    if (u >= n_utt) return;
    const trm_cuda_utterance &d = desc[u];
    const long long n = d.n_out * d.channels;
    const int16_t *p = pcm + d.pcm_offset;
    unsigned long long acc = 0ull;
    for (long long i = threadIdx.x; i < n; i += blockDim.x) acc += (unsigned long long)((long long)p[i] * (2 * i + 1));
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xFFFFFFFFu, acc, o);
    __shared__ unsigned long long part[8];
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long t = 0ull;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += part[w];
        sums[u] = t;
    }
}

extern "C" int trm_k_pcm_checksum(const trm_cuda_utterance *desc, int n_utt, const int16_t *pcm, unsigned long long *sums, cudaStream_t s)
{
    if (n_utt <= 0) return 0;
    pcm_checksum_kernel<<<n_utt, 256, 0, s>>>(desc, n_utt, pcm, sums);
    return (int)cudaGetLastError();
}

// ---- stream pool bookkeeping (trm_cuda_pool_push) ---------------------------------------------------------------------
// One CTA per entry: its waveguide descriptor goes to the slot's place in the array the waveguide kernel indexes, and a
// slot opened since its last launch gets a fresh carried state -- everything zero, the noise generator at its start, the
// "no sample yet" flag set (the state a time-split batch chunk uploads with its tables).
__global__ void pool_prepare_kernel(trm::PoolPrepArgs a)
{
    const int e = blockIdx.x, slot = a.slot[e];
    const unsigned *src = reinterpret_cast<const unsigned *>(a.src + e);
    unsigned *dst = reinterpret_cast<unsigned *>(a.dst + slot);
    for (int i = threadIdx.x; i < (int)(sizeof(trm_cuda_utterance) / 4); i += blockDim.x) dst[i] = src[i];
    if (a.reset[e]) {
        unsigned long long *st = reinterpret_cast<unsigned long long *>(reinterpret_cast<unsigned char *>(a.state) + (size_t)slot * a.state_bytes);
        for (int i = threadIdx.x; i < (int)(a.state_bytes / 8); i += blockDim.x) st[i] = i == 2 ? a.noise_k0 : (i == 3 ? 1ull : 0ull);
    }
}

// One CTA per segment {src, dst, bytes} (ragged lengths): 16-byte accesses when both addresses and the length are
// multiples of 16, 4-byte words otherwise.  A push's history moves and a snapshot's state and history always take the
// 16-byte path (rows start on 32 elements, histories hold a multiple of 4 elements, states are 416 or 800 bytes).
__global__ void segment_copy_kernel(trm::SegCopyArgs a)
{
    const trm::CopySeg g = a.seg[blockIdx.x];
    if (((g.src | g.dst | g.bytes) & 15ull) == 0) {
        const uint4 *src = reinterpret_cast<const uint4 *>(g.src);
        uint4 *dst = reinterpret_cast<uint4 *>(g.dst);
        const long long n = (long long)(g.bytes >> 4);
        for (long long i = threadIdx.x; i < n; i += blockDim.x) dst[i] = src[i];
    } else {
        const unsigned *src = reinterpret_cast<const unsigned *>(g.src);
        unsigned *dst = reinterpret_cast<unsigned *>(g.dst);
        const long long n = (long long)(g.bytes >> 2);
        for (long long i = threadIdx.x; i < n; i += blockDim.x) dst[i] = src[i];
    }
}

extern "C" int trm_k_pool_prepare(const trm::PoolPrepArgs *a, cudaStream_t s)
{
    if (a->n <= 0) return 0;
    pool_prepare_kernel<<<a->n, 128, 0, s>>>(*a);
    return (int)cudaGetLastError();
}

extern "C" int trm_k_segment_copy(const trm::SegCopyArgs *a, cudaStream_t s)
{
    if (a->n <= 0) return 0;
    segment_copy_kernel<<<a->n, 128, 0, s>>>(*a);
    return (int)cudaGetLastError();
}
