// trm_cuda.cu -- C-ABI shim (include/trm_cuda.h): device memory, streams, chunked copy/compute
// pipeline and kernel launches.  No torch types, no C++ in the signatures.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <mutex>
#include <numeric>
#include <string>
#include <tuple>
#include <vector>

#include "kernel_args.h"
#include "trm_cuda.h"

// launchers of the three kernel translation units (launch.cuh): FP64 conformance, FP32 fast, FP64 strict
#define TRM_DECLARE_LAUNCHERS(SUF)                                              \
    int trm_k_configure_##SUF(trm::KernelInfo *);                               \
    int trm_k_upload_##SUF(const double *, int, const unsigned long long *);    \
    int trm_k_tube_wide_##SUF(const trm::TubeArgs *, int, cudaStream_t);        \
    int trm_k_tube_wide_pool_##SUF(const trm::TubeArgs *, int, cudaStream_t);   \
    int trm_k_src_##SUF(const trm::SrcArgs *, int, int, cudaStream_t);          \
    int trm_k_src_ctab_##SUF(const void *, void *, cudaStream_t);               \
    int trm_k_src_pool_##SUF(const trm::SrcPoolArgs *, int, cudaStream_t);     \
    int trm_k_pcm_pool_##SUF(const trm::PcmPoolArgs *, int, cudaStream_t);     \
    int trm_k_pcm_##SUF(const trm::PcmArgs *, long long, cudaStream_t);
extern "C" {
TRM_DECLARE_LAUNCHERS(f64)
TRM_DECLARE_LAUNCHERS(f32)
TRM_DECLARE_LAUNCHERS(f64s)
int trm_k_framegen(const trm::FrameGenArgs *, cudaStream_t);
int trm_k_framegen_pool(const trm::FrameGenPoolArgs *, cudaStream_t);
int trm_k_workload_walk2(unsigned long long, unsigned long long, long long, int, double *, cudaStream_t);
int trm_k_pcm_checksum(const trm_cuda_utterance *, int, const int16_t *, unsigned long long *, cudaStream_t);
int trm_k_pool_prepare(const trm::PoolPrepArgs *, cudaStream_t);
int trm_k_segment_copy(const trm::SegCopyArgs *, cudaStream_t);
}

// precision codes of include/trm.h: 0 = FP64 conformance, 1 = FP32 fast, 2 = FP64 strict
static inline bool prec_is_f64(int precision) { return precision != 1; }
static inline size_t prec_esz(int precision) { return precision != 1 ? sizeof(double) : sizeof(float); }
struct KernelSet {
    int (*tube_wide)(const trm::TubeArgs *, int, cudaStream_t);
    int (*src)(const trm::SrcArgs *, int, int, cudaStream_t);
    int (*pcm)(const trm::PcmArgs *, long long, cudaStream_t);
    int (*src_pool)(const trm::SrcPoolArgs *, int, cudaStream_t);
    int (*tube_wide_pool)(const trm::TubeArgs *, int, cudaStream_t);   // state stored per utterance (tube_wide.cuh)
    int (*pcm_pool)(const trm::PcmPoolArgs *, int, cudaStream_t);
};
static const KernelSet g_kernels[3] = {
    {trm_k_tube_wide_f64, trm_k_src_f64, trm_k_pcm_f64, trm_k_src_pool_f64, trm_k_tube_wide_pool_f64, trm_k_pcm_pool_f64},
    {trm_k_tube_wide_f32, trm_k_src_f32, trm_k_pcm_f32, trm_k_src_pool_f32, trm_k_tube_wide_pool_f32, trm_k_pcm_pool_f32},
    {trm_k_tube_wide_f64s, trm_k_src_f64s, trm_k_pcm_f64s, trm_k_src_pool_f64s, trm_k_tube_wide_pool_f64s, trm_k_pcm_pool_f64s},
};

// FMA-chain kernels used to MEASURE the FP32 / FP64 CUDA-core peak of the device the bench runs on
// (MEASURED_PEAKS.json only carries HBM and bf16 tensor numbers; the waveguide kernel is bound by neither).
template <typename T> __global__ void fp_peak_kernel(T *out, int iters)
{
    T a0 = (T)threadIdx.x * (T)1e-3, a1 = a0 + (T)1, a2 = a0 + (T)2, a3 = a0 + (T)3;
    T a4 = a0 + (T)4, a5 = a0 + (T)5, a6 = a0 + (T)6, a7 = a0 + (T)7;
    const T m = (T)0.999999, c = (T)1e-7;
    for (int i = 0; i < iters; ++i) {
        a0 = a0 * m + c; a1 = a1 * m + c; a2 = a2 * m + c; a3 = a3 * m + c;
        a4 = a4 * m + c; a5 = a5 * m + c; a6 = a6 * m + c; a7 = a7 * m + c;
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
}

namespace {

thread_local std::string g_err;

int fail(const char *what, cudaError_t e)
{
    char buf[512];
    snprintf(buf, sizeof buf, "%s: %s (%d)", what, cudaGetErrorString(e), (int)e);
    g_err = buf;
    return -5;   // TRM_ERR_CUDA
}
int fail_msg(const char *what)
{
    g_err = what;
    return -5;
}
#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t _e = (call);                                                                   \
        if (_e != cudaSuccess) return fail(#call, _e);                                             \
    } while (0)

constexpr int MAX_SLOTS = 16;  // upper bound of chunks in flight (each with its own arena, staging and events)
constexpr int MAX_OUT_GROUPS = 4;   // output groups of a chunk (ChunkPlan::groups)

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Parts of one packed buffer, each from a 256-byte boundary: the same offsets address the device scratch and its host image.
struct Pack { size_t bytes = 0; size_t part(size_t n) { const size_t at = align_up(bytes, 256); bytes = at + n; return at; } };

struct Arena {
    unsigned char *base = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes)
    {
        if (bytes <= cap) return 0;
        if (base) cudaFree(base);
        base = nullptr;
        cap = 0;
        cudaError_t e = cudaMalloc((void **)&base, bytes);
        if (e != cudaSuccess) return fail("cudaMalloc(arena)", e);
        cap = bytes;
        return 0;
    }
    void release()
    {
        if (base) cudaFree(base);
        base = nullptr;
        cap = 0;
    }
};

struct HostStage {
    unsigned char *base = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes)
    {
        if (bytes <= cap) return 0;
        if (base) cudaFreeHost(base);
        base = nullptr;
        cap = 0;
        cudaError_t e = cudaMallocHost((void **)&base, bytes);
        if (e != cudaSuccess) return fail("cudaMallocHost(stage)", e);
        cap = bytes;
        return 0;
    }
    void release()
    {
        if (base) cudaFreeHost(base);
        base = nullptr;
        cap = 0;
    }
};

// Host-side plan of one chunk: rebased descriptors, where its spans live in the caller's arrays, and where its parts live
// in its device scratch.
struct ChunkPlan {
    int u0 = 0, u1 = 0;
    std::vector<trm_cuda_utterance> desc;   // rebased to chunk-local offsets
    std::vector<int> order;
    // resampler work decomposition (src_kernel.cuh): tiles of <= 32 utterances with one converter signature
    std::vector<int> tile_utt, tile_nt;
    std::vector<long long> tile_max_out, tile_first_out, item_base;
    bool frames_dense = true;
    long long frames_lo = 0;                // host frame index of the span start (dense case)
    size_t frame_rows = 0;
    long long tube_lo = 0, out_lo = 0, pcm_lo = 0;   // host element offsets of the spans
    long long tube_n = 0, out_n = 0, pcm_n = 0;      // their lengths (what the copy-outs move)
    size_t tube_elems = 0, out_elems = 0, pcm_elems = 0;
    int src_shape = 0;                      // resampler shape the tiles were built for (KernelInfo::src[])
    // Output groups: contiguous utterance ranges whose resampling + scaling is launched separately, so that the PCM of
    // one group can leave for the host while the next group is still being resampled (tiles never span groups).
    struct Group { int u_begin, u_end; long long item_begin, item_end, max_n_out, pcm_lo, pcm_hi; };
    // Time split: when every utterance of the chunk has the same number of frames, the waveguide runs as two launches
    // (tube samples before / from control frame `split_frame`, recurrence state carried in `state` exactly as
    // a stream pool push does), so that the upload of the later frames overlaps the first launch.  0 = one launch.
    int split_frame = 0, uniform_frames = 0;
    std::vector<trm_cuda_utterance> desc_t[2];
    std::vector<Group> groups;
    long long total_items = 0, max_n_out = 0;
    size_t n_tiles() const { return tile_nt.size(); }
    bool f32_frames = false;                // the caller's frames are float32 rows (64 bytes)
    // Byte offsets of the parts in the chunk's device scratch (chunk_layout).  The uploaded tables come first, [0, up):
    // the pinned staging holds them at the same offsets and receives the maxima back at theirs.  The frame part holds
    // float32 rows when f32_frames (the kernels widen on read); the PCM part exists when want_pcm.
    struct Offsets {
        size_t desc, order, tile_utt, tile_nt, tile_max_out, tile_first_out, item_base, desc_t[2], state;
        size_t maxbits, frames, tube, out, pcm;
    } at{};
    size_t up = 0, arena = 0, stage = 0;
    bool want_pcm = false;
};

}  // namespace

// One compute queue per device, shared by every context (lane) on it: the kernels of concurrent calls run in
// submission order -- waveguide, resampler, PCM of call k, then those of call k+1 -- instead of fighting for the SMs
// (a waveguide launch of call k+1 that slips in front of call k's resampler would delay k's copy-out by a whole
// waveguide kernel).  Copies stay on per-context streams.  The mutex covers the enqueue of one chunk's three kernels.
static cudaStream_t g_run_stream[64];
static std::mutex g_run_mu[64];
// Likewise one copy-in queue per device: the frames of concurrent calls go up one call after the other at full PCIe
// rate (the first call's kernels start after ITS upload, not after everybody's).
static cudaStream_t g_in_stream[64];
static std::mutex g_in_mu[64];

struct trm_cuda_ctx {
    int device = 0;
    int sm_count = 0;
    double *d_wavetables = nullptr;
    int wt_capacity = 0;
    std::vector<double> wt_host;      // what d_wavetables holds
    Arena gen;                        // frame generator: events, descriptors, generated frames
    void *d_tab_f64 = nullptr, *d_tab_f32 = nullptr;
    void *d_ctab_f64 = nullptr, *d_ctab_f32 = nullptr;   // interpolated converter coefficients per time-register fraction
    uint64_t noise_k0 = 0;
    trm::KernelInfo info[3]{};        // by precision code
    const trm::KernelInfo &ki(int precision) const { return info[precision]; }
    cudaStream_t s_out = nullptr;     // copy-out of the chunk pipeline; also wavetable, frame generator and sweep work
    Arena arenas[MAX_SLOTS];
    HostStage stages[MAX_SLOTS];
    int n_slots = 3;              // chunks in flight: one uploading, one computing, one downloading
    cudaEvent_t ev_in[MAX_SLOTS]{}, ev_run[MAX_SLOTS]{}, ev_out[MAX_SLOTS]{};
    cudaEvent_t ev_in2[MAX_SLOTS]{};                    // time split: the later frames are on the device
    cudaEvent_t ev_grp[MAX_SLOTS][MAX_OUT_GROUPS]{};   // a group's PCM is complete (copy-out of the group may start)
};

struct trm_cuda_resident {
    trm_cuda_ctx *ctx = nullptr;
    int precision = 0;
    ChunkPlan plan;
    Arena arena;
    double *d_wavetables = nullptr;     // the batch's glottal tables: the context's set may be replaced by later calls
};

namespace {

int plan_chunk(const trm_cuda_utterance *desc, int u0, int u1, const trm::KernelInfo &ki, ChunkPlan &p, int want_groups = 1)
{
    const int n = u1 - u0;
    // The faster up-sampling shape needs every utterance of the chunk to up-sample with a work-item window that fits it.
    int shape = ki.n_src_shapes > 1 ? 1 : 0;
    for (int u = u0; u < u1 && shape == 1; ++u) {
        const auto &d = desc[u];
        const trm::KernelInfo::SrcShape &s1 = ki.src[1];
        const long long unit = (long long)trm::SRC_CHUNK * (s1.threads / 32);
        if (!d.upsample || d.tri == 0 || (long long)((double)(s1.rows - 3 - 2 * (d.padSize + 1)) * 65536.0 / (double)d.tri) < unit) shape = 0;
    }
    const trm::KernelInfo::SrcShape &sh = ki.src[shape];
    const int tile_width = sh.tile;
    p.src_shape = shape;
    p.u0 = u0;
    p.u1 = u1;
    p.desc.assign(desc + u0, desc + u1);
    // spans in the caller's arrays
    long long f_lo = INT64_MAX, f_hi = 0, f_sum = 0;
    long long t_lo = INT64_MAX, t_hi = 0, o_lo = INT64_MAX, o_hi = 0, c_lo = INT64_MAX, c_hi = 0;
    for (const auto &d : p.desc) {
        f_lo = std::min<long long>(f_lo, d.frame_offset);
        f_hi = std::max<long long>(f_hi, d.frame_offset + d.n_frames);
        f_sum += d.n_frames;
        t_lo = std::min<long long>(t_lo, d.tube_offset);
        t_hi = std::max<long long>(t_hi, d.tube_offset + d.n_tube);
        o_lo = std::min<long long>(o_lo, d.out_offset);
        o_hi = std::max<long long>(o_hi, d.out_offset + d.n_out);
        c_lo = std::min<long long>(c_lo, d.pcm_offset);
        c_hi = std::max<long long>(c_hi, d.pcm_offset + d.n_out * d.channels);
    }
    if (n == 0) { f_lo = t_lo = o_lo = c_lo = 0; }
    p.frames_dense = (f_hi - f_lo) <= f_sum + f_sum / 2 + 64;
    p.frames_lo = f_lo;
    p.tube_lo = t_lo; p.out_lo = o_lo; p.pcm_lo = c_lo;
    p.tube_n = t_hi - t_lo; p.out_n = o_hi - o_lo; p.pcm_n = c_hi - c_lo;
    p.tube_elems = (size_t)align_up((size_t)(t_hi - t_lo), TRM_ALIGN_ELEMS);
    p.out_elems = (size_t)align_up((size_t)(o_hi - o_lo), TRM_ALIGN_ELEMS);
    p.pcm_elems = (size_t)align_up((size_t)(c_hi - c_lo), TRM_ALIGN_ELEMS);
    long long compact = 0;
    p.max_n_out = 0;
    for (int i = 0; i < n; ++i) {
        auto &d = p.desc[i];
        if (p.frames_dense) d.frame_offset -= f_lo;
        else { d.frame_offset = compact; compact += d.n_frames; }
        d.tube_offset -= t_lo;
        d.out_offset -= o_lo;
        d.pcm_offset -= c_lo;
        p.max_n_out = std::max<long long>(p.max_n_out, d.n_out);
    }
    {
        // resampler tiles: utterances that share (time-register increment, pad, direction, phase increment,
        // ratio) share every filter coefficient; longest first so the rows of a tile finish together
        auto key = [&](int a) {
            const auto &d = p.desc[a];
            unsigned long long rb;
            memcpy(&rb, &d.sampleRateRatio, sizeof rb);
            return std::make_tuple(d.tri, d.padSize, d.upsample, d.phaseIncrement, rb);
        };
        // group boundaries: contiguous index ranges with about equal shares of the output samples
        long long out_sum = 0;
        for (const auto &d : p.desc) out_sum += d.n_out;
        const int n_groups = std::max(1, std::min(want_groups, n / std::max(1, tile_width)));
        p.groups.clear();
        p.tile_utt.clear(); p.tile_nt.clear(); p.tile_max_out.clear(); p.tile_first_out.clear(); p.item_base.assign(1, 0);
        int g_at = 0;
        long long acc = 0;
        for (int g = 0; g < n_groups; ++g) {
            int g_end = g_at;
            if (g == n_groups - 1) g_end = n;
            else
                while (g_end < n - (n_groups - 1 - g) && (g_end == g_at || acc + p.desc[g_end].n_out <= out_sum * (g + 1) / n_groups)) acc += p.desc[g_end++].n_out;
            ChunkPlan::Group grp{g_at, g_end, p.item_base.back(), 0, 0, INT64_MAX, 0};
            std::vector<int> idx(g_end - g_at);
            std::iota(idx.begin(), idx.end(), g_at);
            std::stable_sort(idx.begin(), idx.end(), [&](int a, int b) {
                const auto ka = key(a), kb = key(b);
                if (ka != kb) return ka < kb;
                return p.desc[a].n_out > p.desc[b].n_out;
            });
            const int m = (int)idx.size();
            for (int at = 0; at < m;) {
                int end = at;
                while (end < m && end - at < tile_width && key(idx[end]) == key(idx[at])) ++end;
                const auto &d0 = p.desc[idx[at]];
                if (d0.n_out > 0) {
                    const int reach = d0.padSize + 1;
                    // outputs per work item: the input window must fit the staged rows, every warp of the CTA gets the
                    // same whole number of SRC_CHUNK-sized runs
                    const long long unit = d0.upsample ? (long long)trm::SRC_CHUNK * (sh.threads / 32) : (long long)trm::SRC_CHUNK;
                    long long nt = (long long)((double)(sh.rows - 3 - 2 * reach) * 65536.0 / (double)d0.tri);
                    // (libtrm refuses such rate pairs when it derives the descriptor; this guards the C-ABI itself)
                    if (nt < unit) return fail_msg("resampler: the input window of one work item does not fit the staged rows (rate ratio too small)");
                    nt = std::min<long long>(nt, sh.nt_max);
                    nt = nt / unit * unit;
                    long long first = d0.n_out;              // streaming: the tile starts at its earliest missing output
                    for (int r = at; r < end; ++r) first = std::min<long long>(first, p.desc[idx[r]].out_start);
                    first = first / nt * nt;
                    for (int r = 0; r < tile_width; ++r) p.tile_utt.push_back(at + r < end ? idx[at + r] : -1);
                    p.tile_nt.push_back((int)nt);
                    p.tile_max_out.push_back(d0.n_out);
                    p.tile_first_out.push_back(first);
                    p.item_base.push_back(p.item_base.back() + (d0.n_out - first + nt - 1) / nt);
                }
                at = end;
            }
            grp.item_end = p.item_base.back();
            for (int u = g_at; u < g_end; ++u) {
                const auto &d = p.desc[u];
                grp.max_n_out = std::max<long long>(grp.max_n_out, d.n_out);
                grp.pcm_lo = std::min<long long>(grp.pcm_lo, d.pcm_offset);
                grp.pcm_hi = std::max<long long>(grp.pcm_hi, d.pcm_offset + d.n_out * d.channels);
            }
            if (grp.pcm_lo > grp.pcm_hi) grp.pcm_lo = grp.pcm_hi = 0;
            p.groups.push_back(grp);
            g_at = g_end;
        }
        p.total_items = p.item_base.back();
    }
    p.frame_rows = (size_t)(p.frames_dense ? (f_hi - f_lo) : compact);
    // longest utterances first, so the two utterances of a warp (and the warps of a CTA) finish together
    p.order.resize(n);
    std::iota(p.order.begin(), p.order.end(), 0);
    std::stable_sort(p.order.begin(), p.order.end(),
                     [&](int a, int b) { return p.desc[a].n_tube > p.desc[b].n_tube; });
    // time split candidates: dense frames, the same frame count everywhere (so that a frame range is one strided copy) and
    // one control period (so that the split falls on the same tube sample for every utterance)
    p.split_frame = 0;
    p.uniform_frames = 0;
    if (n > 0 && p.frames_dense) {
        const int nf = p.desc[0].n_frames;
        bool uniform = nf > 0;
        for (int i = 0; i < n && uniform; ++i)
            uniform = p.desc[i].n_frames == nf && p.desc[i].frame_offset == (long long)i * nf && p.desc[i].jc0 == 0 && p.desc[i].n_tube > 0 &&
                      p.desc[i].controlPeriod == p.desc[0].controlPeriod;
        if (uniform) p.uniform_frames = nf;
    }
    return 0;
}

// Arms the time split of a planned chunk: launch 0 covers the tube samples before control frame f1 (rounded down to a
// whole 16-sample block per utterance), launch 1 the rest, continuing from the saved state in the middle of a control
// interval (jc0) exactly like a stream pool push.
void arm_time_split(ChunkPlan &p, int f1)
{
    const size_t n = p.desc.size();
    p.split_frame = f1;
    p.desc_t[0].assign(p.desc.begin(), p.desc.end());
    p.desc_t[1].assign(p.desc.begin(), p.desc.end());
    for (size_t u = 0; u < n; ++u) {
        const trm_cuda_utterance &d = p.desc[u];
        const long long cp = d.controlPeriod;
        const long long t1 = ((long long)f1 * cp) / 16 * 16;          // first tube sample of launch 1
        const long long f0 = t1 / cp;                                 // control interval it lies in
        trm_cuda_utterance &a = p.desc_t[0][u], &b = p.desc_t[1][u];
        a.n_tube = t1;
        a.n_frames = f1 + 1;
        b.frame_offset = d.frame_offset + f0;
        b.n_frames = d.n_frames - (int)f0;
        b.jc0 = (int)(t1 - f0 * cp);
        b.tube_offset = d.tube_offset + t1;
        b.n_tube = d.n_tube - t1;
    }
}

// Lays out the chunk's device scratch (ChunkPlan::at), once the plan and its time split are final.
void chunk_layout(ChunkPlan &p, size_t esz, bool want_pcm)
{
    const size_t n = p.desc.size();
    ChunkPlan::Offsets &o = p.at;
    o = {};
    Pack pk;
    o.desc = pk.part(n * sizeof(trm_cuda_utterance));
    o.order = pk.part(n * sizeof(int));
    o.tile_utt = pk.part(p.tile_utt.size() * sizeof(int));
    o.tile_nt = pk.part(p.tile_nt.size() * sizeof(int));
    o.tile_max_out = pk.part(p.tile_max_out.size() * sizeof(long long));
    o.tile_first_out = pk.part(p.tile_first_out.size() * sizeof(long long));
    o.item_base = pk.part(p.item_base.size() * sizeof(long long));
    if (p.split_frame > 0) {
        o.desc_t[0] = pk.part(n * sizeof(trm_cuda_utterance));
        o.desc_t[1] = pk.part(n * sizeof(trm_cuda_utterance));
        o.state = pk.part(n * trm::tube_state_bytes(esz));
    }
    p.up = pk.bytes;
    o.maxbits = pk.part(n * sizeof(unsigned long long));
    p.stage = pk.bytes;
    o.frames = pk.part(p.frame_rows * 128);
    o.tube = pk.part(p.tube_elems * esz);
    o.out = pk.part(p.out_elems * esz);
    if (want_pcm) o.pcm = pk.part(p.pcm_elems * sizeof(int16_t));
    p.arena = pk.bytes;
    p.want_pcm = want_pcm;
}

// The chunk's tables ([0, up) of its layout) -> device in one copy: through the pinned staging `stage` (the pipeline's:
// the copy stays asynchronous), or through a pageable image when there is none.
int upload_plan(const ChunkPlan &p, unsigned char *base, unsigned char *stage, cudaStream_t s, size_t esz = 8, unsigned long long noise_k0 = 0)
{
    const size_t n = p.desc.size();
    if (n == 0) return 0;
    std::vector<unsigned char> image;
    if (!stage) {
        image.resize(p.up);
        stage = image.data();
    }
    auto put = [&](size_t at, const void *src, size_t bytes) { if (bytes) memcpy(stage + at, src, bytes); };
    put(p.at.desc, p.desc.data(), n * sizeof(trm_cuda_utterance));
    put(p.at.order, p.order.data(), n * sizeof(int));
    put(p.at.tile_utt, p.tile_utt.data(), p.tile_utt.size() * sizeof(int));
    put(p.at.tile_nt, p.tile_nt.data(), p.tile_nt.size() * sizeof(int));
    put(p.at.tile_max_out, p.tile_max_out.data(), p.tile_max_out.size() * sizeof(long long));
    put(p.at.tile_first_out, p.tile_first_out.data(), p.tile_first_out.size() * sizeof(long long));
    put(p.at.item_base, p.item_base.data(), p.item_base.size() * sizeof(long long));
    if (p.split_frame > 0) {
        put(p.at.desc_t[0], p.desc_t[0].data(), n * sizeof(trm_cuda_utterance));
        put(p.at.desc_t[1], p.desc_t[1].data(), n * sizeof(trm_cuda_utterance));
        // fresh recurrence state: everything zero, noise generator at its start, "no sample yet" flag set
        const size_t sb = trm::tube_state_bytes(esz);
        memset(stage + p.at.state, 0, n * sb);
        for (size_t u = 0; u < n; ++u) {
            unsigned long long *h = (unsigned long long *)(stage + p.at.state + u * sb);
            h[2] = noise_k0;
            h[3] = 1ull;
        }
    }
    CK(cudaMemcpyAsync(base, stage, p.up, cudaMemcpyHostToDevice, s));
    return 0;
}

int upload_frames(const ChunkPlan &p, unsigned char *base, const trm_cuda_utterance *desc_global, const void *frames_host, cudaStream_t s)
{
    if (p.frame_rows == 0) return 0;
    const size_t row = p.f32_frames ? 64 : 128;                     // bytes per frame in the caller's array and on the device
    unsigned char *dst = base + p.at.frames;
    const unsigned char *src = (const unsigned char *)frames_host;
    if (p.frames_dense) {
        CK(cudaMemcpyAsync(dst, src + (size_t)p.frames_lo * row, p.frame_rows * row, cudaMemcpyDefault, s));
    } else {
        for (size_t i = 0; i < p.desc.size(); ++i) {
            const auto &g = desc_global[p.u0 + i];
            CK(cudaMemcpyAsync(dst + (size_t)p.desc[i].frame_offset * row, src + (size_t)g.frame_offset * row,
                               (size_t)g.n_frames * row, cudaMemcpyDefault, s));
        }
    }
    return 0;
}

// CTAs of the waveguide kernel for a chunk of n utterances: one per SM and wave, at most wide_max_utt utterances each; small
// chunks are spread two utterances per CTA (one feed-forward warp each) over as many SMs as there are pairs.
int wide_groups(const trm_cuda_ctx *ctx, const trm::KernelInfo &ki, int n)
{
    if (n <= 0) return 0;
    const int sm = ctx->sm_count, gmax = ki.wide_max_utt;
    if ((long long)n <= (long long)sm * gmax) return std::max(1, std::min(sm, (n + 1) / 2));
    const int waves = (int)(((long long)n + (long long)sm * gmax - 1) / ((long long)sm * gmax));
    return waves * sm;
}

// One kernel stage of a planned chunk whose scratch starts at `base`; `wavetables` overrides the context's glottal tables
// (device-resident batches keep their own copy), null = the context's.
int launch_stage(trm_cuda_ctx *ctx, int precision, int stage, const ChunkPlan &p, unsigned char *base, const double *wavetables,
                 cudaStream_t s, const ChunkPlan::Group *grp = nullptr, int time_part = -1)
{
    const bool f64 = prec_is_f64(precision);
    const KernelSet &K = g_kernels[precision];
    const int n = (int)p.desc.size();
    const auto *desc = (const trm_cuda_utterance *)(base + p.at.desc);
    auto *maxbits = (unsigned long long *)(base + p.at.maxbits);
    int rc = 0;
    if (stage == TRM_STAGE_TUBE) {
        trm::TubeArgs a{};
        a.desc = desc; a.order = (const int *)(base + p.at.order); a.n_utt = n; a.frames = base + p.at.frames;
        a.frames_f32 = p.f32_frames ? 1 : 0; a.tube = base + p.at.tube;
        a.wavetables = wavetables ? wavetables : ctx->d_wavetables; a.noise_k0 = ctx->noise_k0;
        // time split: launch time_part's descriptors, the recurrence state carried from launch 0 to launch 1
        if (time_part >= 0) { a.desc = (const trm_cuda_utterance *)(base + p.at.desc_t[time_part]); a.state = base + p.at.state; }
        const trm::KernelInfo &ki = ctx->ki(precision);
        const int groups = wide_groups(ctx, ki, n);
        if (groups > 0) rc = K.tube_wide(&a, groups, s);
    } else if (stage == TRM_STAGE_SRC) {
        // (the running maxima are cleared once per chunk: by the ungrouped launch, or by the first group's)
        if (!grp || grp->u_begin == 0) CK(cudaMemsetAsync(maxbits, 0, (size_t)n * sizeof(unsigned long long), s));
        trm::SrcArgs a{};
        a.desc = desc; a.n_utt = n; a.tube = base + p.at.tube; a.out = base + p.at.out; a.maxbits = maxbits;
        a.table = f64 ? ctx->d_tab_f64 : ctx->d_tab_f32;
        a.ctab = f64 ? ctx->d_ctab_f64 : ctx->d_ctab_f32;
        a.tile_utt = (const int *)(base + p.at.tile_utt); a.tile_nt = (const int *)(base + p.at.tile_nt);
        a.tile_max_out = (const long long *)(base + p.at.tile_max_out); a.tile_first_out = (const long long *)(base + p.at.tile_first_out);
        a.item_base = (const long long *)(base + p.at.item_base);
        a.n_tiles = (int)p.n_tiles(); a.total_items = p.total_items;
        if (grp) { a.item_begin = grp->item_begin; a.item_end = grp->item_end; if (a.item_end <= a.item_begin) return 0; }
        const trm::KernelInfo &ki = ctx->ki(precision);
        const int grid = ctx->sm_count * std::max(1, ki.src[p.src_shape].ctas_per_sm);
        rc = K.src(&a, grid, p.src_shape, s);
    } else if (stage == TRM_STAGE_PCM) {
        if (!p.want_pcm) return 0;
        trm::PcmArgs a{};
        a.desc = desc; a.n_utt = grp ? grp->u_end : n; a.u_begin = grp ? grp->u_begin : 0;
        a.out = base + p.at.out; a.maxbits = maxbits; a.pcm = (int16_t *)(base + p.at.pcm);
        const long long longest = grp ? grp->max_n_out : p.max_n_out;
        rc = K.pcm(&a, longest, s);
    }
    if (rc != 0) return fail("kernel launch", (cudaError_t)rc);
    return 0;
}

int chunk_utterances(const trm_cuda_ctx *ctx, int precision, int n, const trm_cuda_utterance *desc, size_t esz)
{
    // Chunk size: the kernels of one chunk run alone on the device, so a chunk must be large enough to fill it --
    // for the batch-throughput waveguide mapping that is >= ~14 utterances per SM (below that its recurrence warp,
    // not the feed-forward work, sets the time) -- and small enough that there are at least two chunks, so that the
    // PCM of one chunk leaves for the host while the next one is computed.  Bounded by scratch memory.
    const char *env = getenv("TRM_CHUNK_UTTERANCES");
    if (env && atoi(env) > 0) return atoi(env);
    // scratch of a chunk = frames + tube-rate + output-rate samples + PCM of its utterances; the bound uses the LARGEST
    // utterance of the batch (ragged batches: an average over a prefix would let one chunk of long utterances overshoot)
    // and what the device can actually give three in-flight chunks per context lane
    size_t per_utt = 1;
    for (int i = 0; i < n; ++i)
        per_utt = std::max(per_utt, (size_t)desc[i].n_frames * 128 + ((size_t)desc[i].n_tube + (size_t)desc[i].n_out) * esz +
                                        (size_t)desc[i].n_out * 2 * desc[i].channels + 1024);
    size_t free_b = 0, total_b = 0, reserved = 0;
    if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) { free_b = (size_t)96 << 30; cudaGetLastError(); }
    for (int i = 0; i < MAX_SLOTS; ++i) reserved += ctx->arenas[i].cap;          // already ours: reused, not needed again
    const size_t budget = std::min<size_t>((size_t)32 << 30, (size_t)(0.85 * (double)(free_b + reserved)) / 3);
    const long long by_mem = std::max<long long>(1, (long long)(budget / per_utt));
    const trm::KernelInfo &ki = ctx->ki(precision);
    const long long lo = (long long)ctx->sm_count * (ki.wide_max_utt / 2), hi = (long long)ctx->sm_count * ki.wide_max_utt;
    // FP64: a launch below ~28 utterances per SM is bound by the latency of its feed-forward warps, so halving a batch
    // costs more kernel time than the overlapped copy-out saves -> one chunk up to the device's capacity.  FP32: the
    // kernels are short next to the PCIe time of their PCM -> two chunks, the first one's PCM hides behind the second.
    long long want = prec_is_f64(precision) ? hi : std::min<long long>(hi, std::max<long long>(lo, (n + 1) / 2));
    long long c = std::max<long long>(1, std::min<long long>(std::min<long long>(want, by_mem), n));
    const long long n_chunks = (n + c - 1) / c;                 // balance the chunks
    return (int)((n + n_chunks - 1) / n_chunks);
}

}  // namespace

extern "C" {

const char *trm_cuda_last_error(void) { return g_err.c_str(); }

// A device's copy-in and compute queues, the copy-out stream of each of its contexts and each stream pool's stream are
// busy at once; with the default of 8 hardware work queues, streams alias onto the same queue and one chunk's kernels
// wait behind another chunk's copies.  Must be set before the CUDA context exists, so it is done on the first entry
// into the library (no effect if the host application already initialised CUDA: such callers set
// CUDA_DEVICE_MAX_CONNECTIONS=32 themselves).
static void want_many_connections() { setenv("CUDA_DEVICE_MAX_CONNECTIONS", "32", 0); }

int trm_cuda_device_count(void)
{
    want_many_connections();
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) { fail("cudaGetDeviceCount", e); return 0; }
    return n;
}

void *trm_cuda_host_alloc(size_t bytes)
{
    want_many_connections();
    void *p = nullptr;
    cudaError_t e = cudaMallocHost(&p, bytes ? bytes : 1);
    if (e != cudaSuccess) { fail("cudaMallocHost", e); return nullptr; }
    return p;
}

void trm_cuda_host_free(void *p) { if (p) cudaFreeHost(p); }

/* Measured FMA peak in TFLOP/s (2 flops per FMA) for precision 0 = FP64, 1 = FP32; best of `reps` runs. */
int trm_cuda_fp_peak(int device, int precision, int reps, double *tflops)
{
    CK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    const int threads = 256, blocks = prop.multiProcessorCount * 8, iters = precision != 1 ? 1 << 14 : 1 << 16;
    void *buf = nullptr;
    CK(cudaMalloc(&buf, (size_t)threads * blocks * sizeof(double)));
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    double best = 0;
    for (int r = 0; r < reps + 1; ++r) {
        CK(cudaEventRecord(e0, 0));
        if (precision != 1) fp_peak_kernel<double><<<blocks, threads>>>((double *)buf, iters);
        else fp_peak_kernel<float><<<blocks, threads>>>((float *)buf, iters);
        CK(cudaEventRecord(e1, 0));
        CK(cudaEventSynchronize(e1));
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, e0, e1));
        const double tf = 2.0 * 8.0 * (double)iters * threads * blocks / (ms * 1e-3) / 1e12;
        if (r > 0 && tf > best) best = tf;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(buf);
    *tflops = best;
    return 0;
}

int trm_cuda_ctx_create(int device, const trm_cuda_tables *t, trm_cuda_ctx **out)
{
    *out = nullptr;
    want_many_connections();
    int ndev = 0;
    CK(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return fail_msg("trm_cuda_ctx_create: no such CUDA device");
    CK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) return fail_msg("trm_cuda_ctx_create: kernels are built for sm_100a only");
    trm_cuda_ctx *c = new trm_cuda_ctx();
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    c->noise_k0 = t->noise_k0;
    int rc;
    if ((rc = trm_k_upload_f64(t->fir_coef, t->fir_taps, (const unsigned long long *)t->noise_pow)) != 0 ||
        (rc = trm_k_upload_f32(t->fir_coef, t->fir_taps, (const unsigned long long *)t->noise_pow)) != 0 ||
        (rc = trm_k_upload_f64s(t->fir_coef, t->fir_taps, (const unsigned long long *)t->noise_pow)) != 0) {
        delete c;
        return rc < 0 ? fail_msg("FIR design is not the 49-tap filter the kernels are built for") : fail("constant upload", (cudaError_t)rc);
    }
    if ((rc = trm_k_configure_f64(&c->info[0])) != 0 || (rc = trm_k_configure_f32(&c->info[1])) != 0 ||
        (rc = trm_k_configure_f64s(&c->info[2])) != 0) {
        delete c;
        return fail("kernel configuration", (cudaError_t)rc);
    }
    // interleaved (h, deltaH) tables in both precisions
    {
        std::vector<trm::HD<double>> td(TRM_SRC_FILTER_LEN);
        std::vector<trm::HD<float>> tf(TRM_SRC_FILTER_LEN);
        // phase-major: entry (l, k) = filter index l + 256 k sits at l * 13 + k, so the 13 taps of one wing are contiguous
        for (int i = 0; i < TRM_SRC_FILTER_LEN; ++i) {
            const int at = (i & 255) * trm::SRC_ZC + (i >> 8);
            td[at].h = t->src_h[i]; td[at].dh = t->src_dh[i];
            tf[at].h = (float)t->src_h[i]; tf[at].dh = (float)t->src_dh[i];
        }
        CK(cudaMalloc(&c->d_tab_f64, td.size() * sizeof(td[0])));
        CK(cudaMalloc(&c->d_tab_f32, tf.size() * sizeof(tf[0])));
        CK(cudaMemcpy(c->d_tab_f64, td.data(), td.size() * sizeof(td[0]), cudaMemcpyHostToDevice));
        CK(cudaMemcpy(c->d_tab_f32, tf.data(), tf.size() * sizeof(tf[0]), cudaMemcpyHostToDevice));
        CK(cudaMalloc(&c->d_ctab_f64, (size_t)65536 * trm::SRC_CLD * sizeof(double)));
        CK(cudaMalloc(&c->d_ctab_f32, (size_t)65536 * trm::SRC_CLD * sizeof(float)));
        if ((rc = trm_k_src_ctab_f64s(c->d_tab_f64, c->d_ctab_f64, 0)) != 0 || (rc = trm_k_src_ctab_f32(c->d_tab_f32, c->d_ctab_f32, 0)) != 0) {
            delete c;
            return fail("converter coefficient table", (cudaError_t)rc);
        }
        CK(cudaDeviceSynchronize());
    }
    {
        // s_out = copy-out of the chunk pipeline (trm_cuda_synthesize_host); frames and kernels go to the device's
        // shared copy-in and compute queues
        {
            std::lock_guard<std::mutex> lk(g_run_mu[device]);
            if (!g_run_stream[device]) CK(cudaStreamCreateWithFlags(&g_run_stream[device], cudaStreamNonBlocking));
            if (!g_in_stream[device]) CK(cudaStreamCreateWithFlags(&g_in_stream[device], cudaStreamNonBlocking));
        }
        int lo = 0, hi = 0;
        CK(cudaDeviceGetStreamPriorityRange(&lo, &hi));          // lo = least (numerically largest)
        CK(cudaStreamCreateWithPriority(&c->s_out, cudaStreamNonBlocking, std::min(lo, hi + 2)));
        const char *env = getenv("TRM_SLOTS");
        if (env && atoi(env) > 0) c->n_slots = std::min(MAX_SLOTS, atoi(env));
        for (int i = 0; i < MAX_SLOTS; ++i) {
            CK(cudaEventCreateWithFlags(&c->ev_in[i], cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&c->ev_run[i], cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&c->ev_out[i], cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&c->ev_in2[i], cudaEventDisableTiming));
            for (int g = 0; g < MAX_OUT_GROUPS; ++g) CK(cudaEventCreateWithFlags(&c->ev_grp[i][g], cudaEventDisableTiming));
        }
    }
    *out = c;
    return 0;
}

int trm_cuda_set_wavetables(trm_cuda_ctx *c, const double *tables, int n_voices)
{
    if (n_voices <= 0) return fail_msg("trm_cuda_set_wavetables: no voices");
    const size_t n = (size_t)n_voices * TRM_TABLE_LENGTH;
    // unchanged since the last call (the usual case: one voice set per application): nothing to do, and in particular
    // no synchronisation that would serialise this call behind another lane's work on the same device
    if (c->wt_host.size() == n && memcmp(c->wt_host.data(), tables, n * sizeof(double)) == 0) return 0;
    CK(cudaSetDevice(c->device));
    CK(cudaStreamSynchronize(c->s_out));   // this context's own work only
    if (n_voices > c->wt_capacity) {
        if (c->d_wavetables) cudaFree(c->d_wavetables);
        c->d_wavetables = nullptr;
        c->wt_capacity = 0;
        CK(cudaMalloc((void **)&c->d_wavetables, n * sizeof(double)));
        c->wt_capacity = n_voices;
    }
    CK(cudaMemcpy(c->d_wavetables, tables, n * sizeof(double), cudaMemcpyHostToDevice));
    c->wt_host.assign(tables, tables + n);
    return 0;
}

void trm_cuda_ctx_destroy(trm_cuda_ctx *c)
{
    if (!c) return;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    if (c->s_out) cudaStreamDestroy(c->s_out);
    for (int i = 0; i < MAX_SLOTS; ++i) {
        if (c->ev_in[i]) cudaEventDestroy(c->ev_in[i]);
        if (c->ev_run[i]) cudaEventDestroy(c->ev_run[i]);
        if (c->ev_out[i]) cudaEventDestroy(c->ev_out[i]);
        if (c->ev_in2[i]) cudaEventDestroy(c->ev_in2[i]);
        for (int g = 0; g < MAX_OUT_GROUPS; ++g) if (c->ev_grp[i][g]) cudaEventDestroy(c->ev_grp[i][g]);
    }
    for (auto &a : c->arenas) a.release();
    c->gen.release();
    for (auto &h : c->stages) h.release();
    if (c->d_wavetables) cudaFree(c->d_wavetables);
    if (c->d_tab_f64) cudaFree(c->d_tab_f64);
    if (c->d_tab_f32) cudaFree(c->d_tab_f32);
    if (c->d_ctab_f64) cudaFree(c->d_ctab_f64);
    if (c->d_ctab_f32) cudaFree(c->d_ctab_f32);
    delete c;
}

int trm_cuda_synthesize_host(trm_cuda_ctx *ctx, int precision, int frame_format, int n, const trm_cuda_utterance *desc,
                             const void *frames_host, int16_t *pcm_host, void *samples_host, double *max_host,
                             void *tube_host, int64_t *launches, void (*enqueued)(void *), void *enqueued_arg)
{
    if (frame_format != 0 && frame_format != 1) return fail_msg("unknown frame format");
    const bool f32_frames = frame_format == 1;
    if (launches) *launches = 0;
    if (n <= 0) return 0;
    CK(cudaSetDevice(ctx->device));
    if (precision < 0 || precision > 2) return fail_msg("unknown precision code");
    const size_t esz = prec_esz(precision);
    const bool want_pcm = pcm_host != nullptr;
    const int per_chunk = chunk_utterances(ctx, precision, n, desc, esz);
    const int n_chunks = (n + per_chunk - 1) / per_chunk;
    const int N_SLOTS = std::min(ctx->n_slots, std::max(n_chunks, 1));
    // Three-stage pipeline over chunks: frames go up on the copy-in stream, the three kernels of a chunk run on the
    // compute stream (one chunk at a time: a waveguide launch fills every SM), PCM / samples come back on the copy-out
    // stream.  H2D of chunk k+1 and D2H of chunk k-1 overlap the kernels of chunk k (full-duplex PCIe).
    cudaStream_t s_in = g_in_stream[ctx->device], s_run = g_run_stream[ctx->device], s_out = ctx->s_out;
    // TRM_TRACE=1: per-chunk timeline of the pipeline stages (CUDA events), printed to stderr
    const bool trace = getenv("TRM_TRACE") != nullptr;
    std::vector<cudaEvent_t> tev;
    static cudaEvent_t t_origin = nullptr;          // one time axis for every traced call of the process
    static std::mutex t_mutex;
    static double t_host0 = 0.0;
    auto now_ms = []() { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return 1e3 * (double)ts.tv_sec + 1e-6 * (double)ts.tv_nsec; };
    auto mark = [&](cudaStream_t st) {
        if (!trace) return;
        cudaEvent_t e;
        cudaEventCreate(&e);
        cudaEventRecord(e, st);
        tev.push_back(e);
    };
    if (trace) {
        std::lock_guard<std::mutex> lk(t_mutex);
        if (!t_origin) { cudaEventCreate(&t_origin); cudaEventRecord(t_origin, s_out); cudaEventSynchronize(t_origin); t_host0 = now_ms(); }
    }
    const double t_enter = trace ? now_ms() - t_host0 : 0.0;
    std::vector<ChunkPlan> plans(N_SLOTS);
    std::vector<int> slot_chunk(N_SLOTS, -1);
    int64_t n_launch = 0;

    auto finish_slot = [&](int slot) -> int {
        // wait for the slot's copy-out, then hand the per-utterance maxima to the caller
        CK(cudaEventSynchronize(ctx->ev_out[slot]));
        const int ci = slot_chunk[slot];
        if (ci >= 0 && max_host) {
            const ChunkPlan &p = plans[slot];
            const unsigned long long *mb = (const unsigned long long *)(ctx->stages[slot].base + p.at.maxbits);
            for (size_t i = 0; i < p.desc.size(); ++i) {
                double v;
                memcpy(&v, &mb[i], sizeof v);
                max_host[p.u0 + i] = v;
            }
        }
        slot_chunk[slot] = -1;
        return 0;
    };

    // An error inside the chunk loop must not return while earlier chunks' copies are still landing in the caller's buffers
    // (the caller may free them as soon as the call fails): drain this call's queues first.
    auto drain = [&]() {
        cudaStreamSynchronize(s_in);
        cudaStreamSynchronize(s_run);
        cudaStreamSynchronize(s_out);
    };
#define CKD(call)                                                                                  \
    do {                                                                                           \
        cudaError_t _e = (call);                                                                   \
        if (_e != cudaSuccess) { drain(); return fail(#call, _e); }                                \
    } while (0)
#define RCD(expr)                                                                                  \
    do {                                                                                           \
        if ((rc = (expr)) != 0) { drain(); return rc; }                                            \
    } while (0)
    for (int ci = 0; ci < n_chunks; ++ci) {
        const int slot = ci % N_SLOTS;
        int rc;
        if (slot_chunk[slot] >= 0) RCD(finish_slot(slot));
        ChunkPlan &p = plans[slot];
        const int u0 = ci * per_chunk, u1 = std::min(n, u0 + per_chunk);
        // large chunks with PCM output are resampled and scaled in up to MAX_OUT_GROUPS output groups
        long long chunk_out = 0;
        for (int u = u0; u < u1; ++u) chunk_out += desc[u].n_out;
        const int want_groups = (want_pcm && !getenv("TRM_NO_OUT_GROUPS")) ? (int)std::min<long long>(MAX_OUT_GROUPS, chunk_out / (64ll << 20)) : 1;
        RCD(plan_chunk(desc, u0, u1, ctx->ki(precision), p, want_groups));
        p.f32_frames = f32_frames;
        const bool grouped = p.groups.size() > 1;
        // long uniform chunks: the waveguide as two launches in time, the later frames uploaded behind the first
        if (p.uniform_frames >= 512 && !getenv("TRM_NO_TIME_SPLIT") &&
            wide_groups(ctx, ctx->ki(precision), u1 - u0) > 0)
            arm_time_split(p, std::max(64, (int)(0.28 * p.uniform_frames)));
        const bool split = p.split_frame > 0;
        chunk_layout(p, esz, want_pcm);
        RCD(ctx->arenas[slot].reserve(p.arena));
        RCD(ctx->stages[slot].reserve(p.stage));
        unsigned char *base = ctx->arenas[slot].base;
        // ---- copy-in -----------------------------------------------------------------------------------------
        {
            std::lock_guard<std::mutex> lk(g_in_mu[ctx->device]);
            mark(s_in);
            RCD(upload_plan(p, base, ctx->stages[slot].base, s_in, esz, ctx->noise_k0));
            if (!split) {
                RCD(upload_frames(p, base, desc, frames_host, s_in));
                CKD(cudaEventRecord(ctx->ev_in[slot], s_in));
            } else {
                // frames [0, f1] of every utterance, then the rest: two strided copies
                const size_t row = f32_frames ? 64 : 128;
                const size_t pitch = (size_t)p.uniform_frames * row, first = (size_t)(p.split_frame + 1) * row;
                const unsigned char *src = (const unsigned char *)frames_host + (size_t)p.frames_lo * row;
                unsigned char *dst = base + p.at.frames;
                CKD(cudaMemcpy2DAsync(dst, pitch, src, pitch, first, (size_t)(u1 - u0), cudaMemcpyDefault, s_in));
                CKD(cudaEventRecord(ctx->ev_in[slot], s_in));
                CKD(cudaMemcpy2DAsync(dst + first, pitch, src + first, pitch, pitch - first, (size_t)(u1 - u0), cudaMemcpyDefault, s_in));
                CKD(cudaEventRecord(ctx->ev_in2[slot], s_in));
            }
            mark(s_in);
        }
        // ---- kernels -----------------------------------------------------------------------------------------
        {
            std::lock_guard<std::mutex> lk(g_run_mu[ctx->device]);
            CKD(cudaStreamWaitEvent(s_run, ctx->ev_in[slot], 0));
            auto waveguide = [&]() -> int {
                if (!split) { ++n_launch; return launch_stage(ctx, precision, TRM_STAGE_TUBE, p, base, nullptr, s_run); }
                int r = launch_stage(ctx, precision, TRM_STAGE_TUBE, p, base, nullptr, s_run, nullptr, 0);
                if (r != 0) return r;
                CKD(cudaStreamWaitEvent(s_run, ctx->ev_in2[slot], 0));
                n_launch += 2;
                return launch_stage(ctx, precision, TRM_STAGE_TUBE, p, base, nullptr, s_run, nullptr, 1);
            };
            if (!grouped) {
                for (int st = 0; st < TRM_STAGE_COUNT; ++st) {
                    if (st == TRM_STAGE_PCM && !want_pcm) { mark(s_run); continue; }
                    if (st == TRM_STAGE_TUBE) rc = waveguide();
                    else { rc = launch_stage(ctx, precision, st, p, base, nullptr, s_run); ++n_launch; }
                    if (rc != 0) { drain(); return rc; }
                    mark(s_run);
                }
            } else {
                // the waveguide over the whole chunk (it needs all of it to fill the device), then resampling + scaling
                // group by group: group g's PCM crosses PCIe while group g+1 is resampled
                RCD(waveguide());
                mark(s_run);
                for (size_t g = 0; g < p.groups.size(); ++g) {
                    RCD(launch_stage(ctx, precision, TRM_STAGE_SRC, p, base, nullptr, s_run, &p.groups[g]));
                    if (g + 1 == p.groups.size()) mark(s_run);
                    RCD(launch_stage(ctx, precision, TRM_STAGE_PCM, p, base, nullptr, s_run, &p.groups[g]));
                    CKD(cudaEventRecord(ctx->ev_grp[slot][g], s_run));
                    n_launch += 2;
                }
                mark(s_run);
            }
            CKD(cudaEventRecord(ctx->ev_run[slot], s_run));
        }
        // ---- copy-out ----------------------------------------------------------------------------------------
        const int16_t *d_pcm = (const int16_t *)(base + p.at.pcm);
        if (grouped) {
            for (size_t g = 0; g < p.groups.size(); ++g) {
                const ChunkPlan::Group &grp = p.groups[g];
                CKD(cudaStreamWaitEvent(s_out, ctx->ev_grp[slot][g], 0));
                if (grp.pcm_hi > grp.pcm_lo)
                    CKD(cudaMemcpyAsync(pcm_host + p.pcm_lo + grp.pcm_lo, d_pcm + grp.pcm_lo, (size_t)(grp.pcm_hi - grp.pcm_lo) * sizeof(int16_t),
                                       cudaMemcpyDeviceToHost, s_out));
            }
        }
        CKD(cudaStreamWaitEvent(s_out, ctx->ev_run[slot], 0));
        if (!grouped && want_pcm && p.pcm_n)
            CKD(cudaMemcpyAsync(pcm_host + p.pcm_lo, d_pcm, (size_t)p.pcm_n * sizeof(int16_t), cudaMemcpyDeviceToHost, s_out));
        if (samples_host && p.out_n)
            CKD(cudaMemcpyAsync((unsigned char *)samples_host + (size_t)p.out_lo * esz, base + p.at.out, (size_t)p.out_n * esz,
                                cudaMemcpyDeviceToHost, s_out));
        if (tube_host && p.tube_n)
            CKD(cudaMemcpyAsync((unsigned char *)tube_host + (size_t)p.tube_lo * esz, base + p.at.tube, (size_t)p.tube_n * esz,
                                cudaMemcpyDeviceToHost, s_out));
        // the maxima come back into the staging at their device offset
        if (max_host)
            CKD(cudaMemcpyAsync(ctx->stages[slot].base + p.at.maxbits, base + p.at.maxbits, p.desc.size() * sizeof(unsigned long long),
                                cudaMemcpyDeviceToHost, s_out));
        CKD(cudaEventRecord(ctx->ev_out[slot], s_out));
        mark(s_out);
        slot_chunk[slot] = ci;
        if (ci == 0 && enqueued) enqueued(enqueued_arg);
    }
    const double t_enqueued = trace ? now_ms() - t_host0 : 0.0;
    for (int slot = 0; slot < N_SLOTS; ++slot) {
        int rc;
        if (slot_chunk[slot] >= 0 && (rc = finish_slot(slot)) != 0) return rc;
    }
    if (trace) {
        std::lock_guard<std::mutex> lk(t_mutex);
        fprintf(stderr, "[trm trace] ctx %p chunk: start h2d_done tube_done src_done pcm_done d2h_done (ms since the first traced call)\n", (void *)ctx);
        for (size_t i = 0; i + 6 <= tev.size(); i += 6) {
            float t[6];
            for (int k = 0; k < 6; ++k) cudaEventElapsedTime(&t[k], t_origin, tev[i + k]);
            fprintf(stderr, "[trm trace] %2zu: %8.2f %8.2f %8.2f %8.2f %8.2f %8.2f\n", i / 6, t[0], t[1], t[2], t[3], t[4], t[5]);
        }
        fprintf(stderr, "[trm trace] host: entered %.2f, everything enqueued %.2f, outputs complete %.2f\n", t_enter, t_enqueued, now_ms() - t_host0);
        for (auto e : tev) cudaEventDestroy(e);
    }
    if (launches) *launches = n_launch;
    return 0;
#undef CKD
#undef RCD
}

int trm_cuda_generate_frames(trm_cuda_ctx *ctx, int n, const trm_cuda_utterance *desc, const trm_cuda_event *events,
                             const int64_t *ev_offset, const int32_t *ev_count, const trm_cuda_framegen *fg, int shared_fg,
                             const double **frames_dev, double *frames_host, float *seed_host)
{
    if (frames_dev) *frames_dev = nullptr;
    if (n <= 0) return 0;
    CK(cudaSetDevice(ctx->device));
    long long n_events = 0, frames_hi = 0;
    for (int u = 0; u < n; ++u) {
        n_events = std::max<long long>(n_events, ev_offset[u] + ev_count[u]);
        frames_hi = std::max<long long>(frames_hi, desc[u].frame_offset + desc[u].n_frames);
    }
    const size_t n_fg = shared_fg ? 1 : (size_t)n;
    std::vector<long long> off(ev_offset, ev_offset + n);
    Pack pk;
    const size_t o_desc = pk.part((size_t)n * sizeof(trm_cuda_utterance)), o_ev = pk.part((size_t)n_events * sizeof(trm_cuda_event)),
                 o_off = pk.part((size_t)n * sizeof(long long)), o_cnt = pk.part((size_t)n * sizeof(int)),
                 o_fg = pk.part(n_fg * sizeof(trm_cuda_framegen)), o_seed = pk.part((size_t)n * sizeof(float)),
                 o_frames = pk.part((size_t)frames_hi * 128);
    int rc;
    if ((rc = ctx->gen.reserve(pk.bytes + 256)) != 0) return rc;
    trm::FrameGenArgs a{};
    unsigned char *d = ctx->gen.base;
    auto *d_desc = (trm_cuda_utterance *)(d + o_desc);
    auto *d_ev = (trm_cuda_event *)(d + o_ev);
    auto *d_off = (long long *)(d + o_off);
    auto *d_cnt = (int *)(d + o_cnt);
    auto *d_fg = (trm_cuda_framegen *)(d + o_fg);
    auto *d_seed = (float *)(d + o_seed);
    auto *d_frames = (double *)(d + o_frames);
    cudaStream_t s = ctx->s_out;
    CK(cudaMemcpyAsync(d_desc, desc, (size_t)n * sizeof(trm_cuda_utterance), cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(d_ev, events, (size_t)n_events * sizeof(trm_cuda_event), cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(d_off, off.data(), (size_t)n * sizeof(long long), cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(d_cnt, ev_count, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(d_fg, fg, n_fg * sizeof(trm_cuda_framegen), cudaMemcpyHostToDevice, s));
    a.desc = d_desc; a.n_utt = n; a.events = d_ev; a.ev_offset = d_off; a.ev_count = d_cnt; a.fg = d_fg; a.shared_fg = shared_fg;
    a.frames = d_frames; a.seed_out = d_seed;
    if ((rc = trm_k_framegen(&a, s)) != 0) return fail("frame generator launch", (cudaError_t)rc);
    if (frames_host) CK(cudaMemcpyAsync(frames_host, d_frames, (size_t)frames_hi * 128, cudaMemcpyDeviceToHost, s));
    if (seed_host) CK(cudaMemcpyAsync(seed_host, d_seed, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    if (frames_dev) *frames_dev = d_frames;
    return 0;
}

/* ------------------------------------------------------------------------------------------------------------
 * stream pool: slots at independent positions, each with its own voice (TRMStream is its lockstep use: n slots of one
 * voice, advanced by the same frames, flushed together)
 * ---------------------------------------------------------------------------------------------------------- */
static long long src_safe_outputs(long long n_in, unsigned tri)
{
    // outputs whose right filter wing lies inside the first n_in input samples: P(n) = (n*tri)>>16 <= n_in-1
    if (n_in <= 0) return 0;
    return (long long)(((unsigned long long)n_in * 65536ull + tri - 1) / tri);
}

struct trm_cuda_pool {
    struct Slot {
        bool open = false;
        bool fresh = false;             // opened since its last waveguide launch: the carried state starts from zero there
        trm_cuda_utterance voice{};     // descriptor template (voice = the slot's wavetable row)
        int cur = 0;                    // history buffer that holds the slot's tube-rate samples
        long long frames_seen = 0;      // control frames pushed so far
        long long s_done = 0;           // tube-rate samples produced so far (multiple of 16 until the flush)
        long long out_done = 0;         // output-rate samples returned so far
        long long in_start = 0;         // first tube-rate sample still in the history buffer (multiple of 4)
        std::vector<double> pending;    // [pend_frames][16]: frames from the control interval in progress on
        long long pend_first = 0;
        int pend_frames = 0;
        // event-fed slots (trm_cuda_pool_open_events): frames are generated on the device, and the pending ones live in
        // row pcur of the slot's two pending-frame rows instead of `pending`
        bool events = false;
        long long ev_count = 0, ev_frames = 0;   // events of the list, frames it expands to
        trm_cuda_framegen fg{};                  // its settings (the device copy is in d_gen[slot].fg)
        int pcur = 0;
    };
    trm_cuda_ctx *ctx = nullptr;
    int precision = 0, cap = 0, max_m = 0;
    size_t esz = 8;
    std::vector<Slot> slots;
    long long stride = 0;               // history elements per slot and buffer
    long long cap_out = 0;              // output samples one slot can return from one push
    unsigned char *d_tube = nullptr;    // [2][cap][stride] tube-rate history, two buffers per slot
    unsigned char *d_out = nullptr;     // [cap * cap_out] outputs of a push, packed entry after entry
    int16_t *d_pcm = nullptr;           // [pcm_cap] PCM16 of a push, packed entry after entry (allocated by the first PCM push)
    long long pcm_cap = 0;
    unsigned char *d_state = nullptr;   // [cap] carried waveguide states
    trm_cuda_utterance *d_desc = nullptr;   // [cap] waveguide descriptors, indexed by slot like the states
    double *d_wavetables = nullptr;     // [cap][512]: row s is slot s's glottal table
    // event-fed slots, allocated by the first trm_cuda_pool_open_events
    std::vector<trm_cuda_event *> d_events;   // [cap] slot s's event list (grow-only, reused by later opens)
    std::vector<long long> events_cap;
    trm::FrameGenPoolState *d_gen = nullptr;  // [cap] generator states
    double *d_pend = nullptr;           // [2][cap][pend_rows][16] pending frames, two rows per slot
    int pend_rows = 0;
    Arena scratch;                      // per-push tables and frames (one upload)
    HostStage stage;
    cudaStream_t st = nullptr;
    long long tube_at(int slot, int buf) const { return ((long long)buf * cap + slot) * stride; }
    unsigned long long tube_addr(long long elem) const { return (unsigned long long)(uintptr_t)(d_tube + (size_t)elem * esz); }
    // device address of pending frame k of row `buf` of a slot
    unsigned long long pend_addr(int slot, int buf, long long k) const
    {
        return (unsigned long long)(uintptr_t)(d_pend + (((size_t)buf * cap + slot) * pend_rows + (size_t)k) * 16);
    }
};

static int pool_err(int code, const char *what)
{
    g_err = what;
    return code;
}

// one entry of a call that names slots: slot s exists, is open and was not named by an earlier entry (named[], one flag
// per slot, records it); `who` names the call in the messages
static int pool_check_slot(const trm_cuda_pool *p, int s, std::vector<unsigned char> &named, const char *who)
{
    if (s < 0 || s >= p->cap) return pool_err(-4, (std::string(who) + ": no such slot").c_str());
    if (!p->slots[s].open) return pool_err(-7, (std::string(who) + ": the slot is not open").c_str());
    if (named[s]) return pool_err(-4, (std::string(who) + ": a slot is named twice").c_str());
    named[s] = 1;
    return 0;
}

int trm_cuda_pool_create(trm_cuda_ctx *ctx, int precision, int capacity, int max_frames_per_push, trm_cuda_pool **out)
{
    *out = nullptr;
    if (capacity <= 0 || max_frames_per_push <= 0 || precision < 0 || precision > 2) return pool_err(-4, "trm_cuda_pool_create: bad sizes");
    CK(cudaSetDevice(ctx->device));
    trm_cuda_pool *p = new trm_cuda_pool();
    p->ctx = ctx; p->precision = precision; p->cap = capacity; p->max_m = max_frames_per_push;
    p->esz = prec_esz(precision);
    p->slots.resize(capacity);
    p->d_events.assign(capacity, nullptr);
    p->events_cap.assign(capacity, 0);
    cudaError_t e = cudaMalloc((void **)&p->d_state, (size_t)capacity * trm::tube_state_bytes(p->esz));
    if (e == cudaSuccess) e = cudaMalloc((void **)&p->d_desc, (size_t)capacity * sizeof(trm_cuda_utterance));
    if (e == cudaSuccess) e = cudaMalloc((void **)&p->d_wavetables, (size_t)capacity * TRM_TABLE_LENGTH * sizeof(double));
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&p->st, cudaStreamNonBlocking);
    if (e != cudaSuccess) { trm_cuda_pool_destroy(p); return fail("trm_cuda_pool_create", e); }
    *out = p;
    return 0;
}

// what one slot of this voice needs: history elements per slot and buffer, samples per push
static void pool_sizes(const trm_cuda_pool *p, const trm_cuda_utterance *v, long long *stride, long long *cap_out)
{
    const long long max_new = (long long)(p->max_m + 1) * v->controlPeriod + 32;
    *stride = (long long)align_up((size_t)(max_new + 128), 32);
    *cap_out = (long long)align_up((size_t)(src_safe_outputs(max_new + 64, v->tri) + 64), 32);
}

// first tube-rate sample the converter still needs once out_total outputs exist (multiple of 4, >= 0)
static long long pool_keep_from(long long out_total, unsigned tri, int pad)
{
    long long next_in = (long long)(((unsigned long long)out_total * tri) >> 16) - 2 * pad - 4;
    if (next_in < 0) next_in = 0;
    return next_in / 4 * 4;
}

// What a push that takes slot sl on to frames_seen frames, flushing it or not, makes of it: the tube-rate samples it has
// then (target), the outputs it has returned (out_total), the first tube-rate sample the converter still needs (next_in),
// and whether that push stays inside one history row of `stride` elements and `cap_out` outputs of one push.
struct PoolAdvance {
    long long target = 0, out_total = 0, next_in = 0;
    bool fits = false;
};

static PoolAdvance pool_advance(const trm_cuda_pool::Slot &sl, long long frames_seen, bool flush, long long stride, long long cap_out)
{
    const unsigned tri = sl.voice.tri;
    const int pad = sl.voice.padSize;
    const long long avail = frames_seen >= 2 ? (frames_seen - 1) * sl.voice.controlPeriod : 0;
    PoolAdvance a;
    a.target = flush ? avail : avail / trm::TB * trm::TB;
    a.out_total = flush ? (long long)(((unsigned long long)(a.target + 2 * pad) * 65536ull + tri - 1) / tri) : src_safe_outputs(a.target, tri);
    a.next_in = std::max(flush ? a.target / 4 * 4 : pool_keep_from(a.out_total, tri, pad), sl.in_start);
    a.fits = a.target - sl.in_start <= stride && a.out_total - sl.out_done <= cap_out;
    return a;
}

int trm_cuda_pool_reserve(trm_cuda_pool *p, const trm_cuda_utterance *v)
{
    if (v->controlPeriod <= 0 || v->tri == 0) return pool_err(-4, "trm_cuda_pool: voice without rates");
    long long stride, cap_out;
    pool_sizes(p, v, &stride, &cap_out);
    CK(cudaSetDevice(p->ctx->device));
    if (stride > p->stride) {
        unsigned char *t = nullptr;
        CK(cudaMalloc((void **)&t, (size_t)2 * p->cap * stride * p->esz));
        if (p->d_tube) {
            // the open slots' histories move to the wider rows (row r = buffer * cap + slot in both layouts)
            cudaError_t e = cudaMemcpy2D(t, (size_t)stride * p->esz, p->d_tube, (size_t)p->stride * p->esz, (size_t)p->stride * p->esz,
                                         (size_t)2 * p->cap, cudaMemcpyDeviceToDevice);
            if (e != cudaSuccess) { cudaFree(t); return fail("trm_cuda_pool_reserve", e); }
            cudaFree(p->d_tube);
        }
        p->d_tube = t;
        p->stride = stride;
    }
    if (cap_out > p->cap_out) {
        if (p->d_out) cudaFree(p->d_out);
        p->d_out = nullptr;
        p->cap_out = 0;
        CK(cudaMalloc((void **)&p->d_out, (size_t)p->cap * cap_out * p->esz));
        p->cap_out = cap_out;
    }
    return 0;
}

// the first slot from `from` on that is not open (p->cap if there is none)
static int pool_free_slot(const trm_cuda_pool *p, int from)
{
    while (from < p->cap && p->slots[from].open) ++from;
    return from;
}

// slot s opened with this voice (its wavetable row is row s), fresh or not; event-fed when ev says so
static trm_cuda_pool::Slot pool_slot(int s, const trm_cuda_utterance &voice, bool fresh, const trm_cuda_pool_event_state *ev)
{
    trm_cuda_pool::Slot sl;
    sl.open = true;
    sl.fresh = fresh;
    sl.voice = voice;
    sl.voice.voice = s;
    if (ev && ev->events) {
        sl.events = true;
        sl.ev_count = ev->n_events;
        sl.ev_frames = ev->ev_frames;
        sl.fg = ev->fg;
        sl.fg.reserved = 0;             // a snapshot stores 0 there, whatever the caller left in it
    }
    return sl;
}

// a free slot for this voice, with the pool's rows reserved for the voice and the slot's wavetable row written; it opens
// when the caller sets its Slot
static int pool_claim(trm_cuda_pool *p, const trm_cuda_utterance *voice, const double *wavetable, const char *full, int *slot)
{
    const int s = pool_free_slot(p, 0);
    if (s == p->cap) return pool_err(-7, full);
    int rc = trm_cuda_pool_reserve(p, voice);
    if (rc != 0) return rc;
    CK(cudaMemcpy(p->d_wavetables + (size_t)s * TRM_TABLE_LENGTH, wavetable, TRM_TABLE_LENGTH * sizeof(double), cudaMemcpyHostToDevice));
    *slot = s;
    return 0;
}

int trm_cuda_pool_open(trm_cuda_pool *p, const trm_cuda_utterance *voice, const double *wavetable, int *slot)
{
    *slot = -1;
    int s;
    const int rc = pool_claim(p, voice, wavetable, "trm_cuda_pool_open: every slot is open", &s);
    if (rc != 0) return rc;
    p->slots[s] = pool_slot(s, *voice, true, nullptr);
    *slot = s;
    return 0;
}

// Between pushes a slot keeps the frames from the control interval its waveguide position s_done lies in: s_done is the
// last whole 16-sample block before the last frame, so at most 1 + ceil(15 / controlPeriod) <= TB frames.  A push
// appends at most max_m more.
static int pool_pend_rows(const trm_cuda_pool *p) { return p->max_m + trm::TB; }

// the event-fed slots' generator states and pending-frame rows, allocated for every slot by the first event-fed open or
// restore
static int pool_event_storage(trm_cuda_pool *p)
{
    if (p->d_gen) return 0;
    const int rows = pool_pend_rows(p);
    trm::FrameGenPoolState *gen = nullptr;
    double *pend = nullptr;
    CK(cudaSetDevice(p->ctx->device));
    cudaError_t e = cudaMalloc((void **)&gen, (size_t)p->cap * sizeof(trm::FrameGenPoolState));
    if (e == cudaSuccess) e = cudaMalloc((void **)&pend, (size_t)2 * p->cap * rows * 128);
    if (e != cudaSuccess) {
        if (gen) cudaFree(gen);
        return fail("pool event storage", e);
    }
    p->d_gen = gen;
    p->d_pend = pend;
    p->pend_rows = rows;
    return 0;
}

// slot s's event list storage, grown to n_events (grow-only: kept for later event-fed opens of the slot)
static int pool_event_list(trm_cuda_pool *p, int s, int64_t n_events)
{
    if (n_events <= p->events_cap[s]) return 0;
    CK(cudaSetDevice(p->ctx->device));
    if (p->d_events[s]) cudaFree(p->d_events[s]);
    p->d_events[s] = nullptr;
    p->events_cap[s] = 0;
    CK(cudaMalloc((void **)&p->d_events[s], (size_t)n_events * sizeof(trm_cuda_event)));
    p->events_cap[s] = n_events;
    return 0;
}

int trm_cuda_pool_open_events(trm_cuda_pool *p, const trm_cuda_utterance *voice, const double *wavetable,
                              const trm_cuda_event *events, int64_t n_events, int64_t n_frames, const trm_cuda_framegen *fg,
                              int *slot)
{
    *slot = -1;
    int s;
    int rc = pool_claim(p, voice, wavetable, "trm_cuda_pool_open_events: every slot is open", &s);
    if (rc == 0) rc = pool_event_storage(p);
    if (rc == 0) rc = pool_event_list(p, s, n_events);
    if (rc != 0) return rc;
    if (n_events > 0) CK(cudaMemcpy(p->d_events[s], events, (size_t)n_events * sizeof(trm_cuda_event), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(&p->d_gen[s].fg, fg, sizeof(trm_cuda_framegen), cudaMemcpyHostToDevice));
    const trm_cuda_pool_event_state ev{1, 0, n_events, n_frames, *fg};
    p->slots[s] = pool_slot(s, *voice, true, &ev);
    *slot = s;
    return 0;
}

int trm_cuda_pool_close(trm_cuda_pool *p, int slot)
{
    if (slot < 0 || slot >= p->cap) return pool_err(-4, "trm_cuda_pool_close: no such slot");
    if (!p->slots[slot].open) return pool_err(-7, "trm_cuda_pool_close: the slot is not open");
    p->slots[slot] = trm_cuda_pool::Slot();
    return 0;
}

int trm_cuda_pool_set_voice(trm_cuda_pool *p, int n, const int32_t *slot, const trm_cuda_utterance *voice,
                            const double *wavetables, int64_t *tube_sample, int64_t *output_sample)
{
    // ---- everything is checked before the pool changes -----------------------------------------------------------------
    if (n < 0 || n > p->cap) return pool_err(-4, "trm_cuda_pool_set_voice: bad entry count");
    if (n > 0 && (!slot || !voice || !wavetables)) return pool_err(-4, "trm_cuda_pool_set_voice: null argument");
    {
        std::vector<unsigned char> named((size_t)p->cap, 0);
        for (int i = 0; i < n; ++i) {
            const int s = slot[i];
            const int rc = pool_check_slot(p, s, named, "trm_cuda_pool_set_voice");
            if (rc != 0) return rc;
            const trm_cuda_utterance &v = voice[i], &c = p->slots[s].voice;
            if (v.controlPeriod != c.controlPeriod || v.sampleRate != c.sampleRate || v.tri != c.tri || v.padSize != c.padSize ||
                v.channels != c.channels)
                return pool_err(-4, "trm_cuda_pool_set_voice: the new voice's rate constants differ from the slot's");
        }
    }
    if (n == 0) return 0;
    // ---- one upload ([segments][rows]), one scatter to the slots' wavetable rows ----------------------------------------
    const size_t wt = TRM_TABLE_LENGTH * sizeof(double);
    Pack pk;
    const size_t o_seg = pk.part((size_t)n * sizeof(trm::CopySeg)), o_wt = pk.part((size_t)n * wt), bytes = pk.bytes;
    CK(cudaSetDevice(p->ctx->device));
    int rc;
    if ((rc = p->scratch.reserve(bytes + 256)) != 0) return rc;
    if ((rc = p->stage.reserve(bytes + 256)) != 0) return rc;
    unsigned char *h = p->stage.base, *d = p->scratch.base;
    trm::CopySeg *seg = (trm::CopySeg *)(h + o_seg);
    memcpy(h + o_wt, wavetables, (size_t)n * wt);
    for (int i = 0; i < n; ++i)
        seg[i] = {(unsigned long long)(uintptr_t)(d + o_wt + (size_t)i * wt),
                  (unsigned long long)(uintptr_t)(p->d_wavetables + (size_t)slot[i] * TRM_TABLE_LENGTH), wt};
    cudaStream_t cs = p->st;
    CK(cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, cs));
    const trm::SegCopyArgs a{(const trm::CopySeg *)(d + o_seg), n};
    if ((rc = trm_k_segment_copy(&a, cs)) != 0) return fail("voice change scatter launch", (cudaError_t)rc);
    CK(cudaStreamSynchronize(cs));
    // ---- the slots change only now that the rows are in place -----------------------------------------------------------
    for (int i = 0; i < n; ++i) {
        trm_cuda_pool::Slot &sl = p->slots[slot[i]];
        sl.voice = voice[i];
        sl.voice.voice = slot[i];
        if (tube_sample) tube_sample[i] = sl.s_done;
        if (output_sample) output_sample[i] = sl.out_done;
    }
    return 0;
}

int64_t trm_cuda_pool_slot_capacity(const trm_cuda_pool *p) { return p->cap_out; }

void trm_cuda_pool_destroy(trm_cuda_pool *p)
{
    if (!p) return;
    cudaSetDevice(p->ctx->device);
    if (p->st) { cudaStreamSynchronize(p->st); cudaStreamDestroy(p->st); }
    if (p->d_tube) cudaFree(p->d_tube);
    if (p->d_out) cudaFree(p->d_out);
    if (p->d_pcm) cudaFree(p->d_pcm);
    if (p->d_state) cudaFree(p->d_state);
    if (p->d_desc) cudaFree(p->d_desc);
    if (p->d_wavetables) cudaFree(p->d_wavetables);
    for (trm_cuda_event *ev : p->d_events)
        if (ev) cudaFree(ev);
    if (p->d_gen) cudaFree(p->d_gen);
    if (p->d_pend) cudaFree(p->d_pend);
    p->scratch.release();
    p->stage.release();
    delete p;
}

// What a PCM push returns instead of samples (trm_cuda_pool_push_pcm16)
struct PoolPcm {
    const double *peak;     // [n]
    int16_t *out;           // packed PCM16, or NULL
    int64_t *offset;        // [n+1]
    double *max;            // [n], or NULL
};

// One push: samples (pcm == nullptr) into samples_host, or PCM16 as `pcm` says.  out_offset receives the packed sample
// offsets either way; d_out holds the samples packed, or in rows of cap_out when out_stride > 0 (samples only).
static int pool_push(trm_cuda_pool *p, int n, const int32_t *slot, const int32_t *n_frames, const double *frames_host,
                     const uint8_t *flush, void *samples_host, int64_t out_stride, int64_t *out_offset, const PoolPcm *pcm)
{
    // ---- arguments: everything is checked before the pool changes -----------------------------------------------
    if (n < 0 || n > p->cap) return pool_err(-4, "trm_cuda_pool_push: bad entry count");
    if (out_stride < 0 || (out_stride > 0 && out_stride < p->cap_out)) return pool_err(-4, "trm_cuda_pool_push: row stride below the slot capacity");
    if (!out_offset || (n > 0 && (!slot || !n_frames))) return pool_err(-4, "trm_cuda_pool_push: null argument");
    if (pcm && (!pcm->offset || (n > 0 && !pcm->peak))) return pool_err(-4, "trm_cuda_pool_push_pcm16: null argument");
    long long total_in = 0;
    {
        std::vector<unsigned char> named((size_t)p->cap, 0);
        for (int i = 0; i < n; ++i) {
            const int s = slot[i];
            const int rc = pool_check_slot(p, s, named, "trm_cuda_pool_push");
            if (rc != 0) return rc;
            if (n_frames[i] < 0 || n_frames[i] > p->max_m) return pool_err(-4, "trm_cuda_pool_push: more frames than the pool was created for");
            if (pcm && !(std::isfinite(pcm->peak[i]) && pcm->peak[i] > 0.0)) return pool_err(-4, "trm_cuda_pool_push_pcm16: a peak is not finite and > 0");
            const trm_cuda_pool::Slot &sl = p->slots[s];
            if (!sl.events) {
                total_in += n_frames[i];
                continue;
            }
            if (sl.frames_seen + n_frames[i] > sl.ev_frames) return pool_err(-4, "trm_cuda_pool_push: more frames than the slot's event list has left");
            if (sl.pend_frames + n_frames[i] > p->pend_rows) return fail_msg("trm_cuda_pool_push: internal capacity (pending frames)");
        }
    }
    if (total_in > 0 && !frames_host) return pool_err(-4, "trm_cuda_pool_push: null frames");
    out_offset[0] = 0;
    if (pcm) pcm->offset[0] = 0;
    if (n == 0) return 0;
    trm_cuda_ctx *ctx = p->ctx;
    CK(cudaSetDevice(ctx->device));

    // ---- per entry, what the push makes of its slot: the samples its frames make computable, the outputs they make
    // safe, the history still needed.  The slots change only in the bookkeeping, once the device work has succeeded. ----
    struct Entry {
        int slot = 0;
        bool flush = false, run = false;
        long long frames_seen = 0;          // the slot's frames after the push
        int pend_frames = 0;                // its pending frames after the push, the waveguide's frames when it runs
        const double *frames = nullptr;     // frame-fed: the push's new frames, in frames_host
        PoolAdvance a;
        long long n_new = 0;
    };
    std::vector<Entry> E((size_t)n);
    const double *fp = frames_host;
    long long wg_frames = 0, total_out = 0, max_ret = 0;
    for (int i = 0; i < n; ++i) {
        Entry &e = E[i];
        e.slot = slot[i];
        e.flush = flush && flush[i];
        const trm_cuda_pool::Slot &sl = p->slots[e.slot];
        e.frames_seen = sl.frames_seen + n_frames[i];
        e.pend_frames = sl.pend_frames + n_frames[i];
        if (!sl.events) {
            e.frames = fp;
            fp += (size_t)n_frames[i] * 16;
        }
        e.a = pool_advance(sl, e.frames_seen, e.flush, p->stride, p->cap_out);
        e.n_new = e.a.target - sl.s_done;
        e.run = !(e.flush && e.frames_seen < 1) && (e.n_new > 0 || (e.flush && e.a.out_total > sl.out_done));
        long long n_ret = 0;
        if (e.run) {
            if (e.n_new > 0) wg_frames += e.pend_frames;
            n_ret = e.a.out_total - sl.out_done;
            if (!e.a.fits) return fail_msg("trm_cuda_pool_push: internal capacity");
        }
        total_out += n_ret > 0 ? n_ret : 0;
        max_ret = std::max(max_ret, n_ret);
        out_offset[i + 1] = total_out;
        if (pcm) pcm->offset[i + 1] = pcm->offset[i] + (n_ret > 0 ? n_ret * sl.voice.channels : 0);
    }

    // ---- host tables of the push, laid out as in the device scratch: one upload ------------------------------------
    std::vector<int> wg;                                  // entries that run the waveguide, longest first
    std::vector<trm_cuda_utterance> rd;                   // resampler views of the entries that return samples
    std::vector<long long> ib(1, 0);                      // work-item prefix
    std::vector<trm::CopySeg> mv;                         // history moves
    std::vector<int> rd_entry;                            // entry of each resampler view
    std::vector<trm::FrameGenPoolEntry> ge;               // event-fed entries that generate frames
    std::vector<trm::CopySeg> fs;                         // event-fed pending frames kept for the next push (other row)
    size_t n_fb = 0;                                      // event-fed entries whose frames the waveguide reads
    long long fed_frames = 0;                             // frames the waveguide reads from frame-fed entries (uploaded)
    for (int i = 0; i < n; ++i) {
        const Entry &e = E[i];
        const trm_cuda_pool::Slot &sl = p->slots[e.slot];
        if (sl.events && n_frames[i] > 0)   // appended after the slot's pending frames; set-up on its first frames
            ge.push_back({(unsigned long long)(uintptr_t)p->d_events[e.slot], sl.ev_count, p->pend_addr(e.slot, sl.pcur, sl.pend_frames),
                          e.slot, n_frames[i], sl.frames_seen == 0 ? 1 : 0, 0});
        if (!e.run) continue;
        if (e.n_new > 0) {
            wg.push_back(i);
            if (sl.events) ++n_fb;
            else fed_frames += e.pend_frames;
        }
        if (sl.events && !e.flush) {
            // the frames before the interval the next push starts in are dropped (bookkeeping below)
            const int drop = (int)(e.a.target / sl.voice.controlPeriod - sl.pend_first), kept = e.pend_frames - drop;
            if (drop > 0 && kept > 0)
                fs.push_back({p->pend_addr(e.slot, sl.pcur, drop), p->pend_addr(e.slot, sl.pcur ^ 1, 0), (unsigned long long)kept * 128});
        }
        const long long n_ret = e.a.out_total - sl.out_done;
        if (n_ret > 0) {
            trm_cuda_utterance r = sl.voice;              // global sample indices of the stream
            r.n_tube = e.a.target;
            r.tube_offset = p->tube_at(e.slot, sl.cur) - sl.in_start;
            r.n_out = e.a.out_total;
            r.out_start = sl.out_done;
            r.in_start = sl.in_start;
            r.out_offset = out_stride > 0 ? i * p->cap_out : out_offset[i];
            r.pcm_offset = pcm ? pcm->offset[i] : 0;
            rd.push_back(r);
            rd_entry.push_back(i);
            ib.push_back(ib.back() + (n_ret + 31) / 32);
        }
        const long long keep = e.a.target - e.a.next_in;
        if (!e.flush && keep > 0)
            mv.push_back({p->tube_addr(p->tube_at(e.slot, sl.cur) + (e.a.next_in - sl.in_start)), p->tube_addr(p->tube_at(e.slot, sl.cur ^ 1)),
                          (unsigned long long)keep * p->esz});
    }
    std::stable_sort(wg.begin(), wg.end(), [&](int a, int b) { return E[a].n_new > E[b].n_new; });
    const size_t n_rd = rd.size(), n_mv = mv.size();
    const size_t n_pk = pcm ? n_rd : 0;                   // PCM: peak and max |y| of each resampler view
    const size_t n_ge = ge.size(), n_fs = fs.size() + n_fb;
    Pack pk;
    const size_t o_dt = pk.part(wg.size() * sizeof(trm_cuda_utterance)), o_ord = pk.part(wg.size() * sizeof(int)),
                 o_rst = pk.part(wg.size() * sizeof(int)), o_rd = pk.part(n_rd * sizeof(trm_cuda_utterance)),
                 o_ib = pk.part(ib.size() * sizeof(long long)), o_mv = pk.part(n_mv * sizeof(trm::CopySeg)),
                 o_pk = pk.part(n_pk * sizeof(double)), o_mx = pk.part(n_pk * sizeof(unsigned long long)),
                 o_ge = pk.part(n_ge * sizeof(trm::FrameGenPoolEntry)), o_fs = pk.part(n_fs * sizeof(trm::CopySeg));
    // the frame region holds the frame-fed entries' frames (uploaded), then the event-fed ones' (copied on the device)
    const size_t o_fr = pk.part((size_t)wg_frames * 128), bytes = pk.bytes, up = o_fr + (size_t)fed_frames * 128;
    if (pcm && p->pcm_cap < 2 * p->cap * p->cap_out) {   // stereo: two int16 per sample
        if (p->d_pcm) cudaFree(p->d_pcm);
        p->d_pcm = nullptr;
        p->pcm_cap = 0;
        CK(cudaMalloc((void **)&p->d_pcm, (size_t)2 * p->cap * p->cap_out * sizeof(int16_t)));
        p->pcm_cap = 2 * (long long)p->cap * p->cap_out;
    }
    int rc;
    if ((rc = p->scratch.reserve(bytes + 256)) != 0) return rc;
    if ((rc = p->stage.reserve(bytes + 256)) != 0) return rc;
    unsigned char *h = p->stage.base;
    {
        trm_cuda_utterance *dt = (trm_cuda_utterance *)(h + o_dt);
        int *ord = (int *)(h + o_ord), *rst = (int *)(h + o_rst);
        double *fr = (double *)(h + o_fr);
        trm::CopySeg *fb = (trm::CopySeg *)(h + o_fs) + fs.size();
        long long f_at = 0, ev_at = fed_frames;
        for (size_t k = 0; k < wg.size(); ++k) {
            const Entry &e = E[wg[k]];
            const trm_cuda_pool::Slot &sl = p->slots[e.slot];
            trm_cuda_utterance d = sl.voice;
            d.frame_offset = sl.events ? ev_at : f_at;
            d.n_frames = e.pend_frames;
            d.n_tube = e.n_new;
            d.tube_offset = p->tube_at(e.slot, sl.cur) + (sl.s_done - sl.in_start);
            d.jc0 = (int)(sl.s_done % sl.voice.controlPeriod);
            d.out_start = 0; d.in_start = 0;
            dt[k] = d;
            ord[k] = e.slot;
            rst[k] = sl.fresh ? 1 : 0;
            // the waveguide reads every pending frame: the slot's first pending frame is the one its position s_done lies in
            if (sl.events) {
                *fb++ = {p->pend_addr(e.slot, sl.pcur, 0), (unsigned long long)(uintptr_t)(p->scratch.base + o_fr + (size_t)ev_at * 128),
                         (unsigned long long)e.pend_frames * 128};
                ev_at += e.pend_frames;
            } else {
                // the slot's pending frames, then the push's new ones
                if (sl.pend_frames) memcpy(fr + (size_t)f_at * 16, sl.pending.data(), (size_t)sl.pend_frames * 128);
                if (n_frames[wg[k]]) memcpy(fr + (size_t)(f_at + sl.pend_frames) * 16, e.frames, (size_t)n_frames[wg[k]] * 128);
                f_at += e.pend_frames;
            }
        }
        if (n_ge) memcpy(h + o_ge, ge.data(), n_ge * sizeof(trm::FrameGenPoolEntry));
        if (!fs.empty()) memcpy(h + o_fs, fs.data(), fs.size() * sizeof(trm::CopySeg));
        if (n_rd) memcpy(h + o_rd, rd.data(), n_rd * sizeof(trm_cuda_utterance));
        memcpy(h + o_ib, ib.data(), ib.size() * sizeof(long long));
        if (n_mv) memcpy(h + o_mv, mv.data(), n_mv * sizeof(trm::CopySeg));
        for (size_t j = 0; j < n_pk; ++j) ((double *)(h + o_pk))[j] = pcm->peak[rd_entry[j]];
        if (n_pk) memset(h + o_mx, 0, n_pk * sizeof(unsigned long long));
    }
    unsigned char *d = p->scratch.base;
    cudaStream_t st = p->st;
    CK(cudaMemcpyAsync(d, h, up, cudaMemcpyHostToDevice, st));
    if (n_ge > 0) {
        // event-fed slots: new frames appended to the pending row, then that row's frames copied where the waveguide
        // reads them and the kept ones to the slot's other row
        const trm::FrameGenPoolArgs a{(const trm::FrameGenPoolEntry *)(d + o_ge), (int)n_ge, p->d_gen};
        if ((rc = trm_k_framegen_pool(&a, st)) != 0) return fail("pool frame generator launch", (cudaError_t)rc);
    }
    if (n_fs > 0) {
        const trm::SegCopyArgs a{(const trm::CopySeg *)(d + o_fs), (int)n_fs};
        if ((rc = trm_k_segment_copy(&a, st)) != 0) return fail("pool frame move launch", (cudaError_t)rc);
    }
    const KernelSet &K = g_kernels[p->precision];
    const trm::KernelInfo &ki = ctx->ki(p->precision);
    const int n_w = (int)wg.size();
    if (n_w > 0) {
        trm::PoolPrepArgs pa{};
        pa.src = (const trm_cuda_utterance *)(d + o_dt); pa.slot = (const int *)(d + o_ord); pa.reset = (const int *)(d + o_rst);
        pa.dst = p->d_desc; pa.state = p->d_state; pa.state_bytes = trm::tube_state_bytes(p->esz); pa.noise_k0 = ctx->noise_k0; pa.n = n_w;
        if ((rc = trm_k_pool_prepare(&pa, st)) != 0) return fail("pool prepare launch", (cudaError_t)rc);
        // one waveguide launch over the slots with new samples; the kernel maps CTA positions to slots through `order`
        trm::TubeArgs a{};
        a.state = p->d_state; a.desc = p->d_desc; a.order = (const int *)(d + o_ord); a.n_utt = n_w;
        a.frames = d + o_fr; a.frames_f32 = 0; a.tube = p->d_tube; a.wavetables = p->d_wavetables; a.noise_k0 = ctx->noise_k0;
        const int gmax = ki.wide_max_utt;
        const int groups = std::max(1, std::min(ctx->sm_count, (n_w + 1) / 2));
        const int g2 = (n_w + groups - 1) / groups > gmax ? (n_w + gmax - 1) / gmax : groups;
        if ((rc = K.tube_wide_pool(&a, g2, st)) != 0) return fail("pool waveguide launch", (cudaError_t)rc);
    }
    if (n_rd > 0) {
        trm::SrcPoolArgs a{};
        a.desc = (const trm_cuda_utterance *)(d + o_rd); a.n = (int)n_rd; a.item_base = (const long long *)(d + o_ib);
        a.total_items = ib.back(); a.tube = p->d_tube; a.out = p->d_out;
        a.table = prec_is_f64(p->precision) ? ctx->d_tab_f64 : ctx->d_tab_f32;
        a.ctab = prec_is_f64(p->precision) ? ctx->d_ctab_f64 : ctx->d_ctab_f32;
        if ((rc = K.src_pool(&a, ctx->sm_count * 8, st)) != 0) return fail("pool resampler launch", (cudaError_t)rc);
    }
    if (n_pk > 0) {
        trm::PcmPoolArgs a{};
        a.desc = (const trm_cuda_utterance *)(d + o_rd); a.n = (int)n_rd; a.item_base = (const long long *)(d + o_ib);
        a.total_items = ib.back(); a.out = p->d_out; a.peak = (const double *)(d + o_pk); a.pcm = p->d_pcm;
        a.maxbits = (unsigned long long *)(d + o_mx);
        if ((rc = K.pcm_pool(&a, ctx->sm_count * 8, st)) != 0) return fail("pool PCM launch", (cudaError_t)rc);
    }
    if (n_mv > 0) {
        const trm::SegCopyArgs a{(const trm::CopySeg *)(d + o_mv), (int)n_mv};
        if ((rc = trm_k_segment_copy(&a, st)) != 0) return fail("pool history move launch", (cudaError_t)rc);
    }
    if (pcm) {
        if (pcm->out && pcm->offset[n] > 0)
            CK(cudaMemcpyAsync(pcm->out, p->d_pcm, (size_t)pcm->offset[n] * sizeof(int16_t), cudaMemcpyDeviceToHost, st));
        // the maxima come back into the staging buffer (its upload precedes this copy on the stream)
        if (pcm->max && n_pk) CK(cudaMemcpyAsync(h + o_mx, d + o_mx, n_pk * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    } else if (samples_host && total_out > 0) {
        if (out_stride > 0)
            CK(cudaMemcpy2DAsync(samples_host, (size_t)out_stride * p->esz, p->d_out, (size_t)p->cap_out * p->esz,
                                 (size_t)max_ret * p->esz, (size_t)n, cudaMemcpyDeviceToHost, st));
        else
            CK(cudaMemcpyAsync(samples_host, p->d_out, (size_t)total_out * p->esz, cudaMemcpyDeviceToHost, st));
    }
    CK(cudaStreamSynchronize(st));
    if (pcm && pcm->max) {
        for (int i = 0; i < n; ++i) pcm->max[i] = 0.0;
        for (size_t j = 0; j < n_pk; ++j) memcpy(&pcm->max[rd_entry[j]], h + o_mx + j * sizeof(unsigned long long), sizeof(double));
    }

    // ---- bookkeeping: the only place a push changes its slots ------------------------------------------------------
    for (int i = 0; i < n; ++i) {
        const Entry &e = E[i];
        trm_cuda_pool::Slot &sl = p->slots[e.slot];
        if (e.flush) { sl = trm_cuda_pool::Slot(); continue; }     // ended: the slot is free again
        sl.frames_seen = e.frames_seen;
        sl.pend_frames = e.pend_frames;
        int drop = 0;
        if (e.run) {
            if (e.n_new > 0) sl.fresh = false;
            sl.in_start = e.a.next_in;
            sl.s_done = e.a.target;
            sl.out_done = e.a.out_total;
            sl.cur ^= 1;
            // frames before the interval the next push starts in are done with
            drop = (int)(sl.s_done / sl.voice.controlPeriod - sl.pend_first);
        }
        if (!sl.events) {
            sl.pending.insert(sl.pending.end(), e.frames, e.frames + (size_t)n_frames[i] * 16);
            sl.pending.erase(sl.pending.begin(), sl.pending.begin() + (size_t)drop * 16);
        } else if (drop > 0 && sl.pend_frames > drop) {
            sl.pcur ^= 1;                                          // the kept frames were copied to the other row
        }
        sl.pend_frames -= drop;
        sl.pend_first += drop;
    }
    return 0;
}

int trm_cuda_pool_push(trm_cuda_pool *p, int n, const int32_t *slot, const int32_t *n_frames, const double *frames_host,
                       const uint8_t *flush, void *samples_host, int64_t out_stride, int64_t *out_offset)
{
    return pool_push(p, n, slot, n_frames, frames_host, flush, samples_host, out_stride, out_offset, nullptr);
}

int trm_cuda_pool_push_pcm16(trm_cuda_pool *p, int n, const int32_t *slot, const int32_t *n_frames, const double *frames_host,
                             const uint8_t *flush, const double *peak, int16_t *pcm_host, int64_t *pcm_offset, double *max_host)
{
    if (n < 0 || n > p->cap) return pool_err(-4, "trm_cuda_pool_push: bad entry count");
    std::vector<int64_t> out_offset((size_t)n + 1);
    const PoolPcm pcm{peak, pcm_host, pcm_offset, max_host};
    return pool_push(p, n, slot, n_frames, frames_host, flush, nullptr, 0, out_offset.data(), &pcm);
}

// ---- snapshots: the part of a slot that is not its voice ------------------------------------------------------------
int trm_cuda_pool_check_state(const trm_cuda_utterance *v, const trm_cuda_pool_slot_state *c)
{
    const long long cp = v->controlPeriod;
    if (cp <= 0 || v->tri == 0) return pool_err(-4, "trm_cuda_pool: voice without rates");
    // what pool_push keeps true between pushes; every index and length a kernel uses after a restore derives from these.
    // 2^32 frames (200 days at 250 Hz) keep the converter's position arithmetic (samples x 65536) inside 64 bits.
    const long long fs = c->frames_seen;
    if (fs < 0 || fs > (1ll << 32) || c->pend_frames < 0 || c->pend_first < 0 || c->pend_first + c->pend_frames != fs)
        return pool_err(-4, "snapshot: the frame counters do not agree");
    const long long avail = fs >= 2 ? (fs - 1) * cp : 0;
    if (c->s_done < 0 || c->s_done % trm::TB != 0 || c->s_done > avail || c->pend_first != c->s_done / cp)
        return pool_err(-4, "snapshot: the waveguide position does not agree with the frames");
    if (c->fresh != (c->s_done == 0 ? 1 : 0))   // the waveguide has run exactly when it has produced samples
        return pool_err(-4, "snapshot: the fresh flag does not agree with the waveguide position");
    if (c->out_done < 0 || c->out_done > src_safe_outputs(c->s_done, v->tri))
        return pool_err(-4, "snapshot: more outputs returned than the waveguide position allows");
    if (c->in_start < 0 || c->in_start % 4 != 0 || c->in_start > c->s_done || c->in_start > pool_keep_from(c->out_done, v->tri, v->padSize))
        return pool_err(-4, "snapshot: the kept history does not cover what the converter reads next");
    return 0;
}

int64_t trm_cuda_pool_slot_bytes(int precision, const trm_cuda_pool_slot_state *c)
{
    const size_t esz = prec_esz(precision);
    return (int64_t)c->pend_frames * 128 + (c->fresh ? 0 : (int64_t)trm::tube_state_bytes(esz)) +
           (int64_t)(c->s_done - c->in_start) * (int64_t)esz;
}

// the generator part of the device state is the FrameGen fields, in the snapshot's order, ahead of the settings
static_assert(offsetof(trm::FrameGenPoolState, fg) == TRM_FRAMEGEN_STATE_BYTES, "generator state layout");
static_assert(sizeof(trm_cuda_event) == 296, "event layout");

static size_t pool_gen_bytes(const trm_cuda_pool_slot_state &c) { return c.frames_seen > 0 ? TRM_FRAMEGEN_STATE_BYTES : 0; }

int64_t trm_cuda_pool_event_bytes(const trm_cuda_pool_slot_state *st, const trm_cuda_pool_event_state *ev)
{
    return ev->events ? (int64_t)pool_gen_bytes(*st) + ev->n_events * (int64_t)sizeof(trm_cuda_event) : 0;
}

// A slot's parts on the device, in the order of its part of the snapshot staging (packed slot after slot from 16-byte
// boundaries): pending frames (event-fed slots: they are on the device), carried state (unless fresh), kept history,
// event list, generator state.  The list precedes the generator so that both the list and everything before it start
// on 16 bytes; the data part orders them the other way.
struct SnapStage {
    enum { PEND, STATE, HIST, LIST, GEN, N_PARTS };
    unsigned long long at[N_PARTS] = {};    // device address
    size_t size[N_PARTS] = {};              // bytes, 0 for a part the slot does not have
    size_t head() const { return size[PEND] + size[STATE] + size[HIST]; }     // the bytes before the list
    size_t bytes() const { return align_up(head() + size[LIST] + size[GEN], 16); }
};

// the parts of slot s, whose history is in buffer sl.cur and pending frames in row sl.pcur, with gen_bytes of its
// generator state
static SnapStage snap_stage(const trm_cuda_pool *p, int s, const trm_cuda_pool::Slot &sl, size_t gen_bytes)
{
    SnapStage g;
    auto part = [&](int k, unsigned long long at, size_t size) { g.at[k] = at; g.size[k] = size; };
    const size_t sb = trm::tube_state_bytes(p->esz);
    if (sl.events) part(SnapStage::PEND, p->pend_addr(s, sl.pcur, 0), (size_t)sl.pend_frames * 128);
    if (!sl.fresh) part(SnapStage::STATE, (unsigned long long)(uintptr_t)(p->d_state + (size_t)s * sb), sb);
    part(SnapStage::HIST, p->tube_addr(p->tube_at(s, sl.cur)), (size_t)(sl.s_done - sl.in_start) * p->esz);
    if (sl.events) {
        part(SnapStage::LIST, (unsigned long long)(uintptr_t)p->d_events[s], (size_t)sl.ev_count * sizeof(trm_cuda_event));
        part(SnapStage::GEN, (unsigned long long)(uintptr_t)(p->d_gen + s), gen_bytes);
    }
    return g;
}

int trm_cuda_pool_save(trm_cuda_pool *p, int n, const int32_t *slot, trm_cuda_pool_slot_state *st,
                       trm_cuda_pool_event_state *ev, void *const *dst)
{
    if (n < 0 || n > p->cap || (n > 0 && (!slot || !st))) return pool_err(-4, "trm_cuda_pool_save: bad arguments");
    {
        std::vector<unsigned char> named((size_t)p->cap, 0);
        for (int i = 0; i < n; ++i) {
            const int s = slot[i];
            const int rc = pool_check_slot(p, s, named, "trm_cuda_pool_save");
            if (rc != 0) return rc;
            if (p->slots[s].events && !ev) return pool_err(-7, "trm_cuda_pool_save: a slot fed from an event list has no version 1 snapshot");
        }
    }
    for (int i = 0; i < n; ++i) {
        const trm_cuda_pool::Slot &sl = p->slots[slot[i]];
        st[i] = trm_cuda_pool_slot_state{sl.frames_seen, sl.s_done, sl.out_done, sl.in_start, sl.pend_first, sl.pend_frames,
                                         sl.fresh ? 1 : 0};
        if (ev) {
            ev[i] = trm_cuda_pool_event_state{};
            if (sl.events) {
                ev[i].events = 1;
                ev[i].n_events = sl.ev_count;
                ev[i].ev_frames = sl.ev_frames;
                ev[i].fg = sl.fg;
            }
        }
    }
    if (!dst || n == 0) return 0;

    // gather every slot's device part into packed staging ([segments][slot 0][slot 1] ..., SnapStage), one copy back
    std::vector<SnapStage> sg((size_t)n);
    std::vector<size_t> at((size_t)n + 1, 0);
    for (int i = 0; i < n; ++i) {
        sg[i] = snap_stage(p, slot[i], p->slots[slot[i]], pool_gen_bytes(st[i]));
        at[i + 1] = at[i] + sg[i].bytes();
    }
    Pack pk;
    const size_t o_seg = pk.part((size_t)SnapStage::N_PARTS * n * sizeof(trm::CopySeg)), o_stg = pk.part(at[n]), bytes = pk.bytes;
    int rc;
    CK(cudaSetDevice(p->ctx->device));
    if ((rc = p->scratch.reserve(bytes + 256)) != 0) return rc;
    if ((rc = p->stage.reserve(bytes + 256)) != 0) return rc;
    unsigned char *h = p->stage.base, *d = p->scratch.base;
    trm::CopySeg *seg = (trm::CopySeg *)(h + o_seg);
    int n_seg = 0;
    for (int i = 0; i < n; ++i) {
        unsigned long long to = (unsigned long long)(uintptr_t)(d + o_stg + at[i]);
        for (int k = 0; k < SnapStage::N_PARTS; ++k)
            if (sg[i].size[k]) {
                seg[n_seg++] = {sg[i].at[k], to, sg[i].size[k]};
                to += sg[i].size[k];
            }
    }
    if (n_seg > 0) {
        cudaStream_t cs = p->st;
        CK(cudaMemcpyAsync(d + o_seg, h + o_seg, (size_t)n_seg * sizeof(trm::CopySeg), cudaMemcpyHostToDevice, cs));
        const trm::SegCopyArgs a{(const trm::CopySeg *)(d + o_seg), n_seg};
        if ((rc = trm_k_segment_copy(&a, cs)) != 0) return fail("snapshot gather launch", (cudaError_t)rc);
        CK(cudaMemcpyAsync(h + o_stg, d + o_stg, at[n], cudaMemcpyDeviceToHost, cs));
        CK(cudaStreamSynchronize(cs));
    }
    // data part: [pending frames][state][history] then, event-fed, [generator][list]
    for (int i = 0; i < n; ++i) {
        const trm_cuda_pool::Slot &sl = p->slots[slot[i]];
        const SnapStage &g = sg[i];
        const size_t list = g.size[SnapStage::LIST], gen = g.size[SnapStage::GEN];
        const unsigned char *from = h + o_stg + at[i];
        unsigned char *o = (unsigned char *)dst[i];
        const size_t host_pend = sl.events ? 0 : (size_t)sl.pend_frames * 128;
        if (host_pend) memcpy(o, sl.pending.data(), host_pend);
        o += host_pend;
        memcpy(o, from, g.head());
        o += g.head();
        if (gen) memcpy(o, from + g.head() + list, gen);
        if (list) memcpy(o + gen, from + g.head(), list);
    }
    return 0;
}

int trm_cuda_pool_restore(trm_cuda_pool *p, int n, const trm_cuda_utterance *voice, const double *wavetables,
                          const trm_cuda_pool_slot_state *st, const trm_cuda_pool_event_state *ev, const void *const *src,
                          int32_t *slot_out)
{
    if (n < 0 || (n > 0 && (!voice || !wavetables || !st || !src || !slot_out)))
        return pool_err(-4, "trm_cuda_pool_restore: bad arguments");
    if (n == 0) return 0;
    // ---- everything is checked before the pool changes ----------------------------------------------------------------
    long long stride = p->stride, cap_out = p->cap_out;     // the sizes after this call's reservations
    bool any_events = false;
    for (int i = 0; i < n; ++i) {
        int rc = trm_cuda_pool_check_state(&voice[i], &st[i]);
        if (rc != 0) return rc;
        long long s, c;
        pool_sizes(p, &voice[i], &s, &c);
        stride = std::max(stride, s);
        cap_out = std::max(cap_out, c);
        if (ev && ev[i].events) {
            if (ev[i].n_events < 0 || st[i].frames_seen > ev[i].ev_frames)
                return pool_err(-4, "trm_cuda_pool_restore: the event part does not agree with the counters");
            // so that pool_push's pending-row capacity check never refuses the restored slot's next push
            if (st[i].pend_frames + p->max_m > pool_pend_rows(p))
                return pool_err(-4, "trm_cuda_pool_restore: a snapshot's pending frames and this pool's next push do not fit its pending-frame rows");
            any_events = true;
        }
    }
    // the slots as they open, in the first n free slots (slot p->cap once there are none left).  The next push of each,
    // with as many frames as this pool takes, flushing or not, must stay inside one history row and one slot's outputs,
    // so that pool_push's capacity check never refuses it.
    std::vector<int> free_slot((size_t)n);
    std::vector<trm_cuda_pool::Slot> made((size_t)n);
    for (int i = 0, s = -1; i < n; ++i) {
        s = free_slot[i] = pool_free_slot(p, std::min(s + 1, p->cap));
        trm_cuda_pool::Slot &sl = made[i] = pool_slot(s, voice[i], st[i].fresh != 0, ev ? &ev[i] : nullptr);
        sl.frames_seen = st[i].frames_seen;
        sl.s_done = st[i].s_done;
        sl.out_done = st[i].out_done;
        sl.in_start = st[i].in_start;
        sl.pend_first = st[i].pend_first;
        sl.pend_frames = st[i].pend_frames;
        for (const bool fl : {false, true})
            if (!pool_advance(sl, sl.frames_seen + p->max_m, fl, stride, cap_out).fits)
                return pool_err(-4, "trm_cuda_pool_restore: a snapshot's history and pending frames do not fit this pool's next push");
    }
    if (free_slot[n - 1] == p->cap) return pool_err(-7, "trm_cuda_pool_restore: fewer free slots than snapshots");

    int rc;
    for (int i = 0; i < n; ++i)
        if ((rc = trm_cuda_pool_reserve(p, &voice[i])) != 0) return rc;
    if (any_events) {
        if ((rc = pool_event_storage(p)) != 0) return rc;
        for (int i = 0; i < n; ++i)
            if (ev[i].events && (rc = pool_event_list(p, free_slot[i], ev[i].n_events)) != 0) return rc;
    }
    // ---- one upload ([segments][wavetables][entry 0's SnapStage, generator with settings] ...), one scatter -----------
    const size_t wt = TRM_TABLE_LENGTH * sizeof(double);
    const size_t gs = sizeof(trm::FrameGenPoolState);   // event-fed: the whole generator state, settings included
    std::vector<SnapStage> sg((size_t)n);
    std::vector<size_t> at((size_t)n + 1, 0);
    for (int i = 0; i < n; ++i) {
        sg[i] = snap_stage(p, free_slot[i], made[i], gs);
        at[i + 1] = at[i] + sg[i].bytes();
    }
    Pack pk;
    const size_t o_seg = pk.part((size_t)(1 + SnapStage::N_PARTS) * n * sizeof(trm::CopySeg)), o_wt = pk.part((size_t)n * wt),
                 o_dev = pk.part(at[n]), bytes = pk.bytes;
    CK(cudaSetDevice(p->ctx->device));
    if ((rc = p->scratch.reserve(bytes + 256)) != 0) return rc;
    if ((rc = p->stage.reserve(bytes + 256)) != 0) return rc;
    unsigned char *h = p->stage.base, *d = p->scratch.base;
    trm::CopySeg *seg = (trm::CopySeg *)(h + o_seg);
    int n_seg = 0;
    memcpy(h + o_wt, wavetables, (size_t)n * wt);
    for (int i = 0; i < n; ++i) {
        const SnapStage &g = sg[i];
        seg[n_seg++] = {(unsigned long long)(uintptr_t)(d + o_wt + (size_t)i * wt),
                        (unsigned long long)(uintptr_t)(p->d_wavetables + (size_t)free_slot[i] * TRM_TABLE_LENGTH), wt};
        unsigned long long from = (unsigned long long)(uintptr_t)(d + o_dev + at[i]);
        for (int k = 0; k < SnapStage::N_PARTS; ++k)
            if (g.size[k]) {
                seg[n_seg++] = {from, g.at[k], g.size[k]};
                from += g.size[k];
            }
        // the data part: [pending frames (frame-fed: they stay on the host)][state][history] then, event-fed, [generator
        // (frames_seen > 0)][list]
        const unsigned char *in = (const unsigned char *)src[i] + (made[i].events ? 0 : (size_t)st[i].pend_frames * 128);
        unsigned char *stg = h + o_dev + at[i];
        memcpy(stg, in, g.head());
        if (!made[i].events) continue;
        const size_t gen_in = pool_gen_bytes(st[i]), list = g.size[SnapStage::LIST];
        memcpy(stg + g.head(), in + g.head() + gen_in, list);
        // a slot with no frames yet sets its generator up on its first push: only the settings matter
        trm::FrameGenPoolState gen{};
        if (gen_in) memcpy(&gen, in + g.head(), gen_in);
        gen.fg = ev[i].fg;
        memcpy(stg + g.head() + list, &gen, gs);
    }
    cudaStream_t cs = p->st;
    CK(cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, cs));
    const trm::SegCopyArgs a{(const trm::CopySeg *)(d + o_seg), n_seg};
    if ((rc = trm_k_segment_copy(&a, cs)) != 0) return fail("snapshot scatter launch", (cudaError_t)rc);
    CK(cudaStreamSynchronize(cs));
    // ---- the slots open only now that the device work has finished without error -------------------------------------
    for (int i = 0; i < n; ++i) {
        trm_cuda_pool::Slot &sl = made[i];
        if (!sl.events) sl.pending.assign((const double *)src[i], (const double *)src[i] + (size_t)st[i].pend_frames * 16);
        p->slots[free_slot[i]] = std::move(sl);
        slot_out[i] = free_slot[i];
    }
    return 0;
}

int trm_cuda_resident_create(trm_cuda_ctx *ctx, int precision, int n, const trm_cuda_utterance *desc,
                             const double *frames_host, trm_cuda_resident **out)
{
    *out = nullptr;
    CK(cudaSetDevice(ctx->device));
    if (precision < 0 || precision > 2) return fail_msg("unknown precision code");
    const size_t esz = prec_esz(precision);
    trm_cuda_resident *r = new trm_cuda_resident();
    r->ctx = ctx;
    r->precision = precision;
    int rc;
    if ((rc = plan_chunk(desc, 0, n, ctx->ki(precision), r->plan)) != 0) { delete r; return rc; }
    chunk_layout(r->plan, esz, true);
    if ((rc = r->arena.reserve(r->plan.arena)) != 0) { delete r; return rc; }
    if ((rc = upload_plan(r->plan, r->arena.base, nullptr, 0)) != 0 || (rc = upload_frames(r->plan, r->arena.base, desc, frames_host, 0)) != 0) {
        r->arena.release();
        delete r;
        return rc;
    }
    CK(cudaMemset(r->arena.base + r->plan.at.maxbits, 0, (size_t)n * sizeof(unsigned long long)));
    if (!ctx->wt_host.empty()) {
        if (cudaMalloc((void **)&r->d_wavetables, ctx->wt_host.size() * sizeof(double)) != cudaSuccess ||
            cudaMemcpy(r->d_wavetables, ctx->wt_host.data(), ctx->wt_host.size() * sizeof(double), cudaMemcpyHostToDevice) != cudaSuccess) {
            if (r->d_wavetables) cudaFree(r->d_wavetables);
            r->arena.release();
            delete r;
            return fail("resident wavetables", cudaGetLastError());
        }
    }
    CK(cudaDeviceSynchronize());
    *out = r;
    return 0;
}

void trm_cuda_resident_destroy(trm_cuda_resident *r)
{
    if (!r) return;
    cudaSetDevice(r->ctx->device);
    cudaDeviceSynchronize();
    r->arena.release();
    if (r->d_wavetables) cudaFree(r->d_wavetables);
    delete r;
}

int trm_cuda_resident_stage(trm_cuda_resident *r, int stage, void *stream)
{
    CK(cudaSetDevice(r->ctx->device));
    return launch_stage(r->ctx, r->precision, stage, r->plan, r->arena.base, r->d_wavetables, (cudaStream_t)stream);
}

int trm_cuda_resident_run(trm_cuda_resident *r, void *stream)
{
    for (int st = 0; st < TRM_STAGE_COUNT; ++st) {
        int rc = trm_cuda_resident_stage(r, st, stream);
        if (rc) return rc;
    }
    return 0;
}

int trm_cuda_resident_fetch(trm_cuda_resident *r, int16_t *pcm_host, void *samples_host, double *max_host, void *tube_host)
{
    CK(cudaSetDevice(r->ctx->device));
    CK(cudaDeviceSynchronize());
    const size_t esz = prec_esz(r->precision);
    const ChunkPlan &p = r->plan;
    const unsigned char *base = r->arena.base;
    if (pcm_host && p.pcm_n) CK(cudaMemcpy(pcm_host + p.pcm_lo, base + p.at.pcm, (size_t)p.pcm_n * sizeof(int16_t), cudaMemcpyDeviceToHost));
    if (samples_host && p.out_n)
        CK(cudaMemcpy((unsigned char *)samples_host + (size_t)p.out_lo * esz, base + p.at.out, (size_t)p.out_n * esz, cudaMemcpyDeviceToHost));
    if (tube_host && p.tube_n)
        CK(cudaMemcpy((unsigned char *)tube_host + (size_t)p.tube_lo * esz, base + p.at.tube, (size_t)p.tube_n * esz, cudaMemcpyDeviceToHost));
    if (max_host && !p.desc.empty()) {
        std::vector<unsigned long long> mb(p.desc.size());
        CK(cudaMemcpy(mb.data(), base + p.at.maxbits, mb.size() * sizeof(mb[0]), cudaMemcpyDeviceToHost));
        for (size_t i = 0; i < mb.size(); ++i) memcpy(&max_host[i], &mb[i], sizeof(double));
    }
    return 0;
}

/*
 * Sweep (BASELINE configs[4], SURVEY.md 8(d) config 5): n utterances of one voice and n_frames frames each, whose control
 * tracks are the walk2 workload (include/trm_workload.h) generated ON THE DEVICE -- utterance k uses index first_index + k
 * of stream `seed` -- synthesized chunk by chunk; the audio never leaves the device: 8 bytes of PCM checksum (and the
 * maximum) per utterance come back.  probe_utt[] (sorted, relative to this call) names utterances whose PCM is copied to
 * probe_pcm (n_probe rows of probe_stride int16) for oracle spot checks.  One stream, no copies inside the loop.
 */
int trm_cuda_sweep(trm_cuda_ctx *ctx, int precision, const trm_cuda_utterance *voice, int32_t n_frames, uint64_t seed,
                   uint64_t first_index, int64_t n, uint64_t *checksums_host, double *max_host, int64_t n_probe,
                   const int64_t *probe_utt, int16_t *probe_pcm, int64_t probe_stride, int64_t *launches, double *kernel_ms)
{
    if (launches) *launches = 0;
    if (kernel_ms) *kernel_ms = 0.0;
    if (n <= 0) return 0;
    if (precision < 0 || precision > 2) return fail_msg("unknown precision code");
    CK(cudaSetDevice(ctx->device));
    const size_t esz = prec_esz(precision);
    const trm::KernelInfo &ki = ctx->ki(precision);
    const int64_t cap = (int64_t)ctx->sm_count * ki.wide_max_utt;          // one full wave of the waveguide kernel
    const int C = (int)std::min<int64_t>(n, cap);
    // one chunk plan, reused: C utterances of the template voice, frames back to back
    std::vector<trm_cuda_utterance> desc((size_t)C, *voice);
    long long tube_at = 0, out_at = 0, pcm_at = 0;
    auto up = [](long long v) { return (v + TRM_ALIGN_ELEMS - 1) / TRM_ALIGN_ELEMS * TRM_ALIGN_ELEMS; };
    for (int u = 0; u < C; ++u) {
        trm_cuda_utterance &d = desc[u];
        d.n_frames = n_frames;
        d.frame_offset = (long long)u * n_frames;
        d.tube_offset = tube_at; d.out_offset = out_at; d.pcm_offset = pcm_at;
        tube_at += up(d.n_tube); out_at += up(d.n_out); pcm_at += up(d.n_out * d.channels);
    }
    ChunkPlan plan;
    int rc;
    if ((rc = plan_chunk(desc.data(), 0, C, ki, plan)) != 0) return rc;
    chunk_layout(plan, esz, true);
    Pack pk{plan.arena};
    const size_t o_sums = pk.part((size_t)C * sizeof(unsigned long long));
    Arena &arena = ctx->arenas[0];
    if ((rc = arena.reserve(pk.bytes)) != 0) return rc;
    unsigned char *base = arena.base;
    auto *d_sums = (unsigned long long *)(base + o_sums);
    const auto *d_desc = (const trm_cuda_utterance *)(base + plan.at.desc);
    const int16_t *d_pcm = (const int16_t *)(base + plan.at.pcm);
    cudaStream_t st = ctx->s_out;
    if ((rc = upload_plan(plan, base, nullptr, st)) != 0) return rc;
    std::vector<unsigned long long> mb((size_t)C);
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    int64_t n_launch = 0, probe_at = 0;
    double ms_total = 0.0;
    for (int64_t at = 0; at < n; at += C) {
        const int m = (int)std::min<int64_t>(C, n - at);
        // (a short last chunk runs the full plan: the utterances beyond m keep the previous chunk's frames and are ignored)
        CK(cudaEventRecord(e0, st));
        if (trm_k_workload_walk2(seed, first_index + (uint64_t)at, m, n_frames, (double *)(base + plan.at.frames), st) != 0) return fail_msg("walk2 launch");
        for (int stage = 0; stage < TRM_STAGE_COUNT; ++stage)
            if ((rc = launch_stage(ctx, precision, stage, plan, base, nullptr, st)) != 0) return rc;
        if (trm_k_pcm_checksum(d_desc, m, d_pcm, d_sums, st) != 0) return fail_msg("checksum launch");
        CK(cudaEventRecord(e1, st));
        n_launch += 5;
        CK(cudaMemcpyAsync(checksums_host + at, d_sums, (size_t)m * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(mb.data(), base + plan.at.maxbits, (size_t)m * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        while (probe_at < n_probe && probe_utt[probe_at] < at + m) {
            const int64_t k = probe_utt[probe_at] - at;
            if (k >= 0) {
                const trm_cuda_utterance &d = plan.desc[(size_t)k];
                const int64_t cnt = std::min<int64_t>(d.n_out * d.channels, probe_stride);
                CK(cudaMemcpyAsync(probe_pcm + probe_at * probe_stride, d_pcm + d.pcm_offset, (size_t)cnt * sizeof(int16_t), cudaMemcpyDeviceToHost, st));
            }
            ++probe_at;
        }
        CK(cudaStreamSynchronize(st));
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, e0, e1));
        ms_total += ms;
        if (max_host)
            for (int i = 0; i < m; ++i) memcpy(&max_host[at + i], &mb[(size_t)i], sizeof(double));
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    if (launches) *launches = n_launch;
    if (kernel_ms) *kernel_ms = ms_total;
    return 0;
}

/* Output-rate samples (and PCM) of ONE utterance of a device-resident batch: what bench.py's in-run oracle check reads. */
int trm_cuda_resident_fetch_utterance(trm_cuda_resident *r, int u, void *samples_host, int16_t *pcm_host, double *max_host)
{
    CK(cudaSetDevice(r->ctx->device));
    CK(cudaDeviceSynchronize());
    if (u < 0 || u >= (int)r->plan.desc.size()) return fail_msg("trm_cuda_resident_fetch_utterance: no such utterance");
    const size_t esz = prec_esz(r->precision);
    const trm_cuda_utterance &d = r->plan.desc[u];
    if (samples_host && d.n_out) CK(cudaMemcpy(samples_host, r->arena.base + r->plan.at.out + (size_t)d.out_offset * esz, (size_t)d.n_out * esz, cudaMemcpyDeviceToHost));
    if (pcm_host && d.n_out) CK(cudaMemcpy(pcm_host, (const int16_t *)(r->arena.base + r->plan.at.pcm) + d.pcm_offset, (size_t)d.n_out * d.channels * sizeof(int16_t), cudaMemcpyDeviceToHost));
    if (max_host) {
        unsigned long long mb = 0;
        CK(cudaMemcpy(&mb, (const unsigned long long *)(r->arena.base + r->plan.at.maxbits) + u, sizeof mb, cudaMemcpyDeviceToHost));
        memcpy(max_host, &mb, sizeof(double));
    }
    return 0;
}

/* Pure copy traffic of one synthesis step, no kernels: `h2d_bytes` from pinned host memory up and `d2h_bytes` down, at the
 * same time on two streams, `reps` times; *ms receives the average time of one repetition.  The ceiling the end-to-end
 * number of a step with these byte counts can reach on this host / PCIe path (tools/pcie_ceiling.py, bench.py e2e.ceiling). */
int trm_cuda_copy_probe(int device, const void *host_in, size_t h2d_bytes, void *host_out, size_t d2h_bytes, int reps, double *ms)
{
    CK(cudaSetDevice(device));
    void *d_in = nullptr, *d_out = nullptr;
    cudaStream_t s_up, s_down;
    cudaEvent_t e0, e1, e2;
    CK(cudaMalloc(&d_in, h2d_bytes ? h2d_bytes : 1));
    CK(cudaMalloc(&d_out, d2h_bytes ? d2h_bytes : 1));
    CK(cudaMemset(d_out, 0, d2h_bytes ? d2h_bytes : 1));
    CK(cudaStreamCreateWithFlags(&s_up, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&s_down, cudaStreamNonBlocking));
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1)); CK(cudaEventCreate(&e2));
    CK(cudaDeviceSynchronize());
    CK(cudaEventRecord(e0, s_up));
    CK(cudaStreamWaitEvent(s_down, e0, 0));
    for (int r = 0; r < reps; ++r) {
        if (h2d_bytes) CK(cudaMemcpyAsync(d_in, host_in, h2d_bytes, cudaMemcpyHostToDevice, s_up));
        if (d2h_bytes) CK(cudaMemcpyAsync(host_out, d_out, d2h_bytes, cudaMemcpyDeviceToHost, s_down));
    }
    CK(cudaEventRecord(e1, s_up));
    CK(cudaEventRecord(e2, s_down));
    CK(cudaStreamSynchronize(s_up));
    CK(cudaStreamSynchronize(s_down));
    float a = 0, b = 0;
    CK(cudaEventElapsedTime(&a, e0, e1));
    CK(cudaEventElapsedTime(&b, e0, e2));
    *ms = (double)(a > b ? a : b) / (reps > 0 ? reps : 1);
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaEventDestroy(e2);
    cudaStreamDestroy(s_up); cudaStreamDestroy(s_down);
    cudaFree(d_in); cudaFree(d_out);
    return 0;
}

}  // extern "C"
