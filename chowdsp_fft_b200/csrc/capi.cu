// The drop-in C ABI (include/chowdsp_fft.h, include/chowdsp_fft_b200.h): plan objects, the process-wide
// device twiddle cache, the pointer-kind policy and the host-staging pipeline.  Replaces the reference's
// dispatcher layer (/root/reference/chowdsp_fft.cpp:63-78, 232-452) and plan construction
// (/root/reference/simd/chowdsp_fft_impl_common.hpp:162-228).  Never throws across the ABI, has no CPU
// compute path: without a CUDA device plan creation fails and says so.
#include <cmath>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <new>
#include <atomic>
#include <chrono>
#include <unordered_map>
#include <vector>

#include <nvtx3/nvToolsExt.h> // header-only; a no-op unless a profiler injects its NVTX library

#include "../../include/chowdsp_fft_b200.h"
#include "dispatch.h"
#include "large_plan.h"

// tracing: every computing entry point of the C ABI is an NVTX range (visible in Nsight Systems / Compute timelines)
namespace
{
struct TraceRange
{
    explicit TraceRange (const char* name) { nvtxRangePushA (name); }
    ~TraceRange() { nvtxRangePop(); }
    TraceRange (const TraceRange&) = delete;
    TraceRange& operator= (const TraceRange&) = delete;
};
} // namespace
#define CFB_TRACE(name) const TraceRange cfb_trace_range_ (name)

#define CFB_API __attribute__ ((visibility ("default")))

namespace
{
using namespace cfb;

// ------------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------------
thread_local char t_error[512] = "";
thread_local char t_last_kernel[96] = ""; // name of the transform kernel this thread launched last (fft_b200_last_kernel)
const char* kKindNames[4] = { "C2C_FWD", "C2C_BWD", "R2C", "C2R" };
void note_kernel (const char* fmt, ...)
{
    va_list ap;
    va_start (ap, fmt);
    vsnprintf (t_last_kernel, sizeof (t_last_kernel), fmt, ap);
    va_end (ap);
}

int fail (int code, const char* fmt, ...)
{
    va_list ap;
    va_start (ap, fmt);
    vsnprintf (t_error, sizeof (t_error), fmt, ap);
    va_end (ap);
    if (getenv ("CHOWDSP_FFT_B200_QUIET") == nullptr)
        fprintf (stderr, "chowdsp_fft_b200: %s\n", t_error);
    return code;
}
int fail_cuda (cudaError_t e, const char* what)
{
    return fail (chowdsp::fft::FFT_B200_ECUDA, "%s: %s", what, cudaGetErrorString (e));
}
#define CFB_CUDA(call)                           \
    do                                           \
    {                                            \
        const cudaError_t e__ = (call);          \
        if (e__ != cudaSuccess)                  \
            return fail_cuda (e__, #call);       \
    } while (0)

bool device_available()
{
    static const bool ok = []
    {
        int n = 0;
        const cudaError_t e = cudaGetDeviceCount (&n);
        if (e != cudaSuccess)
            (void) cudaGetLastError(); // clear the sticky "no device" state
        return e == cudaSuccess && n > 0;
    }();
    return ok;
}

// ------------------------------------------------------------------------------------------------
// device twiddle cache: one immutable table set per (device, complex length, needs-real-split);
// owned by the process, shared by every plan (so pre-allocated handles never leak device memory).
// ------------------------------------------------------------------------------------------------
struct Tables
{
    float2* tw = nullptr;  // stage twiddles
    float2* rtw = nullptr; // real split twiddles (real plans only)
};

std::mutex g_tables_mutex;
std::map<uint64_t, Tables> g_tables;

int get_tables (int device, int logM, bool real, Tables& out, int radix = 16)
{
    const uint64_t key = ((uint64_t) device << 32) | ((uint64_t) (radix == 32 ? 1 : 0) << 16) | ((uint64_t) logM << 1) | (real ? 1u : 0u);
    std::lock_guard<std::mutex> lock (g_tables_mutex);
    auto it = g_tables.find (key);
    if (it != g_tables.end())
    {
        out = it->second;
        return 0;
    }
    Tables t;
    const int len = stage_twiddle_len (logM, radix);
    if (len < 0)
        return fail (chowdsp::fft::FFT_B200_EINVAL, "no kernel for complex length 2^%d", logM);
    std::vector<float2> host ((size_t) len + 1);
    fill_stage_twiddles_rt (logM, radix, host.data());
    CFB_CUDA (cudaMalloc (&t.tw, sizeof (float2) * ((size_t) len + 1)));
    CFB_CUDA (cudaMemcpy (t.tw, host.data(), sizeof (float2) * ((size_t) len + 1), cudaMemcpyHostToDevice));
    if (real)
    {
        const int M = 1 << logM;
        std::vector<float2> hr ((size_t) M / 2 + 1);
        fill_real_twiddles (hr.data(), M);
        CFB_CUDA (cudaMalloc (&t.rtw, sizeof (float2) * hr.size()));
        CFB_CUDA (cudaMemcpy (t.rtw, hr.data(), sizeof (float2) * hr.size(), cudaMemcpyHostToDevice));
    }
    g_tables[key] = t;
    out = t;
    return 0;
}

// tables of the generic mixed-radix kernel, per (device, complex length, needs-real-split)
std::map<uint64_t, Tables> g_mixed_tables;
int get_mixed_tables (int device, int M, bool real, Tables& out)
{
    const uint64_t key = ((uint64_t) device << 40) | ((uint64_t) M << 1) | (real ? 1u : 0u);
    std::lock_guard<std::mutex> lock (g_tables_mutex);
    auto it = g_mixed_tables.find (key);
    if (it != g_mixed_tables.end())
    {
        out = it->second;
        return 0;
    }
    Tables t;
    std::vector<float2> w ((size_t) M);
    fill_mixed_twiddles (w.data(), M);
    CFB_CUDA (cudaMalloc (&t.tw, sizeof (float2) * w.size()));
    CFB_CUDA (cudaMemcpy (t.tw, w.data(), sizeof (float2) * w.size(), cudaMemcpyHostToDevice));
    if (real)
    {
        std::vector<float2> r ((size_t) M / 2 + 1);
        fill_mixed_real_twiddles (r.data(), M);
        CFB_CUDA (cudaMalloc (&t.rtw, sizeof (float2) * r.size()));
        CFB_CUDA (cudaMemcpy (t.rtw, r.data(), sizeof (float2) * r.size(), cudaMemcpyHostToDevice));
    }
    g_mixed_tables[key] = t;
    out = t;
    return 0;
}

// two-level tables W_(2^n)^e = lo[e & mask] * hi[e >> lobits] for the multi-pass (large) transforms
struct BigTables
{
    float2* lo = nullptr;
    float2* hi = nullptr;
    int lobits = 0;
};
std::map<uint64_t, BigTables> g_big_tables;

int get_big_tables (int device, int n, BigTables& out)
{
    const uint64_t key = ((uint64_t) device << 32) | (uint64_t) n;
    std::lock_guard<std::mutex> lock (g_tables_mutex);
    auto it = g_big_tables.find (key);
    if (it != g_big_tables.end())
    {
        out = it->second;
        return 0;
    }
    BigTables t;
    t.lobits = big_twiddle_lobits (n);
    const size_t nlo = (size_t) 1 << t.lobits, nhi = (size_t) 1 << (n - t.lobits);
    std::vector<float2> lo (nlo), hi (nhi);
    fill_big_twiddles (lo.data(), hi.data(), n, t.lobits);
    CFB_CUDA (cudaMalloc (&t.lo, sizeof (float2) * nlo));
    CFB_CUDA (cudaMalloc (&t.hi, sizeof (float2) * nhi));
    CFB_CUDA (cudaMemcpy (t.lo, lo.data(), sizeof (float2) * nlo, cudaMemcpyHostToDevice));
    CFB_CUDA (cudaMemcpy (t.hi, hi.data(), sizeof (float2) * nhi, cudaMemcpyHostToDevice));
    g_big_tables[key] = t;
    out = t;
    return 0;
}

// ------------------------------------------------------------------------------------------------
// plan
// ------------------------------------------------------------------------------------------------
constexpr uint64_t kMagic = 0x4346423230304642ull; // "CFB200FB"
constexpr int kMaxDevices = 16;

struct Plan
{
    uint64_t magic;
    int N;
    int is_complex;
    int logM; // complex length handled by the kernel: log2 N (complex) or log2 N - 1 (real)
    int logW; // unordered layout: 3 = 8-lane, 2 = 4-lane
    int owns_memory;
    int home_device;
    int mixed;   // N = 2^a 3^b 5^c, not a power of two: generic mixed-radix kernel (mixed_kernels.cuh); logM is unused
    int M;       // complex points per transform (N, or N/2 for real plans)
    Tables tables[2][kMaxDevices]; // [radix 16 | 32], filled lazily per device (guarded by g_tables_mutex through get_tables)
    bool have[2][kMaxDevices];
};

int ilog2i (int v)
{
    int l = 0;
    while ((1 << l) < v)
        ++l;
    return l;
}

// reference size rules: common.hpp:168-177 (+ AVX-then-SSE fallback, chowdsp_fft.cpp:262-273);
// powers of two only (north star), one CTA-resident transform (<= 2^14 complex points).
bool is_235 (int N)
{
    if (N <= 0)
        return false;
    for (int r : { 2, 3, 5 })
        while (N % r == 0)
            N /= r;
    return N == 1;
}
int choose_width (int N, bool is_complex, bool use_avx)
{
    if (! is_235 (N))
        return 0;
    for (int W = use_avx ? 8 : 4; W >= 4; W /= 2)
        if (N % (is_complex ? W * W : 2 * W * W) == 0)
            return W;
    return 0;
}

Plan* as_plan (void* setup)
{
    auto* p = static_cast<Plan*> (setup);
    if (p == nullptr || (reinterpret_cast<uintptr_t> (p) & 7) != 0 || p->magic != kMagic)
    {
        fail (chowdsp::fft::FFT_B200_EINVAL, "invalid FFT setup handle %p", setup);
        return nullptr;
    }
    return p;
}

// Points per thread of the single-kernel transform for complex length 2^logM: 32 where that geometry exists and
// pays off, else 16.  Measured on B200 (profiles/r01_radix32_sweep.txt): one exchange fewer is worth +15..25 % at
// 2^13, +5..9 % at 2^14, +2..9 % for the real kinds at 2^10 (STFT config +5 %), and costs 0..5 % at 2^9 and for
// complex 2^10 (fewer resident warps).  Tuning hook "radix32_mask": bit n = complex length 2^n for the complex
// kinds, bit 16+n for the real kinds; -1 restores this default.
constexpr unsigned kRadix32Default = (1u << 13) | (1u << 14) | (1u << (16 + 10)) | (1u << (16 + 13)) | (1u << (16 + 14));
unsigned g_radix32_mask = kRadix32Default;
int radix_for (int logM, bool is_complex) { return (has_radix32 (logM) && ((g_radix32_mask >> (logM + (is_complex ? 0 : 16))) & 1u) != 0) ? 32 : 16; }

int plan_tables (Plan* p, Tables& t, int radix = 16)
{
    int dev = 0;
    CFB_CUDA (cudaGetDevice (&dev));
    if (dev < 0 || dev >= kMaxDevices)
        return fail (chowdsp::fft::FFT_B200_EINVAL, "device index %d out of range", dev);
    if (p->mixed)
        return get_mixed_tables (dev, p->M, ! p->is_complex, t);
    if (p->logM > kMaxLogM)
    {
        t = Tables {};
        return 0; // multi-pass plan: tables are fetched per pass (enqueue_large)
    }
    const int ri = radix == 32 ? 1 : 0;
    {
        // the plan may be shared across threads (chowdsp_fft.h:87-91): its per-device cache is read and written under the mutex
        std::lock_guard<std::mutex> lock (g_tables_mutex);
        if (p->have[ri][dev])
        {
            t = p->tables[ri][dev];
            return 0;
        }
    }
    Tables nt;
    const int rc = get_tables (dev, p->logM, ! p->is_complex, nt, radix);
    if (rc != 0)
        return rc;
    std::lock_guard<std::mutex> lock (g_tables_mutex);
    p->tables[ri][dev] = nt;
    p->have[ri][dev] = true;
    t = nt;
    return 0;
}

// Setup-time table upload for the current device: every table a later transform call on this plan can ask for, so that
// device-pointer calls only enqueue work on the caller's stream -- no cudaMalloc / blocking cudaMemcpy under the tables
// mutex on the first transform, nothing that would invalidate a stream capture (ADVICE r1).  Other devices are still
// filled lazily on first use there.
int preload_large (Plan* p); // multi-pass plans: big twiddle tables + the per-pass stage tables (defined with enqueue_large)
int preload_tables (Plan* p)
{
    Tables t;
    if (p->mixed)
    {
        const int rc = plan_tables (p, t);
        int logP = 0, Q = 0;
        if (rc == 0 && mixq_applies (p->M, logP, Q)) // stage twiddles of the power-of-two sub-transforms (mixq_kernels.cuh)
        {
            int dev = 0;
            CFB_CUDA (cudaGetDevice (&dev));
            return get_tables (dev, logP, false, t, 16);
        }
        return rc;
    }
    if (p->logM > kMaxLogM)
        return preload_large (p);
    int rc = plan_tables (p, t, 16);
    if (rc == 0 && has_radix32 (p->logM))
        rc = plan_tables (p, t, 32); // default radix-32 geometries, the TMA-pipelined kernels (2^13 / 2^14) and wpipe at 2^10
    return rc;
}

size_t reference_bytes (int N, bool is_complex) // sse:67-72 / avx:73-78: 2*Ncvec*W*4 + sizeof(FFT_Setup)
{
    return (size_t) N * (is_complex ? 8 : 4) + 96;
}

// ------------------------------------------------------------------------------------------------
// pointer classification and staging
// ------------------------------------------------------------------------------------------------
enum class Mem
{
    Device,  // device or managed: kernels use it directly
    Pinned,  // page-locked host memory mapped into the device address space
    Pageable // ordinary host memory
};

struct PtrInfo
{
    Mem kind;
    const void* dev; // pointer a kernel may dereference (Device / Pinned)
};

// aligned_malloc blocks are known without asking the driver: base -> (size, pinned, device alias).  Looked up first by
// classify(); a generation counter (bumped by aligned_free) invalidates the per-thread cache of the last ranges seen.
struct HostBlock
{
    size_t bytes;
    bool pinned;
    void* dev; // device alias of a pinned block (cudaHostGetDevicePointer), else nullptr
};
std::mutex g_alloc_mutex;
std::map<uintptr_t, HostBlock> g_allocs;
std::atomic<unsigned long long> g_alloc_generation { 1 };

PtrInfo classify_slow (const void* p)
{
    cudaPointerAttributes a {};
    if (cudaPointerGetAttributes (&a, p) != cudaSuccess)
    {
        (void) cudaGetLastError();
        return { Mem::Pageable, nullptr };
    }
    switch (a.type)
    {
        case cudaMemoryTypeDevice:
        case cudaMemoryTypeManaged: return { Mem::Device, a.devicePointer ? a.devicePointer : p };
        case cudaMemoryTypeHost: return { a.devicePointer ? Mem::Pinned : Mem::Pageable, a.devicePointer };
        default: return { Mem::Pageable, nullptr };
    }
}

// Pointer classification is on the latency path of every drop-in call (two cudaPointerGetAttributes round trips cost more
// than the launch itself for a 1024-point transform, VERDICT r1): blocks handed out by aligned_malloc -- what the
// reference's callers use (test/test.c:19-22, bench/bench.cpp) -- are answered from a thread-local cache of their ranges.
PtrInfo classify (const void* p)
{
    struct Cached
    {
        uintptr_t lo = 1, hi = 0;
        HostBlock blk {};
        unsigned long long generation = 0;
    };
    static thread_local Cached cache[4];
    static thread_local unsigned next = 0;
    const uintptr_t u = reinterpret_cast<uintptr_t> (p);
    const unsigned long long gen = g_alloc_generation.load (std::memory_order_acquire);
    for (const Cached& c : cache)
        if (c.generation == gen && u >= c.lo && u < c.hi)
            return c.blk.pinned ? PtrInfo { Mem::Pinned, static_cast<char*> (c.blk.dev) + (u - c.lo) } : PtrInfo { Mem::Pageable, nullptr };
    {
        std::lock_guard<std::mutex> lock (g_alloc_mutex);
        auto it = g_allocs.upper_bound (u);
        if (it != g_allocs.begin())
        {
            --it;
            if (u < it->first + it->second.bytes)
            {
                Cached& c = cache[next++ & 3u];
                c.lo = it->first;
                c.hi = it->first + it->second.bytes;
                c.blk = it->second;
                c.generation = gen;
                return c.blk.pinned ? PtrInfo { Mem::Pinned, static_cast<char*> (c.blk.dev) + (u - c.lo) } : PtrInfo { Mem::Pageable, nullptr };
            }
        }
    }
    return classify_slow (p);
}

// per-thread staging: two lanes so H2D of chunk c+1, the kernel of chunk c and D2H of chunk c-1 overlap
struct Staging
{
    cudaStream_t stream[2] = { nullptr, nullptr };
    float* buf[2][3] = { { nullptr, nullptr, nullptr }, { nullptr, nullptr, nullptr } };
    size_t cap[2][3] = { { 0, 0, 0 }, { 0, 0, 0 } };
    int device = -1;

    int ensure (int lane, int slot, size_t bytes)
    {
        int dev = 0;
        CFB_CUDA (cudaGetDevice (&dev));
        if (device != dev)
        {
            release();
            device = dev;
        }
        if (stream[lane] == nullptr)
            CFB_CUDA (cudaStreamCreateWithFlags (&stream[lane], cudaStreamNonBlocking));
        if (cap[lane][slot] < bytes)
        {
            if (buf[lane][slot] != nullptr)
            {
                CFB_CUDA (cudaStreamSynchronize (stream[lane]));
                CFB_CUDA (cudaFree (buf[lane][slot]));
                buf[lane][slot] = nullptr;
                cap[lane][slot] = 0;
            }
            const size_t want = bytes < (1u << 20) ? (1u << 20) : bytes;
            CFB_CUDA (cudaMalloc (&buf[lane][slot], want));
            cap[lane][slot] = want;
        }
        return 0;
    }
    void release()
    {
        for (int l = 0; l < 2; ++l)
        {
            for (int s = 0; s < 3; ++s)
            {
                if (buf[l][s] != nullptr)
                    cudaFree (buf[l][s]);
                buf[l][s] = nullptr;
                cap[l][s] = 0;
            }
            if (stream[l] != nullptr)
                cudaStreamDestroy (stream[l]);
            stream[l] = nullptr;
        }
    }
    // Runs when the owning thread exits (thread_local).  A worker thread that used the host-memory path gives its two
    // streams and up to six staging buffers back here -- short-lived audio worker threads would otherwise grow device
    // memory without bound (ADVICE r1).  On the main thread this runs at exit() before any static destructor / atexit
    // handler, i.e. while the runtime is still loaded; if the runtime is already unloading the calls fail with
    // cudaErrorCudartUnloading, which is ignored.
    ~Staging()
    {
        if (device < 0)
            return;
        int cur = -1;
        if (cudaGetDevice (&cur) != cudaSuccess)
        {
            (void) cudaGetLastError();
            return;
        }
        if (cur != device && cudaSetDevice (device) != cudaSuccess)
        {
            (void) cudaGetLastError();
            return;
        }
        for (int l = 0; l < 2; ++l)
            if (stream[l] != nullptr)
                (void) cudaStreamSynchronize (stream[l]);
        release();
        if (cur != device)
            (void) cudaSetDevice (cur);
        (void) cudaGetLastError();
    }
};
thread_local Staging t_staging;

bool g_stft_union = false; // tuning hook "stft_union"
// tuning hook "stft_pipe": persistent TMA-fed frame gather (stft_pipe_kernel) where it applies.  Off by default: at
// hop = N/4 it is 5 % slower on B200 than per-transform loads once the transforms synchronise at warp level (its
// per-item CTA barrier re-couples the warps; profiles/r01_stft.txt); it moves 2.9x fewer L2 -> SM bytes, so it is
// kept for parts / hops where that traffic is the bound
bool g_stft_pipe = false;
// tuning hook "pipe_mask": bit (2 kind + logM - 13) = use the persistent TMA-pipelined kernel (pipe_kernels.cuh) for
// that kind (C2C_FWD, C2C_BWD, R2C, C2R = 0..3) at complex length 2^13 / 2^14, ordered layouts; bits 8..15 the same
// for the 8-lane unordered layout.  Default from the
// A/B sweeps in profiles/r01_pipe_kernel.txt: everything at 2^14 (+20..50 %); at 2^13, where fft_kernel already runs
// two CTAs per SM, +2..7 % except ordered R2C (-3..5 %), which stays with fft_kernel
constexpr unsigned kPipeDefault = 0xFFFFu & ~(1u << 4) & ~(1u << 6); // ordered R2C / C2R at 2^13 stay with fft_kernel<13,32> (C2R since the derived split twiddles: 5.60 vs 5.34 TB/s, profiles/r02_retune.txt)
unsigned g_pipe_mask = kPipeDefault;
bool pipe_enabled (int logM, int kind, int logW)
{
    return has_pipe (logM) && (logW == 0 || logW == 3) && ((g_pipe_mask >> ((logW == 0 ? 0 : 8) + 2 * kind + logM - 13)) & 1u) != 0;
}
// tuning hook "wpipe": which batches of the sizes one warp owns (has_wpipe; forward kinds, 16-byte aligned input rows) go
// through the warp-pipelined kernel (wpipe_kernel): bit 1 = overlapping or windowed frames (STFT analysis), bit 0 = every
// batch, bit 2 = plain batches of N = 2048 real transforms with unordered output (fft_kernel's staging epilogue makes that one
// latency-bound too: 5.6-5.9 -> 6.3 TB/s); bits 8.. = warps per CTA (0 = as many as fit an SM).  Default from
// profiles/r01_wpipe.txt: frames (and that one plain case) only -- their
// re-reads are L2 hits, so fft_kernel is bound by the exposed load latency there (STFT config 4.81 -> 5.30 TB/s), while
// plain batches already run at the HBM roofline with fft_kernel and lose 5..13 % to the landing-buffer round trip.  Bit 3: frames of the
// 2^9-point size too -- off since the burst-mode re-measurement of round 2 (profiles/r02_stft_sizes.txt: N = 1024 frames 4.12 / 4.45 TB/s with /
// without a window through wpipe_kernel<9,16>, 4.44 / 4.95 through stft_kernel / fft_kernel, at 64 .. 1024 channels)
constexpr int kWPipeDefault = 2 | 4;
int g_wpipe = kWPipeDefault;
// tuning hook "wistft": bit 0 = overlap-add synthesis through the warp-pipelined kernel (wistft_kernel) where it applies (N = 2048; bit 1: N = 1024
// too); bits 8.. = warps per CTA (0 = the kernel's maximum)
constexpr int kWIstftDefault = 1;
int g_wistft = kWIstftDefault;
int device_sm_count()
{
    static thread_local int c_dev = -1, c_sms = 148;
    int dev = 0;
    if (cudaGetDevice (&dev) == cudaSuccess && dev != c_dev)
    {
        int n = 0;
        if (cudaDeviceGetAttribute (&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0)
            c_sms = n;
        c_dev = dev;
    }
    return c_sms;
}
int g_pf_ahead = 0;        // tuning hook "pf_ahead": L2 prefetch distance of the single-kernel transforms, in CTAs
// tuning hook "cluster": 1 = complex transforms of 2^15 .. 2^17 points run in ONE pass on a thread-block cluster
// (cluster_kernels.cuh) where the batch layout allows, 0 = always the multi-pass tile path; "cluster_min_batch": batches
// smaller than this stay with the tile path (a cluster kernel runs one transform per cluster: a single transform would
// occupy 4 .. 16 of the 148 SMs)
// Default OFF: measured on B200 (profiles/r02_cluster_kernel.txt) the one-pass cluster kernel reaches 2.9 / 2.6 / 2.3 TB/s at
// 2^15 / 2^16 / 2^17 points against 3.0 / 3.3 / 3.2 TB/s of the two tile passes -- its transform-long critical path (input
// barrier, cluster barrier, exchange barrier, store) is exposed with only two CTAs per SM to overlap it.
constexpr int kClusterDefault = 0, kClusterMinBatchDefault = 8;
int g_cluster = kClusterDefault, g_cluster_min_batch = kClusterMinBatchDefault;

constexpr size_t kZeroCopyBytesDefault = 256 * 1024; // pinned buffers up to this size are used in place (tuning hook zero_copy_kb)
size_t g_zero_copy_bytes = kZeroCopyBytesDefault;
#define kZeroCopyBytes g_zero_copy_bytes
constexpr size_t kChunkBytes = 32ull * 1024 * 1024; // host staging granularity per lane

int kind_of (const Plan* p, int direction)
{
    if (p->is_complex)
        return direction == chowdsp::fft::FFT_FORWARD ? C2C_FWD : C2C_BWD;
    return direction == chowdsp::fft::FFT_FORWARD ? R2C : C2R;
}


// Alignment guard shared by every entry point (ADVICE r1): the kernels move 8-byte complex pairs on ordered data,
// windows and signals and 16-byte vectors on unordered spectra, delay lines and IR partitions.  A misaligned base or
// an odd stride would become cudaErrorMisalignedAddress on the device -- a sticky error that poisons the whole CUDA
// context of the host process -- so it is rejected here with FFT_B200_EINVAL instead.  Strides in floats; a stride only
// matters when more than one row is addressed through it.
bool misaligned (const void* ptr, unsigned align_bytes, long long s0 = 0, long long n0 = 1, long long s1 = 0, long long n1 = 1)
{
    const long long m = (long long) (align_bytes / 4u) - 1;
    return (reinterpret_cast<uintptr_t> (ptr) & (uintptr_t) (align_bytes - 1u)) != 0 || (n0 > 1 && (s0 & m) != 0) || (n1 > 1 && (s1 & m) != 0);
}

// ------------------------------------------------------------------------------------------------
// multi-pass (large) transforms
// ------------------------------------------------------------------------------------------------
// tuning hooks "l2_chunk_mb" (MiB of intermediate per chunk of the L2-chunked schedules, 0 = classic whole-array passes),
// "l2_lanes" (helper streams / ring slots, 1..4) and "l2_policy" (1 = evict_last / evict_first hints on ring / stream accesses)
constexpr int kL2ChunkMbDefault = 16, kL2LanesDefault = 3, kL2PolicyDefault = 1;
int g_l2_chunk_mb = kL2ChunkMbDefault, g_l2_lanes = kL2LanesDefault, g_l2_policy = kL2PolicyDefault;
constexpr int kMaxLanes = 4;
int g_mixq = 1; // tuning hook "mixq"
int g_ristft = 1; // tuning hook "ristft": overlap-add synthesis through ristft_kernel where it applies
constexpr int kTilePfDefault = 0;  // tuning hook "tile_pf" (large_plan.h: tile_pf_distance)
constexpr int kTileTmaDefault = 0; // tuning hook "tile_tma" (large_plan.h: tile_tma_mode)

// helper streams of the chunked schedules: chunks alternate over them so that pass B of one chunk overlaps pass C of the
// previous one; joined back into the caller's stream with events (also legal inside a stream capture)
struct ForkJoin
{
    cudaStream_t lane[kMaxLanes] = { nullptr, nullptr, nullptr, nullptr };
    cudaEvent_t fork = nullptr, join[kMaxLanes] = { nullptr, nullptr, nullptr, nullptr };
    int device = -1;
    int ensure()
    {
        int dev = 0;
        CFB_CUDA (cudaGetDevice (&dev));
        if (device == dev)
            return 0;
        release();
        for (int i = 0; i < kMaxLanes; ++i)
        {
            CFB_CUDA (cudaStreamCreateWithFlags (&lane[i], cudaStreamNonBlocking));
            CFB_CUDA (cudaEventCreateWithFlags (&join[i], cudaEventDisableTiming));
        }
        CFB_CUDA (cudaEventCreateWithFlags (&fork, cudaEventDisableTiming));
        device = dev;
        return 0;
    }
    void release()
    {
        for (int i = 0; i < kMaxLanes; ++i)
        {
            if (lane[i] != nullptr)
                (void) cudaStreamDestroy (lane[i]);
            if (join[i] != nullptr)
                (void) cudaEventDestroy (join[i]);
            lane[i] = nullptr;
            join[i] = nullptr;
        }
        if (fork != nullptr)
            (void) cudaEventDestroy (fork);
        fork = nullptr;
        device = -1;
    }
    ~ForkJoin()
    {
        if (device >= 0)
        {
            release();
            (void) cudaGetLastError();
        }
    }
};
thread_local ForkJoin t_forkjoin;


// fork / join bookkeeping of one schedule run: lane -1 is the caller's stream; the first use of a helper lane makes it
// wait for everything enqueued on the caller's stream so far, join() makes the caller's stream wait for every used lane
struct LaneSet
{
    ForkJoin& fj;
    cudaStream_t main;
    bool forked = false;
    bool used[kMaxLanes] = { false, false, false, false };
    LaneSet (ForkJoin& f, cudaStream_t s) : fj (f), main (s) {}
    cudaStream_t stream_of (int lane, cudaError_t& e)
    {
        if (lane < 0)
            return main;
        if (! forked)
        {
            if (e == cudaSuccess)
                e = cudaEventRecord (fj.fork, main);
            forked = true;
        }
        if (! used[lane])
        {
            if (e == cudaSuccess)
                e = cudaStreamWaitEvent (fj.lane[lane], fj.fork, 0);
            used[lane] = true;
        }
        return fj.lane[lane];
    }
    void join (cudaError_t& e)
    {
        for (int l = 0; l < kMaxLanes; ++l)
            if (used[l])
            {
                if (e == cudaSuccess)
                    e = cudaEventRecord (fj.join[l], fj.lane[l]);
                if (e == cudaSuccess)
                    e = cudaStreamWaitEvent (main, fj.join[l], 0);
                used[l] = false;
            }
        forked = false;
    }
};

// keep freed scratch cached in the stream-ordered pool instead of returning it to the OS at every synchronisation.  The
// release threshold belongs to the device's default pool, so it is set once per device for the whole process, at setup
// time (preload_large): setting it inside a stream capture invalidates the capture, so a multi-pass call must find it set
// even on a thread that never made one before
std::atomic<bool> g_pool_kept[kMaxDevices] {};
void keep_pool_memory (int dev)
{
    if (dev < 0 || dev >= kMaxDevices || g_pool_kept[dev].load (std::memory_order_acquire))
        return;
    cudaMemPool_t pool = nullptr;
    if (cudaDeviceGetDefaultMemPool (&pool, dev) == cudaSuccess)
    {
        unsigned long long keep = ~0ull;
        (void) cudaMemPoolSetAttribute (pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
    (void) cudaGetLastError();
    g_pool_kept[dev].store (true, std::memory_order_release);
}

int tile_radix_for (int logL) { return (tile_radix32() != 0 && logL >= 9) ? 32 : 16; } // must match launch_tile_l (large_inst.cu)

struct LargeTables
{
    BigTables bt;
    Tables pass[3];
};
int large_tables (Plan* p, int dev, const LargeFactors& f, LargeTables& lt)
{
    int rc = get_big_tables (dev, p->is_complex ? p->logM : p->logM + 1, lt.bt);
    const int logs[3] = { f.l1, f.l2, f.l3 };
    for (int i = 0; i < 3 && rc == 0; ++i)
        if (logs[i] != 0)
            rc = get_tables (dev, logs[i], false, lt.pass[i], tile_radix_for (logs[i]));
    return rc;
}
int preload_large (Plan* p)
{
    int dev = 0;
    CFB_CUDA (cudaGetDevice (&dev));
    keep_pool_memory (dev);
    LargeTables lt;
    int rc = large_tables (p, dev, choose_factors (p->logM), lt);
    if (rc == 0 && p->is_complex && has_cluster (p->logM))
    {
        Tables st; // the cluster kernel's local 512-point stage table
        rc = get_tables (dev, 9, false, st, 32);
    }
    return rc;
}

// `batch` transforms larger than a CTA: 2 or 3 tile passes (+ a split / merge pass for real plans) through stream-ordered
// scratch, L2-chunked where that saves HBM sweeps (large_plan.h: build_large_schedule).  Unordered complex layouts are
// folded into the first / last pass.  The reference uses the caller's `work` buffer for the same purpose
// (simd/chowdsp_fft_impl_avx.cpp:1861-1863); here `work` may stay NULL.  Strides in floats.
int enqueue_large (Plan* p, const float* in, float* out, int batch, long long in_stride, long long out_stride, int direction, bool ordered, cudaStream_t stream)
{
    int dev = 0;
    CFB_CUDA (cudaGetDevice (&dev));
    const int n = p->logM;
    const bool fwd = direction == chowdsp::fft::FFT_FORWARD;
    const int dir = fwd ? -1 : +1;
    const LargeFactors f = choose_factors (n);
    const int np = f.passes();
    LargeTables lt;
    int rc = large_tables (p, dev, f, lt);
    if (rc != 0)
        return rc;
    keep_pool_memory (dev);
    const long long npts = 1LL << n;              // float2 per transform
    const size_t bytes = sizeof (float2) << n;
    const bool real = ! p->is_complex;
    // Chunked schedule?  Two-pass plans: only when the batch does not fit in L2 anyway (a single 2^15..2^20-point transform is
    // L2-resident between its passes as it is).  Three-pass plans: always.
    // Measured on B200 (profiles/r02_l2_chunked.txt): +4..8 % up to 2^24 points with 16 MiB chunks on 3 lanes, nothing at
    // 2^26 and -6 % at 2^28 (the chunk unit of 8 k1-rows is 32 MiB there, beyond what L2 keeps for all SMs: 32..40 MB),
    // so the largest transforms keep whole-array passes unless the hook says otherwise (l2_chunk_mb < 0: force chunking)
    long long chunk_elems = (long long) (g_l2_chunk_mb < 0 ? -g_l2_chunk_mb : g_l2_chunk_mb) * (1 << 20) / 8;
    if (np == 2 && (long long) batch * npts <= 2 * chunk_elems)
        chunk_elems = 0;
    if (n > 24 && g_l2_chunk_mb > 0)
        chunk_elems = 0;
    const int lanes = g_l2_lanes < 1 ? 1 : (g_l2_lanes > kMaxLanes ? kMaxLanes : g_l2_lanes);
    // full-size scratch is allocated per super-chunk of the batch (<= 512 MiB per buffer)
    int super = (int) ((512ull << 20) / bytes);
    super = super < 1 ? 1 : (super > batch ? batch : super);
    const long long ring_lane = ring_elems_needed (n, f, super, chunk_elems);
    // real two-pass chunked plans keep the split / merge step inside the chunk: a second sub-slot per lane holds z
    const bool real_in_chunk = real && np == 2 && chunk_elems > 0;
    const bool need_s1 = chunk_elems == 0 || np == 3;
    const bool need_s2 = real && ! real_in_chunk && fwd; // z of a forward real transform, before the split pass (backward: merged into s1)
    float2 *s1 = nullptr, *s2 = nullptr, *ring = nullptr;
    if (need_s1)
        CFB_CUDA (cudaMallocAsync (&s1, bytes * (size_t) super, stream));
    if (need_s2)
        CFB_CUDA (cudaMallocAsync (&s2, bytes * (size_t) super, stream));
    if (chunk_elems > 0)
        CFB_CUDA (cudaMallocAsync (&ring, sizeof (float2) * (size_t) ring_lane * (size_t) lanes * (real_in_chunk ? 2u : 1u), stream));
    ForkJoin& fj = t_forkjoin;
    if (chunk_elems > 0 && (rc = fj.ensure()) != 0)
        return rc;

    RealPassArgs ra {};
    ra.logM = n;
    ra.logW = ordered ? 0 : p->logW;
    ra.tw_lobits = lt.bt.lobits;
    ra.tw_mult = 1;
    ra.tw_lo = lt.bt.lo;
    ra.tw_hi = lt.bt.hi;
    cudaError_t e = cudaSuccess;
    std::vector<LargeLaunch> sched;
    int launches_total = 0;
    for (int b0 = 0; b0 < batch && rc == 0 && e == cudaSuccess; b0 += super)
    {
        const int nb = batch - b0 < super ? batch - b0 : super;
        const float* cin = in + (long long) b0 * in_stride;
        float* cout = out + (long long) b0 * out_stride;
        LargeBuffers bufs {};
        bufs.s1 = s1;
        bufs.ring = ring;
        bufs.ring_lane_elems = ring_lane;
        LaneSet ls (fj, stream);
        auto stream_of = [&] (int lane) -> cudaStream_t { return ls.stream_of (lane, e); };
        auto join = [&] { ls.join (e); };
        if (real_in_chunk)
        {
            // per chunk of k transforms on lane l:  forward  A: src -> ring, C: ring -> z, split: z -> out
            //                                        backward merge: in -> z, A: z -> ring, C: ring -> out
            const long long k = ring_lane / npts;
            int lane = 0;
            for (long long c0 = 0; c0 < nb && e == cudaSuccess; c0 += k, lane = (lane + 1) % lanes)
            {
                const int nc = (int) (nb - c0 < k ? nb - c0 : k);
                float2* slot = ring + (long long) lane * 2 * ring_lane;
                float2* zbuf = slot + ring_lane;
                cudaStream_t st = stream_of (lane);
                LargeBuffers cb {};
                cb.src = fwd ? reinterpret_cast<const float2*> (cin + c0 * in_stride) : zbuf;
                cb.src_bs = fwd ? in_stride / 2 : npts;
                cb.dst = fwd ? zbuf : reinterpret_cast<float2*> (cout + c0 * out_stride);
                cb.dst_bs = fwd ? npts : out_stride / 2;
                cb.s1 = slot;
                build_large_schedule (n, f, nc, cb, 2u, false, false, 0, 0, 1, false, sched);
                const int keep = g_l2_policy ? POLICY_KEEP : POLICY_NORMAL, strm = g_l2_policy ? POLICY_STREAM : POLICY_NORMAL;
                sched[0].pass.args.in_policy = fwd ? strm : keep;
                sched[0].pass.args.out_policy = keep;
                sched[1].pass.args.in_policy = keep;
                sched[1].pass.args.out_policy = fwd ? keep : strm;
                if (! fwd)
                {
                    ra.in = cin + c0 * in_stride;
                    ra.in_bstride = in_stride;
                    ra.out = reinterpret_cast<float*> (zbuf);
                    ra.out_bstride = 2 * npts;
                    if (e == cudaSuccess)
                        e = launch_real_pass (+1, ra, nc, st);
                    ++launches_total;
                }
                for (auto& l : sched)
                {
                    TileArgs& ta = l.pass.args;
                    ta.tw = lt.pass[l.pass.which].tw;
                    ta.tw_lo = lt.bt.lo;
                    ta.tw_hi = lt.bt.hi;
                    ta.tw_lobits = lt.bt.lobits;
                    if (e == cudaSuccess)
                        e = launch_tile_pass (dir, l.pass, st);
                    ++launches_total;
                }
                if (fwd)
                {
                    ra.in = reinterpret_cast<const float*> (zbuf);
                    ra.in_bstride = 2 * npts;
                    ra.out = cout + c0 * out_stride;
                    ra.out_bstride = out_stride;
                    if (e == cudaSuccess)
                        e = launch_real_pass (-1, ra, nc, st);
                    ++launches_total;
                }
            }
            join();
            continue;
        }
        // complex passes:  src -> dst of this super-chunk
        if (real && ! fwd)
        {
            ra.in = cin;
            ra.in_bstride = in_stride;
            ra.out = reinterpret_cast<float*> (s1);
            ra.out_bstride = 2 * npts;
            e = launch_real_pass (+1, ra, nb, stream);
            ++launches_total;
            bufs.src = s1; // pass A then runs in place on s1 (every tile reads all of its elements before it writes them)
            bufs.src_bs = npts;
        }
        else
        {
            bufs.src = reinterpret_cast<const float2*> (cin);
            bufs.src_bs = in_stride / 2;
        }
        if (real && fwd)
        {
            bufs.dst = s2;
            bufs.dst_bs = npts;
        }
        else
        {
            bufs.dst = reinterpret_cast<float2*> (cout);
            bufs.dst_bs = out_stride / 2;
        }
        const bool uio_in = ! real && ! ordered && ! fwd, uio_out = ! real && ! ordered && fwd;
        build_large_schedule (n, f, nb, bufs, real ? 2u : 1u, uio_in, uio_out, p->logW, chunk_elems, lanes, g_l2_policy != 0, sched);
        for (auto& l : sched)
        {
            TileArgs& ta = l.pass.args;
            ta.tw = lt.pass[l.pass.which].tw;
            ta.tw_lo = lt.bt.lo;
            ta.tw_hi = lt.bt.hi;
            ta.tw_lobits = lt.bt.lobits;
            cudaStream_t st = stream_of (l.lane);
            if (e == cudaSuccess)
                e = launch_tile_pass (dir, l.pass, st);
            ++launches_total;
        }
        join();
        if (real && fwd && e == cudaSuccess)
        {
            ra.in = reinterpret_cast<const float*> (s2);
            ra.in_bstride = 2 * npts;
            ra.out = cout;
            ra.out_bstride = out_stride;
            e = launch_real_pass (-1, ra, nb, stream);
            ++launches_total;
        }
    }
    note_kernel ("cfb::tile_fft_kernel<%d|%d|%d,dir %d> %d passes, %s, %d launches", f.l1, f.l2, f.l3, dir, np,
                 chunk_elems > 0 ? (np == 2 ? "L2-chunked (A,C per chunk)" : "L2-chunked (A global; B,C per chunk)") : "whole-array passes", launches_total);
    if (s1 != nullptr)
        CFB_CUDA (cudaFreeAsync (s1, stream));
    if (s2 != nullptr)
        CFB_CUDA (cudaFreeAsync (s2, stream));
    if (ring != nullptr)
        CFB_CUDA (cudaFreeAsync (ring, stream));
    if (e != cudaSuccess)
        return fail_cuda (e, "large transform pass launch");
    return rc;
}

int enqueue_transform (Plan* p, const float* in, float* out, int outer, int inner, long long in_outer, long long in_inner, long long out_outer, long long out_inner, int direction, bool ordered, cudaStream_t stream, const float* window = nullptr)
{
    if (window != nullptr && (p->mixed || p->logM > kMaxLogM || p->is_complex || direction != chowdsp::fft::FFT_FORWARD))
        return fail (chowdsp::fft::FFT_B200_EINVAL, "windowed transforms need a REAL single-kernel power-of-two plan and FFT_FORWARD");
    if (p->mixed)
    {
        if (misaligned (in, 8, in_inner, inner, in_outer, outer) || misaligned (out, 8, out_inner, inner, out_outer, outer))
            return fail (chowdsp::fft::FFT_B200_EINVAL, "mixed-radix transforms need 8-byte aligned buffers and even strides");
        Tables mt;
        const int mrc = plan_tables (p, mt);
        if (mrc != 0)
            return mrc;
        // M = Q 2^p with Q in {3, 5, 9, 15}: the odd factor as one register butterfly around the power-of-two stages
        // (mixq_kernels.cuh); other odd parts keep the generic kernel (tuning hook "mixq" = 0: always the generic kernel)
        int mq_logP = 0, mq_Q = 0;
        if (g_mixq != 0 && mixq_applies (p->M, mq_logP, mq_Q))
        {
            int dev = 0;
            CFB_CUDA (cudaGetDevice (&dev));
            Tables pt;
            const int prc = get_tables (dev, mq_logP, false, pt, 16);
            if (prc != 0)
                return prc;
            MixQArgs qa {};
            qa.tw = pt.tw;
            qa.wtab = mt.tw;
            qa.rtab = mt.rtw;
            qa.kind = kind_of (p, direction);
            qa.W = ordered ? 0 : (1 << p->logW);
            bool ok = true;
            for (int o = 0; o < outer && ok; ++o)
            {
                qa.in = in + (long long) o * in_outer;
                qa.out = out + (long long) o * out_outer;
                qa.in_stride = in_inner;
                qa.out_stride = out_inner;
                qa.batch = inner;
                const cudaError_t qe = launch_mixq (mq_logP, mq_Q, qa, stream);
                if (qe == cudaErrorInvalidConfiguration && o == 0)
                {
                    (void) cudaGetLastError();
                    ok = false; // no such instance: generic kernel below
                }
                else if (qe != cudaSuccess)
                    return fail_cuda (qe, "mixed-radix (Q x 2^p) kernel launch");
            }
            if (ok)
            {
                note_kernel ("cfb::mixq_kernel<%d,%d> M=%d %s W=%d", mq_logP, mq_Q, p->M, kKindNames[qa.kind], qa.W);
                return 0;
            }
        }
        MixedArgs ma {};
        ma.M = p->M;
        ma.nstages = mixed_factor (p->M, ma.radix);
        ma.wtab = mt.tw;
        ma.rtab = mt.rtw;
        ma.kind = kind_of (p, direction);
        ma.W = ordered ? 0 : (1 << p->logW);
        note_kernel ("cfb::mixed_kernel M=%d %s W=%d", p->M, kKindNames[ma.kind], ma.W);
        for (int o = 0; o < outer; ++o) // two-level batches: one launch per outer index
        {
            ma.in = in + (long long) o * in_outer;
            ma.out = out + (long long) o * out_outer;
            ma.in_stride = in_inner;
            ma.out_stride = out_inner;
            ma.batch = inner;
            const cudaError_t me = launch_mixed (ma, stream);
            if (me != cudaSuccess)
                return fail_cuda (me, "mixed-radix kernel launch");
        }
        return 0;
    }
    if (p->logM > kMaxLogM)
    {
        if (misaligned (in, 8, in_inner, inner, in_outer, outer) || misaligned (out, 8, out_inner, inner, out_outer, outer))
            return fail (chowdsp::fft::FFT_B200_EINVAL, "large transforms need 8-byte aligned buffers and even strides");
        // complex 2^15 .. 2^17 points, plain batches with TMA-loadable rows: ONE pass on a thread-block cluster
        // (cluster_kernels.cuh) instead of two tile passes; unordered inputs (inverse) stay with the tile path
        const bool fwd = direction == chowdsp::fft::FFT_FORWARD;
        const long long bstride_in = outer == 1 ? in_inner : in_outer, bstride_out = outer == 1 ? out_inner : out_outer;
        if (g_cluster != 0 && p->is_complex && has_cluster (p->logM) && (outer == 1 || inner == 1) && (ordered || (fwd && p->logW == 3))
            && ! misaligned (in, 16, bstride_in, (long long) outer * inner) && (long long) outer * inner >= g_cluster_min_batch)
        {
            int dev = 0;
            CFB_CUDA (cudaGetDevice (&dev));
            Tables st;
            BigTables bt;
            int rc = get_tables (dev, 9, false, st, 32);
            if (rc == 0)
                rc = get_big_tables (dev, p->logM, bt);
            if (rc != 0)
                return rc;
            ClusterArgs ca {};
            ca.out = out;
            ca.out_stride = bstride_out;
            ca.batch = outer * inner;
            ca.logW = ordered ? 0 : p->logW;
            ca.tw = st.tw;
            ca.tw_lo = bt.lo;
            ca.tw_hi = bt.hi;
            ca.tw_lobits = bt.lobits;
            ca.l2_prefetch = (g_cluster & 2) != 0 ? 0 : 1; // tuning bit 1 switches the L2 prefetch off (A/B)
            const cudaError_t ce = launch_cluster_fft (p->logM, fwd ? -1 : +1, ca.logW, in, bstride_in, ca, stream);
            if (ce == cudaSuccess)
            {
                note_kernel ("cfb::cluster_fft_kernel<%d,%d,%d> (cluster of %d CTAs, one pass)", p->logM - 13, fwd ? -1 : 1, ca.logW, 1 << (p->logM - 13));
                return 0;
            }
            if (ce != cudaErrorInvalidConfiguration && ce != cudaErrorNotSupported)
                return fail_cuda (ce, "cluster fft kernel launch");
            (void) cudaGetLastError();
        }
        for (int o = 0; o < outer; ++o)
        {
            const int rc = enqueue_large (p, in + o * in_outer, out + o * out_outer, inner, in_inner, out_inner, direction, ordered, stream);
            if (rc != 0)
                return rc;
        }
        return 0;
    }
    {
        // the kernels move complex pairs (8 bytes) on the ordered side and 16-byte vectors on the unordered side: reject
        // transforms that do not start on such a boundary instead of faulting on the device (the reference asks for buffers
        // aligned to fft_simd_width_bytes, chowdsp_fft.h:131-136)
        const bool fwd = direction == chowdsp::fft::FFT_FORWARD;
        const unsigned a_in = (! ordered && ! fwd) ? 16u : 8u, a_out = (! ordered && fwd) ? 16u : 8u;
        if (misaligned (in, a_in, in_inner, inner, in_outer, outer) || misaligned (out, a_out, out_inner, inner, out_outer, outer))
            return fail (chowdsp::fft::FFT_B200_EINVAL, "every transform must start on an 8-byte boundary (16-byte for unordered spectra): check the base pointers and strides");
        if (window != nullptr && (reinterpret_cast<uintptr_t> (window) & 7u) != 0)
            return fail (chowdsp::fft::FFT_B200_EINVAL, "the window must be 8-byte aligned");
    }
    Tables t;
    // plain, ordered batches of the two largest single-kernel sizes with 16-byte aligned input rows: persistent
    // TMA-pipelined kernel (32 points per thread)
    const bool use_pipe = window == nullptr && pipe_enabled (p->logM, kind_of (p, direction), ordered ? 0 : p->logW)
                          && (outer == 1 || inner == 1) && (reinterpret_cast<uintptr_t> (in) & 15) == 0
                          && ((outer == 1 ? in_inner : in_outer) & 3) == 0;
    // sizes owned by one warp (2^10 points at 32 per thread, 2^9 at 16), forward kinds, input rows the TMA unit can
    // fetch (16-byte aligned): every warp runs its own prefetch pipeline (wpipe_kernel); covers plain batches and
    // overlapping / windowed frames
    const int wpipe_radix = p->logM == 10 ? 32 : 16;
    const long long row_floats = p->is_complex ? 2LL * p->N : p->N;
    const long long frame_stride = inner > 1 ? in_inner : in_outer;
    const bool frames = window != nullptr || ((long long) outer * inner > 1 && frame_stride > 0 && frame_stride < row_floats);
    const bool unord_real_2048 = ! ordered && ! p->is_complex && p->logM == 10 && (long long) outer * inner >= 4096; // throughput batches only
    const bool use_wpipe = ! use_pipe && ((g_wpipe & 1) != 0 || ((g_wpipe & 2) != 0 && frames && (p->logM == 10 || (g_wpipe & 8) != 0)) || ((g_wpipe & 4) != 0 && unord_real_2048)) && has_wpipe (p->logM, wpipe_radix) && direction == chowdsp::fft::FFT_FORWARD
                           && (reinterpret_cast<uintptr_t> (in) & 15) == 0 && (inner == 1 || (in_inner & 3) == 0) && (outer == 1 || (in_outer & 3) == 0);
    const int radix = use_pipe ? 32 : use_wpipe ? wpipe_radix : radix_for (p->logM, p->is_complex != 0);
    const int rc = plan_tables (p, t, radix);
    if (rc != 0)
        return rc;
    if (use_pipe)
    {
        FftArgs pa {};
        pa.in = in;
        pa.out = out;
        pa.in_inner = outer == 1 ? in_inner : in_outer;
        pa.out_inner = outer == 1 ? out_inner : out_outer;
        pa.inner = pa.batch = outer * inner;
        pa.tw = t.tw;
        pa.rtw = t.rtw;
        note_kernel ("cfb::pipe_kernel<%d,%s,%d>", p->logM, kKindNames[kind_of (p, direction)], ordered ? 0 : p->logW);
        const cudaError_t ep = launch_pipe (p->logM, kind_of (p, direction), ordered ? 0 : p->logW, pa, stream);
        if (ep != cudaSuccess)
            return fail_cuda (ep, "pipelined fft kernel launch");
        return 0;
    }
    FftArgs a {};
    a.in = in;
    a.out = out;
    a.in_inner = in_inner;
    a.in_outer = in_outer;
    a.out_inner = out_inner;
    a.out_outer = out_outer;
    a.inner = inner;
    a.batch = outer * inner;
    a.tw = t.tw;
    a.rtw = t.rtw;
    a.pf_ahead = g_pf_ahead;
    if (use_wpipe)
    {
        a.window = window;
        const int kind = kind_of (p, direction);
        const cudaError_t ew = launch_wpipe (p->logM, kind, ordered ? 0 : p->logW, g_wpipe >> 8, a, stream);
        if (ew != cudaSuccess)
            return fail_cuda (ew, "warp-pipelined fft kernel launch");
        note_kernel ("cfb::wpipe_kernel<%d,%d,%s,%d>", p->logM, radix, kKindNames[kind], ordered ? 0 : p->logW);
        return 0;
    }
    // windowed real frames (STFT analysis) go through the frame-gather kernel; plain overlapping frames only when
    // the union-staging variant is selected (it is slower on B200, see stft_kernel)
    const bool fwd_real = ! p->is_complex && direction == chowdsp::fft::FFT_FORWARD;
    const bool union_ok = in_inner > 0 && in_inner <= p->N;
    // overlapping (or windowed) frames of 16-byte aligned signals: persistent kernel, the union of a CTA's frames
    // arrives by TMA while the previous frames are transformed
    if (g_stft_pipe && fwd_real && union_ok && inner > 1 && (in_inner < p->N || window != nullptr) && (in_inner & 3) == 0 && (in_outer & 3) == 0
        && (reinterpret_cast<uintptr_t> (in) & 15) == 0)
    {
        a.window = window;
        const cudaError_t es = launch_stft_pipe (p->logM, ordered ? 0 : p->logW, radix, a, stream);
        if (es == cudaSuccess)
        {
            note_kernel ("cfb::stft_pipe_kernel<%d,%d,%d>", p->logM, radix, ordered ? 0 : p->logW);
            return 0;
        }
        if (es != cudaErrorInvalidConfiguration) // = does not fit in shared memory at this hop: use the kernels below
            return fail_cuda (es, "persistent stft kernel launch");
        (void) cudaGetLastError();
    }
    if (fwd_real && (in_inner & 1) == 0 && (in_outer & 1) == 0
        && (window != nullptr || (g_stft_union && union_ok && in_inner < p->N && inner > 1 && transforms_per_cta (p->logM, radix) > 1)))
    {
        a.window = window;
        a.union_gather = (g_stft_union && union_ok) ? 1 : 0;
        a.vec4 = ((reinterpret_cast<uintptr_t> (in) & 15) == 0 && (in_inner & 3) == 0 && (in_outer & 3) == 0) ? 1 : 0;
        note_kernel ("cfb::stft_kernel<%d,%d,%d,%s>", p->logM, radix, ordered ? 0 : p->logW, a.union_gather ? "union" : "direct");
        const cudaError_t es = launch_stft (p->logM, ordered ? 0 : p->logW, radix, a, stream);
        if (es != cudaSuccess)
            return fail_cuda (es, "stft kernel launch");
        return 0;
    }
    if (window != nullptr)
        return fail (chowdsp::fft::FFT_B200_EINVAL, "windowed transforms need even hop and channel strides");
    {
        // mirrors small_applies() in fft_inst.cu: dense batches of 16- / 32-point transforms
        const int kd = kind_of (p, direction);
        const long long row = 2LL << p->logM;
        const uintptr_t al = ordered ? 7 : 15;
        const bool small = p->logM <= 5 && radix == 16 && fft_small_mode() != 0 && a.inner >= a.batch
                           && a.in_inner == row && a.out_inner == row && (reinterpret_cast<uintptr_t> (a.in) & al) == 0 && (reinterpret_cast<uintptr_t> (a.out) & al) == 0;
        (void) kd;
        note_kernel (small ? "cfb::fft_small_kernel<%d,%d,%s,%d>" : "cfb::fft_kernel<%d,%d,%s,%d>", p->logM, radix, kKindNames[kd], ordered ? 0 : p->logW);
    }
    const cudaError_t e = launch_fft (p->logM, kind_of (p, direction), ordered ? 0 : p->logW, radix, a, stream);
    if (e != cudaSuccess)
        return fail_cuda (e, "fft kernel launch");
    return 0;
}

// Completion of everything enqueued on `stream` so far.  Small drop-in calls (the reference's single-transform loop,
// bench/bench.cpp:92-97) are latency-bound by the blocking synchronise itself, so for them the stream writes a sequence number
// into a word of mapped pinned memory right behind the kernel (cuStreamWriteValue32, a stream memory operation: no extra
// kernel launch) and the host thread spins on that word; anything larger, or a platform without stream memory operations,
// takes cudaStreamSynchronize.  If the word does not arrive within the spin budget the blocking path reports the outcome.
using WriteValue32Fn = int (*) (void* stream, unsigned long long dptr, unsigned value, unsigned flags);
WriteValue32Fn write_value32()
{
    static WriteValue32Fn fn = []() -> WriteValue32Fn
    {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q = cudaDriverEntryPointSymbolNotFound;
        if (cudaGetDriverEntryPoint ("cuStreamWriteValue32", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess)
        {
            (void) cudaGetLastError();
            return nullptr;
        }
        return reinterpret_cast<WriteValue32Fn> (p);
    }();
    return fn;
}
struct SpinFlag
{
    volatile unsigned* host = nullptr;
    unsigned long long dev = 0;
    unsigned seq = 0;
    int device = -1;
    bool broken = false;
    bool ensure()
    {
        int dv = 0;
        if (broken || cudaGetDevice (&dv) != cudaSuccess)
            return false;
        if (host != nullptr && dv == device)
            return true;
        release();
        void *h = nullptr, *d = nullptr;
        if (cudaHostAlloc (&h, 64, cudaHostAllocMapped) != cudaSuccess || cudaHostGetDevicePointer (&d, h, 0) != cudaSuccess)
        {
            (void) cudaGetLastError();
            if (h != nullptr)
                (void) cudaFreeHost (h);
            broken = true;
            return false;
        }
        host = static_cast<volatile unsigned*> (h);
        *host = 0;
        dev = reinterpret_cast<unsigned long long> (d);
        device = dv;
        return true;
    }
    void release()
    {
        if (host != nullptr)
            (void) cudaFreeHost (const_cast<unsigned*> (host));
        host = nullptr;
    }
    ~SpinFlag()
    {
        release();
        (void) cudaGetLastError();
    }
};
thread_local SpinFlag t_spin;
// tuning hook "spin_sync" (environment CHOWDSP_FFT_B200_SPIN_SYNC=0/1 sets the initial value for callers without the hook)
// Default OFF: measured with the compiled caller (tests/c_caller/latency_bench.c, profiles/r02_latency.txt) the stream-written
// word costs 16.5 us per call against 15.1 us for the blocking synchronise -- the stream memory operation is submitted as its
// own command and adds more than the spin saves.
bool g_spin_sync = []
{
    const char* e = getenv ("CHOWDSP_FFT_B200_SPIN_SYNC");
    return e != nullptr && e[0] == '1';
}();

int wait_stream (cudaStream_t stream, bool small_work)
{
    const WriteValue32Fn wv = (small_work && g_spin_sync) ? write_value32() : nullptr;
    if (wv != nullptr && t_spin.ensure())
    {
        const unsigned seq = ++t_spin.seq;
        if (wv (stream, t_spin.dev, seq, 0) == 0)
        {
            const auto t0 = std::chrono::steady_clock::now();
            for (unsigned i = 1;; ++i)
            {
                if (*t_spin.host == seq)
                {
                    std::atomic_thread_fence (std::memory_order_acquire);
                    return 0;
                }
#if defined(__x86_64__) || defined(__i386__)
                __builtin_ia32_pause();
#endif
                if ((i & 255u) == 0 && std::chrono::steady_clock::now() - t0 > std::chrono::microseconds (500))
                    break; // not a small piece of work after all (or a fault): let the blocking synchronise report it
            }
        }
        else
            t_spin.broken = true; // stream memory operations are not available here: stay on the blocking path
    }
    CFB_CUDA (cudaStreamSynchronize (stream));
    return 0;
}

// Host-resident batch: chunked H2D -> kernel -> D2H on two alternating lanes.
int staged_transform (Plan* p, const float* in, float* out, int batch, long long in_stride, long long out_stride, int direction, bool ordered)
{
    const long long nfl = p->is_complex ? 2LL * p->N : p->N;
    if (batch > 1 && (in_stride < nfl || out_stride < nfl))
        return fail (chowdsp::fft::FFT_B200_EINVAL, "host-memory batches need non-overlapping strides >= %lld floats", nfl);
    // rows are copied with their stride (2-D copy) and packed densely on the device
    const size_t row_bytes = (size_t) nfl * sizeof (float);
    int per_chunk = (int) (kChunkBytes / row_bytes);
    if (per_chunk < 1)
        per_chunk = 1;
    int lane = 0;
    for (int b0 = 0; b0 < batch; b0 += per_chunk, lane ^= 1)
    {
        const int nb = batch - b0 < per_chunk ? batch - b0 : per_chunk;
        Staging& s = t_staging;
        int rc = s.ensure (lane, 0, row_bytes * (size_t) nb);
        if (rc == 0)
            rc = s.ensure (lane, 1, row_bytes * (size_t) nb);
        if (rc != 0)
            return rc;
        cudaStream_t st = s.stream[lane];
        if (batch == 1 || in_stride == nfl) // dense rows: one linear copy
            CFB_CUDA (cudaMemcpyAsync (s.buf[lane][0], in + (long long) b0 * nfl, row_bytes * (size_t) nb, cudaMemcpyHostToDevice, st));
        else
            CFB_CUDA (cudaMemcpy2DAsync (s.buf[lane][0], row_bytes, in + (long long) b0 * in_stride, (size_t) in_stride * sizeof (float), row_bytes, (size_t) nb, cudaMemcpyHostToDevice, st));
        rc = enqueue_transform (p, s.buf[lane][0], s.buf[lane][1], 1, nb, 0, nfl, 0, nfl, direction, ordered, st);
        if (rc != 0)
            return rc;
        if (batch == 1 || out_stride == nfl)
            CFB_CUDA (cudaMemcpyAsync (out + (long long) b0 * nfl, s.buf[lane][1], row_bytes * (size_t) nb, cudaMemcpyDeviceToHost, st));
        else
            CFB_CUDA (cudaMemcpy2DAsync (out + (long long) b0 * out_stride, (size_t) out_stride * sizeof (float), s.buf[lane][1], row_bytes, row_bytes, (size_t) nb, cudaMemcpyDeviceToHost, st));
    }
    for (int l = 0; l < 2; ++l)
        if (t_staging.stream[l] != nullptr)
            CFB_CUDA (cudaStreamSynchronize (t_staging.stream[l]));
    return 0;
}

// Host-resident two-level batches (STFT analysis, fft_transform_strided): transform (o, i) reads in + o in_outer + i in_inner.
// Per outer index (channel) the UNIQUE input span ((inner - 1) in_inner + nfl floats) is uploaded once -- not one copy per
// overlapping frame -- in chunks of channels on two alternating lanes (H2D || kernel || D2H); the device-side output is dense.
// `window` (optional) is a device pointer already.
int staged_two_level (Plan* p, const float* in, float* out, int outer, int inner, long long in_outer, long long in_inner, long long out_outer, long long out_inner,
                      int direction, bool ordered, const float* window_dev)
{
    const long long nfl = p->is_complex ? 2LL * p->N : p->N;
    if (in_inner < 0 || out_inner < nfl || (outer > 1 && out_outer < (long long) (inner - 1) * out_inner + nfl))
        return fail (chowdsp::fft::FFT_B200_EINVAL, "host-memory frame batches need in_inner >= 0 and non-overlapping output rows");
    const long long span_in = (long long) (inner - 1) * in_inner + nfl;  // floats per outer index
    const long long span_in_al = (span_in + 3) & ~3LL;                   // device rows stay 16-byte aligned
    if (outer > 1 && in_outer < span_in && in_outer != 0)
        return fail (chowdsp::fft::FFT_B200_EINVAL, "host-memory frame batches need channel strides >= the channel's span");
    const size_t row_out_bytes = (size_t) inner * (size_t) nfl * sizeof (float);
    int per_chunk = (int) (kChunkBytes / (row_out_bytes > (size_t) span_in_al * 4 ? row_out_bytes : (size_t) span_in_al * 4));
    per_chunk = per_chunk < 1 ? 1 : (per_chunk > outer ? outer : per_chunk);
    int lane = 0;
    for (int o0 = 0; o0 < outer; o0 += per_chunk, lane ^= 1)
    {
        const int no = outer - o0 < per_chunk ? outer - o0 : per_chunk;
        Staging& s = t_staging;
        int rc = s.ensure (lane, 0, (size_t) span_in_al * 4 * (size_t) no);
        if (rc == 0)
            rc = s.ensure (lane, 1, row_out_bytes * (size_t) no);
        if (rc != 0)
            return rc;
        cudaStream_t st = s.stream[lane];
        CFB_CUDA (cudaMemcpy2DAsync (s.buf[lane][0], (size_t) span_in_al * 4, in + (long long) o0 * in_outer, (size_t) (in_outer != 0 ? in_outer : span_in) * 4, (size_t) span_in * 4,
                                     (size_t) (in_outer != 0 ? no : 1), cudaMemcpyHostToDevice, st));
        rc = enqueue_transform (p, s.buf[lane][0], s.buf[lane][1], no, inner, in_outer != 0 ? span_in_al : 0, in_inner, (long long) inner * nfl, nfl, direction, ordered, st, window_dev);
        if (rc != 0)
            return rc;
        if (out_inner == nfl && (no == 1 || out_outer == (long long) inner * nfl))
            CFB_CUDA (cudaMemcpyAsync (out + (long long) o0 * out_outer, s.buf[lane][1], row_out_bytes * (size_t) no, cudaMemcpyDeviceToHost, st));
        else if (out_inner == nfl)
            CFB_CUDA (cudaMemcpy2DAsync (out + (long long) o0 * out_outer, (size_t) out_outer * 4, s.buf[lane][1], row_out_bytes, row_out_bytes, (size_t) no, cudaMemcpyDeviceToHost, st));
        else
            for (int o = 0; o < no; ++o)
                CFB_CUDA (cudaMemcpy2DAsync (out + (long long) (o0 + o) * out_outer, (size_t) out_inner * 4, s.buf[lane][1] + (size_t) o * (size_t) inner * (size_t) nfl, (size_t) nfl * 4,
                                             (size_t) nfl * 4, (size_t) inner, cudaMemcpyDeviceToHost, st));
    }
    for (int l = 0; l < 2; ++l)
        if (t_staging.stream[l] != nullptr)
            CFB_CUDA (cudaStreamSynchronize (t_staging.stream[l]));
    return 0;
}

// a window given as a host pointer is uploaded once (blocking, N floats) into the calling thread's window slot
int window_to_device (const float* window, int n, const float*& dev_out)
{
    dev_out = nullptr;
    if (window == nullptr)
        return 0;
    const PtrInfo wi = classify (window);
    if (wi.kind == Mem::Device)
    {
        dev_out = static_cast<const float*> (wi.dev);
        return 0;
    }
    Staging& s = t_staging;
    const int rc = s.ensure (0, 2, (size_t) n * sizeof (float));
    if (rc != 0)
        return rc;
    CFB_CUDA (cudaMemcpy (s.buf[0][2], window, (size_t) n * sizeof (float), cudaMemcpyHostToDevice));
    dev_out = s.buf[0][2];
    return 0;
}

// shared front end of fft_transform / fft_transform_unordered / fft_transform_batched
int transform_any (void* setup, const float* in, float* out, int batch, long long in_stride, long long out_stride, int direction, bool ordered, cudaStream_t stream, bool force_sync)
{
    Plan* p = as_plan (setup);
    if (p == nullptr)
        return chowdsp::fft::FFT_B200_EINVAL;
    if (in == nullptr || out == nullptr || batch < 0)
        return fail (chowdsp::fft::FFT_B200_EINVAL, "null buffer or negative batch");
    if (batch == 0)
        return 0;
    const long long nfl = p->is_complex ? 2LL * p->N : p->N;
    const PtrInfo pi = classify (in), po = classify (out);
    const bool in_dev = pi.kind == Mem::Device, out_dev = po.kind == Mem::Device;
    if (in_dev != out_dev)
        return fail (chowdsp::fft::FFT_B200_EINVAL, "input and output must both be device memory or both be host memory");
    if (in_dev)
    {
        const int rc = enqueue_transform (p, static_cast<const float*> (pi.dev), static_cast<float*> (const_cast<void*> (po.dev)), 1, batch, 0, in_stride, 0, out_stride, direction, ordered, stream);
        if (rc != 0)
            return rc;
        if (force_sync)
            return wait_stream (stream, (long long) batch * nfl <= 65536);
        return 0;
    }
    // host memory
    const size_t span_in = (size_t) ((batch - 1) * in_stride + nfl) * sizeof (float);
    const size_t span_out = (size_t) ((batch - 1) * out_stride + nfl) * sizeof (float);
    if (pi.kind == Mem::Pinned && po.kind == Mem::Pinned && span_in <= kZeroCopyBytes && span_out <= kZeroCopyBytes)
    {
        // zero-copy: the kernel reads / writes the mapped host buffers over PCIe, one launch, one sync
        cudaStream_t st = cudaStreamPerThread;
        const int rc = enqueue_transform (p, static_cast<const float*> (pi.dev), static_cast<float*> (const_cast<void*> (po.dev)), 1, batch, 0, in_stride, 0, out_stride, direction, ordered, st);
        if (rc != 0)
            return rc;
        return wait_stream (st, true);
    }
    return staged_transform (p, in, out, batch, in_stride, out_stride, direction, ordered);
}

// elementwise front end (convolve / accumulate): operands a, b (read) and ab (read-modify-write)
int elementwise_any (Plan* p, bool convolve, const float* a, const float* b, float* ab, int batch, long long a_stride, long long b_stride, long long ab_stride, long long nfl, float scaling, cudaStream_t stream, bool force_sync)
{
    if (a == nullptr || b == nullptr || ab == nullptr || batch < 0)
        return fail (chowdsp::fft::FFT_B200_EINVAL, "null buffer or negative batch");
    if (batch == 0 || nfl == 0)
        return 0;
    // both kernels move float4 vectors (4 re | 4 im lanes): operands start on 16-byte boundaries, strides are multiples of 4
    if (misaligned (a, 16, a_stride, batch) || misaligned (b, 16, b_stride, batch) || misaligned (ab, 16, ab_stride, batch))
        return fail (chowdsp::fft::FFT_B200_EINVAL, "%s: operands must be 16-byte aligned with strides that are multiples of 4 floats", convolve ? "convolve" : "accumulate");
    const PtrInfo ia = classify (a), ib = classify (b), iab = classify (ab);
    const bool all_dev = ia.kind == Mem::Device && ib.kind == Mem::Device && iab.kind == Mem::Device;
    const bool any_dev = ia.kind == Mem::Device || ib.kind == Mem::Device || iab.kind == Mem::Device;
    if (any_dev && ! all_dev)
        return fail (chowdsp::fft::FFT_B200_EINVAL, "operands must all be device memory or all be host memory");
    auto run = [&] (const float* da, const float* db, float* dab, long long sa, long long sb, long long sab, cudaStream_t st) -> int
    {
        const cudaError_t e = convolve
                                  ? launch_convolve (da, db, dab, sa, sb, sab, (int) nfl, batch, p->logW, ! p->is_complex, scaling, st)
                                  : launch_accumulate (da, db, dab, nfl, st);
        return e == cudaSuccess ? 0 : fail_cuda (e, "elementwise kernel launch");
    };
    if (all_dev)
    {
        const int rc = run (static_cast<const float*> (ia.dev), static_cast<const float*> (ib.dev), static_cast<float*> (const_cast<void*> (iab.dev)), a_stride, b_stride, ab_stride, stream);
        if (rc != 0)
            return rc;
        if (force_sync)
            return wait_stream (stream, (long long) batch * nfl <= 65536);
        return 0;
    }
    const size_t bytes_a = (size_t) ((batch - 1) * a_stride + nfl) * sizeof (float);
    const size_t bytes_b = (size_t) ((batch - 1) * b_stride + nfl) * sizeof (float);
    const size_t bytes_ab = (size_t) ((batch - 1) * ab_stride + nfl) * sizeof (float);
    const bool all_pinned = ia.kind == Mem::Pinned && ib.kind == Mem::Pinned && iab.kind == Mem::Pinned;
    if (all_pinned && bytes_a <= kZeroCopyBytes && bytes_b <= kZeroCopyBytes && bytes_ab <= kZeroCopyBytes)
    {
        cudaStream_t st = cudaStreamPerThread;
        const int rc = run (static_cast<const float*> (ia.dev), static_cast<const float*> (ib.dev), static_cast<float*> (const_cast<void*> (iab.dev)), a_stride, b_stride, ab_stride, st);
        if (rc != 0)
            return rc;
        return wait_stream (st, true);
    }
    // staged: whole operands through lane 0 (aliasing between host operands is preserved by copying
    // each one separately and writing only ab back)
    Staging& s = t_staging;
    int rc = s.ensure (0, 0, bytes_a);
    if (rc == 0)
        rc = s.ensure (0, 1, bytes_b);
    if (rc == 0)
        rc = s.ensure (0, 2, bytes_ab);
    if (rc != 0)
        return rc;
    cudaStream_t st = s.stream[0];
    CFB_CUDA (cudaMemcpyAsync (s.buf[0][0], a, bytes_a, cudaMemcpyHostToDevice, st));
    CFB_CUDA (cudaMemcpyAsync (s.buf[0][1], b, bytes_b, cudaMemcpyHostToDevice, st));
    CFB_CUDA (cudaMemcpyAsync (s.buf[0][2], ab, bytes_ab, cudaMemcpyHostToDevice, st));
    rc = run (s.buf[0][0], s.buf[0][1], s.buf[0][2], a_stride, b_stride, ab_stride, st);
    if (rc != 0)
        return rc;
    CFB_CUDA (cudaMemcpyAsync (ab, s.buf[0][2], bytes_ab, cudaMemcpyDeviceToHost, st));
    CFB_CUDA (cudaStreamSynchronize (st));
    return 0;
}

} // namespace

// ------------------------------------------------------------------------------------------------
// exported C ABI
// ------------------------------------------------------------------------------------------------
extern "C"
{
namespace chowdsp::fft
{
CFB_API size_t fft_bytes_required (int N, fft_transform_t transform, bool)
{
    const size_t ref = reference_bytes (N > 0 ? N : 0, transform == FFT_COMPLEX);
    return ref > sizeof (Plan) + 64 ? ref : sizeof (Plan) + 64;
}

CFB_API void* fft_new_setup_preallocated (int N, fft_transform_t transform, void* data, bool use_avx_if_available)
{
    if (data == nullptr)
    {
        fail (FFT_B200_EINVAL, "fft_new_setup_preallocated: null data block");
        return nullptr;
    }
    const bool is_complex = transform == FFT_COMPLEX;
    const int W = choose_width (N, is_complex, use_avx_if_available);
    const bool pow2 = N > 0 && (N & (N - 1)) == 0;
    const int logM = (W == 0 || ! pow2) ? -1 : ilog2i (N) - (is_complex ? 0 : 1);
    const int M = is_complex ? N : N / 2;
    const bool size_ok = W != 0 && (pow2 ? (logM >= kMinLogM && logM <= kMaxLargeLog - (is_complex ? 0 : 1)) : M <= kMixedMaxM);
    if (! size_ok)
    {
        fail (FFT_B200_EINVAL, "unsupported FFT size N=%d (%s): need %s, as a power of two up to 2^28 or as 2^a 3^b 5^c up to %d",
              N, is_complex ? "complex" : "real", is_complex ? "a multiple of 16" : "a multiple of 32", is_complex ? kMixedMaxM : 2 * kMixedMaxM);
        return nullptr;
    }
    if (! device_available())
    {
        fail (FFT_B200_ENODEVICE, "no usable CUDA device: chowdsp_fft_b200 has no CPU fallback");
        return nullptr;
    }
    auto* p = reinterpret_cast<Plan*> ((reinterpret_cast<uintptr_t> (data) + 7) & ~static_cast<uintptr_t> (7));
    std::memset (p, 0, sizeof (Plan));
    p->N = N;
    p->is_complex = is_complex ? 1 : 0;
    p->logM = logM;
    p->mixed = pow2 ? 0 : 1;
    p->M = M;
    p->logW = W == 8 ? 3 : 2;
    p->owns_memory = 0;
    p->magic = kMagic;
    if (cudaGetDevice (&p->home_device) != cudaSuccess)
    {
        fail (FFT_B200_ECUDA, "cudaGetDevice failed");
        return nullptr;
    }
    if (preload_tables (p) != 0)
    {
        p->magic = 0;
        return nullptr;
    }
    return p;
}

CFB_API void* fft_new_setup (int N, fft_transform_t transform, bool use_avx_if_available)
{
    CFB_TRACE ("fft_new_setup");
    void* block = std::malloc (sizeof (Plan) + 64);
    if (block == nullptr)
        return nullptr;
    void* p = fft_new_setup_preallocated (N, transform, block, use_avx_if_available);
    if (p == nullptr)
    {
        std::free (block);
        return nullptr;
    }
    auto* plan = static_cast<Plan*> (p);
    plan->owns_memory = 1;
    // remember the malloc'd base right behind the plan (the block has 64 spare bytes)
    std::memcpy (reinterpret_cast<char*> (plan) + sizeof (Plan), &block, sizeof (void*));
    return p;
}

CFB_API void fft_destroy_setup (void* setup)
{
    if (setup == nullptr)
        return;
    Plan* p = as_plan (setup);
    if (p == nullptr)
        return;
    p->magic = 0;
    if (p->owns_memory)
    {
        void* block = nullptr;
        std::memcpy (&block, reinterpret_cast<char*> (p) + sizeof (Plan), sizeof (void*));
        std::free (block);
    }
}

CFB_API int fft_simd_width_bytes (void* setup)
{
    Plan* p = as_plan (setup);
    return p == nullptr ? 0 : (p->logW == 3 ? 32 : 16);
}

CFB_API void fft_transform (void* setup, const float* input, float* output, float*, fft_direction_t direction)
{
    CFB_TRACE ("fft_transform");
    const Plan* p = static_cast<const Plan*> (setup);
    const long long nfl = (p != nullptr && p->magic == kMagic) ? (p->is_complex ? 2LL * p->N : p->N) : 0;
    (void) transform_any (setup, input, output, 1, nfl, nfl, direction, true, cudaStreamPerThread, true);
}

CFB_API void fft_transform_unordered (void* setup, const float* input, float* output, float*, fft_direction_t direction)
{
    CFB_TRACE ("fft_transform_unordered");
    const Plan* p = static_cast<const Plan*> (setup);
    const long long nfl = (p != nullptr && p->magic == kMagic) ? (p->is_complex ? 2LL * p->N : p->N) : 0;
    (void) transform_any (setup, input, output, 1, nfl, nfl, direction, false, cudaStreamPerThread, true);
}

CFB_API void fft_convolve_unordered (void* setup, const float* a, const float* b, float* ab, float scaling)
{
    CFB_TRACE ("fft_convolve_unordered");
    Plan* p = as_plan (setup);
    if (p == nullptr)
        return;
    const long long nfl = p->is_complex ? 2LL * p->N : p->N;
    (void) elementwise_any (p, true, a, b, ab, 1, nfl, nfl, nfl, nfl, scaling, cudaStreamPerThread, true);
}

CFB_API void fft_accumulate (void* setup, const float* a, const float* b, float* ab, int N)
{
    CFB_TRACE ("fft_accumulate");
    Plan* p = as_plan (setup);
    if (p == nullptr)
        return;
    if (N < 0 || N % 8 != 0)
    {
        fail (FFT_B200_EINVAL, "fft_accumulate: N=%d must be a non-negative multiple of 8", N);
        return;
    }
    (void) elementwise_any (p, false, a, b, ab, 1, N, N, N, N, 0.f, cudaStreamPerThread, true);
}

CFB_API void* aligned_malloc (size_t nb_bytes)
{
    void* p = nullptr;
    HostBlock blk { nb_bytes > 0 ? nb_bytes : 1, false, nullptr };
    if (device_available())
    {
        if (cudaHostAlloc (&p, blk.bytes, cudaHostAllocPortable | cudaHostAllocMapped) == cudaSuccess
            && cudaHostGetDevicePointer (&blk.dev, p, 0) == cudaSuccess)
            blk.pinned = true;
        else
        {
            (void) cudaGetLastError();
            if (p != nullptr)
                (void) cudaFreeHost (p);
            p = nullptr;
        }
    }
    if (p == nullptr && posix_memalign (&p, 64, blk.bytes) != 0)
        return nullptr;
    std::lock_guard<std::mutex> lock (g_alloc_mutex);
    g_allocs[reinterpret_cast<uintptr_t> (p)] = blk;
    return p;
}

CFB_API void aligned_free (void* p)
{
    if (p == nullptr)
        return;
    bool pinned = false, known = false;
    {
        std::lock_guard<std::mutex> lock (g_alloc_mutex);
        auto it = g_allocs.find (reinterpret_cast<uintptr_t> (p));
        if (it != g_allocs.end())
        {
            pinned = it->second.pinned;
            known = true;
            g_allocs.erase (it);
            g_alloc_generation.fetch_add (1, std::memory_order_acq_rel); // per-thread range caches forget the block
        }
    }
    if (! known)
    {
        fail (FFT_B200_EINVAL, "aligned_free: %p was not returned by aligned_malloc", p);
        return;
    }
    if (pinned)
        cudaFreeHost (p);
    else
        std::free (p);
}

// ---- extensions (chowdsp_fft_b200.h) -----------------------------------------------------------
CFB_API int fft_transform_batched (void* setup, const float* input, float* output, int batch, long long in_stride, long long out_stride, fft_direction_t direction, int ordered, void* stream)
{
    CFB_TRACE ("fft_transform_batched");
    return transform_any (setup, input, output, batch, in_stride, out_stride, direction, ordered != 0, static_cast<cudaStream_t> (stream), false);
}

CFB_API int fft_transform_strided (void* setup, const float* input, float* output, int outer, int inner, long long in_outer, long long in_inner, long long out_outer, long long out_inner, fft_direction_t direction, int ordered, void* stream)
{
    CFB_TRACE ("fft_transform_strided");
    Plan* p = as_plan (setup);
    if (p == nullptr)
        return FFT_B200_EINVAL;
    if (input == nullptr || output == nullptr || outer < 0 || inner < 0 || (long long) outer * inner > 0x7fffffffLL)
        return fail (FFT_B200_EINVAL, "fft_transform_strided: bad arguments");
    if (outer == 0 || inner == 0)
        return 0;
    const PtrInfo pi = classify (input), po = classify (output);
    if ((pi.kind == Mem::Device) != (po.kind == Mem::Device))
        return fail (FFT_B200_EINVAL, "fft_transform_strided: input and output must both be device memory or both be host memory");
    if (pi.kind != Mem::Device) // host buffers: synchronous, the unique input span of every outer index is uploaded once
        return staged_two_level (p, input, output, outer, inner, in_outer, in_inner, out_outer, out_inner, direction, ordered != 0, nullptr);
    return enqueue_transform (p, input, output, outer, inner, in_outer, in_inner, out_outer, out_inner, direction, ordered != 0, static_cast<cudaStream_t> (stream));
}

CFB_API int fft_stft_forward (void* setup, const float* signal, float* spectra, int channels, int frames, long long channel_stride, long long hop, long long out_channel_stride, long long out_frame_stride, const float* window, int ordered, void* stream)
{
    CFB_TRACE ("fft_stft_forward");
    Plan* p = as_plan (setup);
    if (p == nullptr)
        return FFT_B200_EINVAL;
    if (p->is_complex)
        return fail (FFT_B200_EINVAL, "fft_stft_forward needs a REAL plan");
    if (signal == nullptr || spectra == nullptr || channels < 0 || frames < 0 || hop <= 0 || (long long) channels * frames > 0x7fffffffLL)
        return fail (FFT_B200_EINVAL, "fft_stft_forward: bad arguments");
    if (channels == 0 || frames == 0)
        return 0;
    const PtrInfo si = classify (signal), so = classify (spectra);
    if ((si.kind == Mem::Device) != (so.kind == Mem::Device))
        return fail (FFT_B200_EINVAL, "fft_stft_forward: signal and spectra must both be device memory or both be host memory");
    if (si.kind != Mem::Device)
    {
        // host audio (the reference API is host-pointer only, chowdsp_fft.h:138): synchronous; every channel's samples cross
        // PCIe once, the frame overlap is re-read on the device
        const float* wdev = nullptr;
        const int rc = window_to_device (window, p->N, wdev);
        return rc != 0 ? rc : staged_two_level (p, signal, spectra, channels, frames, channel_stride, hop, out_channel_stride, out_frame_stride, FFT_FORWARD, ordered != 0, wdev);
    }
    if (window != nullptr && classify (window).kind != Mem::Device)
        return fail (FFT_B200_EINVAL, "fft_stft_forward: a device signal needs a device window");
    return enqueue_transform (p, signal, spectra, channels, frames, channel_stride, hop, out_channel_stride, out_frame_stride, FFT_FORWARD, ordered != 0, static_cast<cudaStream_t> (stream), window);
}

namespace
{
// overlap-add synthesis on device buffers (arguments validated by the caller)
int istft_enqueue (Plan* p, const float* spectra, float* signal, int channels, int frames, long long spec_channel_stride, long long spec_frame_stride, long long channel_stride, long long hop, const float* window, float scale, int ordered, cudaStream_t stream)
{
    Tables t;
    const int radix = radix_for (p->logM, false);
    const int rc = plan_tables (p, t, radix);
    if (rc != 0)
        return rc;
    // sizes one warp owns, ordered spectra, hop = N/2, N/4 or N/8: every warp is its own pipeline and the overlap-add
    // stays in registers (wistft_kernel).  Items = (channel, segment); pick the segment count that minimises
    // (items per resident warp, rounded up) x (frames per segment + halo).
    {
        const int wr = p->logM == 10 ? 32 : 16;
        const bool hop_ok = hop * 2 == p->N || hop * 4 == p->N || hop * 8 == p->N;
        // (the 2^9-point size only with bit 1 of the hook: ristft_kernel measured 3..6 % faster there, profiles/r02_stft_sizes.txt)
        if ((g_wistft & 1) != 0 && (p->logM == 10 || (g_wistft & 2) != 0) && ordered != 0 && has_wpipe (p->logM, wr) && hop_ok && (spec_frame_stride & 3) == 0 && (spec_channel_stride & 3) == 0
            && (reinterpret_cast<uintptr_t> (spectra) & 15) == 0 && (channel_stride & 1) == 0 && (reinterpret_cast<uintptr_t> (signal) & 7) == 0)
        {
            Tables wt;
            const int wrc = plan_tables (p, wt, wr);
            if (wrc != 0)
                return wrc;
            const int warps = (g_wistft >> 8) > 0 && (g_wistft >> 8) < wistft_warps (p->logM) ? (g_wistft >> 8) : wistft_warps (p->logM);
            const long long total_warps = (long long) device_sm_count() * warps;
            const int halo = (int) (p->N / hop) - 1;
            int nseg = 1, seg_frames = frames;
            long long best = -1;
            for (int cand = 1; cand <= 256 && cand <= (frames + 7) / 8; ++cand)
            {
                const int sf = (frames + cand - 1) / cand;
                const int ns = (frames + sf - 1) / sf;
                const long long items = (long long) channels * ns;
                const long long cost = ((items + total_warps - 1) / total_warps) * (sf + (ns > 1 ? halo : 0));
                if (best < 0 || cost < best)
                {
                    best = cost;
                    nseg = ns;
                    seg_frames = sf;
                }
            }
            FftArgs wa {};
            wa.in = spectra;
            wa.out = signal;
            wa.in_inner = spec_frame_stride;
            wa.in_outer = spec_channel_stride;
            wa.out_inner = hop;
            wa.out_outer = channel_stride;
            wa.inner = frames;
            wa.batch = channels * frames;
            wa.tw = wt.tw;
            wa.rtw = wt.rtw;
            wa.window = window;
            wa.seg_frames = seg_frames;
            wa.nseg = nseg;
            wa.scale = scale;
            note_kernel ("cfb::wistft_kernel<%d,%d,%d>", p->logM, wr, (int) (hop / 64));
            const cudaError_t we = launch_wistft (p->logM, (int) (hop / 64), warps, wa, stream);
            if (we != cudaSuccess)
                return fail_cuda (we, "warp-pipelined istft kernel launch");
            return 0;
        }
    }
    // N = 128 .. 8192, hop = N/2, N/4 or N/8, any layout: the overlap-add stays in the registers of the transform's own
    // thread group (ristft_kernel).  Items = (channel, segment); segment count as above, for the resident transform slots.
    {
        const bool hop_ok = hop * 2 == p->N || hop * 4 == p->N || hop * 8 == p->N;
        const uintptr_t spec_al = ordered != 0 ? 7 : 15;
        if (g_ristft != 0 && p->logM >= 6 && p->logM <= 12 && hop_ok && (spec_frame_stride & (ordered != 0 ? 1 : 3)) == 0 && (spec_channel_stride & (ordered != 0 ? 1 : 3)) == 0
            && (reinterpret_cast<uintptr_t> (spectra) & spec_al) == 0 && (channel_stride & 1) == 0 && (reinterpret_cast<uintptr_t> (signal) & 7) == 0
            && (window == nullptr || (reinterpret_cast<uintptr_t> (window) & 7) == 0))
        {
            Tables rt;
            const int rrc = plan_tables (p, rt, 16);
            if (rrc != 0)
                return rrc;
            const int per_cta16 = transforms_per_cta (p->logM, 16);
            const long long slots = (long long) device_sm_count() * 2 * per_cta16; // two resident CTAs per SM (128 registers)
            const int halo = (int) (p->N / hop) - 1;
            int nseg = 1, seg_frames = frames;
            long long best = -1;
            for (int cand = 1; cand <= 256 && cand <= (frames + 7) / 8; ++cand)
            {
                const int sf = (frames + cand - 1) / cand;
                const int ns = (frames + sf - 1) / sf;
                const long long items = (long long) channels * ns;
                const long long cost = ((items + slots - 1) / slots) * (sf + (ns > 1 ? halo : 0));
                if (best < 0 || cost < best)
                {
                    best = cost;
                    nseg = ns;
                    seg_frames = sf;
                }
            }
            FftArgs ra {};
            ra.in = spectra;
            ra.out = signal;
            ra.in_inner = spec_frame_stride;
            ra.in_outer = spec_channel_stride;
            ra.out_inner = hop;
            ra.out_outer = channel_stride;
            ra.inner = frames;
            ra.batch = channels * frames;
            ra.tw = rt.tw;
            ra.rtw = rt.rtw;
            ra.window = window;
            ra.seg_frames = seg_frames;
            ra.nseg = nseg;
            ra.scale = scale;
            const int hq = (int) (hop * 16 / p->N); // hop / (2 T), T = N / 32: 8, 4 or 2
            const cudaError_t re = launch_ristft (p->logM, hq, ordered != 0 ? 0 : p->logW, ra, stream);
            if (re == cudaSuccess)
            {
                note_kernel ("cfb::ristft_kernel<%d,%d,%d>", p->logM, hq, ordered != 0 ? 0 : p->logW);
                return 0;
            }
            if (re != cudaErrorInvalidConfiguration)
                return fail_cuda (re, "register overlap-add istft kernel launch");
            (void) cudaGetLastError();
        }
    }
    // segmentation: a CTA per (channel, segment of frames).  More segments fill the last wave of CTAs better but
    // every segment after a channel's first recomputes a halo of ceil (N / hop) - 1 frames; segments keep at
    // least 8 groups of frames.  Pick the count with the best (wave occupancy) x (useful fraction of the frames).
    const int per_cta = transforms_per_cta (p->logM, radix);
    const int groups = (frames + per_cta - 1) / per_cta;
    const int halo = (int) ((p->N + hop - 1) / hop) - 1;
    const long long slots = 148LL * (radix == 32 ? 2 : 4);
    int nseg = 1, seg_groups = groups;
    double best = -1.0;
    for (int cand = 1; cand <= 64 && cand <= (groups + 7) / 8; ++cand)
    {
        const int sg = (groups + cand - 1) / cand;
        const int ns = (groups + sg - 1) / sg;
        const long long ctas = (long long) channels * ns;
        const double waves = (double) ((ctas + slots - 1) / slots);
        const double occupancy = (double) ctas / (waves * (double) slots);
        const double useful = (double) frames / ((double) frames + (double) (ns - 1) * halo);
        if (occupancy * useful > best * 1.02) // prefer fewer segments unless clearly better
        {
            best = occupancy * useful;
            nseg = ns;
            seg_groups = sg;
        }
    }
    FftArgs a {};
    a.in = spectra;
    a.out = signal;
    a.in_inner = spec_frame_stride;
    a.in_outer = spec_channel_stride;
    a.out_inner = hop;
    a.out_outer = channel_stride;
    a.inner = frames;
    a.batch = channels * frames;
    a.tw = t.tw;
    a.rtw = t.rtw;
    a.window = window;
    a.seg_frames = seg_groups * per_cta;
    a.nseg = nseg;
    a.scale = scale;
    a.vec4 = ((hop & 3) == 0 && (channel_stride & 3) == 0 && (reinterpret_cast<uintptr_t> (signal) & 15) == 0) ? 1 : 0;
    note_kernel ("cfb::istft_kernel<%d,%d,%d>", p->logM, radix, ordered != 0 ? 0 : p->logW);
    const cudaError_t e = launch_istft (p->logM, ordered != 0 ? 0 : p->logW, radix, a, stream);
    if (e != cudaSuccess)
        return fail_cuda (e, "istft kernel launch");
    return 0;
}
} // namespace

CFB_API int fft_istft_overlap_add (void* setup, const float* spectra, float* signal, int channels, int frames, long long spec_channel_stride, long long spec_frame_stride, long long channel_stride, long long hop, const float* window, float scale, int ordered, void* stream)
{
    CFB_TRACE ("fft_istft_overlap_add");
    Plan* p = as_plan (setup);
    if (p == nullptr)
        return FFT_B200_EINVAL;
    if (p->is_complex || p->mixed || p->logM > 13)
        return fail (FFT_B200_EINVAL, "fft_istft_overlap_add needs a REAL power-of-two plan with N <= 16384 (frame buffers + carried tails must fit in shared memory)");
    if (spectra == nullptr || signal == nullptr || channels < 0 || frames < 0 || hop <= 0 || hop > p->N || (long long) channels * frames > 0x7fffffffLL)
        return fail (FFT_B200_EINVAL, "fft_istft_overlap_add: bad arguments (0 < hop <= N)");
    if (misaligned (spectra, ordered != 0 ? 8 : 16, spec_frame_stride, frames, spec_channel_stride, channels))
        return fail (FFT_B200_EINVAL, "fft_istft_overlap_add: every spectrum frame must start on an 8-byte boundary (16-byte for unordered spectra): check the base pointer and strides");
    if (window != nullptr && misaligned (window, 8))
        return fail (FFT_B200_EINVAL, "fft_istft_overlap_add: the window must be 8-byte aligned");
    if (misaligned (signal, 4))
        return fail (FFT_B200_EINVAL, "fft_istft_overlap_add: the signal must be 4-byte aligned");
    if (channels == 0 || frames == 0)
        return 0;
    const PtrInfo si = classify (spectra), so = classify (signal);
    if ((si.kind == Mem::Device) != (so.kind == Mem::Device))
        return fail (FFT_B200_EINVAL, "fft_istft_overlap_add: spectra and signal must both be device memory or both be host memory");
    if (si.kind != Mem::Device)
    {
        // host buffers: synchronous; chunks of channels on two alternating lanes (H2D spectra || kernel || D2H signal)
        const float* wdev = nullptr;
        int rc = window_to_device (window, p->N, wdev);
        if (rc != 0)
            return rc;
        if (spec_frame_stride < p->N || (channels > 1 && spec_channel_stride < (long long) (frames - 1) * spec_frame_stride + p->N))
            return fail (FFT_B200_EINVAL, "fft_istft_overlap_add: host spectra need non-overlapping frames");
        const long long samples = (long long) (frames - 1) * hop + p->N, samples_al = (samples + 3) & ~3LL;
        const size_t spec_bytes = (size_t) frames * (size_t) p->N * sizeof (float);
        int per_chunk = (int) (kChunkBytes / spec_bytes);
        per_chunk = per_chunk < 1 ? 1 : (per_chunk > channels ? channels : per_chunk);
        int lane = 0;
        for (int c0 = 0; c0 < channels; c0 += per_chunk, lane ^= 1)
        {
            const int nc = channels - c0 < per_chunk ? channels - c0 : per_chunk;
            Staging& sg = t_staging;
            rc = sg.ensure (lane, 0, spec_bytes * (size_t) nc);
            if (rc == 0)
                rc = sg.ensure (lane, 1, (size_t) samples_al * 4 * (size_t) nc);
            if (rc != 0)
                return rc;
            cudaStream_t st = sg.stream[lane];
            for (int c = 0; c < nc; ++c) // frames packed densely on the device
                CFB_CUDA (cudaMemcpy2DAsync (sg.buf[lane][0] + (size_t) c * (size_t) frames * (size_t) p->N, (size_t) p->N * 4, spectra + (long long) (c0 + c) * spec_channel_stride,
                                             (size_t) spec_frame_stride * 4, (size_t) p->N * 4, (size_t) frames, cudaMemcpyHostToDevice, st));
            rc = istft_enqueue (p, sg.buf[lane][0], sg.buf[lane][1], nc, frames, (long long) frames * p->N, p->N, samples_al, hop, wdev, scale, ordered, st);
            if (rc != 0)
                return rc;
            CFB_CUDA (cudaMemcpy2DAsync (signal + (long long) c0 * channel_stride, (size_t) (nc > 1 ? channel_stride : samples) * 4, sg.buf[lane][1], (size_t) samples_al * 4, (size_t) samples * 4,
                                         (size_t) nc, cudaMemcpyDeviceToHost, st));
        }
        for (int l = 0; l < 2; ++l)
            if (t_staging.stream[l] != nullptr)
                CFB_CUDA (cudaStreamSynchronize (t_staging.stream[l]));
        return 0;
    }
    if (window != nullptr && classify (window).kind != Mem::Device)
        return fail (FFT_B200_EINVAL, "fft_istft_overlap_add: device spectra need a device window");
    return istft_enqueue (p, spectra, signal, channels, frames, spec_channel_stride, spec_frame_stride, channel_stride, hop, window, scale, ordered, static_cast<cudaStream_t> (stream));
}

// ---- JUCE-convention wrappers (reference chowdsp_fft_juce/chowdsp_fft_juce.cpp:32-86), batched ----
namespace
{
int juce_launch (Plan* p, int kind, const float* in, float* out, int batch, long long in_stride, long long out_stride, cudaStream_t stream)
{
    if (p->mixed || p->logM > kMaxLogM)
        return fail (FFT_B200_EINVAL, "the JUCE-convention entry points need a single-kernel power-of-two plan (N <= 16384 complex, 32768 real)");
    if (misaligned (in, 8, in_stride, batch) || misaligned (out, 8, out_stride, batch))
        return fail (FFT_B200_EINVAL, "the JUCE-convention entry points need 8-byte aligned buffers and even strides");
    if (batch == 0)
        return 0;
    if (classify (in).kind != Mem::Device || classify (out).kind != Mem::Device)
        return fail (FFT_B200_EINVAL, "the JUCE-convention entry points need device pointers");
    Tables t;
    const int radix = radix_for (p->logM, p->is_complex != 0);
    const int rc = plan_tables (p, t, radix);
    if (rc != 0)
        return rc;
    FftArgs a {};
    a.in = in;
    a.out = out;
    a.in_inner = in_stride;
    a.out_inner = out_stride;
    a.inner = a.batch = batch;
    a.tw = t.tw;
    a.rtw = t.rtw;
    note_kernel ("cfb::fft_kernel_juce<%d,%d,%s>", p->logM, radix, kKindNames[kind]);
    const cudaError_t e = launch_fft_juce (p->logM, kind, radix, a, stream);
    return e == cudaSuccess ? 0 : fail_cuda (e, "JUCE-convention kernel launch");
}
} // namespace

CFB_API int fft_juce_perform_batched (void* setup, const float* input, float* output, int batch, long long in_stride, long long out_stride, int inverse, void* stream)
{
    CFB_TRACE ("fft_juce_perform_batched");
    Plan* p = as_plan (setup);
    if (p == nullptr)
        return FFT_B200_EINVAL;
    if (! p->is_complex || input == nullptr || output == nullptr || batch < 0)
        return fail (FFT_B200_EINVAL, "fft_juce_perform_batched needs a COMPLEX plan and non-null buffers");
    if (! inverse) // forward: the conventions coincide with fft_transform
        return transform_any (setup, input, output, batch, in_stride, out_stride, FFT_FORWARD, true, static_cast<cudaStream_t> (stream), false);
    return juce_launch (p, C2C_BWD, input, output, batch, in_stride, out_stride, static_cast<cudaStream_t> (stream));
}

CFB_API int fft_juce_real_forward_batched (void* setup, float* inout, int batch, long long stride, int ignore_negative_freqs, void* stream)
{
    CFB_TRACE ("fft_juce_real_forward_batched");
    Plan* p = as_plan (setup);
    if (p == nullptr)
        return FFT_B200_EINVAL;
    if (p->is_complex || inout == nullptr || batch < 0 || (batch > 1 && stride < (ignore_negative_freqs ? p->N + 2 : 2LL * p->N)))
        return fail (FFT_B200_EINVAL, "fft_juce_real_forward_batched needs a REAL plan and rows of at least %s floats", ignore_negative_freqs ? "N + 2" : "2 N");
    int rc = juce_launch (p, R2C, inout, inout, batch, stride, stride, static_cast<cudaStream_t> (stream));
    if (rc != 0 || ignore_negative_freqs || batch == 0)
        return rc;
    const cudaError_t e = launch_juce_mirror (inout, stride, p->N / 2, batch, static_cast<cudaStream_t> (stream));
    return e == cudaSuccess ? 0 : fail_cuda (e, "negative-frequency mirror launch");
}

CFB_API int fft_juce_real_inverse_batched (void* setup, float* inout, int batch, long long stride, void* stream)
{
    CFB_TRACE ("fft_juce_real_inverse_batched");
    Plan* p = as_plan (setup);
    if (p == nullptr)
        return FFT_B200_EINVAL;
    if (p->is_complex || inout == nullptr || batch < 0 || (batch > 1 && stride < p->N + 2))
        return fail (FFT_B200_EINVAL, "fft_juce_real_inverse_batched needs a REAL plan and rows of at least N + 2 floats");
    return juce_launch (p, C2R, inout, inout, batch, stride, stride, static_cast<cudaStream_t> (stream));
}

CFB_API int fft_convolve_unordered_batched (void* setup, const float* a, const float* b, float* ab, int batch, long long a_stride, long long b_stride, long long ab_stride, float scaling, void* stream)
{
    CFB_TRACE ("fft_convolve_unordered_batched");
    Plan* p = as_plan (setup);
    if (p == nullptr)
        return FFT_B200_EINVAL;
    const long long nfl = p->is_complex ? 2LL * p->N : p->N;
    return elementwise_any (p, true, a, b, ab, batch, a_stride, b_stride, ab_stride, nfl, scaling, static_cast<cudaStream_t> (stream), false);
}

CFB_API int fft_partitioned_convolve_step (void* setup, const float* windows, long long window_stride, const float* ir, long long ir_channel_stride, float* fdl, long long fdl_channel_stride, float* output, long long output_stride, int channels, int partitions, int block_index, float scaling, void* stream)
{
    CFB_TRACE ("fft_partitioned_convolve_step");
    Plan* p = as_plan (setup);
    if (p == nullptr)
        return FFT_B200_EINVAL;
    if (p->is_complex)
        return fail (FFT_B200_EINVAL, "fft_partitioned_convolve_step needs a REAL plan");
    if (p->mixed || p->logM > kMaxLogM)
        return fail (FFT_B200_EINVAL, "fft_partitioned_convolve_step: block size N=%d must be a power of two up to the single-kernel limit 32768", p->N);
    if (windows == nullptr || ir == nullptr || fdl == nullptr || output == nullptr || channels < 0 || partitions < 1 || block_index < 0)
        return fail (FFT_B200_EINVAL, "fft_partitioned_convolve_step: bad arguments");
    if (channels == 0)
        return 0;
    // windows / output move float2 pairs; the delay line and the IR partitions (N floats each, N % 32 == 0) move float4 vectors
    if (misaligned (windows, 8, window_stride, channels) || misaligned (output, 8, output_stride, channels)
        || misaligned (ir, 16, ir_channel_stride, channels) || misaligned (fdl, 16, fdl_channel_stride, channels))
        return fail (FFT_B200_EINVAL, "fft_partitioned_convolve_step: windows / output must be 8-byte aligned with even strides, ir / fdl 16-byte aligned with strides that are multiples of 4 floats");
    if (classify (windows).kind != Mem::Device || classify (ir).kind != Mem::Device || classify (fdl).kind != Mem::Device || classify (output).kind != Mem::Device)
        return fail (FFT_B200_EINVAL, "fft_partitioned_convolve_step needs device pointers");
    Tables t;
    const int rc = plan_tables (p, t);
    if (rc != 0)
        return rc;
    PConvArgs a {};
    a.in = windows;
    a.in_stride = window_stride;
    a.ir = ir;
    a.ir_ch_stride = ir_channel_stride;
    a.fdl = fdl;
    a.fdl_ch_stride = fdl_channel_stride;
    a.out = output;
    a.out_stride = output_stride;
    a.channels = channels;
    a.P = partitions;
    a.t = block_index;
    a.scaling = scaling;
    a.tw = t.tw;
    a.rtw = t.rtw;
    note_kernel ("cfb::pconv_kernel<%d,%d>", p->logM, p->logW);
    const cudaError_t e = launch_pconv (p->logM, p->logW, a, static_cast<cudaStream_t> (stream));
    return e == cudaSuccess ? 0 : fail_cuda (e, "partitioned convolution kernel launch");
}

// ---- streaming convolver with non-uniform partitions (fft_convolver_*; schedule: conv_schedule in pconv_kernel.cuh) ----
namespace
{
constexpr uint64_t kConvMagic = 0x434642434f4e5631ull; // "CFBCONV1"
constexpr int kConvMaxSegments = 16;                   // B = 16 up to Bmax = 16384 needs 11
constexpr int kConvMaxBlockDefault = 16384;            // the largest block of the fused step's real plans
int g_conv_max_block = kConvMaxBlockDefault;           // tuning hook "convolver_max_block"

struct ConvSegment
{
    int Bk = 0, P = 0;    // block size, partitions
    long long start = 0;  // first tap (also the output delay for k >= 1)
    Plan* plan = nullptr; // real plan of 2 Bk points
    Tables tables;
    float* fdl = nullptr; // [channels][P][2 Bk] frequency-delay line
};

// the state that depends on the IR; the input history and the delay lines depend on the input only and are shared by both banks
struct ConvBank
{
    float* ir[kConvMaxSegments] = {}; // per segment [channels or 1][P][2 Bk] IR spectra, unordered layout
    float* acc = nullptr;             // [channels][ring] output accumulator
    float* S = nullptr;               // [channels][2 Bmax] partial spectrum of a sliced last segment (P > 1), else null
};

struct ConvCtx
{
    uint64_t magic;
    int channels = 0, B = 0, Bmax = 0, nseg = 0, device = 0;
    bool shared_ir = false;
    long long L = 0;       // IR length at create: the schedule covers it, and later IRs may not be longer
    ConvSegment seg[kConvMaxSegments];
    ConvBank bank[2];      // bank[cur] holds the IR in use; bank[1 - cur] takes the next one (allocated by the first set_ir)
    int cur = 0;
    float* scratch = nullptr; // set_ir's IR partition gather buffer (scratch_floats), allocated with the second bank
    size_t scratch_floats = 0;
    float* hist = nullptr; // [channels][2 ring] mirrored input history, ring = 2 Bmax
    long long ring = 0;
    long long t = 0;       // calls since create / reset
    int fade = 0;          // > 0: calls [fade_t0, fade_t0 + fade) crossfade from bank[cur] to bank[1 - cur]
    long long fade_t0 = 0;
};

ConvCtx* as_conv (void* ctx)
{
    auto* d = static_cast<ConvCtx*> (ctx);
    if (d == nullptr || (reinterpret_cast<uintptr_t> (d) & 7) != 0 || d->magic != kConvMagic)
    {
        fail (chowdsp::fft::FFT_B200_EINVAL, "invalid convolver context %p", ctx);
        return nullptr;
    }
    return d;
}

// block index for the fused step: the slot written is t % P and min(t + 1, P) partitions are summed, so a running count can be
// folded to keep it in int range
int fold_index (long long t, int P) { return t < P ? (int) t : (int) (t % P) + P; }

void conv_bank_free (ConvBank& b)
{
    for (float*& p : b.ir)
    {
        (void) cudaFree (p);
        p = nullptr;
    }
    (void) cudaFree (b.acc);
    (void) cudaFree (b.S);
    b.acc = b.S = nullptr;
}

int conv_bank_alloc (const ConvCtx* d, ConvBank& b)
{
    const size_t C = (size_t) d->channels, Cir = d->shared_ir ? 1 : C;
    for (int k = 0; k < d->nseg; ++k)
        CFB_CUDA (cudaMalloc (&b.ir[k], sizeof (float) * Cir * 2 * (size_t) d->seg[k].Bk * (size_t) d->seg[k].P));
    CFB_CUDA (cudaMalloc (&b.acc, sizeof (float) * C * (size_t) d->ring));
    const ConvSegment& last = d->seg[d->nseg - 1];
    if (d->nseg > 1 && last.P > 1)
        CFB_CUDA (cudaMalloc (&b.S, sizeof (float) * C * 2 * (size_t) last.Bk));
    return 0;
}

void conv_free (ConvCtx* d)
{
    for (int k = 0; k < d->nseg; ++k)
    {
        (void) cudaFree (d->seg[k].fdl);
        if (d->seg[k].plan != nullptr)
            chowdsp::fft::fft_destroy_setup (d->seg[k].plan);
    }
    conv_bank_free (d->bank[0]);
    conv_bank_free (d->bank[1]);
    (void) cudaFree (d->scratch);
    (void) cudaFree (d->hist);
    d->magic = 0;
    delete d;
}

int conv_zero (ConvCtx* d, cudaStream_t st)
{
    const size_t C = (size_t) d->channels;
    const ConvBank& b = d->bank[d->cur];
    for (int k = 0; k < d->nseg; ++k)
        CFB_CUDA (cudaMemsetAsync (d->seg[k].fdl, 0, sizeof (float) * C * (size_t) d->seg[k].P * 2 * (size_t) d->seg[k].Bk, st));
    CFB_CUDA (cudaMemsetAsync (d->hist, 0, sizeof (float) * C * 2 * (size_t) d->ring, st));
    CFB_CUDA (cudaMemsetAsync (b.acc, 0, sizeof (float) * C * (size_t) d->ring, st));
    if (b.S != nullptr)
        CFB_CUDA (cudaMemsetAsync (b.S, 0, sizeof (float) * C * 2 * (size_t) d->Bmax, st));
    d->t = 0;
    return 0;
}

// IR spectra of bank b: zero-padded partitions [Bk taps | Bk zeros] gathered into tmp, forward-transformed in the plan's
// unordered layout.  create and set_ir run this same sequence, so equal IRs give bitwise equal spectra.
int conv_prepare_ir (const ConvCtx* d, ConvBank& b, const float* ir, long long L, long long ir_stride, float* tmp, cudaStream_t st)
{
    const int Cir = d->shared_ir ? 1 : d->channels;
    for (int k = 0; k < d->nseg; ++k)
    {
        const ConvSegment& g = d->seg[k];
        const ConvIrArgs ga { ir, ir_stride, tmp, L, g.start, Cir, g.P, g.Bk };
        const cudaError_t e = launch_conv_ir_gather (ga, st);
        if (e != cudaSuccess)
            return fail_cuda (e, "IR partition gather");
        const int rc = chowdsp::fft::fft_transform_batched (g.plan, tmp, b.ir[k], Cir * g.P, 2LL * g.Bk, 2LL * g.Bk, chowdsp::fft::FFT_FORWARD, 0, st);
        if (rc != 0)
            return rc;
    }
    return 0;
}

int conv_build (ConvCtx* d, const float* ir, long long L, long long ir_stride, cudaStream_t st)
{
    int blocks[kConvMaxSegments];
    long long parts[kConvMaxSegments], starts[kConvMaxSegments];
    d->nseg = conv_schedule (d->B, L, d->Bmax, blocks, parts, starts, kConvMaxSegments);
    if (d->nseg > kConvMaxSegments)
        return fail (chowdsp::fft::FFT_B200_EINVAL, "fft_convolver_create: schedule of %d segments", d->nseg);
    d->L = L;
    const size_t C = (size_t) d->channels, Cir = d->shared_ir ? 1 : C;
    for (int k = 0; k < d->nseg; ++k)
    {
        if (parts[k] > (1 << 24))
            return fail (chowdsp::fft::FFT_B200_EINVAL, "fft_convolver_create: ir_length %lld needs too many partitions", L);
        ConvSegment& g = d->seg[k];
        g.Bk = blocks[k];
        g.P = (int) parts[k];
        g.start = starts[k];
        const size_t n = 2 * (size_t) g.Bk * (size_t) g.P;
        d->scratch_floats = d->scratch_floats > Cir * n ? d->scratch_floats : Cir * n;
        CFB_CUDA (cudaMalloc (&g.fdl, sizeof (float) * C * n));
        g.plan = static_cast<Plan*> (chowdsp::fft::fft_new_setup (2 * g.Bk, chowdsp::fft::FFT_REAL, true));
        if (g.plan == nullptr)
            return chowdsp::fft::FFT_B200_ECUDA;
        const int rc = plan_tables (g.plan, g.tables);
        if (rc != 0)
            return rc;
    }
    d->ring = 2LL * d->Bmax;
    CFB_CUDA (cudaMalloc (&d->hist, sizeof (float) * C * 2 * (size_t) d->ring));
    int rc = conv_bank_alloc (d, d->bank[0]);
    if (rc == 0)
        rc = conv_zero (d, st);
    if (rc != 0)
        return rc;
    float* tmp = nullptr;
    CFB_CUDA (cudaMalloc (&tmp, sizeof (float) * d->scratch_floats));
    rc = conv_prepare_ir (d, d->bank[0], ir, L, ir_stride, tmp, st);
    const cudaError_t es = cudaStreamSynchronize (st);
    (void) cudaFree (tmp);
    if (rc != 0)
        return rc;
    return es == cudaSuccess ? 0 : fail_cuda (es, "fft_convolver_create");
}

long long conv_ir_stride (const ConvCtx* d, const ConvSegment& g) { return d->shared_ir ? 0 : (long long) g.P * 2 * g.Bk; }

// slice [pair0, pair0 + pairs) of bank b's partial spectrum S for firing q of the last segment k
cudaError_t conv_slice (const ConvCtx* d, const ConvBank& b, int k, long long q, int pair0, int pairs, cudaStream_t st)
{
    const ConvSegment& g = d->seg[k];
    const PConvSliceArgs sa { b.ir[k], conv_ir_stride (d, g), g.fdl, (long long) g.P * 2 * g.Bk, b.S, 2LL * g.Bk,
                              d->channels, g.P, 2 * g.Bk, g.plan->logW, (int) (q % g.P), pair0, pairs };
    return launch_pconv_slice (sa, st);
}

// firing q of segment k >= 1 with bank b: adds its Bk results into the bank's ring at [end, end + Bk).  from_fdl takes X_q from
// the delay line (written by the current bank's firing, or by the firing being re-run) instead of transforming the window.
cudaError_t conv_fire (const ConvCtx* d, const ConvBank& b, int k, long long q, long long end, bool from_fdl, cudaStream_t st)
{
    const ConvSegment& g = d->seg[k];
    const bool sliced = k == d->nseg - 1 && g.P > 1;
    PConvArgs a {};
    a.in = d->hist + d->ring + end - 2LL * g.Bk;
    a.in_stride = 2 * d->ring;
    a.ir = b.ir[k];
    a.ir_ch_stride = conv_ir_stride (d, g);
    a.fdl = g.fdl;
    a.fdl_ch_stride = (long long) g.P * 2 * g.Bk;
    a.out = b.acc + end;
    a.out_stride = d->ring;
    a.channels = d->channels;
    a.P = g.P;
    a.t = fold_index (q, g.P);
    a.scaling = 1.f / (float) (2 * g.Bk);
    a.tw = g.tables.tw;
    a.rtw = g.tables.rtw;
    const PConvAcc x { nullptr, 0, b.S, 2LL * g.Bk };
    return launch_pconv_acc (g.plan->logM, g.plan->logW, PCONV_ADD, sliced, from_fdl, a, x, st);
}
} // namespace

CFB_API int fft_convolver_create (int channels, int block_size, const float* ir, long long ir_length, long long ir_channel_stride, void* stream, void** ctx_out)
{
    CFB_TRACE ("fft_convolver_create");
    if (ctx_out == nullptr)
        return fail (FFT_B200_EINVAL, "fft_convolver_create: null ctx_out");
    *ctx_out = nullptr;
    if (channels < 1 || block_size < 16 || block_size > kConvMaxBlockDefault || (block_size & (block_size - 1)) != 0 || ir == nullptr || ir_length < 1
        || ir_channel_stride < 0 || (ir_channel_stride != 0 && ir_channel_stride < ir_length))
        return fail (FFT_B200_EINVAL, "fft_convolver_create: bad arguments (channels >= 1, block_size a power of two in [16, 16384], ir_length >= 1, ir_channel_stride 0 or >= ir_length)");
    if (misaligned (ir, 4))
        return fail (FFT_B200_EINVAL, "fft_convolver_create: the IR must be 4-byte aligned");
    if (! device_available())
        return fail (FFT_B200_ENODEVICE, "no usable CUDA device: chowdsp_fft_b200 has no CPU fallback");
    if (classify (ir).kind != Mem::Device)
        return fail (FFT_B200_EINVAL, "fft_convolver_create needs a device pointer for the IR");
    auto* d = new (std::nothrow) ConvCtx();
    if (d == nullptr)
        return fail (FFT_B200_ECUDA, "out of host memory");
    d->magic = kConvMagic;
    d->channels = channels;
    d->B = block_size;
    d->Bmax = g_conv_max_block > block_size ? g_conv_max_block : block_size;
    d->shared_ir = ir_channel_stride == 0;
    const cudaError_t e = cudaGetDevice (&d->device);
    const int rc = e != cudaSuccess ? fail_cuda (e, "cudaGetDevice") : conv_build (d, ir, ir_length, ir_channel_stride, static_cast<cudaStream_t> (stream));
    if (rc != 0)
    {
        (void) cudaStreamSynchronize (static_cast<cudaStream_t> (stream));
        conv_free (d);
        return rc;
    }
    *ctx_out = d;
    return 0;
}

CFB_API int fft_convolver_process (void* ctx, const float* input, long long input_stride, float* output, long long output_stride, void* stream_)
{
    CFB_TRACE ("fft_convolver_process");
    ConvCtx* d = as_conv (ctx);
    if (d == nullptr)
        return FFT_B200_EINVAL;
    const int C = d->channels, B = d->B;
    if (input == nullptr || output == nullptr)
        return fail (FFT_B200_EINVAL, "fft_convolver_process: null buffer");
    if (misaligned (input, 8, input_stride, C) || misaligned (output, 8, output_stride, C))
        return fail (FFT_B200_EINVAL, "fft_convolver_process: input / output must be 8-byte aligned with even strides");
    if (classify (input).kind != Mem::Device || classify (output).kind != Mem::Device)
        return fail (FFT_B200_EINVAL, "fft_convolver_process needs device pointers");
    int dev = 0;
    CFB_CUDA (cudaGetDevice (&dev));
    if (dev != d->device)
        return fail (FFT_B200_EINVAL, "fft_convolver_process: the context lives on device %d, the current device is %d", d->device, dev);
    cudaStream_t st = static_cast<cudaStream_t> (stream_);
    const long long t = d->t, ring = d->ring;
    const long long pos = (t * B) % ring, end = (pos + B) % ring; // ring position of this block and of the sample after it
    // during a crossfade the next bank runs every step after the current one, on the delay-line spectra the current one stores
    const int banks = d->fade > 0 ? 2 : 1;
    cudaError_t e = launch_conv_input (ConvInputArgs { input, input_stride, d->hist, 2 * ring, C, B / 2, pos, ring }, st);
    // segments k >= 1 fire when their block of Bk samples is complete and add their Bk results to the ring at [end, end + Bk):
    // strictly after the block emitted now, and never wrapping (end is a multiple of Bk, ring = 2 Bmax)
    for (int k = d->nseg - 1; k >= 1 && e == cudaSuccess; --k)
    {
        const ConvSegment& g = d->seg[k];
        const int D = g.Bk / B;
        const long long q = t / D; // the firing this call belongs to; it fires on the period's last call
        const bool sliced = k == d->nseg - 1 && g.P > 1;
        for (int i = 0; i < banks && e == cudaSuccess; ++i)
        {
            const ConvBank& b = d->bank[d->cur ^ i];
            if (sliced)
                e = conv_slice (d, b, k, q, (int) (t % D) * (B / 4), B / 4, st);
            if ((t + 1) % D == 0 && e == cudaSuccess)
                e = conv_fire (d, b, k, q, end, i == 1, st);
        }
    }
    if (e == cudaSuccess)
    {
        // segment 0 (block B, every call): output = its result + the ring's [pos, pos + B), which it clears
        const ConvSegment& g = d->seg[0];
        PConvArgs a {};
        a.in = d->hist + ring + end - 2LL * B;
        a.in_stride = 2 * ring;
        a.ir = d->bank[d->cur].ir[0];
        a.ir_ch_stride = conv_ir_stride (d, g);
        a.fdl = g.fdl;
        a.fdl_ch_stride = (long long) g.P * 2 * B;
        a.out = output;
        a.out_stride = output_stride;
        a.channels = C;
        a.P = g.P;
        a.t = fold_index (t, g.P);
        a.scaling = 1.f / (float) (2 * B);
        a.tw = g.tables.tw;
        a.rtw = g.tables.rtw;
        if (d->nseg == 1) // uniform: nothing is ever added to the ring, the plain step writes the output
            e = launch_pconv (g.plan->logM, g.plan->logW, a, st);
        else
            e = launch_pconv_acc (g.plan->logM, g.plan->logW, PCONV_EMIT, false, false, a, PConvAcc { d->bank[d->cur].acc + pos, ring, nullptr, 0 }, st);
        if (banks == 2 && e == cudaSuccess)
        {
            // the new IR's output mixed over it: weight (n - fade_t0 B + 1) / (fade B) at output sample n (the uniform
            // schedule's ring stays zero, so the same mode serves it)
            const ConvBank& nb = d->bank[d->cur ^ 1];
            const double span = (double) d->fade * B;
            a.ir = nb.ir[0];
            const PConvAcc x { nb.acc + pos, ring, nullptr, 0, (float) ((double) ((t - d->fade_t0) * B + 1) / span), (float) (1.0 / span) };
            e = launch_pconv_acc (g.plan->logM, g.plan->logW, PCONV_EMIT_MIX, false, true, a, x, st);
        }
    }
    note_kernel ("cfb::pconv_acc_kernel: streaming convolver, %d segments", d->nseg);
    if (e != cudaSuccess)
        return fail_cuda (e, "convolver launch");
    d->t = t + 1;
    if (banks == 2 && d->t == d->fade_t0 + d->fade) // the crossfade is complete: the new IR's bank becomes the current one
    {
        d->cur ^= 1;
        d->fade = 0;
    }
    return 0;
}

CFB_API int fft_convolver_set_ir (void* ctx, const float* ir, long long ir_length, long long ir_channel_stride, int fade_blocks, void* stream)
{
    CFB_TRACE ("fft_convolver_set_ir");
    ConvCtx* d = as_conv (ctx);
    if (d == nullptr)
        return FFT_B200_EINVAL;
    if (d->fade > 0)
        return fail (FFT_B200_EINVAL, "fft_convolver_set_ir: a crossfade is still running (%lld of %d calls left)", d->fade_t0 + d->fade - d->t, d->fade);
    if (ir == nullptr || ir_length < 1 || ir_length > d->L || (d->shared_ir ? ir_channel_stride != 0 : ir_channel_stride < ir_length) || fade_blocks < 0
        || (long long) fade_blocks * d->B > (1LL << 24))
        return fail (FFT_B200_EINVAL, "fft_convolver_set_ir: bad arguments (1 <= ir_length <= %lld, ir_channel_stride %s, fade_blocks >= 0 and fade_blocks * %d <= 2^24)",
                     d->L, d->shared_ir ? "0 (shared IR)" : ">= ir_length (per-channel IRs)", d->B);
    if (misaligned (ir, 4))
        return fail (FFT_B200_EINVAL, "fft_convolver_set_ir: the IR must be 4-byte aligned");
    if (classify (ir).kind != Mem::Device)
        return fail (FFT_B200_EINVAL, "fft_convolver_set_ir needs a device pointer for the IR");
    int dev = 0;
    CFB_CUDA (cudaGetDevice (&dev));
    if (dev != d->device)
        return fail (FFT_B200_EINVAL, "fft_convolver_set_ir: the context lives on device %d, the current device is %d", d->device, dev);
    cudaStream_t st = static_cast<cudaStream_t> (stream);
    ConvBank& nb = d->bank[d->cur ^ 1];
    if (nb.acc == nullptr) // first call: the second bank and the gather scratch (cudaMalloc may synchronise)
    {
        int rc = conv_bank_alloc (d, nb);
        if (rc == 0 && cudaMalloc (&d->scratch, sizeof (float) * d->scratch_floats) != cudaSuccess)
            rc = fail (FFT_B200_ECUDA, "fft_convolver_set_ir: out of device memory");
        if (rc != 0)
        {
            conv_bank_free (nb);
            (void) cudaFree (d->scratch);
            d->scratch = nullptr;
            return rc;
        }
    }
    int rc = conv_prepare_ir (d, nb, ir, ir_length, ir_channel_stride, d->scratch, st);
    if (rc != 0)
        return rc;
    const size_t C = (size_t) d->channels;
    const long long t0 = d->t, B = d->B, ring = d->ring;
    CFB_CUDA (cudaMemsetAsync (nb.acc, 0, sizeof (float) * C * (size_t) ring, st));
    // Re-prime: the ring and S of a context that had run with the new IR since call 0.  Only each segment's most recent firing
    // (t_f = floor(t0 / D) D - 1) adds to samples >= t0 B; re-run it in descending k, the order in which a fresh context made
    // those additions.  X_q comes from the delay line: the window of the largest segment's firing may already be overwritten in
    // the input ring.
    cudaError_t e = cudaSuccess;
    for (int k = d->nseg - 1; k >= 1 && e == cudaSuccess; --k)
    {
        const ConvSegment& g = d->seg[k];
        const long long D = g.Bk / B, m = t0 / D; // m - 1: the most recent firing, m: the current period
        const bool sliced = k == d->nseg - 1 && g.P > 1;
        if (m >= 1)
        {
            if (sliced)
                e = conv_slice (d, nb, k, m - 1, 0, g.Bk / 4, st);
            if (e == cudaSuccess)
                e = conv_fire (d, nb, k, m - 1, (m * g.Bk) % ring, true, st);
        }
        if (sliced && e == cudaSuccess) // S of the current period in full; the remaining slices of the period rewrite the same values
            e = conv_slice (d, nb, k, m, 0, g.Bk / 4, st);
    }
    if (e != cudaSuccess)
        return fail_cuda (e, "fft_convolver_set_ir: re-prime launch");
    if (d->nseg > 1)
    {
        // the re-run firings also added into [t0 B - Bmax, t0 B), already emitted; a fresh context holds zeros there
        const long long from = (t0 * B + d->Bmax) % ring, n1 = from + d->Bmax <= ring ? d->Bmax : ring - from;
        CFB_CUDA (cudaMemset2DAsync (nb.acc + from, sizeof (float) * ring, 0, sizeof (float) * n1, C, st));
        if (n1 < d->Bmax)
            CFB_CUDA (cudaMemset2DAsync (nb.acc, sizeof (float) * ring, 0, sizeof (float) * (d->Bmax - n1), C, st));
    }
    if (fade_blocks == 0)
        d->cur ^= 1;
    else
    {
        d->fade = fade_blocks;
        d->fade_t0 = t0;
    }
    return 0;
}

CFB_API int fft_convolver_reset (void* ctx, void* stream)
{
    CFB_TRACE ("fft_convolver_reset");
    ConvCtx* d = as_conv (ctx);
    if (d == nullptr)
        return FFT_B200_EINVAL;
    if (d->fade > 0) // a running crossfade ends at the new IR
    {
        d->cur ^= 1;
        d->fade = 0;
    }
    return conv_zero (d, static_cast<cudaStream_t> (stream));
}

CFB_API int fft_convolver_segments (void* ctx, int* block_sizes, int* partitions, int max_segments)
{
    ConvCtx* d = as_conv (ctx);
    if (d == nullptr)
        return FFT_B200_EINVAL;
    for (int k = 0; k < d->nseg && k < max_segments; ++k)
    {
        if (block_sizes != nullptr)
            block_sizes[k] = d->seg[k].Bk;
        if (partitions != nullptr)
            partitions[k] = d->seg[k].P;
    }
    return d->nseg;
}

CFB_API int fft_convolver_destroy (void* ctx)
{
    ConvCtx* d = as_conv (ctx);
    if (d == nullptr)
        return FFT_B200_EINVAL;
    (void) cudaDeviceSynchronize(); // work queued on any stream may still use the buffers
    conv_free (d);
    (void) cudaGetLastError();
    return 0;
}

// ---- streaming STFT: analysis and overlap-add synthesis contexts (chowdsp_fft_b200.h: fft_stft_stream_*) ----------------
namespace
{
constexpr uint64_t kStftStreamMagic = 0x4346425354465331ull; // "CFBSTFS1"

struct StftStreamCtx
{
    uint64_t magic;
    int channels = 0, max_frames = 0, device = 0;
    bool ordered = false;
    long long N = 0, hop = 0;
    float scale = 1.f;
    Plan* plan = nullptr;           // the context's own REAL plan of N points (same unordered layout as the caller's)
    Tables tables;                  // its radix-16 tables (ristft_carry_kernel)
    float* awin = nullptr;          // copies of the windows (N floats each), nullptr = rectangular
    float* swin = nullptr;
    // analysis: mirrored input ring per channel, [ring | ring | max_frames hop] floats at hist + c * hist_stride.  Padded-signal
    // sample q (N - hop zeros, then the input) is stored at q % ring and q % ring + ring, by one conv_input_kernel launch per call
    float* hist = nullptr;
    long long ring = 0, hist_stride = 0;
    long long a_frames = 0;         // spectra produced since create / reset
    // synthesis: the N - hop carried overlap-add sums per channel (ristft_carry_kernel's accumulators)
    float* carry = nullptr;
};

StftStreamCtx* as_stft_stream (void* ctx)
{
    auto* d = static_cast<StftStreamCtx*> (ctx);
    if (d == nullptr || (reinterpret_cast<uintptr_t> (d) & 7) != 0 || d->magic != kStftStreamMagic)
    {
        fail (chowdsp::fft::FFT_B200_EINVAL, "invalid streaming STFT context %p", ctx);
        return nullptr;
    }
    return d;
}

void stft_stream_free (StftStreamCtx* d)
{
    (void) cudaFree (d->awin);
    (void) cudaFree (d->swin);
    (void) cudaFree (d->hist);
    (void) cudaFree (d->carry);
    if (d->plan != nullptr)
        chowdsp::fft::fft_destroy_setup (d->plan);
    d->magic = 0;
    delete d;
}

int stft_stream_zero (StftStreamCtx* d, cudaStream_t st)
{
    const size_t C = (size_t) d->channels;
    CFB_CUDA (cudaMemsetAsync (d->hist, 0, sizeof (float) * C * (size_t) d->hist_stride, st));
    CFB_CUDA (cudaMemsetAsync (d->carry, 0, sizeof (float) * C * (size_t) (d->N - d->hop), st));
    d->a_frames = 0;
    return 0;
}

int stft_stream_check_device (const StftStreamCtx* d, const char* fn)
{
    int dev = 0;
    CFB_CUDA (cudaGetDevice (&dev));
    if (dev != d->device)
        return fail (chowdsp::fft::FFT_B200_EINVAL, "%s: the context lives on device %d, the current device is %d", fn, d->device, dev);
    return 0;
}
} // namespace

CFB_API int fft_stft_stream_create (void* setup, int channels, long long hop, int max_frames, const float* analysis_window, const float* synthesis_window, float scale,
                                    int ordered, void* stream, void** ctx_out)
{
    CFB_TRACE ("fft_stft_stream_create");
    if (ctx_out == nullptr)
        return fail (FFT_B200_EINVAL, "fft_stft_stream_create: null ctx_out");
    *ctx_out = nullptr;
    Plan* p = as_plan (setup);
    if (p == nullptr)
        return FFT_B200_EINVAL;
    if (p->is_complex || p->mixed || p->logM < 6 || p->logM > 12)
        return fail (FFT_B200_EINVAL, "fft_stft_stream_create needs a REAL power-of-two plan with 128 <= N <= 8192");
    if (hop * 2 != p->N && hop * 4 != p->N && hop * 8 != p->N)
        return fail (FFT_B200_EINVAL, "fft_stft_stream_create: hop %lld is not N/2, N/4 or N/8 (N = %d)", hop, p->N);
    if (channels < 1 || max_frames < 1 || (long long) channels * max_frames > 0x7fffffffLL || (long long) max_frames * hop > (1LL << 28))
        return fail (FFT_B200_EINVAL, "fft_stft_stream_create: bad arguments (channels >= 1, max_frames >= 1)");
    for (const float* w : { analysis_window, synthesis_window })
        if (w != nullptr && misaligned (w, 4))
            return fail (FFT_B200_EINVAL, "fft_stft_stream_create: the windows must be 4-byte aligned");
    if (! device_available())
        return fail (FFT_B200_ENODEVICE, "no usable CUDA device: chowdsp_fft_b200 has no CPU fallback");
    auto* d = new (std::nothrow) StftStreamCtx();
    if (d == nullptr)
        return fail (FFT_B200_ECUDA, "out of host memory");
    d->magic = kStftStreamMagic;
    d->channels = channels;
    d->max_frames = max_frames;
    d->ordered = ordered != 0;
    d->N = p->N;
    d->hop = hop;
    d->scale = scale;
    // ring >= (N - hop) + 2 max_frames hop: a call's frames span (N - hop) + frames hop samples, and a call whose span crosses
    // the ring's end reads the low copy, whose entries for that span no earlier call can have wrapped over (see analyze).
    // A multiple of 4 floats: every frame start keeps the 16-byte alignment of an offline frame at f hop.
    const long long span_max = (long long) max_frames * hop;
    d->ring = (p->N - hop + 2 * span_max + 3) & ~3LL;
    d->hist_stride = 2 * d->ring + span_max;
    cudaStream_t st = static_cast<cudaStream_t> (stream);
    const size_t C = (size_t) channels, wbytes = sizeof (float) * (size_t) p->N;
    int rc = 0;
    cudaError_t e = cudaGetDevice (&d->device);
    if (e == cudaSuccess)
    {
        d->plan = static_cast<Plan*> (chowdsp::fft::fft_new_setup (p->N, chowdsp::fft::FFT_REAL, p->logW == 3));
        if (d->plan == nullptr || d->plan->logW != p->logW)
            rc = fail (FFT_B200_ECUDA, "fft_stft_stream_create: could not create the context's plan");
    }
    if (e == cudaSuccess && rc == 0)
        rc = plan_tables (d->plan, d->tables, 16);
    if (e == cudaSuccess && rc == 0 && analysis_window != nullptr && (e = cudaMalloc (&d->awin, wbytes)) == cudaSuccess)
        e = cudaMemcpyAsync (d->awin, analysis_window, wbytes, cudaMemcpyDefault, st);
    if (e == cudaSuccess && rc == 0 && synthesis_window != nullptr && (e = cudaMalloc (&d->swin, wbytes)) == cudaSuccess)
        e = cudaMemcpyAsync (d->swin, synthesis_window, wbytes, cudaMemcpyDefault, st);
    if (e == cudaSuccess && rc == 0 && (e = cudaMalloc (&d->hist, sizeof (float) * C * (size_t) d->hist_stride)) == cudaSuccess)
        e = cudaMalloc (&d->carry, sizeof (float) * C * (size_t) (p->N - hop));
    if (e == cudaSuccess && rc == 0)
        rc = stft_stream_zero (d, st);
    if (e == cudaSuccess && rc == 0)
        e = cudaStreamSynchronize (st); // the windows may be freed by the caller once create returns
    if (e != cudaSuccess && rc == 0)
        rc = fail_cuda (e, "fft_stft_stream_create");
    if (rc != 0)
    {
        (void) cudaStreamSynchronize (st);
        stft_stream_free (d);
        return rc;
    }
    *ctx_out = d;
    return 0;
}

CFB_API int fft_stft_stream_analyze (void* ctx, const float* input, long long input_stride, int frames, float* spectra, long long spec_channel_stride, long long spec_frame_stride,
                                     void* stream)
{
    CFB_TRACE ("fft_stft_stream_analyze");
    StftStreamCtx* d = as_stft_stream (ctx);
    if (d == nullptr)
        return FFT_B200_EINVAL;
    const int C = d->channels;
    if (input == nullptr || spectra == nullptr || frames < 1 || frames > d->max_frames)
        return fail (FFT_B200_EINVAL, "fft_stft_stream_analyze: bad arguments (non-null buffers, 1 <= frames <= max_frames = %d)", d->max_frames);
    if (misaligned (input, 8, input_stride, C))
        return fail (FFT_B200_EINVAL, "fft_stft_stream_analyze: the input must be 8-byte aligned with an even channel stride");
    if (misaligned (spectra, d->ordered ? 8 : 16, spec_frame_stride, frames, spec_channel_stride, C))
        return fail (FFT_B200_EINVAL, "fft_stft_stream_analyze: every spectrum must start on an 8-byte boundary (16-byte for unordered spectra): check the base pointer and strides");
    if (classify (input).kind != Mem::Device || classify (spectra).kind != Mem::Device)
        return fail (FFT_B200_EINVAL, "fft_stft_stream_analyze needs device pointers");
    int rc = stft_stream_check_device (d, "fft_stft_stream_analyze");
    if (rc != 0)
        return rc;
    cudaStream_t st = static_cast<cudaStream_t> (stream);
    // this call's frames cover padded samples [P0, P0 + span), the new ones are the last frames hop of them
    const long long hop = d->hop, ring = d->ring, n_new = (long long) frames * hop, span = d->N - hop + n_new;
    const long long P0 = d->a_frames * hop, b = P0 % ring, w = (P0 + d->N - hop) % ring;
    // The high copy [ring, 2 ring) always holds the newest sample of every residue (a write that crosses the ring's end lands
    // its wrapped part there through the low copy's overflow).  A span that crosses the end reads the low copy instead:
    // then b > ring - span >= ring - (N - hop) - max_frames hop >= max_frames hop, so a write that wrapped at P0 - b ended
    // before P0, and every sample of [P0, P0 + ring - b) sits at its own place in the low copy.
    const long long base = b + span <= ring ? ring + b : b;
    const cudaError_t e = launch_conv_input (ConvInputArgs { input, input_stride, d->hist, d->hist_stride, C, (int) (n_new / 2), w, ring }, st);
    if (e != cudaSuccess)
        return fail_cuda (e, "streaming STFT input launch");
    rc = enqueue_transform (d->plan, d->hist + base, spectra, C, frames, d->hist_stride, hop, spec_channel_stride, spec_frame_stride, FFT_FORWARD, d->ordered, st, d->awin);
    if (rc != 0)
        return rc;
    d->a_frames += frames;
    return 0;
}

CFB_API int fft_stft_stream_synthesize (void* ctx, const float* spectra, long long spec_channel_stride, long long spec_frame_stride, int frames, float* output, long long output_stride,
                                        void* stream)
{
    CFB_TRACE ("fft_stft_stream_synthesize");
    StftStreamCtx* d = as_stft_stream (ctx);
    if (d == nullptr)
        return FFT_B200_EINVAL;
    const int C = d->channels;
    if (spectra == nullptr || output == nullptr || frames < 1 || frames > d->max_frames)
        return fail (FFT_B200_EINVAL, "fft_stft_stream_synthesize: bad arguments (non-null buffers, 1 <= frames <= max_frames = %d)", d->max_frames);
    if (misaligned (spectra, d->ordered ? 8 : 16, spec_frame_stride, frames, spec_channel_stride, C))
        return fail (FFT_B200_EINVAL, "fft_stft_stream_synthesize: every spectrum must start on an 8-byte boundary (16-byte for unordered spectra): check the base pointer and strides");
    if (misaligned (output, 8, output_stride, C))
        return fail (FFT_B200_EINVAL, "fft_stft_stream_synthesize: the output must be 8-byte aligned with an even channel stride");
    if (classify (spectra).kind != Mem::Device || classify (output).kind != Mem::Device)
        return fail (FFT_B200_EINVAL, "fft_stft_stream_synthesize needs device pointers");
    const int rc = stft_stream_check_device (d, "fft_stft_stream_synthesize");
    if (rc != 0)
        return rc;
    FftArgs a {};
    a.in = spectra;
    a.out = output;
    a.in_inner = spec_frame_stride;
    a.in_outer = spec_channel_stride;
    a.out_inner = d->hop;
    a.out_outer = output_stride;
    a.inner = frames;
    a.batch = C * frames;
    a.tw = d->tables.tw;
    a.rtw = d->tables.rtw;
    a.window = d->swin;
    a.seg_frames = frames;
    a.nseg = 1;
    a.scale = d->scale;
    const int logW = d->ordered ? 0 : d->plan->logW, hq = (int) (d->hop * 16 / d->N);
    const cudaError_t e = launch_ristft (d->plan->logM, hq, logW, a, static_cast<cudaStream_t> (stream), reinterpret_cast<float2*> (d->carry));
    if (e != cudaSuccess)
        return fail_cuda (e, "streaming overlap-add synthesis launch");
    note_kernel ("cfb::ristft_carry_kernel<%d,%d,%d>", d->plan->logM, hq, logW);
    return 0;
}

CFB_API int fft_stft_stream_reset (void* ctx, void* stream)
{
    CFB_TRACE ("fft_stft_stream_reset");
    StftStreamCtx* d = as_stft_stream (ctx);
    if (d == nullptr)
        return FFT_B200_EINVAL;
    const int rc = stft_stream_check_device (d, "fft_stft_stream_reset");
    return rc != 0 ? rc : stft_stream_zero (d, static_cast<cudaStream_t> (stream));
}

CFB_API int fft_stft_stream_destroy (void* ctx)
{
    StftStreamCtx* d = as_stft_stream (ctx);
    if (d == nullptr)
        return FFT_B200_EINVAL;
    (void) cudaDeviceSynchronize(); // work queued on any stream may still use the buffers
    stft_stream_free (d);
    (void) cudaGetLastError();
    return 0;
}

CFB_API int fft_large_factors (void* setup, int* l1, int* l2, int* l3)
{
    Plan* p = as_plan (setup);
    if (p == nullptr)
        return FFT_B200_EINVAL;
    if (p->logM <= kMaxLogM)
        return fail (FFT_B200_EINVAL, "fft_large_factors: N=%d is a single-kernel plan", p->N);
    const LargeFactors f = choose_factors (p->logM);
    if (l1 != nullptr)
        *l1 = f.l1;
    if (l2 != nullptr)
        *l2 = f.l2;
    if (l3 != nullptr)
        *l3 = f.l3;
    return 0;
}

CFB_API int fft_dist_phase (void* setup, int phase, int rank, int world, const float* in, float* out, fft_direction_t direction, void* stream)
{
    CFB_TRACE ("fft_dist_phase");
    Plan* p = as_plan (setup);
    if (p == nullptr)
        return FFT_B200_EINVAL;
    if (! p->is_complex || p->logM <= kMaxLogM)
        return fail (FFT_B200_EINVAL, "fft_dist_phase needs a complex multi-pass plan");
    if (in == nullptr || out == nullptr || phase < 0 || phase > 2 || rank < 0 || rank >= world)
        return fail (FFT_B200_EINVAL, "fft_dist_phase: bad arguments");
    const LargeFactors f = choose_factors (p->logM);
    TilePass tp;
    if (! build_dist_phase (p->logM, f, phase, rank, world, tp))
        return fail (FFT_B200_EINVAL, "fft_dist_phase: N=2^%d cannot be split over %d ranks (needs a three-pass plan, power-of-two world, L1/world >= 8)", p->logM, world);
    int dev = 0;
    CFB_CUDA (cudaGetDevice (&dev));
    BigTables bt;
    int rc = get_big_tables (dev, p->logM, bt);
    if (rc != 0)
        return rc;
    Tables st;
    rc = get_tables (dev, tp.logL, false, st, tile_radix_for (tp.logL));
    if (rc != 0)
        return rc;
    tp.args.tw = st.tw;
    tp.args.tw_lo = bt.lo;
    tp.args.tw_hi = bt.hi;
    tp.args.tw_lobits = bt.lobits;
    tp.args.in = reinterpret_cast<const float2*> (in);
    tp.args.out = reinterpret_cast<float2*> (out);
    const cudaError_t e = launch_tile (tp.logL, tp.C, direction == FFT_FORWARD ? -1 : +1, tp.load_j_fast, 0, tp.args, static_cast<cudaStream_t> (stream));
    return e == cudaSuccess ? 0 : fail_cuda (e, "distributed phase launch");
}

CFB_API int fft_dist_phase0_peer (void* setup, int rank, int world, const float* in, float* const* peer_recv, fft_direction_t direction, void* stream)
{
    CFB_TRACE ("fft_dist_phase0_peer");
    Plan* p = as_plan (setup);
    if (p == nullptr)
        return FFT_B200_EINVAL;
    if (! p->is_complex || p->logM <= kMaxLogM)
        return fail (FFT_B200_EINVAL, "fft_dist_phase0_peer needs a complex multi-pass plan");
    if (in == nullptr || peer_recv == nullptr || world < 1 || world > 8 || rank < 0 || rank >= world)
        return fail (FFT_B200_EINVAL, "fft_dist_phase0_peer: bad arguments (world <= 8)");
    const LargeFactors f = choose_factors (p->logM);
    TilePass tp;
    if (! build_dist_phase (p->logM, f, 0, rank, world, tp))
        return fail (FFT_B200_EINVAL, "fft_dist_phase0_peer: N=2^%d cannot be split over %d ranks", p->logM, world);
    int dev = 0;
    CFB_CUDA (cudaGetDevice (&dev));
    BigTables bt;
    int rc = get_big_tables (dev, p->logM, bt);
    if (rc != 0)
        return rc;
    Tables st;
    rc = get_tables (dev, tp.logL, false, st, tile_radix_for (tp.logL));
    if (rc != 0)
        return rc;
    int wl = 0;
    while ((1 << wl) < world)
        ++wl;
    tp.args.tw = st.tw;
    tp.args.tw_lo = bt.lo;
    tp.args.tw_hi = bt.hi;
    tp.args.tw_lobits = bt.lobits;
    tp.args.in = reinterpret_cast<const float2*> (in);
    tp.args.out = nullptr;
    tp.args.peer_row_log = f.l1 - wl;
    for (int h = 0; h < world; ++h)
    {
        if (peer_recv[h] == nullptr)
            return fail (FFT_B200_EINVAL, "fft_dist_phase0_peer: null receive buffer for rank %d", h);
        tp.args.peer_out[h] = reinterpret_cast<float2*> (peer_recv[h]);
    }
    const cudaError_t e = launch_tile (tp.logL, tp.C, direction == FFT_FORWARD ? -1 : +1, tp.load_j_fast, 0, tp.args, static_cast<cudaStream_t> (stream));
    return e == cudaSuccess ? 0 : fail_cuda (e, "distributed phase 0 (peer stores) launch");
}

// ---- distributed transform as ONE call per rank (the reference's contract is one fft_transform call,
// /root/reference/chowdsp_fft.cpp:318-356; here every rank makes one fft_dist_transform call) ------------------------
namespace
{
constexpr uint64_t kDistMagic = 0x4346424449535431ull; // "CFBDIST1"
constexpr int kDistBlobHandles = 4;                    // recv[0], recv[1], natural, flags
struct DistCtx
{
    uint64_t magic;
    Plan* plan;
    int rank, world, device;
    LargeFactors f;
    long long L1, S1, rows, cols;
    size_t local_bytes;                 // this rank's share of the transform: N / world complex values
    float2* recv[2] = { nullptr, nullptr };
    float2* nat = nullptr;
    unsigned long long* flags = nullptr; // [2][8] step counters + status word behind them
    int* status = nullptr;
    float2* peer_recv[2][8];
    float2* peer_nat[8];
    unsigned long long* peer_flags[8];
    std::vector<void*> mapped;
    float2* scratch = nullptr;           // phases 1 + 2: whole-array intermediate or the ring of the chunked schedule, kept across calls
    size_t scratch_bytes = 0;
    bool connected = false;
    unsigned long long step = 0;
    float phase_ms[4] = { 0.f, 0.f, 0.f, 0.f };
    cudaEvent_t ev[5] = { nullptr, nullptr, nullptr, nullptr, nullptr };
};
DistCtx* as_dist (void* ctx)
{
    auto* d = static_cast<DistCtx*> (ctx);
    if (d == nullptr || d->magic != kDistMagic)
    {
        fail (chowdsp::fft::FFT_B200_EINVAL, "invalid distributed context %p", ctx);
        return nullptr;
    }
    return d;
}
} // namespace

CFB_API int fft_dist_create (void* setup, int rank, int world, void** ctx_out)
{
    CFB_TRACE ("fft_dist_create");
    Plan* p = as_plan (setup);
    if (p == nullptr || ctx_out == nullptr)
        return FFT_B200_EINVAL;
    *ctx_out = nullptr;
    if (! p->is_complex || p->logM <= kMaxLogM)
        return fail (FFT_B200_EINVAL, "fft_dist_create needs a complex multi-pass plan");
    if (world < 1 || world > 8 || rank < 0 || rank >= world)
        return fail (FFT_B200_EINVAL, "fft_dist_create: 0 <= rank < world <= 8");
    const LargeFactors f = choose_factors (p->logM);
    TilePass probe;
    if (! build_dist_phase (p->logM, f, 0, rank, world, probe) || f.l3 < ilog2i (world))
        return fail (FFT_B200_EINVAL, "fft_dist_create: N=2^%d cannot be split over %d ranks (needs a three-pass plan, power-of-two world, L1/world >= 16)", p->logM, world);
    auto* d = new (std::nothrow) DistCtx();
    if (d == nullptr)
        return fail (FFT_B200_ECUDA, "out of host memory");
    d->magic = kDistMagic;
    d->plan = p;
    d->rank = rank;
    d->world = world;
    d->f = f;
    d->L1 = 1LL << f.l1;
    d->S1 = 1LL << (f.l2 + f.l3);
    d->rows = d->L1 / world;
    d->cols = d->S1 / world;
    d->local_bytes = sizeof (float2) * (size_t) (d->L1 * d->cols);
    cudaError_t e = cudaGetDevice (&d->device);
    for (int b = 0; b < 2 && e == cudaSuccess; ++b)
        e = cudaMalloc (&d->recv[b], d->local_bytes);
    if (e == cudaSuccess)
        e = cudaMalloc (&d->nat, d->local_bytes);
    if (e == cudaSuccess)
        e = cudaMalloc (&d->flags, 256);
    if (e == cudaSuccess)
        e = cudaMemset (d->flags, 0, 256);
    for (int i = 0; i < 5 && e == cudaSuccess; ++i)
        e = cudaEventCreate (&d->ev[i]);
    if (e != cudaSuccess)
    {
        fail_cuda (e, "fft_dist_create");
        for (auto* q : { (void*) d->recv[0], (void*) d->recv[1], (void*) d->nat, (void*) d->flags })
            if (q != nullptr)
                (void) cudaFree (q);
        delete d;
        return FFT_B200_ECUDA;
    }
    d->status = reinterpret_cast<int*> (d->flags + 16);
    for (int h = 0; h < 8; ++h)
    {
        d->peer_recv[0][h] = d->peer_recv[1][h] = d->peer_nat[h] = nullptr;
        d->peer_flags[h] = nullptr;
    }
    d->peer_recv[0][rank] = d->recv[0];
    d->peer_recv[1][rank] = d->recv[1];
    d->peer_nat[rank] = d->nat;
    d->peer_flags[rank] = d->flags;
    d->connected = world == 1;
    if (preload_large (p) != 0)
    {
        fft_dist_destroy (d);
        return FFT_B200_ECUDA;
    }
    *ctx_out = d;
    return 0;
}

CFB_API size_t fft_dist_blob_bytes (void) { return 64 * kDistBlobHandles; }

CFB_API int fft_dist_export (void* ctx, void* blob)
{
    DistCtx* d = as_dist (ctx);
    if (d == nullptr || blob == nullptr)
        return FFT_B200_EINVAL;
    void* blocks[kDistBlobHandles] = { d->recv[0], d->recv[1], d->nat, d->flags };
    for (int i = 0; i < kDistBlobHandles; ++i)
    {
        cudaIpcMemHandle_t h;
        CFB_CUDA (cudaIpcGetMemHandle (&h, blocks[i]));
        std::memcpy (static_cast<char*> (blob) + 64 * i, &h, 64);
    }
    return 0;
}

CFB_API int fft_dist_connect (void* ctx, const void* blobs)
{
    CFB_TRACE ("fft_dist_connect");
    DistCtx* d = as_dist (ctx);
    if (d == nullptr || (blobs == nullptr && d->world > 1))
        return FFT_B200_EINVAL;
    if (d->connected)
        return 0;
    for (int h = 0; h < d->world; ++h)
    {
        if (h == d->rank)
            continue;
        void* mapped[kDistBlobHandles];
        for (int i = 0; i < kDistBlobHandles; ++i)
        {
            cudaIpcMemHandle_t hd;
            std::memcpy (&hd, static_cast<const char*> (blobs) + (size_t) h * fft_dist_blob_bytes() + 64 * i, 64);
            mapped[i] = nullptr;
            CFB_CUDA (cudaIpcOpenMemHandle (&mapped[i], hd, cudaIpcMemLazyEnablePeerAccess));
            d->mapped.push_back (mapped[i]);
        }
        d->peer_recv[0][h] = static_cast<float2*> (mapped[0]);
        d->peer_recv[1][h] = static_cast<float2*> (mapped[1]);
        d->peer_nat[h] = static_cast<float2*> (mapped[2]);
        d->peer_flags[h] = static_cast<unsigned long long*> (mapped[3]);
    }
    d->connected = true;
    return 0;
}

CFB_API float* fft_dist_natural_buffer (void* ctx)
{
    DistCtx* d = as_dist (ctx);
    return d == nullptr ? nullptr : reinterpret_cast<float*> (d->nat);
}

CFB_API int fft_dist_status (void* ctx)
{
    DistCtx* d = as_dist (ctx);
    if (d == nullptr)
        return FFT_B200_EINVAL;
    int st = 0;
    CFB_CUDA (cudaMemcpy (&st, d->status, sizeof (int), cudaMemcpyDeviceToHost));
    return st == 0 ? 0 : fail (FFT_B200_ECUDA, "distributed transform: a peer did not reach the exchange barrier in time");
}

CFB_API int fft_dist_phase_ms (void* ctx, float* ms4)
{
    DistCtx* d = as_dist (ctx);
    if (d == nullptr || ms4 == nullptr)
        return FFT_B200_EINVAL;
    for (int i = 0; i < 4; ++i)
        ms4[i] = d->phase_ms[i];
    return 0;
}

CFB_API int fft_dist_transform (void* ctx, const float* input, float* output, fft_direction_t direction, int natural_order, int timed, void* stream_)
{
    CFB_TRACE ("fft_dist_transform");
    DistCtx* d = as_dist (ctx);
    if (d == nullptr)
        return FFT_B200_EINVAL;
    if (! d->connected)
        return fail (FFT_B200_EINVAL, "fft_dist_transform: call fft_dist_connect first");
    if (input == nullptr || (output == nullptr && ! natural_order))
        return fail (FFT_B200_EINVAL, "fft_dist_transform: null buffer");
    if (misaligned (input, 8) || (output != nullptr && misaligned (output, 8)))
        return fail (FFT_B200_EINVAL, "fft_dist_transform: buffers must be 8-byte aligned");
    if (classify (input).kind != Mem::Device || (output != nullptr && classify (output).kind != Mem::Device))
        return fail (FFT_B200_EINVAL, "fft_dist_transform needs device pointers");
    cudaStream_t stream = static_cast<cudaStream_t> (stream_);
    Plan* p = d->plan;
    const int n = p->logM, dir = direction == FFT_FORWARD ? -1 : +1, world = d->world;
    LargeTables lt;
    int rc = large_tables (p, d->device, d->f, lt);
    if (rc != 0)
        return rc;
    const unsigned long long step = ++d->step;
    const int b = (int) (step & 1);
    cudaError_t e = cudaSuccess;
    auto mark = [&] (int i)
    {
        if (timed && e == cudaSuccess)
            e = cudaEventRecord (d->ev[i], stream);
    };
    auto barrier = [&] (int which)
    {
        if (world == 1)
            return;
        DistBarrierArgs ba {};
        for (int h = 0; h < world; ++h)
            ba.peer_flags[h] = d->peer_flags[h];
        ba.own_flags = d->flags;
        ba.status = d->status;
        ba.rank = d->rank;
        ba.world = world;
        ba.which = which;
        ba.step = step;
        ba.timeout_ns = 20ull * 1000 * 1000 * 1000;
        if (e == cudaSuccess)
            e = launch_dist_barrier (ba, stream);
    };
    mark (0);
    {   // phase 0: column FFTs + twiddle, every output row block stored straight into its owner's receive buffer
        TilePass tp;
        build_dist_phase (n, d->f, 0, d->rank, world, tp);
        int wl = 0;
        while ((1 << wl) < world)
            ++wl;
        tp.args.tw = lt.pass[0].tw;
        tp.args.tw_lo = lt.bt.lo;
        tp.args.tw_hi = lt.bt.hi;
        tp.args.tw_lobits = lt.bt.lobits;
        tp.args.in = reinterpret_cast<const float2*> (input);
        tp.args.out = nullptr;
        tp.args.peer_row_log = d->f.l1 - wl;
        for (int h = 0; h < world; ++h)
            tp.args.peer_out[h] = d->peer_recv[b][h];
        e = launch_tile (tp.logL, tp.C, dir, tp.load_j_fast, 0, tp.args, stream);
    }
    mark (1);
    barrier (0);
    mark (2);
    // phases 1 + 2 on this rank's rows, L2-chunked
    long long chunk_elems = (long long) (g_l2_chunk_mb < 0 ? -g_l2_chunk_mb : g_l2_chunk_mb) * (1 << 20) / 8;
    if (n > 24 && g_l2_chunk_mb > 0)
        chunk_elems = 0; // same policy as the single-GPU path: beyond 2^24 points the chunk unit (8 k1-rows) outgrows L2
    const int lanes = g_l2_lanes < 1 ? 1 : (g_l2_lanes > kMaxLanes ? kMaxLanes : g_l2_lanes);
    const int c_last = tile_c (d->f.l3, true);
    long long nrc = chunk_elems / d->S1;
    nrc -= nrc % c_last;
    if (chunk_elems > 0 && nrc < c_last)
        nrc = c_last;
    const long long ring_lane = chunk_elems > 0 ? (nrc > d->rows ? d->rows : nrc) * d->S1 : 0;
    // the intermediate of phases 1 + 2 belongs to the context (no allocation on the transform path after the first call)
    const size_t need = chunk_elems <= 0 ? d->local_bytes : sizeof (float2) * (size_t) ring_lane * (size_t) lanes;
    if (d->scratch_bytes < need)
    {
        if (d->scratch != nullptr)
        {
            CFB_CUDA (cudaDeviceSynchronize());
            CFB_CUDA (cudaFree (d->scratch));
            d->scratch = nullptr;
            d->scratch_bytes = 0;
        }
        CFB_CUDA (cudaMalloc (&d->scratch, need));
        d->scratch_bytes = need;
    }
    float2* s1 = chunk_elems <= 0 ? d->scratch : nullptr;
    float2* ring = chunk_elems <= 0 ? nullptr : d->scratch;
    ForkJoin& fj = t_forkjoin;
    if ((rc = fj.ensure()) != 0)
        return rc;
    std::vector<LargeLaunch> sched;
    float2* dst = natural_order ? nullptr : reinterpret_cast<float2*> (output);
    if (! build_dist_schedule (n, d->f, d->rank, world, d->recv[b], dst, d->peer_nat, natural_order != 0, s1, ring, ring_lane, chunk_elems, lanes, g_l2_policy != 0, sched))
        return fail (FFT_B200_EINVAL, "fft_dist_transform: cannot schedule N=2^%d over %d ranks", n, world);
    LaneSet ls (fj, stream);
    for (auto& l : sched)
    {
        TileArgs& ta = l.pass.args;
        ta.tw = lt.pass[l.pass.which].tw;
        ta.tw_lo = lt.bt.lo;
        ta.tw_hi = lt.bt.hi;
        ta.tw_lobits = lt.bt.lobits;
        cudaStream_t st = ls.stream_of (l.lane, e);
        if (e == cudaSuccess)
            e = launch_tile_pass (dir, l.pass, st);
    }
    ls.join (e);
    mark (3);
    if (natural_order)
    {
        barrier (1); // every rank's pass-C stores into this rank's natural block have landed
        if (output != nullptr && reinterpret_cast<float2*> (output) != d->nat && e == cudaSuccess)
            e = cudaMemcpyAsync (output, d->nat, d->local_bytes, cudaMemcpyDeviceToDevice, stream);
    }
    mark (4);
    note_kernel ("cfb::tile_fft_kernel<%d|%d|%d,dir %d> distributed over %d ranks: phase 0 with peer stores, in-stream flag barrier, %s (B,C)%s",
                 d->f.l1, d->f.l2, d->f.l3, dir, world, chunk_elems > 0 ? "L2-chunked" : "whole-array", natural_order ? ", natural order by peer stores" : "");
    if (e != cudaSuccess)
        return fail_cuda (e, "distributed transform launch");
    if (timed)
    {
        CFB_CUDA (cudaEventSynchronize (d->ev[4]));
        for (int i = 0; i < 4; ++i)
            CFB_CUDA (cudaEventElapsedTime (&d->phase_ms[i], d->ev[i], d->ev[i + 1]));
    }
    return 0;
}

CFB_API int fft_dist_destroy (void* ctx)
{
    DistCtx* d = as_dist (ctx);
    if (d == nullptr)
        return FFT_B200_EINVAL;
    (void) cudaDeviceSynchronize();
    for (void* m : d->mapped)
        (void) cudaIpcCloseMemHandle (m);
    for (auto* q : { (void*) d->recv[0], (void*) d->recv[1], (void*) d->nat, (void*) d->flags, (void*) d->scratch })
        if (q != nullptr)
            (void) cudaFree (q);
    for (auto& ev : d->ev)
        if (ev != nullptr)
            (void) cudaEventDestroy (ev);
    d->magic = 0;
    delete d;
    (void) cudaGetLastError();
    return 0;
}

// Peer-memory plumbing for the fused exchange: plain cudaMalloc blocks (IPC handles need whole allocations)
CFB_API void* fft_dist_alloc (size_t bytes)
{
    void* p = nullptr;
    if (cudaMalloc (&p, bytes > 0 ? bytes : 1) != cudaSuccess)
    {
        fail_cuda (cudaGetLastError(), "fft_dist_alloc");
        return nullptr;
    }
    return p;
}
CFB_API void fft_dist_free (void* p)
{
    if (p != nullptr)
        (void) cudaFree (p);
}
CFB_API int fft_dist_ipc_export (void* p, void* handle64)
{
    static_assert (sizeof (cudaIpcMemHandle_t) == 64, "IPC handles are exchanged as 64 opaque bytes");
    if (p == nullptr || handle64 == nullptr)
        return fail (FFT_B200_EINVAL, "fft_dist_ipc_export: null argument");
    cudaIpcMemHandle_t h;
    CFB_CUDA (cudaIpcGetMemHandle (&h, p));
    std::memcpy (handle64, &h, 64);
    return 0;
}
CFB_API void* fft_dist_ipc_open (const void* handle64)
{
    if (handle64 == nullptr)
        return nullptr;
    cudaIpcMemHandle_t h;
    std::memcpy (&h, handle64, 64);
    void* p = nullptr;
    const cudaError_t e = cudaIpcOpenMemHandle (&p, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess)
    {
        fail_cuda (e, "cudaIpcOpenMemHandle");
        return nullptr;
    }
    return p;
}
CFB_API void fft_dist_ipc_close (void* p)
{
    if (p != nullptr)
        (void) cudaIpcCloseMemHandle (p);
}

CFB_API int fft_accumulate_batched (void* setup, const float* a, const float* b, float* ab, long long n, void* stream)
{
    CFB_TRACE ("fft_accumulate_batched");
    Plan* p = as_plan (setup);
    if (p == nullptr)
        return FFT_B200_EINVAL;
    if (n < 0 || n % 8 != 0)
        return fail (FFT_B200_EINVAL, "fft_accumulate_batched: n must be a non-negative multiple of 8");
    return elementwise_any (p, false, a, b, ab, 1, n, n, n, n, 0.f, static_cast<cudaStream_t> (stream), false);
}

CFB_API int fft_b200_set_tuning (const char* key, int value)
{
    if (key != nullptr && std::strcmp (key, "spin_sync") == 0 && value >= -1 && value <= 1)
    {
        g_spin_sync = value == 1;
        return 0;
    }
    if (key != nullptr && std::strcmp (key, "ristft") == 0 && value >= -1 && value <= 1)
    {
        g_ristft = value == -1 ? 1 : value;
        return 0;
    }
    if (key != nullptr && std::strcmp (key, "small") == 0 && value >= -1 && value <= 1)
    {
        fft_small_mode() = value == -1 ? 1 : value;
        return 0;
    }
    if (key != nullptr && std::strcmp (key, "mixq") == 0 && value >= -1 && value <= 1)
    {
        g_mixq = value == -1 ? 1 : value;
        return 0;
    }
    if (key != nullptr && std::strcmp (key, "tile_stream") == 0 && value >= -1 && value <= 3)
    {
        tile_stream_mode() = value == -1 ? 0 : value;
        return 0;
    }
    if (key != nullptr && std::strcmp (key, "tile_pf") == 0 && value >= -1)
    {
        tile_pf_distance() = value == -1 ? kTilePfDefault : value;
        return 0;
    }
    if (key != nullptr && std::strcmp (key, "zero_copy_kb") == 0 && value >= -1)
    {
        g_zero_copy_bytes = value == -1 ? kZeroCopyBytesDefault : (size_t) value * 1024;
        return 0;
    }
    if (key != nullptr && std::strcmp (key, "cluster") == 0 && value >= -1 && value <= 3)
    {
        g_cluster = value == -1 ? kClusterDefault : value;
        return 0;
    }
    if (key != nullptr && std::strcmp (key, "cluster_min_batch") == 0 && value >= -1)
    {
        g_cluster_min_batch = value == -1 ? kClusterMinBatchDefault : value;
        return 0;
    }
    if (key != nullptr && std::strcmp (key, "l2_chunk_mb") == 0 && value >= -256 && value <= 256)
    {
        g_l2_chunk_mb = value == -1 ? kL2ChunkMbDefault : value; // -1 = default; other negative values: |value| MiB, also beyond 2^24 points
        return 0;
    }
    if (key != nullptr && std::strcmp (key, "l2_lanes") == 0 && (value == -1 || (value >= 1 && value <= kMaxLanes)))
    {
        g_l2_lanes = value == -1 ? kL2LanesDefault : value;
        return 0;
    }
    if (key != nullptr && std::strcmp (key, "l2_policy") == 0 && value >= -1 && value <= 1)
    {
        g_l2_policy = value == -1 ? kL2PolicyDefault : value;
        return 0;
    }
    if (key != nullptr && std::strcmp (key, "tile_tma") == 0 && value >= -1 && value <= 1)
    {
        tile_tma_mode() = value == -1 ? kTileTmaDefault : value;
        return 0;
    }
    if (key != nullptr && std::strcmp (key, "tile_r") == 0 && value >= -1 && value <= 1)
    {
        tile_radix32() = value == -1 ? 0 : value;
        return 0;
    }
    if (key != nullptr && std::strcmp (key, "tile_c") == 0 && (value == -1 || value == 0 || value == 8 || value == 16))
    {
        tile_c_override() = value == -1 ? 0 : value;
        return 0;
    }
    if (key != nullptr && std::strcmp (key, "tile_c_jfast") == 0 && (value == -1 || value == 0 || value == 8 || value == 16))
    {
        tile_c_jfast_override() = value == -1 ? 0 : value;
        return 0;
    }
    if (key != nullptr && std::strcmp (key, "pipe_mask") == 0)
    {
        g_pipe_mask = value == -1 ? kPipeDefault : (unsigned) value;
        return 0;
    }
    if (key != nullptr && std::strcmp (key, "radix32_mask") == 0)
    {
        g_radix32_mask = value == -1 ? kRadix32Default : (unsigned) value;
        return 0;
    }
    if (key != nullptr && std::strcmp (key, "pf_ahead") == 0 && value >= -1)
    {
        g_pf_ahead = value == -1 ? 0 : value;
        return 0;
    }
    if (key != nullptr && std::strcmp (key, "wistft") == 0)
    {
        g_wistft = value == -1 ? kWIstftDefault : value;
        return 0;
    }
    if (key != nullptr && std::strcmp (key, "wpipe") == 0)
    {
        g_wpipe = value == -1 ? kWPipeDefault : value;
        return 0;
    }
    if (key != nullptr && std::strcmp (key, "stft_pipe") == 0)
    {
        g_stft_pipe = value != 0;
        return 0;
    }
    if (key != nullptr && std::strcmp (key, "convolver_max_block") == 0 && (value == -1 || (value >= 16 && value <= kConvMaxBlockDefault && (value & (value - 1)) == 0)))
    {
        g_conv_max_block = value == -1 ? kConvMaxBlockDefault : value;
        return 0;
    }
    if (key != nullptr && std::strcmp (key, "stft_union") == 0)
    {
        g_stft_union = value != 0;
        return 0;
    }
    return fail (FFT_B200_EINVAL, "fft_b200_set_tuning: unknown key or value");
}

CFB_API const char* fft_b200_last_error (void) { return t_error; }
CFB_API const char* fft_b200_last_kernel (void) { return t_last_kernel; }
CFB_API void fft_b200_clear_error (void) { t_error[0] = 0; }
CFB_API unsigned long long fft_b200_launch_count (void) { return cfb::launch_count(); }
CFB_API int fft_b200_device_available (void) { return device_available() ? 1 : 0; }
} // namespace chowdsp::fft
}
