// Persistent, TMA-pipelined single-kernel transform for the largest CTA-resident sizes (2^13 and 2^14 complex
// points per transform, i.e. C2C N = 8192 / 16384 and real N = 16384 / 32768).
//
// Why a second kernel for these sizes: a 2^14-point transform fills half of an SM's register file, so
// fft_kernel (fft_kernels.cuh) runs ONE CTA per SM and its load -> compute -> store phases cannot overlap
// (ncu, profiles/r01_ncu_c2c16384.txt: DRAM 49 %, issue slots 25 % busy, long-scoreboard stalls dominate).  Here
// one CTA per SM stays resident and loops over its share of the batch; the NEXT transform's input is fetched by
// the TMA unit (cp.async.bulk global -> shared, completion on an mbarrier) into a landing buffer while the
// current transform is in registers, so HBM reads, butterflies and HBM writes of neighbouring transforms overlap
// inside one SM.
//
// Shared memory (2^14: 217..226 KB, per kind): landing buffer (8 M bytes) + exchange region (4 M bytes) + the
// last stage's twiddle rows.  The transform is 32 x 32 x r_last.  The stage-0 exchange is an ordinary padded 64-bit exchange that
// borrows the (already consumed) landing buffer; the TMA for the next transform is issued right after it.  The
// stage-1 exchange runs while that copy is in flight, so it only has the half-size region: it moves the data in
// two balanced rounds of 16 registers per thread (round_scatter / round_gather).  [A first version moved real and
// imaginary parts separately through the half-size region for both exchanges: twice the LDS/STS instructions,
// MIO-queue bound, 5.0 TB/s at 2^14 -- profiles/r01_pipe_kernel.txt.]
//
// Unordered (8-lane) layouts: an unordered INPUT lands as the padded staging image fft_kernel uses (the TMA copies it
// in 512-byte pieces, one per thread, so that the 32-byte gaps of the bank-spreading pad appear on the fly); an
// unordered OUTPUT is staged and drained in two halves through the exchange region.  The 4-lane layout stays with
// fft_kernel.
//
// Replaces the same reference pipeline as fft_kernel (simd/chowdsp_fft_impl_avx.cpp:1848-1935); layouts, signs
// and scaling are identical to it (natural-order complex, pffft-packed real spectra; SURVEY.md §8a-L).
#pragma once
#include "fft_kernels.cuh"

namespace cfb
{
#ifdef CFB_PIPE_RTW_TABLE // A/B switch (tools/ only)
constexpr bool kPipeDeriveRtw = false;
#else
constexpr bool kPipeDeriveRtw = true;
#endif

// geometry and shared-memory layout of pipe_kernel<LOGM, KIND, LOGW> (LOGW = 0 ordered, 3 = 8-lane unordered)
template <int LOGM, int KIND = C2C_FWD, int LOGW = 0>
struct PipeGeo
{
    using G = Geo<LOGM, 32>;
    static constexpr int M = G::M, T = G::T, R = 32;
    static_assert (LOGW == 0 || LOGW == 3, "ordered or 8-lane unordered");
    static_assert (G::S == 3 && G::radix (1) == 32, "written for 32 x 32 x r_last");
    static_assert (G::T % 32 == 0 && G::R == 32, "the addressing below assumes 32 points per thread");
    static constexpr bool IN_UNORD = LOGW != 0 && (KIND == C2C_BWD || KIND == C2R);
    static constexpr bool OUT_UNORD = LOGW != 0 && (KIND == C2C_FWD || KIND == R2C);
    // landing buffer = TMA destination: one transform, linear; or the padded unordered staging image (one 8-float
    // gap per 128 floats, upad())
    static constexpr int LAND_BYTES = IN_UNORD ? (2 * M + (2 * M >> 4)) * 4 : M * 8;
    static constexpr int CHUNK_FLOATS = 128;                 // unordered input: floats per TMA piece (2 W^2)
    static constexpr int NCHUNK = 2 * M / CHUNK_FLOATS;      // <= T
    // exchange region: M/2 float2 (stage-1 rounds, unpadded; half-spectrum exchange of the real split / merge
    // steps), or half of a padded unordered staging image for unordered outputs; the padded stage-0 exchange
    // (M + M/32 float2) spans the landing buffer and the start of this region
    static constexpr int HALF_IMAGE_FLOATS = M + (M >> 4);
    static constexpr int XCH_BYTES = OUT_UNORD ? HALF_IMAGE_FLOATS * 4 : M * 4;
    static_assert (LAND_BYTES + XCH_BYTES >= (M + (M >> 5)) * 8, "stage-0 exchange does not fit");
    // last-stage twiddle rows kept in shared memory: q = 1, 2, 3 and 4, 8, .. (the other powers are one register
    // product each, as in the full-radix stages).  Out of L1 they would not fit next to a > 200 KB carve-out, and
    // every L2 round trip stalls one of only four warps per scheduler.
    static constexpr int RL = G::RLAST;
    static constexpr int TW_ROWS = RL <= 4 ? RL - 1 : 3 + (RL / 4 - 1);
    static constexpr int TW_OFFSET = LAND_BYTES + XCH_BYTES;
    static constexpr int TW1_OFFSET = TW_OFFSET + TW_ROWS * T * 8; // stage-1 rows w^4 .. w^28, 32 entries each
    static constexpr int BAR_OFFSET = TW1_OFFSET + 7 * 32 * 8;
    static constexpr int SMEM_BYTES = BAR_OFFSET + 16;
    static constexpr int CTAS_PER_SM = (2 * (SMEM_BYTES + 1024) <= 228 * 1024 && 2 * T <= 512) ? 2 : 1;
    static_assert (SMEM_BYTES <= 227 * 1024, "landing + exchange buffers exceed the shared memory of an SM");
    static_assert (RL >= 4, "expects a short last stage of radix >= 4");
    static FFT_CX int tw_row_q (int i) { return i < 3 ? i + 1 : 4 * (i - 2); } // smem row i holds power q
    static FFT_CX int tw_row_of (int q) { return q < 4 ? q - 1 : q / 4 + 2; }  // its inverse (q < 4 or q % 4 == 0)
};

// ---------------------------------------------------------------------------------------------
// mbarrier + bulk-copy helpers (sm_90+ PTX; SASS: SYNCS.*, UBLKCP.S.G).  One barrier phase = one transform:
// mbar_expect arms it with the transform's byte count (one thread), bulk_copy starts a piece (any thread), mbar_wait
// blocks until phase `it` has received all of its bytes.
// ---------------------------------------------------------------------------------------------
#ifdef CHOWDSP_EMU
// the emulator runs every CUDA thread as an OS thread: the "TMA" is a memcpy by the issuing thread followed by a
// release add of the byte count to the barrier word, the wait spins on the running total
FFT_HD void mbar_init (unsigned long long* bar) { __atomic_store_n (bar, 0ull, __ATOMIC_RELEASE); }
FFT_HD void mbar_expect (unsigned long long*, unsigned) {}
FFT_HD void bulk_copy (void* dst, const void* src, unsigned bytes, unsigned long long* bar)
{
    std::memcpy (dst, src, bytes);
    __atomic_fetch_add (bar, (unsigned long long) bytes, __ATOMIC_RELEASE);
}
FFT_HD void mbar_wait (unsigned long long* bar, unsigned it, unsigned bytes_per_phase)
{
    while (__atomic_load_n (bar, __ATOMIC_ACQUIRE) < (unsigned long long) (it + 1) * bytes_per_phase)
        std::this_thread::yield();
}
#else
FFT_HD unsigned smem_addr (const void* p) { return (unsigned) __cvta_generic_to_shared (p); }
FFT_HD void mbar_init (unsigned long long* bar)
{
    asm volatile ("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_addr (bar)) : "memory");
    asm volatile ("fence.mbarrier_init.release.cluster;" ::: "memory");
}
FFT_HD void mbar_expect (unsigned long long* bar, unsigned bytes)
{
    asm volatile ("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr (bar)), "r"(bytes) : "memory");
}
FFT_HD void bulk_copy (void* dst, const void* src, unsigned bytes, unsigned long long* bar)
{
    asm volatile ("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                  ::"r"(smem_addr (dst)), "l"(src), "r"(bytes), "r"(smem_addr (bar)) : "memory");
}
FFT_HD void mbar_wait (unsigned long long* bar, unsigned it, unsigned)
{
    const unsigned addr = smem_addr (bar), parity = it & 1u;
    unsigned done;
    do
    {
        asm volatile ("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                      : "=r"(done) : "r"(addr), "r"(parity) : "memory");
    } while (done == 0);
}
#endif

// ---------------------------------------------------------------------------------------------
// Persistent frame-gather (STFT analysis) kernel: R2C of OVERLAPPING windows of one signal, times an optional window,
// any single-kernel size.  Work item = PER_CTA consecutive frames of one channel (as in stft_kernel); a resident CTA
// loops over items blockIdx.x, blockIdx.x + gridDim.x, ...  The UNION of an item's frames ((PER_CTA - 1) hop + N floats
// instead of PER_CTA N) is brought in by one TMA bulk copy into a landing buffer while the previous item is being
// transformed; every transform takes its stage-0 registers from there.  Against fft_kernel / stft_kernel this
// hides the load latency (ncu on the STFT config: 28 % of the stall samples sat on the first use of the loaded
// registers, 16 warps per SM) and cuts the L2 -> SM bytes by the overlap factor without spending LSU instructions
// on the staging.  Needs 0 < hop <= N, hop and channel stride multiples of 4 floats, 16-byte aligned signal.
// Shared memory: [landing: a.land_bytes][mbarrier, 16 bytes][PER_CTA exchange buffers].
// ---------------------------------------------------------------------------------------------
template <int LOGM, int R, int LOGW>
struct StftPipeGeo
{
    using G = Geo<LOGM, R>;
    using L = Launch<LOGM, R>;
    static constexpr int NFL = 2 * G::M;
    static constexpr int SMEM_F2 = LOGW != 0 ? G::SMEM_F2_UNORD : G::SMEM_F2;
    static constexpr int XCH_BYTES = L::PER_CTA * SMEM_F2 * 8;
    static int land_bytes (long long hop) { return (int) (((L::PER_CTA - 1) * hop + NFL) * 4); } // hop % 4 == 0: multiple of 16
    static int smem_bytes (long long hop) { return land_bytes (hop) + 16 + XCH_BYTES; }
};

template <int LOGM, int R, int LOGW>
FFT_HD void stft_pipe_body (const FftArgs& a)
{
    using SP = StftPipeGeo<LOGM, R, LOGW>;
    using G = typename SP::G;
    constexpr int T = G::T, NFL = SP::NFL, PER_CTA = SP::L::PER_CTA;
    FFT_DYN_SMEM (char, smem);
    float2* land = reinterpret_cast<float2*> (smem);
    unsigned long long* bar = reinterpret_cast<unsigned long long*> (smem + a.land_bytes);
    float2* xch = reinterpret_cast<float2*> (smem + a.land_bytes + 16);

    const int tid = (int) threadIdx.x;
    const int j = tid & (T - 1);
    const int lt = tid / T;
    const long long items = (long long) (a.batch / a.inner) * a.groups;
    const long long step = (long long) gridDim.x;
    const int hop = (int) a.in_inner;

    // item -> (channel, first frame, frames); span = floats of the union of its frames
    auto fetch = [&] (long long item)
    {
        const long long o = item / a.groups;
        const int f0 = (int) (item - o * a.groups) * PER_CTA;
        const int nact = a.inner - f0 < PER_CTA ? a.inner - f0 : PER_CTA;
        const unsigned bytes = (unsigned) ((nact - 1) * hop + NFL) * 4u;
        mbar_expect (bar, bytes);
        bulk_copy (land, a.in + o * a.in_outer + (long long) f0 * hop, bytes, bar);
    };
    long long item = (long long) blockIdx.x;
    if (tid == 0)
    {
        mbar_init (bar);
        if (item < items)
            fetch (item);
    }
    __syncthreads();
#ifdef CHOWDSP_EMU
    unsigned long long emu_bytes = 0; // the emulated barrier counts bytes: running total expected after each item
#endif
    for (unsigned it = 0; item < items; item += step, ++it)
    {
        const long long o = item / a.groups;
        const int f0 = (int) (item - o * a.groups) * PER_CTA;
        const int nact = a.inner - f0 < PER_CTA ? a.inner - f0 : PER_CTA;
        const bool active = lt < nact;
        const int ltc = active ? lt : nact - 1; // idle transforms of a channel's last group redo its last frame, no store
#ifdef CHOWDSP_EMU
        emu_bytes += (unsigned long long) ((nact - 1) * hop + NFL) * 4u;
        while (__atomic_load_n (bar, __ATOMIC_ACQUIRE) < emu_bytes)
            std::this_thread::yield();
#else
        mbar_wait (bar, it, 0);
#endif
        float* out = a.out + o * a.out_outer + (long long) (f0 + ltc) * a.out_inner;
        const auto input_consumed = [&]
        {
            if (tid == 0 && item + step < items)
                fetch (item + step);
        };
        fft_core<LOGM, R, R2C, LOGW, false, false, false, true> (nullptr, out, active, j, xch + lt * SP::SMEM_F2, a.tw, a.rtw,
                                                                 land + ltc * (hop / 2), reinterpret_cast<const float2*> (a.window), input_consumed);
        if constexpr (G::S == 1)
        {
            __syncthreads(); // single-stage transforms have no barrier of their own after the input reads
            input_consumed();
        }
    }
}

template <int LOGM, int R, int LOGW>
__global__ void __launch_bounds__ (Launch<LOGM, R>::THREADS, Launch<LOGM, R>::MIN_BLOCKS) stft_pipe_kernel (const FftArgs a)
{
    stft_pipe_body<LOGM, R, LOGW> (a);
}

// ---------------------------------------------------------------------------------------------
// Warp-pipelined transform (wpipe_kernel) for the sizes one warp owns (T = M / R = 32: 2^10 points at 32 per thread,
// 2^9 at 16): every warp of a resident CTA is its own software pipeline over transforms of the CTA's share of the batch
//   * the warp's NEXT input (8 M bytes, contiguous) is fetched by the TMA unit into a landing buffer private to the warp
//     (cp.async.bulk + the warp's own mbarrier) as soon as the stage-0 registers of the current transform have been
//     read out of it, i.e. the copy has a whole transform's butterflies, exchanges and stores to complete;
//   * nothing is CTA-wide: the only barriers are __syncwarp and the warp's mbarrier wait, so the warps of an SM drift
//     apart and their LSU / FMA / store phases interleave.
// Against fft_kernel this removes the exposed load latency that bounds the STFT config (ncu: 36 % of the stall samples on
// the first use of the loaded registers at 16 resident warps per SM, DRAM 60 %): every resident warp keeps 8 M bytes in
// flight all the time instead of during a third of its life.
// Plain and two-level (frame gather, optional window) batches, kinds R2C / C2C_FWD, every layout.  Every transform's
// input must be 16-byte aligned (the launcher checks base, in_inner and in_outer).
// Shared memory: per warp [landing 8 M bytes][exchange buffer][mbarrier, next-transform slot: 16 bytes]; then the CTA's
// work counter (16 bytes).
// ---------------------------------------------------------------------------------------------
#ifndef CFB_WPIPE_ALIAS
#define CFB_WPIPE_ALIAS 1 // A/B switch (tools/ only)
#endif
template <int LOGM, int R, int LOGW>
struct WPipeGeo
{
    using G = Geo<LOGM, R>;
    static_assert (G::T == 32, "wpipe_kernel: one warp per transform");
    static constexpr int IN_BYTES = 2 * G::M * 4;
    static constexpr int SMEM_F2 = LOGW != 0 ? G::SMEM_F2_UNORD : G::SMEM_F2;
    // ALIAS: the landing buffer doubles as the exchange buffer -- the next input copy starts only after the gather of the
    // last exchange instead of right after the stage-0 reads (a shorter prefetch window), but a warp needs half the shared
    // memory, so 16 warps (4 per scheduler) are resident instead of 13.  Ordered layouts only (their epilogues do not
    // stage anything in shared memory).
    static constexpr bool ALIAS = CFB_WPIPE_ALIAS != 0 && LOGW == 0;
    static constexpr int XCH_OFFSET = ALIAS ? 0 : IN_BYTES;
    static constexpr int BAR_OFFSET = XCH_OFFSET + (SMEM_F2 * 8 > IN_BYTES || ! ALIAS ? SMEM_F2 * 8 : IN_BYTES);
    static constexpr int WARP_BYTES = BAR_OFFSET + 16;
    static constexpr int CTA_EXTRA_BYTES = 16; // the work counter
    static constexpr int MAX_WARPS = (227 * 1024 - CTA_EXTRA_BYTES) / WARP_BYTES < 16 ? (227 * 1024 - CTA_EXTRA_BYTES) / WARP_BYTES : 16;
    static constexpr int smem_bytes (int warps) { return warps * WARP_BYTES + CTA_EXTRA_BYTES; }
    static_assert (WARP_BYTES % 16 == 0, "landing buffers must stay 16-byte aligned");
};

// shared-memory work counter of a CTA (one lane per warp asks for the warp's next transform)
FFT_HD unsigned smem_take (unsigned* counter)
{
#ifdef CHOWDSP_EMU
    return __atomic_fetch_add (counter, 1u, __ATOMIC_RELAXED);
#else
    return atomicAdd (counter, 1u);
#endif
}

template <int LOGM, int R, int KIND, int LOGW>
FFT_HD void wpipe_body (const FftArgs& a)
{
    using WP = WPipeGeo<LOGM, R, LOGW>;
    static_assert (KIND == R2C || KIND == C2C_FWD, "wpipe_kernel: kinds whose input is a contiguous natural-order row");
    FFT_DYN_SMEM (char, smem);
    const int tid = (int) threadIdx.x;
    const int lane = tid & 31, warp = tid >> 5;
    const int wpc = (int) blockDim.x >> 5;
    char* wbase = smem + (size_t) warp * WP::WARP_BYTES;
    float2* land = reinterpret_cast<float2*> (wbase);
    float2* xch = reinterpret_cast<float2*> (wbase + WP::XCH_OFFSET);
    unsigned long long* bar = reinterpret_cast<unsigned long long*> (wbase + WP::BAR_OFFSET);
    volatile unsigned* wnext = reinterpret_cast<volatile unsigned*> (bar + 1); // the warp's next transform, written by lane 0
    unsigned* counter = reinterpret_cast<unsigned*> (smem + (size_t) wpc * WP::WARP_BYTES);
    constexpr bool ALIAS = WP::ALIAS;

    // The CTA owns the contiguous range [first, first + count) of the batch (neighbouring frames of an STFT are then
    // fetched close together in time: their overlap is an L2 hit); inside the CTA the warps take transforms one at a
    // time from a shared counter, so a warp that shares its scheduler with more warps than the others just takes fewer.
    const long long first = (long long) a.batch * (long long) blockIdx.x / (long long) gridDim.x;
    const unsigned count = (unsigned) ((long long) a.batch * ((long long) blockIdx.x + 1) / (long long) gridDim.x - first);
    const bool two_level = a.inner < a.batch;
    auto locate = [&] (unsigned i, long long& xo, long long& xi)
    {
        const long long t = first + i;
        xo = 0;
        xi = t;
        if (two_level)
        {
            xo = (long long) ((unsigned) t / (unsigned) a.inner);
            xi = t - xo * a.inner;
        }
    };
    auto fetch = [&] (unsigned i)
    {
        long long xo, xi;
        locate (i, xo, xi);
        mbar_expect (bar, (unsigned) WP::IN_BYTES);
        bulk_copy (land, a.in + xo * a.in_outer + xi * a.in_inner, (unsigned) WP::IN_BYTES, bar);
    };
    if (tid == 0)
        *counter = 0u;
    __syncthreads();
    if (lane == 0)
    {
        mbar_init (bar);
        const unsigned i = smem_take (counter);
        *wnext = i;
        if (i < count)
            fetch (i);
    }
    tsync<32, true>();
    unsigned cur = *wnext;
    for (unsigned it = 0; cur < count; ++it)
    {
        long long xo, xi;
        locate (cur, xo, xi);
        float* out = a.out + xo * a.out_outer + xi * a.out_inner;
        mbar_wait (bar, it, (unsigned) WP::IN_BYTES);
        // runs after the warp-level barrier that follows the stage-0 reads: the landing buffer is free again, and every
        // lane has read *wnext for this trip
        const auto next_fetch = [&]
        {
            if (lane == 0)
            {
                const unsigned i = smem_take (counter);
                *wnext = i;
                if (i < count)
                    fetch (i);
            }
        };
        if constexpr (ALIAS)
        {
            fft_core<LOGM, R, KIND, LOGW, false, false, false, 2, NoHook, false, 0, decltype (next_fetch)> (nullptr, out, true, lane, xch, a.tw, a.rtw, land,
                                                                                                      reinterpret_cast<const float2*> (a.window), NoHook(), nullptr, next_fetch);
            tsync<32, true>(); // lane 0's *wnext is visible to the warp
        }
        else
            fft_core<LOGM, R, KIND, LOGW, false, false, false, 2> (nullptr, out, true, lane, xch, a.tw, a.rtw, land,
                                                                   reinterpret_cast<const float2*> (a.window), next_fetch);
        cur = *wnext; // a warp-level barrier lies between lane 0's write and this read
    }
}

template <int LOGM, int R, int KIND, int LOGW>
__global__ void __launch_bounds__ (WPipeGeo<LOGM, R, LOGW>::MAX_WARPS * 32, 1) wpipe_kernel (const FftArgs a)
{
    wpipe_body<LOGM, R, KIND, LOGW> (a);
}

// ---------------------------------------------------------------------------------------------
// Warp-pipelined overlap-add synthesis (wistft_kernel): the inverse STFT for the sizes one warp owns, hop = N / 2, N / 4
// or N / 8.  out[c][t] = scale * sum over frames f of window[t - f hop] * C2R (spectrum (c, f)) [t - f hop], as istft_kernel,
// but a WARP walks through the frames [fs, fe) of one (channel, segment) item on its own:
//   * the next frame's spectrum arrives by the warp's own bulk copy while the current one is transformed (as wpipe_kernel);
//   * thread j's result registers are the samples 2 (j + 32 m) (+1), and hop / 2 = 32 HQ, so the overlap-add never
//     leaves the thread: the N - hop samples a frame shares with its successors live in R - HQ accumulator REGISTERS
//     that shift by HQ per frame; the hop samples that are final are stored straight from registers.  No shared-memory
//     traffic, no barrier and no atomics for the overlap-add; the sums are formed in frame order (bit-reproducible).
// Segments other than a channel's first start N / hop - 1 frames early (halo, recomputed, not stored).  Items are
// distributed like wpipe_kernel's transforms (contiguous share per CTA, shared-memory counter inside).
// Ordered (pffft-packed) spectra, 16-byte aligned frames, 8-byte aligned signals.
// ---------------------------------------------------------------------------------------------
template <int LOGM, int R, int HQ>
FFT_HD void wistft_body (const FftArgs& a)
{
    using WP = WPipeGeo<LOGM, R, 0>;
    static_assert (HQ >= 1 && 2 * HQ <= R, "hop <= N / 2");
    constexpr int NACC = R - HQ;            // float2 accumulators per thread: the N - hop carried samples
    constexpr int HOP2 = 32 * HQ;           // hop in float2 units
    constexpr int HALO = R / HQ - 1;
    FFT_DYN_SMEM (char, smem);
    const int tid = (int) threadIdx.x;
    const int lane = tid & 31, warp = tid >> 5;
    const int wpc = (int) blockDim.x >> 5;
    char* wbase = smem + (size_t) warp * WP::WARP_BYTES;
    float2* land = reinterpret_cast<float2*> (wbase);
    float2* xch = reinterpret_cast<float2*> (wbase + WP::XCH_OFFSET);
    unsigned long long* bar = reinterpret_cast<unsigned long long*> (wbase + WP::BAR_OFFSET);
    volatile unsigned* wnext = reinterpret_cast<volatile unsigned*> (bar + 1);
    unsigned* counter = reinterpret_cast<unsigned*> (smem + (size_t) wpc * WP::WARP_BYTES);

    const int frames = a.inner;
    const long long items = (long long) (a.batch / a.inner) * a.nseg;
    const long long first = items * (long long) blockIdx.x / (long long) gridDim.x;
    const unsigned count = (unsigned) (items * ((long long) blockIdx.x + 1) / (long long) gridDim.x - first);
    const float2* __restrict__ win2 = reinterpret_cast<const float2*> (a.window);
    const float2 scale2 = make_float2 (a.scale, a.scale);

    auto decode = [&] (unsigned i, int& c, int& fs, int& fe)
    {
        const long long t = first + i;
        c = (int) (t / a.nseg);
        fs = (int) (t - (long long) c * a.nseg) * a.seg_frames;
        fe = fs + a.seg_frames < frames ? fs + a.seg_frames : frames;
    };
    auto fetch = [&] (int c, int f)
    {
        mbar_expect (bar, (unsigned) WP::IN_BYTES);
        bulk_copy (land, a.in + (long long) c * a.in_outer + (long long) f * a.in_inner, (unsigned) WP::IN_BYTES, bar);
    };
    if (tid == 0)
        *counter = 0u;
    __syncthreads();
    if (lane == 0)
    {
        mbar_init (bar);
        const unsigned i = smem_take (counter);
        *wnext = i;
        if (i < count)
        {
            int c, fs, fe;
            decode (i, c, fs, fe);
            fetch (c, fs - HALO > 0 ? fs - HALO : 0);
        }
    }
    tsync<32, true>();
    unsigned cur = *wnext;
    if (cur >= count)
        return;
    int c, fs, fe;
    decode (cur, c, fs, fe);
    int f = fs - HALO > 0 ? fs - HALO : 0;
    float2 acc[NACC];
#pragma unroll
    for (int i = 0; i < NACC; ++i)
        acc[i] = make_float2 (0.f, 0.f);
    for (unsigned it = 0;; ++it)
    {
        mbar_wait (bar, it, (unsigned) WP::IN_BYTES);
        const bool last_of_item = f + 1 == fe;
        const auto input_consumed = [&]
        {
            if (lane == 0)
            {
                if (! last_of_item)
                    fetch (c, f + 1);
                else
                {
                    const unsigned i = smem_take (counter);
                    *wnext = i;
                    if (i < count)
                    {
                        int c2, fs2, fe2;
                        decode (i, c2, fs2, fe2);
                        fetch (c2, fs2 - HALO > 0 ? fs2 - HALO : 0);
                    }
                }
            }
        };
        float2 v[R];
        if constexpr (WP::ALIAS)
        {
            fft_core<LOGM, R, C2R, 0, false, false, false, 2, NoHook, true, 0, decltype (input_consumed)> (nullptr, nullptr, true, lane, xch, a.tw, a.rtw, land, nullptr, NoHook(), v,
                                                                                                     input_consumed);
            tsync<32, true>(); // lane 0's *wnext is visible to the warp
        }
        else
            fft_core<LOGM, R, C2R, 0, false, false, false, 2, decltype (input_consumed), true> (nullptr, nullptr, true, lane, xch, a.tw, a.rtw, land, nullptr, input_consumed, v);
#pragma unroll
        for (int m = 0; m < R; ++m)
        {
            v[m] = f2_mul (v[m], scale2);
            if (win2 != nullptr)
                v[m] = f2_mul (v[m], __ldg (win2 + lane + 32 * m));
        }
        // overlap-add in registers: slot m of this frame is slot m - HQ of the next one
        float2* __restrict__ sig2 = reinterpret_cast<float2*> (a.out + (long long) c * a.out_outer) + (long long) f * HOP2 + lane;
        if (f >= fs)
        {
#pragma unroll
            for (int m = 0; m < HQ; ++m)
                sig2[32 * m] = f2_add (acc[m], v[m]);
        }
#pragma unroll
        for (int i = 0; i < NACC; ++i)
            acc[i] = i + HQ < NACC ? f2_add (acc[i + HQ], v[i + HQ]) : v[i + HQ];
        if (! last_of_item)
        {
            ++f;
            continue;
        }
        if (fe == frames) // end of the channel: the carried samples are output too
        {
#pragma unroll
            for (int i = 0; i < NACC; ++i)
                sig2[HOP2 + 32 * i] = acc[i];
        }
        cur = *wnext;
        if (cur >= count)
            break;
        decode (cur, c, fs, fe);
        f = fs - HALO > 0 ? fs - HALO : 0;
#pragma unroll
        for (int i = 0; i < NACC; ++i)
            acc[i] = make_float2 (0.f, 0.f);
    }
}

template <int LOGM, int R>
struct WIstftGeo
{
    // 64 result + up to 56 accumulator registers per thread on top of the transform's temporaries: 10 resident warps
    // (168 registers per thread; 12 warps measured 9 % slower: 28 KB of L1 left for window + twiddles) for 32 points per
    // thread, 16 (128) for 16
    static constexpr int MAX_WARPS = R == 32 ? (WPipeGeo<LOGM, R, 0>::ALIAS ? 12 : 10) : 16;
};
template <int LOGM, int R, int HQ>
__global__ void __launch_bounds__ (WIstftGeo<LOGM, R>::MAX_WARPS * 32, 1) wistft_kernel (const FftArgs a)
{
    wistft_body<LOGM, R, HQ> (a);
}

// start the copy of one transform into the landing buffer (called by every thread of the CTA)
template <class P>
FFT_HD void pipe_fetch (char* land, const float* src, int j, unsigned long long* bar)
{
    if constexpr (! P::IN_UNORD)
    {
        if (j == 0)
        {
            mbar_expect (bar, (unsigned) P::LAND_BYTES);
            bulk_copy (land, src, (unsigned) P::LAND_BYTES, bar);
        }
    }
    else
    {
        // piece c of 128 floats goes to float offset 136 c: the staging image's pad appears during the copy
        if (j == 0)
            mbar_expect (bar, (unsigned) (2 * P::M * 4));
        if (j < P::NCHUNK)
            bulk_copy (land + (size_t) j * (P::CHUNK_FLOATS + 8) * 4, src + (size_t) j * P::CHUNK_FLOATS, (unsigned) P::CHUNK_FLOATS * 4, bar);
    }
}

// ---------------------------------------------------------------------------------------------
// exchange after stage 1 (Ns = 32, radix 32) in TWO balanced rounds through a buffer of M/2 float2: round h moves
// the outputs q in [16 h, 16 h + 16) of every thread.  Position p = w 1024 + q 32 + l (writer thread 32 w + l) maps to
// slot w 512 + (q - 16 h) 32 + l; reader j needs p = j + m T, which lies in round h iff ((m mod D) div (D/2)) == h
// with D = 1024 / T, at slot (m div D) 512 + (m mod D mod D/2) T + j.  Every thread stores 16 and loads 16 values per
// round (so 32 complex registers stay live), all accesses are unit stride across a warp: conflict free, no padding.
// ---------------------------------------------------------------------------------------------
template <class G, int H>
FFT_HD void round_scatter (const float2 (&v)[32], int j, float2* xs)
{
    float2* sb = xs + (j >> 5) * 512 + (j & 31);
#pragma unroll
    for (int q = 0; q < 16; ++q)
        sts2 (sb + q * 32, v[16 * H + q]);
}
template <class G, int H>
FFT_HD void round_gather (float2 (&v)[32], int j, const float2* xs)
{
    constexpr int D = 1024 / G::T;
    static_assert (D >= 2 && G::T * D == 1024, "expects 256 or 512 threads per transform");
    const float2* rb = xs + j;
#pragma unroll
    for (int m = 0; m < 32; ++m)
        if ((m % D) / (D / 2) == H)
            v[m] = lds2 (rb + (m / D) * 512 + ((m % D) % (D / 2)) * G::T);
}

// stage 1 (Ns = 32, radix 32): its ten twiddle rows depend on the lane only (k = j mod 32), so the persistent loop
// fetches them once per kernel instead of once per transform (as L1 loads they were 20 % of all stall samples,
// profiles/r01_pipe_kernel.txt): w^1, w^2, w^3 stay in registers, w^4, w^8, .., w^28 in shared memory (ten
// register pairs would spill under the 128-register cap of a 512-thread CTA)
struct Stage1Tw
{
    float2 w1, w2, w3;
};
template <class G>
FFT_HD Stage1Tw load_stage1_tw (int j, const float2* __restrict__ tw, float2* tw1s)
{
    constexpr int Ns = 32;
    const float2* __restrict__ t = tw + G::tw_off (1) + (j & (Ns - 1));
    Stage1Tw r;
    r.w1 = __ldg (t);
    r.w2 = __ldg (t + Ns);
    r.w3 = __ldg (t + 2 * Ns);
    if (j < Ns)
    {
#pragma unroll
        for (int a4 = 1; a4 < 8; ++a4)
            sts2 (tw1s + (a4 - 1) * Ns + j, __ldg (t + (2 + a4) * Ns));
    }
    return r;
}
template <int DIR>
FFT_HD void pipe_stage1 (float2 (&v)[32], const Stage1Tw& w, const float2* tw1s_lane)
{
    v[1] = cmul_dir<DIR> (v[1], w.w1);
    v[2] = cmul_dir<DIR> (v[2], w.w2);
    v[3] = cmul_dir<DIR> (v[3], w.w3);
#pragma unroll
    for (int a4 = 1; a4 < 8; ++a4)
    {
        const float2 wa = lds2 (tw1s_lane + (a4 - 1) * 32);
        v[4 * a4] = cmul_dir<DIR> (v[4 * a4], wa);
        v[4 * a4 + 1] = cmul_dir<DIR> (v[4 * a4 + 1], cmul_dir<-1> (w.w1, wa));
        v[4 * a4 + 2] = cmul_dir<DIR> (v[4 * a4 + 2], cmul_dir<-1> (w.w2, wa));
        v[4 * a4 + 3] = cmul_dir<DIR> (v[4 * a4 + 3], cmul_dir<-1> (w.w3, wa));
    }
    RegFft<32, DIR, 1>::run (&v[0]);
}

// last (short) stage with the twiddle rows in shared memory: butterfly u of this thread has k = j + u T and
// W^(k q) = W^(j q) W_R^(u q); W^(j q) for q not in the table is one product of two rows
template <class P, int DIR>
FFT_HD void pipe_last_stage (float2 (&v)[32], int j, const float2* tws)
{
    using G = typename P::G;
    constexpr int r = P::RL, SUB = 32 / r, T = G::T;
    float2 w[r];
    const float2* tj = tws + j;
    last_stage_tw<r> (w, [&] (int q) { return lds2 (tj + P::tw_row_of (q) * T); });
#pragma unroll
    for (int q = 1; q < r; ++q)
    {
#pragma unroll
        for (int u = 0; u < SUB; ++u)
        {
            const float2 x = cmul_dir<DIR> (v[u + q * SUB], w[q]);
            v[u + q * SUB] = mul_w32_rt<DIR> (x, u * q);
        }
    }
#pragma unroll
    for (int u = 0; u < SUB; ++u)
        RegFft<r, DIR, SUB>::run (&v[u]);
}

// linear 128-bit drain of one half of the padded unordered staging image (M floats) to global memory
template <class P>
FFT_HD void half_drain (const float* sf, float* __restrict__ out, int j)
{
#pragma unroll
    for (int i = 0; i < P::M / (4 * P::T); ++i)
    {
        const int q = j + i * P::T;
        reinterpret_cast<float4*> (out)[q] = lds4 (sf + upad (4 * q, 3));
    }
}

// ---------------------------------------------------------------------------------------------
// the kernel: grid = min (batch, SMs * CTAS_PER_SM), blockDim = T = M / 32, dynamic smem = PipeGeo::SMEM_BYTES.
// Plain batches only (transform x reads in + x in_inner, writes out + x out_inner); the input rows must be
// 16-byte aligned (TMA), which the launcher checks.
// ---------------------------------------------------------------------------------------------
// result stores of the ordered epilogue: streaming (st.global.cs, evict-first) at 2^14 points, plain at 2^13 -- burst-mode A/B on
// B200 (profiles/r02_retune.txt): +1.5 % at 2^14 (one resident CTA per SM), -3.5 % at 2^13 (two)
template <int LOGM>
FFT_HD void pipe_stg (float2* p, float2 v)
{
#if ! defined(CHOWDSP_EMU) && ! defined(CFB_PIPE_NO_STCS)
    if constexpr (LOGM >= 14)
        __stcs (p, v);
    else
        *p = v;
#else
    *p = v;
#endif
}

template <int LOGM, int KIND, int LOGW>
FFT_HD void pipe_body (const FftArgs& a)
{
    using P = PipeGeo<LOGM, KIND, LOGW>;
    using G = typename P::G;
    constexpr int R = 32, T = G::T, M = G::M;
    constexpr int DIR = (KIND == C2C_FWD || KIND == R2C) ? -1 : +1;
    constexpr int WL = 8;                                    // lanes of the unordered layout
    constexpr unsigned PHASE_BYTES = P::IN_UNORD ? 2u * M * 4u : (unsigned) P::LAND_BYTES;
    FFT_DYN_SMEM (char, smem);
    float2* land = reinterpret_cast<float2*> (smem);
    float2* xs = reinterpret_cast<float2*> (smem + P::LAND_BYTES);
    float2* xh = xs - M / 2;                                 // half-spectrum exchange: bin k >= M/2 at xh[k], unit stride
    float2* tws = reinterpret_cast<float2*> (smem + P::TW_OFFSET);
    float2* tw1s = reinterpret_cast<float2*> (smem + P::TW1_OFFSET);
    unsigned long long* bar = reinterpret_cast<unsigned long long*> (smem + P::BAR_OFFSET);

    const int j = (int) threadIdx.x;
    const UPos<G, 3> up (j);
    {   // last-stage twiddle rows: global table row q-1 (T entries each, see Geo) -> shared row i
        const float2* __restrict__ tl = a.tw + G::tw_off (G::S - 1) + j;
#pragma unroll
        for (int i = 0; i < P::TW_ROWS; ++i)
            sts2 (tws + i * T + j, __ldg (tl + (P::tw_row_q (i) - 1) * T));
    }
    // real split / merge twiddle of this thread's first bin, w_j / 2; the others are w_(j + m T) = w_j W_64^m
    float2 wj = make_float2 (0.f, 0.f);
    if constexpr (KIND == R2C || KIND == C2R)
        wj = __ldg (a.rtw + j);
    const Stage1Tw w1t = load_stage1_tw<G> (j, a.tw, tw1s);
    const long long step = (long long) gridDim.x;
    long long x = (long long) blockIdx.x;
    if (j == 0)
        mbar_init (bar);
    __syncthreads();
    if (x < a.batch)
        pipe_fetch<P> (smem, a.in + x * a.in_inner, j, bar);

    for (unsigned it = 0; x < a.batch; x += step, ++it)
    {
        float2 v[R];
        mbar_wait (bar, it, PHASE_BYTES);
        // ---- prologue: stage-0 registers v[m] = input element j + m T, from the landing buffer ----
        if constexpr (KIND == C2C_FWD || KIND == R2C || (KIND == C2C_BWD && ! P::IN_UNORD))
        {
            const float2* lj = land + j;
#pragma unroll
            for (int m = 0; m < R; ++m)
                v[m] = lds2 (lj + m * T);
        }
        else if constexpr (KIND == C2C_BWD)
        {
            const float* lf = reinterpret_cast<const float*> (land);
#pragma unroll
            for (int m = 0; m < R; ++m)
                v[m] = staged_load (lf, up.cplx (m), WL);
        }
        else
        {
            // merge step  Z'[k] = (X[k] + X*[M-k]) + i conj(w_k) (X[k] - X*[M-k]),  w_k = e^{-2 pi i k / 2M}, as fft_kernel
            // forms it (same bits): the pair (k, M-k), k = j + m T < M/2, comes from the landing buffer (ordered) or the
            // staging image; Z'[k] is this thread's register m, Z'[M-k] belongs to thread T-j and crosses the exchange region
            const float* lf = reinterpret_cast<const float*> (land);
            const float2 two = make_float2 (2.f, 2.f);
            __syncthreads(); // the previous iteration's last round_gather is done everywhere: xh may be overwritten
#pragma unroll
            for (int m = 0; m < R / 2; ++m)
            {
                const bool special = (m == 0 && j == 0);
                float2 xa, xm;
                if constexpr (P::IN_UNORD)
                {
                    xa = staged_load (lf, up.real_lo (m), WL);
                    xm = staged_load (lf, special ? W_HALF_ROW<3>() : up.real_hi (m), WL);
                }
                else
                {
                    xa = lds2 (land + j + m * T);
                    xm = lds2 (special ? land + M / 2 : land + (M - m * T) - j);
                }
                const float2 wh = real_tw<32, kPipeDeriveRtw> (wj, a.rtw + j + m * T, m);
                const float2 cm = make_float2 (xm.x, -xm.y);
                const float2 e = f2_add (xa, cm), d = f2_sub (xa, cm);
                const float2 wd = cmul_dir<+1> (d, wh);
                float2 zk = f2_fma (make_float2 (-wd.y, wd.x), two, e);
                float2 zm = f2_fma (make_float2 (wd.y, wd.x), two, make_float2 (e.x, -e.y));
                if (special)
                {
                    zk = make_float2 (xa.x + xa.y, xa.x - xa.y);   // Z'[0] from (DC, Nyquist)
                    zm = make_float2 (2.f * xm.x, -2.f * xm.y);    // Z'[M/2] = 2 conj X[M/2]
                }
                v[m] = zk;
                sts2 (special ? xh + M / 2 : xh + (M - m * T) - j, zm);
            }
            __syncthreads();
#pragma unroll
            for (int m = R / 2; m < R; ++m)
                v[m] = lds2 (xh + j + m * T);
        }
        // ---- stage 0, full 64-bit exchange through [landing | exchange] (padded, M + M/32 slots) ----
        stage_compute<G, DIR, 0> (v, j, a.tw);
        __syncthreads(); // the landing buffer has been consumed, and the previous iteration is done with xs
        stage_scatter<G, 0> (v, j, land);
        __syncthreads();
        gather_natural<G, 0, R> (v, j, land);
        __syncthreads(); // landing buffer free again: fetch the next transform while this one finishes
        if (x + step < a.batch)
            pipe_fetch<P> (smem, a.in + (x + step) * a.in_inner, j, bar);
        // ---- stage 1, two-round exchange through the exchange region alone ----
        pipe_stage1<DIR> (v, w1t, tw1s + (j & 31));
        {
            float2 n[R]; // the gathered values land in fresh registers: v[16..31] are still needed by round 1
            round_scatter<G, 0> (v, j, xs);
            __syncthreads();
            round_gather<G, 0> (n, j, xs);
            __syncthreads();
            round_scatter<G, 1> (v, j, xs);
            __syncthreads();
            round_gather<G, 1> (n, j, xs);
#pragma unroll
            for (int m = 0; m < R; ++m)
                v[m] = n[m];
        }
        // ---- last stage ----
        pipe_last_stage<P, DIR> (v, j, tws);

        // ---- epilogue ----
        float* out = a.out + x * a.out_inner;
        if constexpr (KIND == C2C_BWD || KIND == C2R || (KIND == C2C_FWD && ! P::OUT_UNORD))
        {
            float2* __restrict__ out2 = reinterpret_cast<float2*> (out) + j;
#pragma unroll
            for (int m = 0; m < R; ++m)
                pipe_stg<LOGM> (out2 + m * T, v[m]);
        }
        else if constexpr (KIND == C2C_FWD && CFB_UNORD_DIRECT != 0)
        {
            // unordered complex output straight from registers (as fft_core's UDIRECT path): threads j, j+1 swap one float, the
            // even one stores (re_j, re_j+1), the odd one (im_j, im_j+1) -- contiguous 8-byte pairs of the unordered layout
            constexpr int UW = 8, ULT = R / UW;
            const int u_odd = j & 1;
            float* __restrict__ ob = out + (((j & ~1) >> 3) * 2 * UW * UW) + ((j & ~1) & (UW - 1)) + (u_odd ? UW : 0);
#pragma unroll
            for (int m = 0; m < R; ++m)
            {
                const float recv = shfl1 (u_odd ? v[m].x : v[m].y, (j ^ 1) & 31, 32);
                const float2 o = u_odd ? make_float2 (recv, v[m].y) : make_float2 (v[m].x, recv);
                *reinterpret_cast<float2*> (ob + (m % ULT) * (T / UW) * 2 * UW * UW + (m / ULT) * 2 * UW) = o;
            }
        }
        else if constexpr (KIND == C2C_FWD)
        {
            // unordered output, staged and drained in two halves of the (padded) image: bin j + m T lies in half
            // (m mod 4) / 2 (UPos::cplx: block index = j / 8 + (m mod 4) T / 8, M / 64 blocks per half)
            float* sf = reinterpret_cast<float*> (xs);
#pragma unroll
            for (int h = 0; h < 2; ++h)
            {
                __syncthreads(); // the exchange region (or the previous half) has been read by everyone
#pragma unroll
                for (int m = 0; m < R; ++m)
                    if ((m % 4) / 2 == h)
                        staged_store (sf, up.cplx (m) - h * P::HALF_IMAGE_FLOATS, WL, v[m]);
                __syncthreads();
                half_drain<P> (sf, out + h * M, j);
            }
        }
        else
        {
            // split step  X[k] = E - i w_k D,  X[M-k] = conj(E + i w_k D),  E,D = (Z[k] +- Z*[M-k]) / 2.
            // Z[k], k = j + m T < M/2, is register m; Z[M-k] is register R-1-m of thread T-j: the upper half of the
            // spectrum crosses the exchange region (unit stride on both sides, no padding needed).
            __syncthreads();
#pragma unroll
            for (int m = R / 2; m < R; ++m)
                sts2 (xh + j + m * T, v[m]);
            __syncthreads();
            float2 zb[R / 2];
#pragma unroll
            for (int m = 0; m < R / 2; ++m)
                zb[m] = lds2 ((m == 0 && j == 0) ? xh + M / 2 : xh + (M - m * T) - j);
            float2* __restrict__ lo = reinterpret_cast<float2*> (out) + j;
            float2* __restrict__ hi = reinterpret_cast<float2*> (out) + (M - T) - j;
            float2 xlo[P::OUT_UNORD ? R / 2 : 1], xhi[P::OUT_UNORD ? R / 2 : 1];
#pragma unroll
            for (int m = 0; m < R / 2; ++m)
            {
                const float2 za = v[m], zm = zb[m];
                const float2 wh = real_tw<32, kPipeDeriveRtw> (wj, a.rtw + j + m * T, m);
                const float2 cm = make_float2 (zm.x, -zm.y);
                const float2 e = f2_add (za, cm), d = f2_sub (za, cm);
                const float2 wd = cmul_dir<-1> (d, wh);
                float2 xa = f2_fma (e, make_float2 (0.5f, 0.5f), make_float2 (wd.y, -wd.x));
                float2 xm = f2_fma (e, make_float2 (0.5f, -0.5f), make_float2 (-wd.y, -wd.x));
                const bool special = (m == 0 && j == 0);
                if (special)
                {
                    xa = make_float2 (za.x + za.y, za.x - za.y);
                    xm = make_float2 (zm.x, -zm.y);
                }
                if constexpr (P::OUT_UNORD)
                {
                    xlo[m] = xa;
                    xhi[m] = xm;
                }
                else
                {
                    lo[m * T] = xa;
                    float2* ph = special ? reinterpret_cast<float2*> (out) + M / 2 : hi - m * T + T;
                    *ph = xm;
                }
            }
            if constexpr (P::OUT_UNORD)
            {
                // which half of the image a bin falls in depends on the thread for a few bins (the reversed odd rows
                // wrap at thread 0), so the half is tested on the position itself
                float* sf = reinterpret_cast<float*> (xs);
#pragma unroll
                for (int h = 0; h < 2; ++h)
                {
                    __syncthreads();
#pragma unroll
                    for (int m = 0; m < R / 2; ++m)
                    {
                        const int plo = up.real_lo (m);
                        const int phi = (m == 0 && j == 0) ? W_HALF_ROW<3>() : up.real_hi (m);
                        if ((plo >= P::HALF_IMAGE_FLOATS) == (h == 1))
                            staged_store (sf, plo - h * P::HALF_IMAGE_FLOATS, WL, xlo[m]);
                        else
                        {
                            smem_skip();
                            smem_skip();
                        }
                        if ((phi >= P::HALF_IMAGE_FLOATS) == (h == 1))
                            staged_store (sf, phi - h * P::HALF_IMAGE_FLOATS, WL, xhi[m]);
                        else
                        {
                            smem_skip();
                            smem_skip();
                        }
                    }
                    __syncthreads();
                    half_drain<P> (sf, out + h * M, j);
                }
            }
        }
    }
}

template <int LOGM, int KIND, int LOGW>
__global__ void __launch_bounds__ (PipeGeo<LOGM>::T, PipeGeo<LOGM, KIND, LOGW>::CTAS_PER_SM) pipe_kernel (const FftArgs a)
{
    pipe_body<LOGM, KIND, LOGW> (a);
}
} // namespace cfb
