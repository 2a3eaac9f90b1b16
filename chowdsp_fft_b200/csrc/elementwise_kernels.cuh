// Unordered-domain elementwise kernels: the frequency-domain multiply-accumulate behind
// fft_convolve_unordered and the plain sum behind fft_accumulate, and the streaming convolver's helpers
// (argument structs in pconv_kernel.cuh).  Pure HBM streaming.
#pragma once
#include "fft_kernels.cuh"
#include "pconv_kernel.cuh"

namespace cfb
{
// ---------------------------------------------------------------------------------------------
// unordered-domain elementwise kernels
// ---------------------------------------------------------------------------------------------
struct ConvArgs
{
    const float* a;
    const float* b;
    float* ab;
    long long a_stride, b_stride, ab_stride; // floats between consecutive spectra (0 = shared operand)
    int nfloats;                             // floats per spectrum (N real, 2N complex)
    int batch;
    int logW;
    int is_real;                             // DC / Nyquist are two real products (avx:1974-1978)
    float scaling;
};

// ab += a * b * scaling on (W re | W im) vector pairs -- pffft_convolve_internal,
// /root/reference/simd/chowdsp_fft_impl_avx.cpp:1937-1979.  One thread per 4 re + 4 im floats.
__global__ void __launch_bounds__ (256) convolve_kernel (const ConvArgs p)
{
    const int W = 1 << p.logW;
    const int quads = p.nfloats >> 3; // work items per spectrum
    const long long total = (long long) quads * p.batch;
    for (long long i = (long long) blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long) gridDim.x * blockDim.x)
    {
        const long long x = i / quads;
        const int q = (int) (i - x * quads);
        // W = 8: two quads per 16-float chunk;  W = 4: one quad per 8-float chunk
        const int off = p.logW == 3 ? ((q >> 1) * 16 + (q & 1) * 4) : q * 8;
        // plain loads: a, b and ab may alias (chowdsp_fft.h:153)
        const float4 ar = *reinterpret_cast<const float4*> (p.a + x * p.a_stride + off);
        const float4 ai = *reinterpret_cast<const float4*> (p.a + x * p.a_stride + off + W);
        const float4 br = *reinterpret_cast<const float4*> (p.b + x * p.b_stride + off);
        const float4 bi = *reinterpret_cast<const float4*> (p.b + x * p.b_stride + off + W);
        float4* pr = reinterpret_cast<float4*> (p.ab + x * p.ab_stride + off);
        float4* pi = reinterpret_cast<float4*> (p.ab + x * p.ab_stride + off + W);
        float4 cr = *pr, ci = *pi;
        const float s = p.scaling;
        const float dc = cr.x + (ar.x * br.x) * s, ny = ci.x + (ai.x * bi.x) * s;
        cr.x += (ar.x * br.x - ai.x * bi.x) * s; ci.x += (ar.x * bi.x + ai.x * br.x) * s;
        cr.y += (ar.y * br.y - ai.y * bi.y) * s; ci.y += (ar.y * bi.y + ai.y * br.y) * s;
        cr.z += (ar.z * br.z - ai.z * bi.z) * s; ci.z += (ar.z * bi.z + ai.z * br.z) * s;
        cr.w += (ar.w * br.w - ai.w * bi.w) * s; ci.w += (ar.w * bi.w + ai.w * br.w) * s;
        if (p.is_real && q == 0)
        {
            cr.x = dc;
            ci.x = ny;
        }
        *pr = cr;
        *pi = ci;
    }
}

// ab = a + b -- fft_accumulate_internal, avx:1981-1994
__global__ void __launch_bounds__ (256) accumulate_kernel (const float* a, const float* b, float* ab, long long n4)
{
    for (long long i = (long long) blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long) gridDim.x * blockDim.x)
    {
        const float4 x = reinterpret_cast<const float4*> (a)[i], y = reinterpret_cast<const float4*> (b)[i];
        reinterpret_cast<float4*> (ab)[i] = make_float4 (x.x + y.x, x.y + y.y, x.z + y.z, x.w + y.w);
    }
}

// JUCE convention for real spectra when the caller wants the redundant negative frequencies as well
// (chowdsp_fft_juce.cpp:58-61): bin M + i = conj (bin M - i), i = 1 .. M-1, rows of 2 M complex bins
__global__ void __launch_bounds__ (256) juce_mirror_kernel (float* data, long long stride, int M, long long total)
{
    for (long long t = (long long) blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long) gridDim.x * blockDim.x)
    {
        const long long row = t / (M - 1);
        const int i = 1 + (int) (t - row * (M - 1));
        float2* d = reinterpret_cast<float2*> (data + row * stride);
        const float2 v = d[M - i];
        d[M + i] = make_float2 (v.x, -v.y);
    }
}

// ---------------------------------------------------------------------------------------------
// streaming convolver (fft_convolver_*)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__ (256) pconv_slice_kernel (const PConvSliceArgs a)
{
    const long long item = (long long) blockIdx.x * blockDim.x + threadIdx.x;
    if (item >= (long long) a.channels * a.pairs)
        return;
    const int c = (int) (item / a.pairs), pr = a.pair0 + (int) (item % a.pairs);
    const int W = 1 << a.logW, lq = a.logW - 2;
    const int off = ((pr >> lq) << (a.logW + 1)) + ((pr & ((1 << lq) - 1)) << 2);
    const float* irc = a.ir + (long long) c * a.ir_ch_stride + off;
    const float* fdlc = a.fdl + (long long) c * a.fdl_ch_stride + off;
    float4 ar = make_float4 (0.f, 0.f, 0.f, 0.f), ai = ar;
    float dc = 0.f, ny = 0.f;
    int g = (a.q - 1 + a.P) % a.P; // slot of X_(q-1)
    for (int p = 1; p < a.P; ++p)
    {
        const float* h = irc + (long long) p * a.N;
        const float* xs = fdlc + (long long) g * a.N;
        const float4 hr = ld_stream4 (h), hi = ld_stream4 (h + W), xr = ld_stream4 (xs), xi = ld_stream4 (xs + W);
        dc = fmaf (xr.x, hr.x, dc);
        ny = fmaf (xi.x, hi.x, ny);
        cmac4 (ar, ai, xr, xi, hr, hi);
        g = g == 0 ? a.P - 1 : g - 1;
    }
    if (pr == 0)
    {
        ar.x = dc;
        ai.x = ny;
    }
    float* sc = a.S + (long long) c * a.s_stride + off;
    *reinterpret_cast<float4*> (sc) = ar;
    *reinterpret_cast<float4*> (sc + W) = ai;
}

__global__ void __launch_bounds__ (256) conv_input_kernel (const ConvInputArgs a)
{
    const long long item = (long long) blockIdx.x * blockDim.x + threadIdx.x;
    if (item >= (long long) a.channels * a.half_block)
        return;
    const long long c = item / a.half_block, k = item % a.half_block;
    const float2 v = *reinterpret_cast<const float2*> (a.in + c * a.in_stride + 2 * k);
    float* h = a.hist + c * a.hist_stride + a.pos + 2 * k;
    *reinterpret_cast<float2*> (h) = v;
    *reinterpret_cast<float2*> (h + a.mirror) = v;
}

__global__ void __launch_bounds__ (256) conv_ir_gather_kernel (const ConvIrArgs a)
{
    const long long n2 = 2LL * a.Bk, total = (long long) a.channels * a.P * n2;
    for (long long item = (long long) blockIdx.x * blockDim.x + threadIdx.x; item < total; item += (long long) gridDim.x * blockDim.x)
    {
        const long long i = item % n2, cp = item / n2, p = cp % a.P, c = cp / a.P;
        const long long tap = a.start + p * a.Bk + i;
        a.dst[item] = (i < a.Bk && tap < a.length) ? a.ir[c * a.ir_stride + tap] : 0.f;
    }
}
} // namespace cfb
