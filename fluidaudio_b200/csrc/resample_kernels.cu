// Device-side AudioConverter stage: PCM (float32 / int16, any channel count, planar or interleaved, any rate) ->
// mono float32 at the model rate, written straight into the buffer the log-mel kernel reads (no host round trip).
// See resample_plan.h for the reference lines and the filter design.
#include "resample_plan.h"

#include <algorithm>
#include <cmath>
#include <numeric>

namespace fa {
namespace resample {

#define FA_CUDA_TRY(expr)                                                                   \
    do {                                                                                    \
        cudaError_t e__ = (expr);                                                           \
        if (e__ != cudaSuccess) {                                                           \
            fa::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
            return FA_CUDA_ERROR;                                                           \
        }                                                                                   \
    } while (0)

// ------------------------------------------------------------------------------------------------ design (host)
bool rational_ratio(double in_rate, double out_rate, long long &L, long long &M) {
    double scale = 1.0;
    if (std::fabs(in_rate - std::round(in_rate)) > 1e-9 || std::fabs(out_rate - std::round(out_rate)) > 1e-9) scale = 1000.0;
    const long long a = (long long)std::llround(out_rate * scale), b = (long long)std::llround(in_rate * scale);
    if (a <= 0 || b <= 0) return false;
    const long long g = std::gcd(a, b);
    L = a / g;
    M = b / g;
    return std::fabs((double)a / scale - out_rate) < 1e-6 && std::fabs((double)b / scale - in_rate) < 1e-6;
}

static double bessel_i0(double x) {   // power series, converges for every x; 60 terms are exact to double for x <= 20
    double sum = 1.0, term = 1.0;
    const double q = 0.25 * x * x;
    for (int k = 1; k < 200; ++k) {
        term *= q / ((double)k * (double)k);
        sum += term;
        if (term < 1e-18 * sum) break;
    }
    return sum;
}

int make_design(double in_rate, double out_rate, Design &d) {
    if (!(in_rate > 0) || !(out_rate > 0)) return FA_INVALID_ARGUMENT;
    if (!rational_ratio(in_rate, out_rate, d.L, d.M)) {
        fa::set_error("sample rates %.6f -> %.6f are not on a 1/1000 Hz grid", in_rate, out_rate);
        return FA_UNSUPPORTED;
    }
    const double lower = std::min(1.0, (double)d.L / (double)d.M);
    d.fc = lower * kRolloff;
    d.half = (int)std::ceil((double)kZeros / lower);
    d.taps = 2 * d.half;
    d.exact = d.L <= kMaxExactPhases;
    d.phases = d.exact ? (int)d.L : kInterpPhases;
    if ((255.0 * (double)d.M / (double)d.L + d.taps + 8) * sizeof(float) > 200.0 * 1024.0) {
        fa::set_error("resampling ratio %lld/%lld needs a filter window larger than shared memory", d.L, d.M);
        return FA_UNSUPPORTED;
    }
    const int rows = d.exact ? d.phases : d.phases + 1;
    d.row_stride = (d.taps + 3) & ~3;   // rows padded with zero taps to whole float4s (16-byte aligned coefficient loads)
    d.table.assign((size_t)rows * d.row_stride, 0.0f);
    const double pi = 3.14159265358979323846, i0b = bessel_i0(kBeta);
    std::vector<double> row(d.taps);
    for (int p = 0; p < rows; ++p) {
        const double frac = (double)p / (double)d.phases;
        double sum = 0.0;
        for (int k = 0; k < d.taps; ++k) {
            const double t = (double)(k - d.half + 1) - frac;   // input sample n0 - H + 1 + k sits at offset t from the output
            double g = 0.0;
            if (std::fabs(t) < (double)d.half) {
                const double x = pi * d.fc * t;
                const double s = std::fabs(x) < 1e-12 ? 1.0 : std::sin(x) / x;
                const double u = t / (double)d.half;
                g = d.fc * s * bessel_i0(kBeta * std::sqrt(std::max(0.0, 1.0 - u * u))) / i0b;
            }
            row[k] = g;
            sum += g;
        }
        for (int k = 0; k < d.taps; ++k) d.table[(size_t)p * d.row_stride + k] = (float)(row[k] / sum);
    }
    return FA_OK;
}

long long output_count(long long frames, double in_rate, double out_rate) {
    if (in_rate == out_rate) return frames;
    const double ratio = in_rate / out_rate;
    return (long long)((double)frames / ratio);   // AudioConverter.swift:417-418
}

bool is_identity(const AudioFormat &f) {
    return f.in_rate == f.out_rate && f.channels == 1 && f.format == kPcmF32;
}

int resolve_algorithm(const AudioFormat &f) {
    if (f.algorithm == kAlgoSinc || f.algorithm == kAlgoLinear) return f.algorithm;
    return f.channels > 2 ? kAlgoLinear : kAlgoSinc;
}

long long outputs_ready(const AudioFormat &f, const Design &d, long long frames, long long frames_avail,
                        long long out_total) {
    if (frames_avail >= frames) return out_total;
    long long ready;
    if (f.in_rate == f.out_rate) ready = frames_avail;
    else if (resolve_algorithm(f) == kAlgoLinear) ready = (long long)((double)(frames_avail - 2) / (f.in_rate / f.out_rate)) - 1;
    else ready = ((frames_avail - d.half - 1) * d.L) / d.M - 1;   // n0(i) + H < frames_avail
    return std::max(0LL, std::min(ready, out_total));
}

// ------------------------------------------------------------------------------------------------ kernels
struct Source {
    const void *pcm;
    long long frames;
    int channels;
    int format;
    int interleaved;
    float weight;   // 1 / channels (float32, AudioConverter.swift:401)
};

// mono sample n: float32 sum over channels in channel order, times 1/channels (AudioConverter.swift:403-409).
// int16 is widened like AVAudioPCMBuffer's int16 -> float conversion: v / 32768.
__device__ __forceinline__ float mono_at(const Source &s, long long n) {
    if (s.channels == 1)   // the common mono cases without the channel loop
        return s.format == kPcmI16 ? (float)__ldg(reinterpret_cast<const short *>(s.pcm) + n) * (1.0f / 32768.0f)
                                   : __ldg(reinterpret_cast<const float *>(s.pcm) + n);
    if (s.channels == 2 && s.interleaved && s.format == kPcmI16) {   // stereo WAV: one 32-bit load per frame
        const short2 v = __ldg(reinterpret_cast<const short2 *>(s.pcm) + n);
        return __fmul_rn(__fadd_rn(__fadd_rn(0.0f, (float)v.x * (1.0f / 32768.0f)), (float)v.y * (1.0f / 32768.0f)), s.weight);
    }
    float sum = 0.0f;
    for (int c = 0; c < s.channels; ++c) {
        const long long at = s.interleaved ? n * s.channels + c : (long long)c * s.frames + n;
        const float v = s.format == kPcmI16 ? (float)__ldg(reinterpret_cast<const short *>(s.pcm) + at) * (1.0f / 32768.0f)
                                            : __ldg(reinterpret_cast<const float *>(s.pcm) + at);
        sum = __fadd_rn(sum, v);
    }
    return s.channels == 1 ? sum : __fmul_rn(sum, s.weight);
}

// same rate: mixdown / format conversion only
__global__ void __launch_bounds__(256) mixdown_kernel(Source s, float *out, long long o_begin, long long o_end) {
    const long long i = o_begin + (long long)blockIdx.x * 256 + threadIdx.x;
    if (i < o_end) out[i] = i < s.frames ? mono_at(s, i) : 0.0f;
}

// AudioConverter.linearResample (:417-434), float32 operations individually rounded, source position in double
__global__ void __launch_bounds__(256) linear_kernel(Source s, double ratio, float *out, long long o_begin, long long o_end) {
    const long long i = o_begin + (long long)blockIdx.x * 256 + threadIdx.x;
    if (i >= o_end) return;
    const double src = (double)i * ratio;
    const long long idx = (long long)src;
    const float frac = (float)(src - (double)idx);
    float v = 0.0f;
    if (idx < s.frames - 1)
        v = __fadd_rn(__fmul_rn(mono_at(s, idx), __fsub_rn(1.0f, frac)), __fmul_rn(mono_at(s, idx + 1), frac));
    else if (idx < s.frames)
        v = mono_at(s, idx);
    out[i] = v;
}

// Kaiser-windowed-sinc polyphase.  One CTA = 256 consecutive outputs; their input span (mixed down, widened) is staged
// in shared memory once, every thread then runs its 2H-tap dot product out of shared memory: coefficients as 16-byte
// loads through the read-only path (a single row when L == 1, i.e. integer decimation: every lane reads the same
// address), four independent accumulators, index arithmetic of type U relative to one 64-bit division per CTA.
// A thread's phase numerator is base_ph + threadIdx.x * M < L + 255 M.  Integer rates keep that below 2^32 (U = unsigned,
// 32-bit division); rates on the 1/1000 Hz grid do not (44100.001 Hz -> 16 kHz: L = 16 000 000, M = 44 100 001, and
// 255 M ~ 1.1e10), so those take U = unsigned long long (see sinc_needs_64bit).
template <typename U>
__global__ void __launch_bounds__(256)
sinc_kernel(Source s, long long L, long long M, int half, int phases, int exact, int row_stride,
            const float *__restrict__ tab, float *out, long long o_begin, long long o_end) {
    extern __shared__ float xs[];
    __shared__ long long base_n0;
    __shared__ U base_ph;
    const long long i0 = o_begin + (long long)blockIdx.x * 256;
    if (threadIdx.x == 0) {
        const long long num = i0 * M;
        base_n0 = num / L;
        base_ph = (U)(num - base_n0 * L);
    }
    __syncthreads();
    const U uL = (U)L, uM = (U)M;
    const int last = (int)(min(i0 + 255, o_end - 1) - i0);
    const long long n_lo = base_n0 - half + 1;
    const int span = (int)((base_ph + (U)last * uM) / uL) + 2 * half;
    for (int j = threadIdx.x; j < span + 4; j += 256) {
        const long long n = n_lo + j;
        xs[j] = (j < span && n >= 0 && n < s.frames) ? mono_at(s, n) : 0.0f;
    }
    __syncthreads();
    const long long i = i0 + threadIdx.x;
    if (i >= o_end) return;
    const U t = base_ph + (U)threadIdx.x * uM;
    const U dn = t / uL, ph = t - dn * uL;
    const float *x = xs + dn;          // input n0 - H + 1 + k sits at xs[dn + k]
    const int nq = row_stride >> 2;
    float a0 = 0.0f, a1 = 0.0f, a2 = 0.0f, a3 = 0.0f;
    if (exact) {
        const float4 *row = reinterpret_cast<const float4 *>(tab + (size_t)ph * row_stride);
#pragma unroll 4
        for (int q = 0; q < nq; ++q) {
            const float4 c = __ldg(row + q);
            a0 = fmaf(c.x, x[4 * q], a0);
            a1 = fmaf(c.y, x[4 * q + 1], a1);
            a2 = fmaf(c.z, x[4 * q + 2], a2);
            a3 = fmaf(c.w, x[4 * q + 3], a3);
        }
    } else {
        const double pos = (double)ph / (double)L * (double)phases;
        const int p = (int)pos;
        const float a = (float)(pos - (double)p);
        const float4 *r0 = reinterpret_cast<const float4 *>(tab + (size_t)p * row_stride), *r1 = r0 + nq;
#pragma unroll 2
        for (int q = 0; q < nq; ++q) {
            const float4 c0 = __ldg(r0 + q), c1 = __ldg(r1 + q);
            a0 = fmaf(fmaf(a, c1.x - c0.x, c0.x), x[4 * q], a0);
            a1 = fmaf(fmaf(a, c1.y - c0.y, c0.y), x[4 * q + 1], a1);
            a2 = fmaf(fmaf(a, c1.z - c0.z, c0.z), x[4 * q + 2], a2);
            a3 = fmaf(fmaf(a, c1.w - c0.w, c0.w), x[4 * q + 3], a3);
        }
    }
    out[i] = (a0 + a1) + (a2 + a3);
}

// L + 255 M (the largest phase numerator of a CTA, see sinc_kernel) does not fit 32 bits
static bool sinc_needs_64bit(const Design &d) { return (unsigned long long)d.L + 255ull * (unsigned long long)d.M > 0xffffffffull; }

int launch_convert(const void *d_pcm, long long frames, const AudioFormat &f, const Design &d, const float *d_tab,
                   float *d_out, long long o_begin, long long o_end, cudaStream_t stream, long long *launches) {
    if (o_end <= o_begin) return FA_OK;
    Source s{d_pcm, frames, f.channels, f.format, f.interleaved, 1.0f / (float)f.channels};
    const unsigned grid = (unsigned)((o_end - o_begin + 255) / 256);
    if (f.in_rate == f.out_rate) {
        mixdown_kernel<<<grid, 256, 0, stream>>>(s, d_out, o_begin, o_end);
    } else if (resolve_algorithm(f) == kAlgoLinear) {
        linear_kernel<<<grid, 256, 0, stream>>>(s, f.in_rate / f.out_rate, d_out, o_begin, o_end);
    } else {
        const size_t smem = sizeof(float) * (size_t)((255 * d.M) / d.L + d.taps + 12);
        auto *kernel = sinc_needs_64bit(d) ? sinc_kernel<unsigned long long> : sinc_kernel<unsigned>;
        if (smem > 48 * 1024)
            FA_CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kernel<<<grid, 256, smem, stream>>>(s, d.L, d.M, d.half, d.phases, d.exact ? 1 : 0, d.row_stride, d_tab, d_out,
                                            o_begin, o_end);
    }
    FA_CUDA_TRY(cudaGetLastError());
    if (launches) ++*launches;
    return FA_OK;
}

} // namespace resample
} // namespace fa
