// Fused log-mel frontend for sm_100a:  pre-emphasis -> Hann window -> 512-point real FFT -> |.|^2 ->
// Slaney mel filterbank -> log, one persistent CTA per SM.
//
// Re-implements Sources/FluidAudio/Shared/AudioMelSpectrogram.swift:325-456 (computeFlatTransposed),
// :185-292 (computeFlat) and :132-178 (compute) — the three differ only in (pad, window offset, pre-emphasis,
// output layout), which are kernel parameters here.
//
// Data flow per tile of kTileFrames (16) frames, two CTAs of 8 warps per SM so that one CTA's FP64 transform phase
// overlaps the other's float32 mel/log phase and barrier waits:
//   HBM --cp.async.bulk (TMA 1-D, mbarrier complete_tx)--> raw[2]   double-buffered, prefetched one tile ahead
//   raw --pre-emphasis--> ptile                                       all threads
//   ptile --one warp per frame: FFT256 + recombination--> power[32][257]
//   power --lane = frame, warp = mel: banded dot + log--> otile / HBM
// The transform runs in FP64 (see mel_core.cuh for why), everything the reference does in float32 stays float32.
// HBM traffic is the algorithmic minimum: every sample is read once (plus a 352-sample halo per tile) and
// every log-mel value is written once, both fully coalesced.
//
// The mel filterbank is applied as a BANDED contraction on the FP32 pipe, not as a tensor-core GEMM: each
// FFT bin feeds at most two triangular filters, so the dense [T x 257] x [257 x nMels] product is >97 % zeros
// (514 useful MACs per frame out of 20 560 at 80 mels), and bf16 operands cannot meet the 1e-4 log-mel parity
// bound (SURVEY.md §7 H3).  See DESIGN.md §4.
#include "mel_core.cuh"
#include "mel_plan.h"

#include <cuda_runtime.h>
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

namespace fa {
namespace mel {

// ------------------------------------------------------------------------------------------------ PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {
    }
}
// 1-D bulk copy global -> shared (TMA engine), completion signalled on an mbarrier.  SASS: UBLKCP.
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ------------------------------------------------------------------------------------------------ kernel
struct TileGeom {
    int unit;          // index into units[]
    long long f0;      // first frame of the tile (absolute frame index inside the clip)
    int nf;            // frames in this tile (1..32)
    long long a0;      // audio index of ptile[0]  (= f0*hop - pad)
    long long base;    // audio index of raw[0]    (= floor4(a0 - 1), may be negative)
    long long gs, ge;  // bulk-copied audio range [gs, ge), both multiples of 4 (empty if ge <= gs)
};

__device__ __forceinline__ const MelUnit &unit_at(const MelLaunch &P, int idx) { return P.inline_unit ? P.unit0 : P.units[idx]; }

__device__ __forceinline__ TileGeom tile_geom(const MelLaunch &P, int tile) {
    // units are sorted by tile_begin; binary search for the unit that owns this tile
    int lo = 0, hi = P.inline_unit ? 0 : P.num_units - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (P.units[mid].tile_begin <= tile) lo = mid; else hi = mid - 1;
    }
    const MelUnit &u = P.inline_unit ? P.unit0 : P.units[lo];
    TileGeom g;
    g.unit = lo;
    g.f0 = u.frame_begin + (long long)kTileFrames * (tile - u.tile_begin);
    const long long rem = u.frame_begin + u.frame_count - g.f0;
    g.nf = rem < kTileFrames ? (int)rem : kTileFrames;
    g.a0 = g.f0 * P.hop - P.pad;
    const long long need0 = g.a0 - 1;
    g.base = (need0 >= 0) ? (need0 & ~3LL) : -(((-need0) + 3) & ~3LL);
    long long ge = (g.a0 + P.pt_len + 3) & ~3LL;
    const long long n4 = u.n & ~3LL;
    if (ge > n4) ge = n4;
    g.gs = g.base < 0 ? 0 : g.base;
    g.ge = ge;
    if (!P.use_tma) g.ge = g.gs;   // nothing is bulk-copied: every sample comes through the read-only path
    return g;
}

// Geometry + the unit fields a tile needs, computed ONCE per tile by thread 0 and broadcast through shared memory (three
// rotating slots): every thread recomputing it (binary search, 64-bit index math, a 56-byte struct copy) three times per
// tile was 6 % of the kernel's instructions (profiles/r02_mel.md).
struct TileInfo {
    TileGeom g;
    long long audio_off, n, out_off, out_stride;
    float last;
    int pad_;
};
__device__ __forceinline__ void make_tile_info(const MelLaunch &P, int tile, TileInfo &ti) {
    ti.g = tile_geom(P, tile);
    const MelUnit &u = unit_at(P, ti.g.unit);
    ti.audio_off = u.audio_off;
    ti.n = u.n;
    ti.out_off = u.out_off;
    ti.out_stride = u.out_stride;
    ti.last = u.last;
}

template <int kWarps, typename V, int kLayout>   // kLayout: 0 time-major [T x nMels], 1 mel-major [nMels x stride]
__global__ void __launch_bounds__(kWarps * 32, 2) mel512_kernel(const MelLaunch P) {
    constexpr int kF = vtraits<V>::kFrames;   // frames one warp transforms together (2: packed float32 pairs)
    extern __shared__ __align__(128) unsigned char smem[];
    float *raw0 = reinterpret_cast<float *>(smem);
    float *raw1 = raw0 + P.raw_cap;
    float *ptile = raw1 + P.raw_cap;
    cpxv<V> *fftbuf = reinterpret_cast<cpxv<V> *>(ptile + P.pt_cap);   // kWarps * kFftPad complex values (16 bytes each)
    float *power = reinterpret_cast<float *>(fftbuf + kWarps * kFftPad);   // (kTileFrames / 2) pair rows x kPairStride
    float *otile = power + (kTileFrames / 2) * kPairStride;  // kTileFrames rows of ot_stride floats
    const int ot_stride = P.ot_stride;                       // n_mels + 4 (rows stay 16-byte aligned) or n_mels + 1
    float *fbw = otile + kTileFrames * ot_stride;            // fb_nnz_cap
    int4 *fbmeta = reinterpret_cast<int4 *>(fbw + P.fb_cap);   // n_slots x {first bin, quads, weight offset, mel bin or -1}
    uint64_t *bars = reinterpret_cast<uint64_t *>(fbmeta + P.n_slots);
    TileInfo *tinfo = reinterpret_cast<TileInfo *>(bars + 2);   // [3]

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    if (tid == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int i = tid; i < P.fb_nnz; i += kWarps * 32) fbw[i] = P.fb_w[i];
    for (int i = tid; i < P.n_slots; i += kWarps * 32) fbmeta[i] = P.fb_slots[i];
    for (int i = tid; i < (kTileFrames / 2) * kPairStride; i += kWarps * 32) power[i] = 0.0f;   // rows of partial tiles, pad columns
    // per-lane constants (window slots, twiddles, butterfly addresses): built on the host once per plan (FP64 sin / cos
    // inlined here cost ~3 % of the kernel and 9 000 SASS lines), one struct copy per thread
    const LaneTables<V> T = reinterpret_cast<const LaneTables<V> *>(P.lane_tab)[lane];
    __syncthreads();

    cpxv<V> *buf = fftbuf + warp * kFftPad;

    auto issue = [&](int tile, int buf, TileInfo &slot) {   // thread 0 only: publishes the tile's info, starts its bulk copy
        make_tile_info(P, tile, slot);
        const TileGeom &g = slot.g;
        float *dst = buf ? raw1 : raw0;
        if (g.ge > g.gs) {
            const uint32_t bytes = (uint32_t)((g.ge - g.gs) * 4);
            mbar_expect_tx(&bars[buf], bytes);
            bulk_g2s(dst + (g.gs - g.base), P.audio + slot.audio_off + g.gs, bytes, &bars[buf]);
        } else {
            mbar_arrive(&bars[buf]);
        }
    };

    // pre-emphasis of one tile from its raw buffer into ptile (zero outside [0, n))
    auto preemphasize = [&](const TileInfo &u, const float *raw) {   // u.n / u.last / u.audio_off: the owning clip
        const TileGeom &g = u.g;
        const float a = P.preemph;
        const bool interior = g.a0 >= 1 && g.a0 - 1 >= g.gs && g.a0 + P.pt_len <= g.ge && g.a0 + P.pt_len <= u.n;
        if (interior) {
            // every sample of the tile and its predecessor came through the bulk copy (conflict-free, unit stride)
            const float *src = raw + (g.a0 - g.base);   // src[t] = x(a0 + t), src[-1] valid
            if (((g.a0 - g.base) & 3) == 0 && (P.pt_len & 3) == 0) {   // 16-byte aligned rows: four samples per step
                const float4 *s4 = reinterpret_cast<const float4 *>(src);
                float4 *d4 = reinterpret_cast<float4 *>(ptile);
                for (int q = tid; q < (P.pt_len >> 2); q += kWarps * 32) {
                    const float4 x = s4[q];
                    float4 y = x;
                    const float prev = src[4 * q - 1];   // (a shuffle from the neighbour lane saves 4 wavefronts per frame but costs
                                                         //  more instructions than it saves: measured 0.3135 vs 0.3096 ms)
                    if (a != 0.0f) {
                        y.x = preemph_rest(x.x, prev, a);
                        y.y = preemph_rest(x.y, x.x, a);
                        y.z = preemph_rest(x.z, x.y, a);
                        y.w = preemph_rest(x.w, x.z, a);
                    }
                    d4[q] = y;
                }
            } else if (a == 0.0f) {
                for (int t = tid; t < P.pt_len; t += kWarps * 32) ptile[t] = src[t];
            } else {
                for (int t = tid; t < P.pt_len; t += kWarps * 32) ptile[t] = preemph_rest(src[t], src[t - 1], a);
            }
        } else {
            const float *gaudio = P.audio + u.audio_off;
            auto sample = [&](long long i) -> float {   // x(i) for -1 <= i < n
                if (i >= g.gs && i < g.ge) return raw[i - g.base];
                if (i < 0) return u.last;
                return __ldg(gaudio + i);
            };
            for (int t = tid; t < P.pt_len; t += kWarps * 32) {
                const long long i = g.a0 + t;
                float v = 0.0f;
                if (i >= 0 && i < u.n) {
                    const float x = sample(i);
                    if (a == 0.0f) v = x;
                    else if (i == 0) v = preemph_first(x, u.last, a);
                    else v = preemph_rest(x, sample(i - 1), a);
                }
                ptile[t] = v;
            }
        }
    };
    // time-major tile is contiguous in HBM: nf rows of n_mels floats; flat, fully coalesced copy out of otile
    auto copy_out = [&](float *dst, int total) {
        if (P.vec_out) {   // rows are whole float4s and dst is 16-byte aligned (the unit's output is, and f0 is a multiple of 16)
            float4 *d4 = reinterpret_cast<float4 *>(dst);
            for (int q = tid; q < (total >> 2); q += kWarps * 32) {
                const int e = 4 * q;
                const int row = (int)__umulhi((unsigned)e, P.inv_n_mels);                  // e / n_mels
                d4[q] = *reinterpret_cast<const float4 *>(otile + e + 4 * row);             // row stride n_mels + 4: one LDS.128
            }
        } else {
            const int row_pad = ot_stride - P.n_mels;                        // 1, or 4 when a caller's output is not 16-byte aligned
            for (int idx = tid; idx < total; idx += kWarps * 32) {
                // idx / n_mels (exact for idx < 2^16); ceil(2^32 / 1) does not fit the 32-bit reciprocal
                const int fi = P.n_mels == 1 ? idx : (int)__umulhi((unsigned)idx, P.inv_n_mels);
                dst[idx] = otile[idx + fi * row_pad];                        // padded row stride n_mels + row_pad
            }
        }
    };

    // Software pipeline over the CTA's tiles, two block barriers per tile:
    //   phase A(i): copy-out of tile i-1 (otile -> HBM)  +  FFT of tile i (ptile -> power)
    //   phase B(i): mel + log of tile i (power -> otile)  +  pre-emphasis of tile i+1 (raw -> ptile), TMA for tile i+2
    // The bulk copy of a tile is issued two phases B ahead of its use, its raw buffer was last read one phase B earlier.
    const int first = blockIdx.x, stride = gridDim.x;
    if (first >= P.total_tiles) return;
    if (tid == 0) {
        issue(first, 0, tinfo[0]);
        if (first + stride < P.total_tiles) issue(first + stride, 1, tinfo[1]);
    }
    __syncthreads();
    mbar_wait(&bars[0], 0);
    preemphasize(tinfo[0], raw0);
    __syncthreads();
    float *pending_dst = nullptr;
    int pending_total = 0;
    int it = 0, slot = 0;   // slot = it % 3
    for (int tile = first; tile < P.total_tiles; tile += stride, ++it, slot = slot == 2 ? 0 : slot + 1) {
        const TileInfo &u = tinfo[slot];
        const int nf = u.g.nf;

        // ---- phase A: previous tile's copy-out, then one warp per frame (pair): FFT256 + recombination + power ----
        if (pending_dst) copy_out(pending_dst, pending_total);
        for (int fi = warp * kF; fi < nf; fi += kWarps * kF) {   // kF == 2: frames fi and fi + 1 (kTileFrames is even)
            const float *pf = ptile + fi * P.hop;
            V re[8], im[8];
            if (P.mid_full) pass1<true>(lane, pf, P.hop, T, buf); else pass1<false>(lane, pf, P.hop, T, buf);
            __syncwarp();
            pass2_load(lane, buf, re, im);
            __syncwarp();
            pass2_store(lane, T, re, im, buf);
            __syncwarp();
            pass3_post(lane, buf, T, power + (fi >> 1) * kPairStride + (fi & 1));   // pair row (+ slot on the FP64 path)
            __syncwarp();
        }
        __syncthreads();

        // ---- phase B: mel filterbank + log; a warp covers kTileFrames frames x (32 / kTileFrames) mel bins -------
        const int next = tile + stride;
        const int slot1 = slot == 2 ? 0 : slot + 1, slot2 = slot1 == 2 ? 0 : slot1 + 1;
        if (tid == 0 && next + stride < P.total_tiles) {
            fence_proxy_async();   // generic-proxy reads of this raw buffer (pre-emphasis, previous phase B) precede the async write
            issue(next + stride, it & 1, tinfo[slot2]);   // slot2 held tile it-1: nobody reads it any more
        }
        {
            constexpr int kPairs = kTileFrames / 2, kGroup = 32 / kPairs;   // lane = (frame pair, one of kGroup mel bins)
            const int pl = lane % kPairs, mg = lane / kPairs;
            const float *prow = power + pl * kPairStride;
            float *orow = otile + (2 * pl) * ot_stride;
            float *gout = kLayout == 1 ? P.out + u.out_off + u.g.f0 + 2 * pl : nullptr;   // mel-major: this pair's columns
            // slots, not mel bins: the plan deals the groups of four filters to the warps by band width (LPT), so that the
            // warp with the widest (highest) filters does not hold the block barrier; md.w = the slot's mel bin, -1 = empty
            for (int slot = warp * kGroup + mg; slot < P.n_slots; slot += kWarps * kGroup) {
                const int4 md = fbmeta[slot];
                // two frames per lane on packed FFMA2; rows beyond the tile's last frame hold finite leftovers: computed and
                // dropped, no divergent branch
                const float2 a2 = mel_dot_pairs(reinterpret_cast<const float4 *>(prow + 2 * md.x),
                                                reinterpret_cast<const float4 *>(fbw + md.z), md.y);
                const float v0 = log_value(a2.x, P.log_floor, P.log_clamped, P.log_normal),
                            v1 = log_value(a2.y, P.log_floor, P.log_clamped, P.log_normal);
                const int m = md.w;
                if (m < 0) continue;
                if (kLayout == 0) {
                    orow[m] = v0;
                    orow[ot_stride + m] = v1;
                } else {
                    float *g = gout + (long long)m * u.out_stride;
                    if (2 * pl < nf) g[0] = v0;
                    if (2 * pl + 1 < nf) g[1] = v1;
                }
            }
        }
        if (kLayout == 0) {
            pending_dst = P.out + u.out_off + u.g.f0 * P.n_mels;
            pending_total = nf * P.n_mels;
        }
        if (next < P.total_tiles) {
            const int nb = (it + 1) & 1;
            mbar_wait(&bars[nb], (uint32_t)((it + 1) >> 1) & 1u);
            preemphasize(tinfo[slot1], nb ? raw1 : raw0);
        }
        __syncthreads();
    }
    if (pending_dst) copy_out(pending_dst, pending_total);
}


// ------------------------------------------------------------------------------------------------ any-nFFT kernel
// AudioMelSpectrogram is parametric (AudioMelSpectrogram.swift:59-70) and LS-EEND derives nFFT = nextPow2(winLength)
// (Diarizer/LS-EEND/LSEENDTypes.swift:55-57): nFFT other than 512, or an odd hop, take this kernel.  Same contract, same
// unit / tile bookkeeping and the same packed filterbank as mel512_kernel; one warp per frame, the transform an FP64
// radix-2 decimation-in-time FFT of the real frame in shared memory (twiddles from an FP64 table), power rounded once
// to float32.  A correctness-first path: ~6x the instructions per frame of the specialised kernel.
struct GenericParams {
    int n_fft, log2n, bins, prow;      // prow: floats per power row (bins rounded up to quads + 4)
    const cpxd *tw;                    // W_n^k, k < n/2
    int warps;
};

__global__ void __launch_bounds__(256) mel_generic_kernel(const MelLaunch P, const GenericParams G) {
    extern __shared__ __align__(16) unsigned char smem[];
    cpxd *tw = reinterpret_cast<cpxd *>(smem);                                   // n/2
    cpxd *fft = tw + G.n_fft / 2;                                                // warps x n
    float *power = reinterpret_cast<float *>(fft + (size_t)G.warps * G.n_fft);   // warps x prow
    float *win = power + (size_t)G.warps * G.prow;                               // n (0 outside the window)
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nthreads = G.warps * 32;
    for (int i = tid; i < G.n_fft / 2; i += nthreads) tw[i] = G.tw[i];
    for (int i = tid; i < G.n_fft; i += nthreads) win[i] = P.in_tab[i] ? P.win_tab[i] : 0.0f;
    for (int i = tid; i < G.warps * G.prow; i += nthreads) power[i] = 0.0f;
    __syncthreads();
    cpxd *buf = fft + (size_t)warp * G.n_fft;
    float *prow = power + (size_t)warp * G.prow;
    const float a = P.preemph;
    for (int tile = blockIdx.x; tile < P.total_tiles; tile += gridDim.x) {
        const TileGeom g = tile_geom(P, tile);
        const MelUnit u = unit_at(P, g.unit);
        const float *x = P.audio + u.audio_off;
        for (int fi = warp; fi < g.nf; fi += G.warps) {
            const long long f = g.f0 + fi;
            const long long base = f * P.hop - P.pad;
            // pre-emphasis + window into bit-reversed order
            for (int j = lane; j < G.n_fft; j += 32) {
                const long long i = base + j;
                float v = 0.0f;
                if (i >= 0 && i < u.n && P.in_tab[j]) {
                    const float xi = __ldg(x + i);
                    if (a == 0.0f) v = xi;
                    else if (i == 0) v = preemph_first(xi, u.last, a);
                    else v = preemph_rest(xi, __ldg(x + i - 1), a);
                    v = __fmul_rn(v, win[j]);
                }
                cpxd z;
                z.x = (double)v;
                z.y = 0.0;
                buf[__brev((unsigned)j) >> (32 - G.log2n)] = z;
            }
            __syncwarp();
            for (int s = 0; s < G.log2n; ++s) {
                const int half = 1 << s, step = G.n_fft >> (s + 1);
                for (int t = lane; t < G.n_fft / 2; t += 32) {
                    const int j = t & (half - 1);
                    const int ia = ((t >> s) << (s + 1)) + j, ib = ia + half;
                    const cpxd w = tw[j * step], zb = buf[ib], za = buf[ia];
                    const double tr = zb.x * w.x - zb.y * w.y, ti = zb.x * w.y + zb.y * w.x;
                    cpxd o;
                    o.x = za.x - tr;
                    o.y = za.y - ti;
                    buf[ib] = o;
                    o.x = za.x + tr;
                    o.y = za.y + ti;
                    buf[ia] = o;
                }
                __syncwarp();
            }
            for (int b = lane; b < G.bins; b += 32) {
                const float xr = (float)buf[b].x, xi = (float)buf[b].y;
                prow[b] = 4.0f * __fadd_rn(__fmul_rn(xr, xr), __fmul_rn(xi, xi));   // the packed weights carry 1/4
            }
            __syncwarp();
            for (int m = lane; m < P.n_mels; m += 32) {
                const int lo = P.fb_lo[m], nq = (P.fb_hi[m] - lo) >> 2;
                const float v = log_value(mel_dot_quads(reinterpret_cast<const float4 *>(prow + lo),
                                                        reinterpret_cast<const float4 *>(P.fb_w + P.fb_off[m]), nq),
                                          P.log_floor, P.log_clamped);
                if (P.layout == 0) P.out[u.out_off + f * P.n_mels + m] = v;
                else P.out[u.out_off + (long long)m * u.out_stride + f] = v;
            }
            __syncwarp();
        }
    }
}

// ------------------------------------------------------------------------------------------------ host plan
static float swift_float_pi() {
    const uint32_t bits = 0x40490FDAu;   // Swift's Float.pi is rounded toward zero
    float f;
    std::memcpy(&f, &bits, 4);
    return f;
}

// AudioMelSpectrogram.swift:553-562
void build_window(int length, bool periodic, std::vector<float> &w) {
    w.resize(length);
    const float divisor = periodic ? (float)length : (float)(length - 1);
    const float pi = swift_float_pi();
    for (int i = 0; i < length; ++i) {
        const float phase = 2.0f * pi * (float)i / divisor;
        w[i] = 0.5f * (1.0f - cosf(phase));
    }
}

// AudioMelSpectrogram.swift:564-642 (Slaney mel scale, Slaney area normalisation, Float32 arithmetic)
void build_filterbank(int n_fft, int n_mels, int sample_rate, std::vector<float> &fb) {
    const int bins = n_fft / 2 + 1;
    const float f_sp = 200.0f / 3.0f, min_log_hz = 1000.0f;
    const float min_log_mel = min_log_hz / f_sp;
    const float log_step = logf(6.4f) / 27.0f;
    auto to_mel = [&](float hz) { return hz >= min_log_hz ? min_log_mel + logf(hz / min_log_hz) / log_step : hz / f_sp; };
    auto to_hz = [&](float mel) {
        return mel >= min_log_mel ? min_log_hz * expf(log_step * (mel - min_log_mel)) : f_sp * mel;
    };
    const float mel_lo = to_mel(0.0f), mel_hi = to_mel((float)sample_rate / 2.0f);
    std::vector<float> edge(n_mels + 2), freq(bins);
    for (int i = 0; i < n_mels + 2; ++i) edge[i] = to_hz(mel_lo + (float)i * (mel_hi - mel_lo) / (float)(n_mels + 1));
    for (int i = 0; i < bins; ++i) freq[i] = (float)i * (float)sample_rate / (float)n_fft;
    fb.assign((size_t)n_mels * bins, 0.0f);
    for (int m = 0; m < n_mels; ++m) {
        const float l = edge[m], c = edge[m + 1], r = edge[m + 2];
        const float norm = 2.0f / (r - l);
        for (int b = 0; b < bins; ++b) {
            const float f = freq[b];
            if (f >= l && f < c) fb[(size_t)m * bins + b] = norm * (f - l) / (c - l);
            else if (f >= c && f <= r) fb[(size_t)m * bins + b] = norm * (r - f) / (r - c);
        }
    }
}

#define FA_CUDA_TRY(expr)                                                                   \
    do {                                                                                    \
        cudaError_t e__ = (expr);                                                           \
        if (e__ != cudaSuccess) {                                                           \
            fa::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
            return FA_CUDA_ERROR;                                                           \
        }                                                                                   \
    } while (0)

static constexpr int kWarpsPerCta = 8;
static constexpr int kCtasPerSm = 2;

// Dynamic shared memory of mel512_kernel (the layout at the top of the kernel) and the tile extents it is made of.
static size_t mel512_smem_bytes(int hop, int n_mels, int fb_nnz, int n_slots, int *pt_len_out = nullptr,
                                int *pt_cap_out = nullptr, int *raw_cap_out = nullptr, int *fb_cap_out = nullptr) {
    const int pt_len = (kTileFrames - 1) * hop + kNfft;
    const int pt_cap = (pt_len + 31) & ~31;
    const int raw_cap = (pt_len + 1 + 3 + 3 + 31) & ~31;   // whole 128-byte lines: the pre-emphasised tile behind it stays line-aligned
    const int fb_cap = (fb_nnz + 3) & ~3;
    if (pt_len_out) *pt_len_out = pt_len;
    if (pt_cap_out) *pt_cap_out = pt_cap;
    if (raw_cap_out) *raw_cap_out = raw_cap;
    if (fb_cap_out) *fb_cap_out = fb_cap;
    return sizeof(float) * ((size_t)2 * raw_cap + pt_cap + 0 +
                            (size_t)(kTileFrames / 2) * kPairStride + (size_t)kTileFrames * (n_mels + 4) + fb_cap) +
           sizeof(cpxd) * (size_t)kWarpsPerCta * kFftPad + sizeof(int) * 4 * (size_t)n_slots + 8 +
           2 * sizeof(uint64_t) + 3 * sizeof(TileInfo) + 16;
}

MelPlan::~MelPlan() { release(); }

void MelPlan::release() {
    auto fr = [](auto *&p) {
        if (p) cudaFree(p);
        p = nullptr;
    };
    for (int m = 0; m < 2; ++m) {
        fr(d_win_tab_mode[m]);
        fr(d_in_tab_mode[m]);
        fr(d_lane_tab[m][0]);
        fr(d_lane_tab[m][1]);
    }
    fr(d_fb_w);
    fr(d_fb_slots);
    fr(d_fb_lo);
    fr(d_fb_hi);
    fr(d_fb_off);
    fr(d_units);
    fr(d_audio);
    fr(d_out);
    fr(d_pcm);
    fr(d_rs_tab);
    fr(d_generic_tw);
    d_pcm_cap = 0;
    rs_in = rs_out = 0.0;
    d_audio_cap = d_out_cap = 0;
    if (h_units) cudaFreeHost(h_units);
    h_units = nullptr;
    units_cap = 0;
    for (auto &s : streams)
        if (s) cudaStreamDestroy(s), s = nullptr;
    for (auto &e : events)
        if (e) cudaEventDestroy(e);
    events.clear();
    for (auto &e : timer)
        if (e) cudaEventDestroy(e), e = nullptr;
}

int MelPlan::init(const MelConfig &c) {
    cfg = c;
    if (cfg.pad_to < 1) cfg.pad_to = 1;   // AudioMelSpectrogram.swift:72
    if (cfg.n_mels <= 0 || cfg.hop_length <= 0 || cfg.win_length <= 0 || cfg.n_fft <= 0 || cfg.sample_rate <= 0) {
        fa::set_error("mel config: all sizes must be positive");
        return FA_INVALID_ARGUMENT;
    }
    const bool pow2 = cfg.n_fft >= 32 && cfg.n_fft <= 4096 && (cfg.n_fft & (cfg.n_fft - 1)) == 0;
    if (!pow2 || cfg.win_length > cfg.n_fft || cfg.n_mels > 512 || cfg.hop_length > 65536) {
        fa::set_error("mel config unsupported by the sm_100a kernels: need nFFT a power of two in 32..4096, win <= nFFT, "
                      "nMels <= 512 (got nFFT=%d hop=%d win=%d nMels=%d)",
                      cfg.n_fft, cfg.hop_length, cfg.win_length, cfg.n_mels);
        return FA_UNSUPPORTED;
    }
    // the specialised kernel covers every in-repo caller's shape; anything else takes mel_generic_kernel (so do hops
    // whose tile does not fit the specialised kernel's shared memory, decided below)
    generic = cfg.n_fft != kNfft || (cfg.hop_length & 1) || cfg.hop_length > 1024;
    const int n_fft = cfg.n_fft, bins = n_fft / 2 + 1;
    build_window(cfg.win_length, cfg.window_periodic != 0, window);
    build_filterbank(cfg.n_fft, cfg.n_mels, cfg.sample_rate, filterbank);

    // banded filterbank: per mel the contiguous range of non-zero bins, widened with explicit zero weights to whole
    // bin quads.  Weights are stored times 1/4 because the kernel's power tile holds 4|X|^2 (mel_core.cuh).
    std::vector<int> lo(cfg.n_mels), hi(cfg.n_mels), off(cfg.n_mels);
    int nnz = 0;
    for (int m = 0; m < cfg.n_mels; ++m) {
        int a = bins, b = 0;
        for (int k = 0; k < bins; ++k)
            if (filterbank[(size_t)m * bins + k] != 0.0f) {
                a = std::min(a, k);
                b = k + 1;
            }
        if (b == 0) a = 0;
        a &= ~3;                       // whole bin quads: 16-byte aligned reads of the power row (pair rows, kPairStride)
        b = (b + 3) & ~3;              // may reach 260 > 257: the tile's pad columns are zero, so are these weights
        lo[m] = a;
        hi[m] = b;
        off[m] = nnz;                  // a multiple of four: 16-byte aligned weight quads
        nnz += b - a;
    }
    fb_nnz = nnz;
    // filterbank-stage schedule of mel512_kernel: groups of four consecutive filters, dealt to the 8 warps longest first
    // (cost = widest band of the group, in quads); slot = (iteration * 8 + warp) * 4 + member
    std::vector<int4> slots;
    {
        const int groups = (cfg.n_mels + 3) / 4;
        std::vector<int> cost(groups, 0), order(groups);
        for (int g = 0; g < groups; ++g) {
            for (int m = 4 * g; m < std::min(cfg.n_mels, 4 * g + 4); ++m) cost[g] = std::max(cost[g], (hi[m] - lo[m]) >> 2);
            order[g] = g;
        }
        std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return cost[a] > cost[b]; });
        std::vector<std::vector<int>> mine(kWarpsPerCta);
        std::vector<long long> load(kWarpsPerCta, 0);
        // warp 0's lane 0 also computes the next tile's geometry and issues its bulk copy in this phase: measured, that is
        // worth more than a full share of the filterbank work (handicap 0 / 6 / 12 / 24 quads: 0.3109 / 0.3049 / 0.2996 /
        // 0.2982 ms per audio-hour, identical output; profiles/r02_mel.md), so warp 0 only takes a group when the others
        // are this far ahead
        load[0] = 24;
        if (const char *h = std::getenv("FA_MEL_ISSUE_HANDICAP")) load[0] = std::atoi(h);   // tuning hook (schedule only)
        for (int g : order) {
            int best = 0;
            for (int wv = 1; wv < kWarpsPerCta; ++wv)
                if (load[wv] + 2 * (long long)mine[wv].size() < load[best] + 2 * (long long)mine[best].size()) best = wv;
            mine[best].push_back(g);
            load[best] += cost[g] + 4;   // + per-iteration control
        }
        size_t iters = 0;
        for (auto &v : mine) iters = std::max(iters, v.size());
        slots.assign(iters * kWarpsPerCta * 4, make_int4(0, 0, 0, -1));
        for (int wv = 0; wv < kWarpsPerCta; ++wv)
            for (size_t it = 0; it < mine[wv].size(); ++it)
                for (int q = 0; q < 4; ++q) {
                    const int m = 4 * mine[wv][it] + q;
                    if (m < cfg.n_mels) slots[(it * kWarpsPerCta + wv) * 4 + q] = make_int4(lo[m], (hi[m] - lo[m]) >> 2, off[m], m);
                }
    }
    n_slots = (int)slots.size();

    int dev = 0;
    FA_CUDA_TRY(cudaGetDevice(&dev));
    cudaDeviceProp prop;
    FA_CUDA_TRY(cudaGetDeviceProperties(&prop, dev));
    num_sms = prop.multiProcessorCount;
    if (prop.major != 10) {
        fa::set_error("fluidaudio_b200 requires an sm_100a device, found sm_%d%d", prop.major, prop.minor);
        return FA_NO_DEVICE;
    }
    // mel512_kernel stages 15 hops + 512 samples three times (two raw buffers + the pre-emphasised tile): long even hops
    // do not fit the per-CTA opt-in limit (on B200 from hop ~890 at 80 mels, ~680 at 512 mels) and take the any-nFFT
    // kernel, which computes the same values
    if (!generic && mel512_smem_bytes(cfg.hop_length, cfg.n_mels, fb_nnz, n_slots) > (size_t)prop.sharedMemPerBlockOptin)
        generic = true;

    // weights packed in the order the kernel finds the bins in its power tile: mel512_kernel swizzles inside each bin
    // quad (pow_pos, mel_core.cuh), the any-nFFT kernel keeps the natural order
    std::vector<float> w;
    w.reserve(fb_nnz);
    for (int m = 0; m < cfg.n_mels; ++m)
        for (int k = lo[m]; k < hi[m]; ++k) {
            const int src = generic ? k : ((k & ~3) | ((k & 3) ^ ((k >> 4) & 3)));   // position k holds bin src: pow_pos is an involution
            w.push_back(src < bins ? 0.25f * filterbank[(size_t)m * bins + src] : 0.0f);
        }

    std::vector<float> win_tab(n_fft, 0.0f);
    std::vector<uint8_t> in_tab(n_fft, 0);
    for (int mode = 0; mode < 2; ++mode) {   // 0: centred window (offset (nFFT-win)/2); 1: legacy compute(), offset 0
        const int off_w = mode == 0 ? (cfg.n_fft - cfg.win_length) / 2 : 0;
        std::fill(win_tab.begin(), win_tab.end(), 0.0f);
        std::fill(in_tab.begin(), in_tab.end(), 0);
        for (int j = 0; j < cfg.win_length; ++j) {
            win_tab[off_w + j] = window[j];
            in_tab[off_w + j] = 1;
        }
        FA_CUDA_TRY(cudaMalloc(&d_win_tab_mode[mode], n_fft * sizeof(float)));
        FA_CUDA_TRY(cudaMalloc(&d_in_tab_mode[mode], n_fft));
        FA_CUDA_TRY(cudaMemcpy(d_win_tab_mode[mode], win_tab.data(), n_fft * sizeof(float), cudaMemcpyHostToDevice));
        FA_CUDA_TRY(cudaMemcpy(d_in_tab_mode[mode], in_tab.data(), n_fft, cudaMemcpyHostToDevice));
    }
    if (!generic) {
        for (int mode = 0; mode < 2; ++mode) {
            const int off_w = mode == 0 ? (cfg.n_fft - cfg.win_length) / 2 : 0;
            std::fill(win_tab.begin(), win_tab.end(), 0.0f);
            std::fill(in_tab.begin(), in_tab.end(), 0);
            for (int j = 0; j < cfg.win_length; ++j) {
                win_tab[off_w + j] = window[j];
                in_tab[off_w + j] = 1;
            }
            std::vector<LaneTables<double>> t64(32);
            std::vector<LaneTables<f32x2>> t32(32);
            for (int l = 0; l < 32; ++l) {
                load_lane_tables(l, win_tab.data(), in_tab.data(), t64[l]);
                load_lane_tables(l, win_tab.data(), in_tab.data(), t32[l]);
            }
            FA_CUDA_TRY(cudaMalloc(&d_lane_tab[mode][0], 32 * sizeof(LaneTables<double>)));
            FA_CUDA_TRY(cudaMalloc(&d_lane_tab[mode][1], 32 * sizeof(LaneTables<f32x2>)));
            FA_CUDA_TRY(cudaMemcpy(d_lane_tab[mode][0], t64.data(), 32 * sizeof(LaneTables<double>), cudaMemcpyHostToDevice));
            FA_CUDA_TRY(cudaMemcpy(d_lane_tab[mode][1], t32.data(), 32 * sizeof(LaneTables<f32x2>), cudaMemcpyHostToDevice));
        }
    }
    FA_CUDA_TRY(cudaMalloc(&d_fb_w, std::max<size_t>(1, w.size()) * sizeof(float)));
    FA_CUDA_TRY(cudaMalloc(&d_fb_slots, std::max<size_t>(1, slots.size()) * sizeof(int4)));
    if (!slots.empty())
        FA_CUDA_TRY(cudaMemcpy(d_fb_slots, slots.data(), slots.size() * sizeof(int4), cudaMemcpyHostToDevice));
    FA_CUDA_TRY(cudaMalloc(&d_fb_lo, cfg.n_mels * sizeof(int)));
    FA_CUDA_TRY(cudaMalloc(&d_fb_hi, cfg.n_mels * sizeof(int)));
    FA_CUDA_TRY(cudaMalloc(&d_fb_off, cfg.n_mels * sizeof(int)));
    if (!w.empty()) FA_CUDA_TRY(cudaMemcpy(d_fb_w, w.data(), w.size() * sizeof(float), cudaMemcpyHostToDevice));
    FA_CUDA_TRY(cudaMemcpy(d_fb_lo, lo.data(), cfg.n_mels * sizeof(int), cudaMemcpyHostToDevice));
    FA_CUDA_TRY(cudaMemcpy(d_fb_hi, hi.data(), cfg.n_mels * sizeof(int), cudaMemcpyHostToDevice));
    FA_CUDA_TRY(cudaMemcpy(d_fb_off, off.data(), cfg.n_mels * sizeof(int), cudaMemcpyHostToDevice));

    for (auto &st : streams) FA_CUDA_TRY(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    if (generic) {
        // FP64 twiddle table W_n^k and the shared-memory budget: as many warps per CTA as fit beside it
        std::vector<cpxd> tw(n_fft / 2);
        for (int k = 0; k < n_fft / 2; ++k) tw[k] = unit_root(k, n_fft);
        FA_CUDA_TRY(cudaMalloc(&d_generic_tw, tw.size() * sizeof(cpxd)));
        FA_CUDA_TRY(cudaMemcpy(d_generic_tw, tw.data(), tw.size() * sizeof(cpxd), cudaMemcpyHostToDevice));
        generic_prow = ((bins + 3) & ~3) + 4;
        int log2n = 0;
        while ((1 << log2n) < n_fft) ++log2n;
        generic_log2n = log2n;
        const size_t fixed = (size_t)(n_fft / 2) * sizeof(cpxd) + (size_t)n_fft * sizeof(float);
        const size_t per_warp = (size_t)n_fft * sizeof(cpxd) + (size_t)generic_prow * sizeof(float);
        generic_warps = (int)std::min<size_t>(8, ((size_t)prop.sharedMemPerBlockOptin - fixed - 1024) / per_warp);
        if (generic_warps < 1) {
            fa::set_error("mel config: nFFT %d does not fit shared memory", n_fft);
            return FA_UNSUPPORTED;
        }
        smem_bytes = fixed + per_warp * generic_warps;
        FA_CUDA_TRY(cudaFuncSetAttribute(mel_generic_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes));
        return FA_OK;
    }
    smem_bytes = mel512_smem_bytes(cfg.hop_length, cfg.n_mels, fb_nnz, n_slots, &pt_len, &pt_cap, &raw_cap, &fb_cap);
    FA_CUDA_TRY(cudaFuncSetAttribute(mel512_kernel<kWarpsPerCta, double, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes));
    FA_CUDA_TRY(cudaFuncSetAttribute(mel512_kernel<kWarpsPerCta, double, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes));
    FA_CUDA_TRY(cudaFuncSetAttribute(mel512_kernel<kWarpsPerCta, f32x2, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes));
    FA_CUDA_TRY(cudaFuncSetAttribute(mel512_kernel<kWarpsPerCta, f32x2, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes));
    return FA_OK;
}

long long MelPlan::frame_count(long long n, int mode, long long expected) const {
    long long computed;   // C++ integer division truncates toward zero exactly like Swift's Int '/'
    if (mode == 0) computed = 1 + (n + 2 * (long long)(cfg.n_fft / 2) - cfg.win_length) / cfg.hop_length;
    else if (mode == 1) computed = std::max<long long>(0, (n - cfg.n_fft) / cfg.hop_length + 1);
    else computed = 1 + (n - cfg.win_length) / cfg.hop_length;
    return expected >= 0 ? expected : computed;
}

int MelPlan::ensure_units(int count) {
    if (count <= units_cap) return FA_OK;
    if (d_units) cudaFree(d_units);
    if (h_units) cudaFreeHost(h_units);
    d_units = nullptr;
    h_units = nullptr;
    units_cap = std::max(count, 64);
    FA_CUDA_TRY(cudaMalloc(&d_units, units_cap * sizeof(MelUnit)));
    FA_CUDA_TRY(cudaMallocHost(&h_units, units_cap * sizeof(MelUnit)));
    return FA_OK;
}

int MelPlan::ensure_staging(size_t audio_floats, size_t out_floats) {
    if (audio_floats > d_audio_cap) {
        if (d_audio) cudaFree(d_audio);
        d_audio = nullptr;
        d_audio_cap = 0;
        FA_CUDA_TRY(cudaMalloc(&d_audio, audio_floats * sizeof(float)));
        d_audio_cap = audio_floats;
    }
    if (out_floats > d_out_cap) {
        if (d_out) cudaFree(d_out);
        d_out = nullptr;
        d_out_cap = 0;
        FA_CUDA_TRY(cudaMalloc(&d_out, out_floats * sizeof(float)));
        d_out_cap = out_floats;
    }
    return FA_OK;
}

int MelPlan::ensure_events(size_t count) {
    while (events.size() < count) {
        cudaEvent_t e;
        FA_CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        events.push_back(e);
    }
    return FA_OK;
}

int MelPlan::launch(const float *d_audio_base, float *d_out_base, int first, int count, int total_tiles, int mode,
                    int layout, cudaStream_t stream, bool aligned16) {
    if (total_tiles <= 0) return FA_OK;
    MelLaunch P{};
    P.audio = d_audio_base;
    P.out = d_out_base;
    P.units = d_units + first;
    P.num_units = count;
    P.inline_unit = (inline_unit && count == 1) ? 1 : 0;
    if (P.inline_unit) P.unit0 = h_units[first];
    P.total_tiles = total_tiles;
    P.hop = cfg.hop_length;
    P.pad = mode == 0 ? cfg.n_fft / 2 : 0;
    P.preemph = mode == 2 ? 0.0f : cfg.preemph;
    P.n_mels = cfg.n_mels;
    P.log_floor = cfg.log_floor;
    P.log_clamped = cfg.log_floor_mode;
    P.ot_stride = (cfg.n_mels & 3) == 0 ? cfg.n_mels + 4 : cfg.n_mels + 1;
    // float4 row stores need a 16-byte aligned output: a caller's device pointer, batch output offsets or pinned view may
    // not be (the units' descriptors are still in h_units)
    P.vec_out = (cfg.n_mels & 3) == 0 && (reinterpret_cast<uintptr_t>(d_out_base) & 15) == 0;
    for (int u = first; u < first + count && P.vec_out; ++u) P.vec_out = (h_units[u].out_off & 3) == 0;
    P.log_normal = cfg.log_floor >= 1e-37f ? 1 : 0;   // mel energies are >= 0: log's argument is then never a denormal
    P.layout = layout;
    P.lane_tab = d_lane_tab[mode == 2 ? 1 : 0][precision == 1 ? 1 : 0];
    P.win_tab = d_win_tab_mode[mode == 2 ? 1 : 0];
    P.in_tab = d_in_tab_mode[mode == 2 ? 1 : 0];
    P.fb_w = d_fb_w;
    P.fb_slots = reinterpret_cast<const int4 *>(d_fb_slots);
    P.n_slots = n_slots;
    P.fb_lo = d_fb_lo;
    P.fb_hi = d_fb_hi;
    P.fb_off = d_fb_off;
    P.fb_nnz = fb_nnz;
    P.fb_cap = fb_cap;
    P.pt_len = pt_len;
    P.pt_cap = pt_cap;
    P.raw_cap = raw_cap;
    P.use_tma = aligned16 ? 1 : 0;
    {
        const int off_w = mode == 2 ? 0 : (cfg.n_fft - cfg.win_length) / 2;
        P.mid_full = (off_w <= 64 && off_w + cfg.win_length >= 448) ? 1 : 0;
    }
    P.inv_n_mels = (unsigned)((0x100000000ull + (unsigned)cfg.n_mels - 1) / (unsigned)cfg.n_mels);   // 0 for n_mels == 1
    if (generic) {
        GenericParams G{cfg.n_fft, generic_log2n, cfg.n_fft / 2 + 1, generic_prow, reinterpret_cast<const cpxd *>(d_generic_tw),
                        generic_warps};
        const int ggrid = std::min(total_tiles, num_sms * std::max(1, 16 / generic_warps));
        mel_generic_kernel<<<ggrid, generic_warps * 32, smem_bytes, stream>>>(P, G);
        FA_CUDA_TRY(cudaGetLastError());
        ++launches;
        return FA_OK;
    }
    const int grid = std::min(total_tiles, num_sms * kCtasPerSm);
    const dim3 blk(kWarpsPerCta * 32);
    if (precision == 1) {
        if (layout == 0) mel512_kernel<kWarpsPerCta, f32x2, 0><<<grid, blk, smem_bytes, stream>>>(P);
        else mel512_kernel<kWarpsPerCta, f32x2, 1><<<grid, blk, smem_bytes, stream>>>(P);
    } else {
        if (layout == 0) mel512_kernel<kWarpsPerCta, double, 0><<<grid, blk, smem_bytes, stream>>>(P);
        else mel512_kernel<kWarpsPerCta, double, 1><<<grid, blk, smem_bytes, stream>>>(P);
    }
    FA_CUDA_TRY(cudaGetLastError());
    ++launches;
    return FA_OK;
}

static inline long long ceil_to(long long v, long long m) { return ((v + m - 1) / m) * m; }
static inline int tiles_of(long long frames) { return (int)((frames + kTileFrames - 1) / kTileFrames); }

// Shape rules shared by every entry point.  Returns false for the reference's "empty" guard
// (AudioMelSpectrogram.swift:135-137, :199-201, :349-351).
static bool shape_of(const MelPlan &p, long long n, int mode, long long expected, long long &T, long long &Tp) {
    T = p.frame_count(n, mode, mode == 0 || mode == 1 ? expected : -1);
    if (T <= 0 || n <= 0) return false;
    Tp = mode == 2 ? T : ceil_to(T, p.cfg.pad_to);
    return true;
}

int MelPlan::compute_device(const float *d_in, long long n, float last, int mode, long long expected, int layout,
                            float *d_out_buf, long long out_len, long long *mel_length, long long *num_frames,
                            cudaStream_t stream) {
    long long T, Tp;
    if (!shape_of(*this, n, mode, expected, T, Tp)) {
        if (mel_length) *mel_length = 0;
        if (num_frames) *num_frames = mode == 2 ? 0 : 1;
        if (mode != 2) {
            if (out_len < cfg.n_mels) return FA_OUTPUT_TOO_SMALL;
            FA_CUDA_TRY(cudaMemsetAsync(d_out_buf, 0, cfg.n_mels * sizeof(float), stream));
        }
        return FA_OK;
    }
    if (mel_length) *mel_length = T;
    if (num_frames) *num_frames = Tp;
    if (out_len < Tp * cfg.n_mels) {
        fa::set_error("mel output needs %lld floats, buffer has %lld", Tp * cfg.n_mels, out_len);
        return FA_OUTPUT_TOO_SMALL;
    }
    int st = ensure_units(1);
    if (st != FA_OK) return st;
    if (Tp > T) FA_CUDA_TRY(cudaMemsetAsync(d_out_buf, 0, Tp * cfg.n_mels * sizeof(float), stream));
    h_units[0] = MelUnit{0, n, 0, Tp, 0, T, last, 0};
    FA_CUDA_TRY(cudaMemcpyAsync(d_units, h_units, sizeof(MelUnit), cudaMemcpyHostToDevice, stream));
    const bool aligned = (reinterpret_cast<uintptr_t>(d_in) & 15) == 0;
    return launch(d_in, d_out_buf, 0, 1, tiles_of(T), mode, layout, stream, aligned);
}

int MelPlan::compute_batch_device(const float *d_in, const long long *offsets, int count, const float *last, int mode,
                                  int layout, float *d_out_buf, const long long *out_offsets, long long *mel_lengths,
                                  long long *num_frames, cudaStream_t stream) {
    int st = ensure_units(count);
    if (st != FA_OK) return st;
    int tiles = 0, used = 0;
    bool aligned = (reinterpret_cast<uintptr_t>(d_in) & 15) == 0;
    for (int i = 0; i < count; ++i) {
        const long long n = offsets[i + 1] - offsets[i];
        long long T, Tp;
        if (!shape_of(*this, n, mode, -1, T, Tp)) {
            if (mel_lengths) mel_lengths[i] = 0;
            if (num_frames) num_frames[i] = mode == 2 ? 0 : 1;
            if (mode != 2) FA_CUDA_TRY(cudaMemsetAsync(d_out_buf + out_offsets[i], 0, cfg.n_mels * sizeof(float), stream));
            continue;
        }
        if (mel_lengths) mel_lengths[i] = T;
        if (num_frames) num_frames[i] = Tp;
        if (Tp > T) FA_CUDA_TRY(cudaMemsetAsync(d_out_buf + out_offsets[i], 0, Tp * cfg.n_mels * sizeof(float), stream));
        if (offsets[i] & 3) aligned = false;
        h_units[used] = MelUnit{offsets[i], n, out_offsets[i], Tp, 0, T, last ? last[i] : 0.0f, tiles};
        tiles += tiles_of(T);
        ++used;
    }
    if (!used) return FA_OK;
    FA_CUDA_TRY(cudaMemcpyAsync(d_units, h_units, used * sizeof(MelUnit), cudaMemcpyHostToDevice, stream));
    return launch(d_in, d_out_buf, 0, used, tiles, mode, layout, stream, aligned);
}

// A pinned (page-locked, mapped) host buffer has a device alias under UVA: the kernel can then store its output rows
// straight into host memory (coalesced 16-byte stores become posted PCIe writes), which removes the D2H copy stage and its
// cross-stream hand-offs from the pipeline.  Pageable memory returns nullptr and takes the staged copy.
static float *device_alias_if_pinned(float *host) {
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, host) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return (a.type == cudaMemoryTypeHost && a.devicePointer) ? static_cast<float *>(a.devicePointer) : nullptr;
}

// Host buffers in, host buffers out.  A long clip is cut into units of `chunk` frames: unit c's samples are copied
// on the H2D stream while unit c-1 runs on the compute stream and unit c-2's rows return on the D2H stream.
// FA_MEL_TRACE_PIPELINE=1: device timestamps (timing events) at the end of every unit's H2D, kernels and D2H, printed to
// stderr after the call — the tool behind profiles/r02_mel.md's pipeline timeline.  Off: no events, no cost.
struct PipelineTrace {
    bool on = false;
    cudaEvent_t t0 = nullptr;
    std::vector<cudaEvent_t> ev;
    std::vector<int> tag;   // unit * 4 + stage (0 H2D done, 1 kernels done, 2 D2H done)
    PipelineTrace() {
        static const bool want = [] { const char *e = std::getenv("FA_MEL_TRACE_PIPELINE"); return e && *e && *e != '0'; }();
        on = want;
    }
    void start(cudaStream_t s) {
        if (!on) return;
        cudaEventCreate(&t0);
        cudaEventRecord(t0, s);
    }
    void mark(cudaStream_t s, int unit, int stage) {
        if (!on) return;
        cudaEvent_t e;
        cudaEventCreate(&e);
        cudaEventRecord(e, s);
        ev.push_back(e);
        tag.push_back(unit * 4 + stage);
    }
    void dump(const char *what) {
        if (!on) return;
        static const char *names[3] = {"h2d", "kern", "d2h"};
        std::fprintf(stderr, "[pipeline %s]", what);
        for (size_t i = 0; i < ev.size(); ++i) {
            float ms = 0.0f;
            cudaEventElapsedTime(&ms, t0, ev[i]);
            std::fprintf(stderr, " u%d.%s=%.3f", tag[i] / 4, names[tag[i] & 3], ms);
            cudaEventDestroy(ev[i]);
        }
        std::fprintf(stderr, "\n");
        cudaEventDestroy(t0);
    }
};

// Frame ranges of the pipeline's units.  The pipeline's fixed cost is its ramp: nothing can be computed before the first
// unit's samples have landed, and the last unit's kernel + D2H run after the last byte of input.  So the units at both ends
// are small (1 : 2 : 4 ... 4 : 2 : 1) and the ones in between large enough to amortise the per-transfer cost.  Bounds are
// multiples of the tile height; no unit is shorter than min_unit frames (fewer units otherwise).
static std::vector<long long> unit_bounds(long long T, long long max_units, long long min_unit) {
    std::vector<long long> b{0};
    long long K = std::max<long long>(1, std::min(max_units, T / std::max<long long>(1, min_unit)));
    auto weight = [&](long long c, long long k) -> long long {
        if (k < 6) return 4;
        const long long e = std::min(c, k - 1 - c);
        return e == 0 ? 1 : (e == 1 ? 2 : 4);
    };
    for (; K > 1; --K) {   // the smallest unit must still hold min_unit frames
        long long sum = 0;
        for (long long c = 0; c < K; ++c) sum += weight(c, K);
        if (T * weight(0, K) / sum >= min_unit) break;
    }
    long long sum = 0, acc = 0;
    for (long long c = 0; c < K; ++c) sum += weight(c, K);
    for (long long c = 0; c + 1 < K; ++c) {
        acc += weight(c, K);
        const long long e = std::min(T, ceil_to((long long)((double)T * (double)acc / (double)sum), kTileFrames));
        if (e > b.back() && e < T) b.push_back(e);
    }
    b.push_back(T);
    return b;
}

int MelPlan::compute_host(const float *audio, long long n, float last, int mode, long long expected, int layout,
                          float *out, long long out_len, long long *mel_length, long long *num_frames) {
    long long T, Tp;
    if (!shape_of(*this, n, mode, expected, T, Tp)) {
        if (mel_length) *mel_length = 0;
        if (num_frames) *num_frames = mode == 2 ? 0 : 1;
        if (mode != 2) {
            if (out_len < cfg.n_mels) return FA_OUTPUT_TOO_SMALL;
            for (int m = 0; m < cfg.n_mels; ++m) out[m] = 0.0f;   // padValue
        }
        return FA_OK;
    }
    if (mel_length) *mel_length = T;
    if (num_frames) *num_frames = Tp;
    const long long need = Tp * cfg.n_mels;
    if (out_len < need) {
        fa::set_error("mel output needs %lld floats, buffer has %lld", need, out_len);
        return FA_OUTPUT_TOO_SMALL;
    }
    int st = ensure_staging((size_t)n + 8, (size_t)need);
    if (st != FA_OK) return st;
    const std::vector<long long> bounds = unit_bounds(T, pipeline_chunks, 4096);
    const int chunks = (int)bounds.size() - 1;
    float *out_alias = (zero_copy_out && layout == 0 && chunks > 1) ? device_alias_if_pinned(out) : nullptr;
    float *k_out = out_alias ? out_alias : d_out;   // where the kernel writes
    if (out_alias && Tp > T) std::memset(out + T * cfg.n_mels, 0, (size_t)(Tp - T) * cfg.n_mels * sizeof(float));
    st = ensure_units(chunks);
    if (st != FA_OK) return st;
    cudaStream_t s_in = streams[0], s_k = streams[1], s_out = streams[2];
    if (chunks == 1) {
        // the streaming callers' shape (a few thousand samples, SortformerDiarizer.swift:857-905): nothing to overlap, so
        // one stream, no events, the unit descriptor passed in the kernel parameters, one synchronisation
        FA_CUDA_TRY(cudaMemcpyAsync(d_audio, audio, n * sizeof(float), cudaMemcpyHostToDevice, s_k));
        if (Tp > T) FA_CUDA_TRY(cudaMemsetAsync(d_out, 0, need * sizeof(float), s_k));
        h_units[0] = MelUnit{0, n, 0, Tp, 0, T, last, 0};
        inline_unit = true;
        st = launch(d_audio, d_out, 0, 1, tiles_of(T), mode, layout, s_k, true);
        inline_unit = false;
        if (st != FA_OK) return st;
        FA_CUDA_TRY(cudaMemcpyAsync(out, d_out, need * sizeof(float), cudaMemcpyDeviceToHost, s_k));
        FA_CUDA_TRY(cudaStreamSynchronize(s_k));
        return FA_OK;
    }
    st = ensure_events(2 * (size_t)chunks);
    if (st != FA_OK) return st;
    for (int c = 0; c < chunks; ++c) h_units[c] = MelUnit{0, n, 0, Tp, bounds[c], bounds[c + 1] - bounds[c], last, 0};
    FA_CUDA_TRY(cudaMemcpyAsync(d_units, h_units, chunks * sizeof(MelUnit), cudaMemcpyHostToDevice, s_k));
    if (Tp > T && !out_alias) FA_CUDA_TRY(cudaMemsetAsync(d_out, 0, need * sizeof(float), s_k));
    const long long pad = mode == 0 ? cfg.n_fft / 2 : 0;
    long long copied = 0;
    for (int c = 0; c < chunks; ++c) {
        const long long f_end = h_units[c].frame_begin + h_units[c].frame_count;            // exclusive
        long long s_end = std::min(n, (f_end - 1) * cfg.hop_length + cfg.n_fft - pad);          // samples needed so far
        if (c == chunks - 1) s_end = n;
        if (s_end > copied) {
            FA_CUDA_TRY(cudaMemcpyAsync(d_audio + copied, audio + copied, (s_end - copied) * sizeof(float),
                                        cudaMemcpyHostToDevice, s_in));
            copied = s_end;
        }
        FA_CUDA_TRY(cudaEventRecord(events[2 * c], s_in));
        FA_CUDA_TRY(cudaStreamWaitEvent(s_k, events[2 * c], 0));
        st = launch(d_audio, k_out, c, 1, tiles_of(h_units[c].frame_count), mode, layout, s_k, true);
        if (st != FA_OK) return st;
        if (out_alias) continue;   // the kernel stored its rows in the caller's pinned buffer: no D2H stage
        FA_CUDA_TRY(cudaEventRecord(events[2 * c + 1], s_k));
        FA_CUDA_TRY(cudaStreamWaitEvent(s_out, events[2 * c + 1], 0));
        const long long fb = h_units[c].frame_begin, fc = h_units[c].frame_count;
        if (layout == 0) {
            const long long rows = (c == chunks - 1) ? (Tp - fb) : fc;   // last unit also returns the zero pad rows
            FA_CUDA_TRY(cudaMemcpyAsync(out + fb * cfg.n_mels, d_out + fb * cfg.n_mels, rows * cfg.n_mels * sizeof(float),
                                        cudaMemcpyDeviceToHost, s_out));
        } else {
            const long long cols = (c == chunks - 1) ? (Tp - fb) : fc;
            FA_CUDA_TRY(cudaMemcpy2DAsync(out + fb, Tp * sizeof(float), d_out + fb, Tp * sizeof(float),
                                          cols * sizeof(float), cfg.n_mels, cudaMemcpyDeviceToHost, s_out));
        }
    }
    FA_CUDA_TRY(cudaStreamSynchronize(s_out));
    FA_CUDA_TRY(cudaStreamSynchronize(s_k));
    return FA_OK;
}

int MelPlan::ensure_resampler(double in_rate, double out_rate) {
    if (in_rate == out_rate || (in_rate == rs_in && out_rate == rs_out && d_rs_tab)) return FA_OK;
    resample::Design d;
    const int st = resample::make_design(in_rate, out_rate, d);
    if (st != FA_OK) return st;
    if (d_rs_tab) cudaFree(d_rs_tab);
    d_rs_tab = nullptr;
    FA_CUDA_TRY(cudaMalloc(&d_rs_tab, d.table.size() * sizeof(float)));
    FA_CUDA_TRY(cudaMemcpy(d_rs_tab, d.table.data(), d.table.size() * sizeof(float), cudaMemcpyHostToDevice));
    rs_design = std::move(d);
    rs_in = in_rate;
    rs_out = out_rate;
    return FA_OK;
}

// AudioConverter.resample + computeFlatTransposed as one device pipeline.  The PCM is copied in chunks; as soon as a
// chunk has landed the compute stream converts the samples it completes (mixdown + polyphase / linear, see
// resample_kernels.cu) into the float buffer the mel kernel reads, runs the frames those samples complete, and the D2H
// stream returns their rows — H2D of chunk c+1, kernels of chunk c and D2H of chunk c-1 overlap.
int MelPlan::compute_host_pcm(const void *pcm, long long frames, const resample::AudioFormat &f, float last, int mode,
                              int layout, float *out, long long out_len, long long *mel_length, long long *num_frames,
                              long long *resampled) {
    const long long n = resample::output_count(frames, f.in_rate, f.out_rate);
    if (resampled) *resampled = n;
    long long T, Tp;
    if (!shape_of(*this, n, mode, -1, T, Tp)) {
        if (mel_length) *mel_length = 0;
        if (num_frames) *num_frames = mode == 2 ? 0 : 1;
        if (mode != 2) {
            if (out_len < cfg.n_mels) return FA_OUTPUT_TOO_SMALL;
            for (int m = 0; m < cfg.n_mels; ++m) out[m] = 0.0f;
        }
        return FA_OK;
    }
    if (mel_length) *mel_length = T;
    if (num_frames) *num_frames = Tp;
    const long long need = Tp * cfg.n_mels;
    if (out_len < need) {
        fa::set_error("mel output needs %lld floats, buffer has %lld", need, out_len);
        return FA_OUTPUT_TOO_SMALL;
    }
    int st = ensure_resampler(f.in_rate, f.out_rate);
    if (st != FA_OK) return st;
    st = ensure_staging((size_t)n + 8, (size_t)need);
    if (st != FA_OK) return st;
    const size_t bps = f.format == resample::kPcmI16 ? 2 : 4;
    const size_t pcm_bytes = (size_t)frames * f.channels * bps;
    if (pcm_bytes + 16 > d_pcm_cap) {
        if (d_pcm) cudaFree(d_pcm);
        d_pcm = nullptr;
        d_pcm_cap = 0;
        FA_CUDA_TRY(cudaMalloc(&d_pcm, pcm_bytes + 16));
        d_pcm_cap = pcm_bytes + 16;
    }
    // pipeline depth: ~10 MB of PCM per chunk (the copy engines' fixed cost per transfer and the host's enqueue rate make
    // finer chunks slower: int16 hour 3.08 ms at 8-12 chunks, 3.44 at 24, 3.61 at 96 — profiles/r02_mel.md)
    const long long kMaxChunks = std::max<long long>(1, std::min<long long>(pipeline_chunks, (long long)(pcm_bytes / (10u << 20)) + 1));
    const std::vector<long long> bounds = unit_bounds(T, kMaxChunks, 4096);
    const int chunks = (int)bounds.size() - 1;
    float *out_alias = (zero_copy_out && layout == 0) ? device_alias_if_pinned(out) : nullptr;
    float *k_out = out_alias ? out_alias : d_out;   // where the kernel writes
    if (out_alias && Tp > T) std::memset(out + T * cfg.n_mels, 0, (size_t)(Tp - T) * cfg.n_mels * sizeof(float));
    st = ensure_units(chunks);
    if (st != FA_OK) return st;
    st = ensure_events(2 * (size_t)chunks);
    if (st != FA_OK) return st;
    cudaStream_t s_in = streams[0], s_k = streams[1], s_out = streams[2];
    for (int c = 0; c < chunks; ++c) h_units[c] = MelUnit{0, n, 0, Tp, bounds[c], bounds[c + 1] - bounds[c], last, 0};
    FA_CUDA_TRY(cudaMemcpyAsync(d_units, h_units, chunks * sizeof(MelUnit), cudaMemcpyHostToDevice, s_k));
    if (Tp > T && !out_alias) FA_CUDA_TRY(cudaMemsetAsync(d_out, 0, need * sizeof(float), s_k));
    const long long pad = mode == 0 ? cfg.n_fft / 2 : 0;
    const resample::Design &D = rs_design;
    const bool linear = f.in_rate != f.out_rate && resample::resolve_algorithm(f) == resample::kAlgoLinear;
    long long in_copied = 0, converted = 0;
    PipelineTrace trace;
    trace.start(s_in);
    for (int c = 0; c < chunks; ++c) {
        const long long f_end = h_units[c].frame_begin + h_units[c].frame_count;
        long long s_end = std::min(n, (f_end - 1) * cfg.hop_length + cfg.n_fft - pad);   // model-rate samples needed so far
        if (c == chunks - 1) s_end = n;
        // input frames those samples depend on
        long long in_need = frames;
        if (c != chunks - 1) {
            if (f.in_rate == f.out_rate) in_need = s_end;
            else if (linear) in_need = (long long)((double)(s_end + 1) * (f.in_rate / f.out_rate)) + 4;
            else in_need = ((s_end + 2) * D.M) / D.L + D.half + 3;
            in_need = std::min(frames, std::max(in_need, in_copied));
        }
        if (in_need > in_copied) {
            const char *src = reinterpret_cast<const char *>(pcm);
            char *dst = reinterpret_cast<char *>(d_pcm);
            if (f.interleaved || f.channels == 1) {
                const size_t a = (size_t)in_copied * f.channels * bps, b = (size_t)in_need * f.channels * bps;
                FA_CUDA_TRY(cudaMemcpyAsync(dst + a, src + a, b - a, cudaMemcpyHostToDevice, s_in));
            } else {
                for (int ch = 0; ch < f.channels; ++ch) {
                    const size_t a = ((size_t)ch * frames + in_copied) * bps, b = ((size_t)ch * frames + in_need) * bps;
                    FA_CUDA_TRY(cudaMemcpyAsync(dst + a, src + a, b - a, cudaMemcpyHostToDevice, s_in));
                }
            }
            in_copied = in_need;
        }
        FA_CUDA_TRY(cudaEventRecord(events[2 * c], s_in));
        trace.mark(s_in, c, 0);
        FA_CUDA_TRY(cudaStreamWaitEvent(s_k, events[2 * c], 0));
        long long ready = resample::outputs_ready(f, D, frames, in_copied, n);
        if (ready < s_end) {
            fa::set_error("internal: resampler window accounting (%lld < %lld)", ready, s_end);
            return FA_RUNTIME_ERROR;
        }
        ready = c == chunks - 1 ? n : s_end;
        st = resample::launch_convert(d_pcm, frames, f, D, d_rs_tab, d_audio, converted, ready, s_k, &launches);
        if (st != FA_OK) return st;
        converted = std::max(converted, ready);
        st = launch(d_audio, k_out, c, 1, tiles_of(h_units[c].frame_count), mode, layout, s_k, true);
        if (st != FA_OK) return st;
        trace.mark(s_k, c, 1);
        if (out_alias) continue;   // the kernel stored its rows in the caller's pinned buffer: no D2H stage
        FA_CUDA_TRY(cudaEventRecord(events[2 * c + 1], s_k));
        FA_CUDA_TRY(cudaStreamWaitEvent(s_out, events[2 * c + 1], 0));
        const long long fb = h_units[c].frame_begin, fc = h_units[c].frame_count;
        if (layout == 0) {
            const long long rows = (c == chunks - 1) ? (Tp - fb) : fc;
            FA_CUDA_TRY(cudaMemcpyAsync(out + fb * cfg.n_mels, d_out + fb * cfg.n_mels, rows * cfg.n_mels * sizeof(float),
                                        cudaMemcpyDeviceToHost, s_out));
        } else {
            const long long cols = (c == chunks - 1) ? (Tp - fb) : fc;
            FA_CUDA_TRY(cudaMemcpy2DAsync(out + fb, Tp * sizeof(float), d_out + fb, Tp * sizeof(float),
                                          cols * sizeof(float), cfg.n_mels, cudaMemcpyDeviceToHost, s_out));
        }
        trace.mark(s_out, c, 2);
    }
    FA_CUDA_TRY(cudaStreamSynchronize(s_out));
    FA_CUDA_TRY(cudaStreamSynchronize(s_k));
    trace.dump("pcm");
    return FA_OK;
}

// Batch of clips, host buffers: clips are grouped so that copies and kernels of successive groups overlap.
int MelPlan::compute_batch_host(const float *audio, const long long *offsets, int count, const float *last, int mode,
                                int layout, float *out, const long long *out_offsets, long long *mel_lengths,
                                long long *num_frames) {
    if (count <= 0) return FA_OK;
    // device-side packing: clip i starts at a 4-float aligned offset so that every tile can use the TMA path
    // When every clip already starts at a multiple of four floats in the caller's buffer, the device copy keeps the
    // caller's layout and a whole group of clips travels in ONE transfer (a bulk copy may read up to three floats past a
    // clip's end: the neighbour's samples or the pad below, never used: the kernel masks by the clip length).  512 clips
    // cost 1 024 cudaMemcpyAsync calls otherwise: ~4 ms of host enqueue time on a 25 ms batch.
    bool same_layout = true;
    for (int i = 0; i < count; ++i) same_layout = same_layout && ((offsets[i] - offsets[0]) & 3) == 0 && offsets[i + 1] >= offsets[i];
    std::vector<long long> doff(count + 1), dout(count + 1);
    long long a = 0, o = 0;
    std::vector<long long> Ts(count), Tps(count);
    for (int i = 0; i < count; ++i) {
        const long long n = offsets[i + 1] - offsets[i];
        doff[i] = same_layout ? offsets[i] - offsets[0] : a;
        a = same_layout ? ceil_to(offsets[i + 1] - offsets[0], 4) + 4 : a + ceil_to(n, 4) + 4;
        dout[i] = o;
        long long T, Tp;
        if (!shape_of(*this, n, mode, -1, T, Tp)) {
            Ts[i] = 0;
            Tps[i] = 0;
            o += cfg.n_mels;
        } else {
            Ts[i] = T;
            Tps[i] = Tp;
            o += Tp * cfg.n_mels;
        }
    }
    doff[count] = a;
    dout[count] = o;
    int st = ensure_staging((size_t)a + 8, (size_t)o);
    if (st != FA_OK) return st;
    st = ensure_units(count);
    if (st != FA_OK) return st;
    const int groups = std::min(count, 32);   // one H2D, one launch, one D2H per group: the last group's kernel + D2H is the pipeline's tail
    st = ensure_events(2 * (size_t)groups);
    if (st != FA_OK) return st;
    cudaStream_t s_in = streams[0], s_k = streams[1], s_out = streams[2];
    // all unit descriptors first (one small copy), then per group: H2D, kernel, D2H
    std::vector<int> g_first(groups + 1), g_units(groups + 1, 0), g_tiles(groups, 0);
    int used = 0;
    for (int g = 0; g < groups; ++g) {
        const int c0 = (int)((long long)count * g / groups), c1 = (int)((long long)count * (g + 1) / groups);
        g_first[g] = used;
        int tiles = 0;
        for (int i = c0; i < c1; ++i) {
            if (mel_lengths) mel_lengths[i] = Ts[i];
            if (num_frames) num_frames[i] = Ts[i] ? Tps[i] : (mode == 2 ? 0 : 1);
            if (!Ts[i]) continue;
            h_units[used] = MelUnit{doff[i], offsets[i + 1] - offsets[i], dout[i], Tps[i], 0, Ts[i], last ? last[i] : 0.0f, tiles};
            tiles += tiles_of(Ts[i]);
            ++used;
        }
        g_tiles[g] = tiles;
    }
    g_first[groups] = used;
    if (used) FA_CUDA_TRY(cudaMemcpyAsync(d_units, h_units, used * sizeof(MelUnit), cudaMemcpyHostToDevice, s_k));
    FA_CUDA_TRY(cudaMemsetAsync(d_out, 0, (size_t)o * sizeof(float), s_k));
    for (int g = 0; g < groups; ++g) {
        const int c0 = (int)((long long)count * g / groups), c1 = (int)((long long)count * (g + 1) / groups);
        if (same_layout) {
            const long long n = offsets[c1] - offsets[c0];
            if (n > 0)
                FA_CUDA_TRY(cudaMemcpyAsync(d_audio + doff[c0], audio + offsets[c0], n * sizeof(float), cudaMemcpyHostToDevice, s_in));
        } else {
            for (int i = c0; i < c1; ++i) {
                const long long n = offsets[i + 1] - offsets[i];
                if (n > 0)
                    FA_CUDA_TRY(cudaMemcpyAsync(d_audio + doff[i], audio + offsets[i], n * sizeof(float), cudaMemcpyHostToDevice, s_in));
            }
        }
        FA_CUDA_TRY(cudaEventRecord(events[2 * g], s_in));
        FA_CUDA_TRY(cudaStreamWaitEvent(s_k, events[2 * g], 0));
        st = launch(d_audio, d_out, g_first[g], g_first[g + 1] - g_first[g], g_tiles[g], mode, layout, s_k, true);
        if (st != FA_OK) return st;
        FA_CUDA_TRY(cudaEventRecord(events[2 * g + 1], s_k));
        FA_CUDA_TRY(cudaStreamWaitEvent(s_out, events[2 * g + 1], 0));
        bool out_contiguous = c1 > c0;   // the caller's output offsets follow the packed device layout: one transfer
        for (int i = c0; i < c1 && out_contiguous; ++i) out_contiguous = out_offsets[i] - out_offsets[c0] == dout[i] - dout[c0];
        if (out_contiguous) {
            FA_CUDA_TRY(cudaMemcpyAsync(out + out_offsets[c0], d_out + dout[c0], (dout[c1] - dout[c0]) * sizeof(float),
                                        cudaMemcpyDeviceToHost, s_out));
        } else {
            for (int i = c0; i < c1; ++i) {
                const long long len = dout[i + 1] - dout[i];
                FA_CUDA_TRY(cudaMemcpyAsync(out + out_offsets[i], d_out + dout[i], len * sizeof(float), cudaMemcpyDeviceToHost, s_out));
            }
        }
    }
    FA_CUDA_TRY(cudaStreamSynchronize(s_out));
    FA_CUDA_TRY(cudaStreamSynchronize(s_k));
    return FA_OK;
}

} // namespace mel
} // namespace fa
