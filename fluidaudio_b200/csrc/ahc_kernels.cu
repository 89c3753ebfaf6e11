// Centroid-linkage agglomerative clustering on one B200, bit-compatible with the reference's
// fastcluster_compute_centroid_linkage (Sources/FastClusterWrapper/FastClusterWrapper.cpp:196-244 driving
// fastcluster_internal.hpp:1625-1800).
//
// Why it can be bit-exact: every squared distance is accumulated exactly as the C++ does it
// (FastClusterWrapper.cpp:44-52): sum = sum + (a[k]-b[k])*(a[k]-b[k]) for k = 0..D-1 in order, each operation
// individually rounded (__dsub_rn/__dmul_rn/__dadd_rn: no FMA contraction, no tree reduction); merged
// centroids use (a*wa + b*wb)/(wa+wb) with the same four roundings (:89-100); and the pair chosen at every
// step comes out of the same heap rules (ahc_core.cuh).  Parallelism is ACROSS pairs, never inside one sum:
// one thread owns one (i,j) chain.
//
// Kernels
//   ahc_stage_kernel      input rows -> node store (row-major) + scan copy (k-major, coalesced across nodes)
//   ahc_init_nn_kernel    N(N-1)/2 distances, tiled: 128 i-threads x 16 j-accumulators, k-chunks through smem;
//                         per (i, j-range) lexicographic (distance, j) minimum
//   ahc_init_reduce_kernel  per-i minimum over j-ranges -> nearest neighbour + key of the heap
//   ahc_merge_kernel      persistent, cooperative: CTA 0 = master (heap, live list, merge log; one warp),
//                         CTAs 1.. = workers (one node per thread).  Per merge step the master publishes one
//                         command (release store), workers build the new centroid, scan their nodes against
//                         it (256-long chain each, node data streamed from L2), reduce to one candidate per
//                         CTA and signal (release add); the master folds the <=147 candidates and updates
//                         the heap.  N-1 dependent steps, no kernel launch or host round trip inside.
#include "ahc_core.cuh"
#include "ahc_plan.h"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <mutex>
#include <new>
#include <vector>

namespace fa {
namespace ahc {

#define FA_CUDA_TRY(expr)                                                                               \
    do {                                                                                                \
        cudaError_t e__ = (expr);                                                                       \
        if (e__ != cudaSuccess) {                                                                       \
            fa::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
            return e__ == cudaErrorMemoryAllocation ? FA_ALLOCATION_FAILURE : FA_CUDA_ERROR;            \
        }                                                                                               \
    } while (0)

// ------------------------------------------------------------------------------------------------ sync helpers
__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned *p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_u32(unsigned *p, unsigned v) {
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void red_release_add_u32(unsigned *p, unsigned v) {
    asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

__device__ __forceinline__ double sq_step(double sum, double a, double b) {
    const double diff = __dsub_rn(a, b);
    return __dadd_rn(sum, __dmul_rn(diff, diff));
}

// ------------------------------------------------------------------------------------------------ staging
// in: [N x D] row-major.  rows[0..N) = in; cols[k*Ns + i] = in[i*D + k].
__global__ void ahc_stage_kernel(const double *__restrict__ in, double *__restrict__ rows, double *__restrict__ cols,
                                 int N, int D, int Ns) {
    __shared__ double tile[32][33];
    const int i0 = blockIdx.x * 32, k0 = blockIdx.y * 32;
    const int tx = threadIdx.x, ty = threadIdx.y;   // 32 x 8
    for (int r = ty; r < 32; r += 8) {
        const int i = i0 + r, k = k0 + tx;
        double v = 0.0;
        if (i < N && k < D) {
            v = in[(size_t)i * D + k];
            rows[(size_t)i * D + k] = v;
        }
        tile[r][tx] = v;
    }
    __syncthreads();
    for (int r = ty; r < 32; r += 8) {
        const int k = k0 + r, i = i0 + tx;
        if (k < D && i < Ns) cols[(size_t)k * Ns + i] = tile[tx][r];
    }
}

// ------------------------------------------------------------------------------------------------ initial NN
constexpr int kTI = 128;   // i per CTA (one thread each)
constexpr int kTJ = 16;    // j accumulators per thread
constexpr int kKC = 32;    // k chunk staged in shared memory
constexpr int kJR = 512;   // j range per CTA (grid.y)

__global__ void __launch_bounds__(kTI) ahc_init_nn_kernel(const double *__restrict__ cols, int N, int D, int Ns,
                                                           Cand *__restrict__ partial, int *error) {
    __shared__ double sj[kKC][kTJ];
    const int t = threadIdx.x;
    const int i = blockIdx.x * kTI + t;
    const int jr0 = blockIdx.y * kJR;
    const int i_last = min(N, (int)(blockIdx.x + 1) * kTI) - 1;   // largest i of this CTA
    double best = INFINITY;
    int arg = INT_MAX;
    if (jr0 < i_last) {
        const int jr1 = min(jr0 + kJR, i_last);   // pairs need j < i <= i_last
        bool bad = false;
        for (int j0 = jr0; j0 < jr1; j0 += kTJ) {
            double acc[kTJ];
#pragma unroll
            for (int jj = 0; jj < kTJ; ++jj) acc[jj] = 0.0;
            for (int k0 = 0; k0 < D; k0 += kKC) {
                __syncthreads();
#pragma unroll
                for (int u = 0; u < (kKC * kTJ) / kTI; ++u) {
                    const int idx = t + kTI * u;
                    const int kk = idx / kTJ, jj = idx % kTJ;
                    const int k = k0 + kk, j = j0 + jj;
                    sj[kk][jj] = (k < D && j < N) ? cols[(size_t)k * Ns + j] : 0.0;
                }
                __syncthreads();
                if (i < N) {
                    const int kn = min(kKC, D - k0);
#pragma unroll 4
                    for (int kk = 0; kk < kn; ++kk) {
                        const double xi = cols[(size_t)(k0 + kk) * Ns + i];
#pragma unroll
                        for (int jj = 0; jj < kTJ; ++jj) acc[jj] = sq_step(acc[jj], xi, sj[kk][jj]);
                    }
                }
            }
            if (i < N) {
#pragma unroll
                for (int jj = 0; jj < kTJ; ++jj) {
                    const int j = j0 + jj;
                    if (j < i && j < jr1) {
                        const double d = acc[jj];
                        if (d != d) bad = true;
                        if (d < best) {   // ascending j + strict '<'  ==  lexicographic (d, j) minimum
                            best = d;
                            arg = j;
                        }
                    }
                }
            }
        }
        if (bad) atomicExch(error, 1);
    }
    if (i < N) {
        Cand c;
        c.d = best;
        c.id = arg;
        partial[(size_t)blockIdx.y * N + i] = c;
    }
}

__global__ void ahc_init_reduce_kernel(const Cand *__restrict__ partial, int N, int ranges, double *key, int *nn,
                                       int *node_weight) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    node_weight[i] = 1;
    if (i < 1) {
        key[0] = INFINITY;
        nn[0] = 0;
        return;
    }
    double best = INFINITY;
    int arg = 0;   // reference initialises idx = 0 and min = +inf (fastcluster_internal.hpp:1654-1656)
    for (int r = 0; r < ranges; ++r) {
        const Cand c = partial[(size_t)r * N + i];
        if (c.id != INT_MAX && c.d < best) {
            best = c.d;
            arg = c.id;
        }
    }
    key[i] = best;
    nn[i] = arg;
}

// ------------------------------------------------------------------------------------------------ initial NN, filtered
// The exact pass above evaluates all N(N-1)/2 bit-exact chains (3.6 ms at N = 10 000, FP64 pipe 76 % busy).  The filter
// path finds the same (min, argmin) per row with far fewer chains:
//   1. d2~(i,j) = |x_i|^2 + |x_j|^2 - 2 <x_i, x_j>, the inner product in float32 (tiled SIMT GEMM on float copies), with a
//      RIGOROUS error bound E_ij = c1 r_i r_j + c2 (n_i + n_j): c1 = 2.02 (D + 3) 2^-24 covers the float conversion of the
//      inputs and a D-term float32 accumulation in any order (|fl(sum) - sum| <= gamma_D sum |x y| <= gamma_D r_i r_j), c2
//      covers the double arithmetic of the combination and the rounding of the exact chain itself;
//   2. U_i = min_j (d2~ + E) is an upper bound of row i's true minimum; every j with d2~ - E <= U_i is a CANDIDATE (the
//      true argmin, and every exact tie of it, always is);
//   3. only the candidates run the reference's sequential chain (same sq_step arithmetic as the exact pass), and the
//      lexicographic (distance, j) minimum over them is the reference's (min, first argmin).
// Two passes over the lower-triangular 64 x 64 tiles (the float32 products are recomputed rather than stored: N^2 / 2
// floats would be 200 MB at N = 10 000).  Non-finite or huge inputs, or a candidate list that overflows (thousands of
// exact duplicates), fall back to the exact pass — the result is bit-identical either way.
constexpr int kFT = 64;    // tile edge
constexpr int kFK = 16;    // k chunk
struct FilterBufs {
    float *cf;                      // [D x Ns] float copy of cols
    double *nrm2;                   // [N] |x_i|^2
    float *rn;                      // [N] |x_i| rounded up
    unsigned long long *U;          // [N] bits of the row's upper bound (non-negative doubles order like their bits)
    unsigned long long *best_d;     // [N] bits of the exact minimum
    int *best_j;                    // [N]
    int2 *cand;                     // [cap] (i, j)
    double *cand_d;                 // [cap]
    int *counters;                  // [0] candidates appended, [1] bad input, [2] overflow
    float *tmin;                    // [N x NT] per (row, column tile): min_j (d2~ - E) rounded down, or nullptr (not kept)
    int nt;                         // column tiles per row
    int cap;
    double c1, c2;
};

__global__ void ahc_filter_prep_kernel(const double *__restrict__ cols, int N, int D, int Ns, FilterBufs F) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= Ns) return;
    double n = 0.0;
    bool bad = false;
    for (int k = 0; k < D; ++k) {
        const double v = i < N ? cols[(size_t)k * Ns + i] : 0.0;
        F.cf[(size_t)k * Ns + i] = (float)v;
        n = fma(v, v, n);
        if (!(fabs(v) <= 1e17)) bad = true;   // also NaN / Inf
    }
    for (int k = D; k < ((D + 7) & ~7); ++k) F.cf[(size_t)k * Ns + i] = 0.0f;
    if (i < N) {
        F.nrm2[i] = n;
        F.rn[i] = __fmul_ru(__double2float_ru(sqrt(n)), 1.000001f);
        F.U[i] = ~0ull;
        F.best_d[i] = ~0ull;
        F.best_j[i] = INT_MAX;
        if (bad) atomicExch(&F.counters[1], 1);
    }
}

template <bool kCollect>
__global__ void __launch_bounds__(256) ahc_filter_tile_kernel(int N, int D, int Ns, FilterBufs F) {
    __shared__ __align__(16) float As[kFK][kFT], Bs[kFK][kFT];
    // lower-triangular tile pair (ti >= tj) from the linear block index
    const int b = blockIdx.x;
    int ti = (int)((sqrt(8.0 * (double)b + 1.0) - 1.0) * 0.5);
    while ((long long)ti * (ti + 1) / 2 > b) --ti;
    while ((long long)(ti + 1) * (ti + 2) / 2 <= b) ++ti;
    const int tj = b - (int)((long long)ti * (ti + 1) / 2);
    const int i0 = ti * kFT, j0 = tj * kFT;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    if (kCollect && F.tmin) {   // skip tiles in which no row can have a candidate (almost all of them)
        int any = 0;
        if (threadIdx.x < kFT) {
            const int i = i0 + threadIdx.x;
            if (i < N && i > j0) any = (double)F.tmin[(size_t)i * F.nt + tj] <= __longlong_as_double((long long)F.U[i]);
        }
        if (!__syncthreads_or(any)) return;
    }
    float acc[4][4];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[a][c] = 0.0f;
    for (int k0 = 0; k0 < D; k0 += kFK) {
        __syncthreads();
        for (int idx = threadIdx.x; idx < kFK * kFT; idx += 256) {
            const int kk = idx / kFT, ii = idx % kFT, k = k0 + kk;
            As[kk][ii] = (k < D && i0 + ii < Ns) ? F.cf[(size_t)k * Ns + i0 + ii] : 0.0f;
            Bs[kk][ii] = (k < D && j0 + ii < Ns) ? F.cf[(size_t)k * Ns + j0 + ii] : 0.0f;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < kFK; ++kk) {
            const float4 a4 = *reinterpret_cast<const float4 *>(&As[kk][ty * 4]);
            const float4 b4 = *reinterpret_cast<const float4 *>(&Bs[kk][tx * 4]);
            const float av[4] = {a4.x, a4.y, a4.z, a4.w}, bv[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
            for (int a = 0; a < 4; ++a)
#pragma unroll
                for (int c = 0; c < 4; ++c) acc[a][c] = fmaf(av[a], bv[c], acc[a][c]);
        }
    }
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        const int i = i0 + ty * 4 + a;
        double rowmin = 1.7976931348623157e308, rowlo = 1.7976931348623157e308;
        const double ni = i < N ? F.nrm2[i] : 0.0;
        const double ri = i < N ? (double)F.rn[i] : 0.0;
        const double Ui = (kCollect && i < N) ? __longlong_as_double((long long)F.U[i]) : 0.0;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int j = j0 + tx * 4 + c;
            if (i < N && j < i) {
                const double nj = F.nrm2[j];
                const double approx = (ni + nj) - 2.0 * (double)acc[a][c];
                const double E = F.c1 * ri * (double)F.rn[j] + F.c2 * (ni + nj);
                if (!kCollect) {
                    rowmin = fmin(rowmin, fmax(approx + E, 0.0));
                    rowlo = fmin(rowlo, approx - E);
                } else if (approx - E <= Ui) {
                    const int slot = atomicAdd(&F.counters[0], 1);
                    if (slot < F.cap) F.cand[slot] = make_int2(i, j);
                    else F.counters[2] = 1;
                }
            }
        }
        if (!kCollect) {   // the 16 threads of a row group are one half-warp: fold, one atomic per (row, tile)
#pragma unroll
            for (int o = 8; o >= 1; o >>= 1) {
                rowmin = fmin(rowmin, __shfl_xor_sync(0xffffffffu, rowmin, o));
                rowlo = fmin(rowlo, __shfl_xor_sync(0xffffffffu, rowlo, o));
            }
            if (tx == 0 && i < N) {
                if (rowmin < 1.7976931348623157e308) atomicMin(&F.U[i], (unsigned long long)__double_as_longlong(rowmin));
                // what pass 2 needs to know about this (row, tile): can any pair in it be a candidate?
                if (F.tmin) F.tmin[(size_t)i * F.nt + tj] = rowlo < 1.7976931348623157e308 ? __double2float_rd(rowlo) : 3.0e38f;
            }
        }
    }
}

// Pass 1 at full SIMT rate: 128 x 128 tiles of the lower triangle, 8 x 8 inner products per thread held as packed
// float pairs (FFMA2: one issue slot per two FMAs), k in chunks of eight through double-buffered shared memory with the
// next chunk's two float4 global loads in flight during the arithmetic.  Rows / columns of a thread: {ty*4..+3, 64+ty*4..+3}
// x {tx*4..+3, 64+tx*4..+3}, so the per-k operand loads are four LDS.128 (two of them warp-wide broadcasts) for 32 FFMA2.
// The bounds keep the 64-column granularity of pass 2: a tile feeds column tiles 2*TJ and 2*TJ+1.
constexpr int kGT = 128, kGK = 8;

__device__ __forceinline__ void cp_async16_zfill(void *smem, const void *gmem, bool valid) {
    const unsigned dst = (unsigned)__cvta_generic_to_shared(smem);
    const int bytes = valid ? 16 : 0;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(gmem), "r"(bytes) : "memory");
}

__device__ __forceinline__ float2 ffma2_bcast(float a, float2 b, float2 c) {
    return __ffma2_rn(make_float2(a, a), b, c);
}

__global__ void __launch_bounds__(256, 2) ahc_filter_tile128_kernel(int N, int D, int Ns, FilterBufs F) {
    __shared__ __align__(16) float As[2][kGK][kGT], Bs[2][kGK][kGT];
    const int b = blockIdx.x;
    int ti = (int)((sqrt(8.0 * (double)b + 1.0) - 1.0) * 0.5);
    while ((long long)ti * (ti + 1) / 2 > b) --ti;
    while ((long long)(ti + 1) * (ti + 2) / 2 <= b) ++ti;
    const int tj = b - (int)((long long)ti * (ti + 1) / 2);
    const int i0 = ti * kGT, j0 = tj * kGT;
    const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
    const int lk = t >> 5, lc = (t & 31) * 4;   // this thread's float4 of a [8 x 128] chunk
    // Ns is a multiple of 32: a float4 is inside or outside the matrix as a whole; cf has its row count rounded up to a
    // multiple of eight with zero rows, so k needs no bound check
    const int a_bytes = i0 + lc < Ns ? 16 : 0, b_bytes = j0 + lc < Ns ? 16 : 0;
    const float *ga = a_bytes ? F.cf + (size_t)lk * Ns + i0 + lc : F.cf;
    const float *gb = b_bytes ? F.cf + (size_t)lk * Ns + j0 + lc : F.cf;
    const size_t gstep = a_bytes ? (size_t)kGK * Ns : 0, gstep_b = b_bytes ? (size_t)kGK * Ns : 0;
    const unsigned sa = (unsigned)__cvta_generic_to_shared(&As[0][lk][lc]), sb = (unsigned)__cvta_generic_to_shared(&Bs[0][lk][lc]);
    constexpr unsigned kBufBytes = kGK * kGT * sizeof(float);
    float2 acc[8][4];
#pragma unroll
    for (int a = 0; a < 8; ++a)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[a][c] = make_float2(0.0f, 0.0f);
    // chunk -> buffer: asynchronous 16-byte copies straight into shared memory (zero-filled outside the matrix): the
    // prefetch holds no registers
    auto stage = [&](int bufi) {
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(sa + bufi * kBufBytes), "l"(ga), "r"(a_bytes) : "memory");
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(sb + bufi * kBufBytes), "l"(gb), "r"(b_bytes) : "memory");
        asm volatile("cp.async.commit_group;" ::: "memory");
        ga += gstep;
        gb += gstep_b;
    };
    stage(0);
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();
    int buf = 0;
    for (int k0 = 0; k0 < D; k0 += kGK) {
        const bool more = k0 + kGK < D;
        if (more) stage(buf ^ 1);   // that buffer was last read a full chunk (and a barrier) ago
#pragma unroll
        for (int kk = 0; kk < kGK; ++kk) {
            const float4 a0 = *reinterpret_cast<const float4 *>(&As[buf][kk][ty * 4]);
            const float4 a1 = *reinterpret_cast<const float4 *>(&As[buf][kk][64 + ty * 4]);
            const float4 b0 = *reinterpret_cast<const float4 *>(&Bs[buf][kk][tx * 4]);
            const float4 b1 = *reinterpret_cast<const float4 *>(&Bs[buf][kk][64 + tx * 4]);
            const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
            const float2 bv[4] = {make_float2(b0.x, b0.y), make_float2(b0.z, b0.w), make_float2(b1.x, b1.y),
                                  make_float2(b1.z, b1.w)};
#pragma unroll
            for (int a = 0; a < 8; ++a)
#pragma unroll
                for (int c = 0; c < 4; ++c) acc[a][c] = ffma2_bcast(av[a], bv[c], acc[a][c]);
        }
        if (more) {
            asm volatile("cp.async.wait_group 0;" ::: "memory");
            __syncthreads();
            buf ^= 1;
        }
    }
    // Bounds per (row, 64-column tile) in float32 INTERVAL arithmetic (every operation rounded towards the safe side), so
    // that the epilogue is ~12 instructions per pair instead of ~35 in double: with s = n_i + n_j,
    //   lo = RD(RD(-2 dot + RD(s)) - E^),  hi = RU(RU(-2 dot + RU(s)) + E^),  E^ = RU(c1r_i^ r_j + RU(c2^ RU(s))) >= E.
    // Rounding the bounds to float widens the band by < 1 % of E (2^-24 * 4 against c1 ~ 3e-5).  The columns' norms go
    // through shared memory (the operand buffers are free now); the 16 tx threads of a row group are one half-warp.
    __syncthreads();
    float *nlo = &As[0][0][0], *nhi = nlo + kGT, *rj = nhi + kGT;   // [128] each
    if (t < kGT) {
        const int j = j0 + t;
        const double nj = j < N ? F.nrm2[j] : 0.0;
        nlo[t] = __double2float_rd(nj);
        nhi[t] = __double2float_ru(nj);
        rj[t] = j < N ? F.rn[j] : 0.0f;
    }
    __syncthreads();
    const float c1up = __double2float_ru(F.c1), c2up = __double2float_ru(F.c2);
    const float kInf = __int_as_float(0x7f800000);
#pragma unroll
    for (int a = 0; a < 8; ++a) {
        const int i = i0 + (a >> 2) * 64 + ty * 4 + (a & 3);
        const double ni = i < N ? F.nrm2[i] : 0.0;
        const float ni_lo = __double2float_rd(ni), ni_hi = __double2float_ru(ni);
        const float c1ri = __fmul_ru(c1up, i < N ? F.rn[i] : 0.0f);
        float rowmin = kInf;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            float rowlo = kInf;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const int jl = h * 64 + tx * 4 + c, j = j0 + jl;
                const float2 p = acc[a][h * 2 + (c >> 1)];
                const float dot = (c & 1) ? p.y : p.x;
                const float s_lo = __fadd_rd(ni_lo, nlo[jl]), s_hi = __fadd_ru(ni_hi, nhi[jl]);
                const float e = __fmaf_ru(c1ri, rj[jl], __fmul_ru(c2up, s_hi));
                const float hi = __fadd_ru(__fmaf_ru(-2.0f, dot, s_hi), e);
                const float lo = __fsub_rd(__fmaf_rd(-2.0f, dot, s_lo), e);
                const bool live = i < N && j < i;
                rowmin = fminf(rowmin, live ? fmaxf(hi, 0.0f) : kInf);
                rowlo = fminf(rowlo, live ? lo : kInf);
            }
            if (F.tmin) {
#pragma unroll
                for (int o = 8; o >= 1; o >>= 1) rowlo = fminf(rowlo, __shfl_xor_sync(0xffffffffu, rowlo, o));
                const int t64 = 2 * tj + h;
                if (tx == 0 && i < N && t64 < F.nt) F.tmin[(size_t)i * F.nt + t64] = rowlo < kInf ? rowlo : 3.0e38f;
            }
        }
#pragma unroll
        for (int o = 8; o >= 1; o >>= 1) rowmin = fminf(rowmin, __shfl_xor_sync(0xffffffffu, rowmin, o));
        if (tx == 0 && i < N && rowmin < kInf)
            atomicMin(&F.U[i], (unsigned long long)__double_as_longlong((double)rowmin));
    }
}

// Pass 2, sparse form (when pass 1 kept its per (row, column tile) lower bounds): one warp per row.  The warp scans its
// row's bounds (a few of ~N/64 tiles can hold a candidate), and for every such tile evaluates the row's 64 float32 inner
// products itself (two columns per lane, x_i from shared memory, the columns coalesced from the k-major float copy) and
// appends the pairs inside the band.  Re-running the dense tile GEMM and exiting early still recomputed ~half the tiles
// (any of a tile's 64 rows keeps it alive); this does ~1.5 tiles' worth of one row per row.
__global__ void __launch_bounds__(256) ahc_filter_rows_kernel(int N, int D, int Ns, FilterBufs F) {
    extern __shared__ float xrow[];   // [8 warps x D]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int i = blockIdx.x * 8 + warp;
    if (i >= N || i < 1) return;
    float *xi = xrow + (size_t)warp * D;
    for (int k = lane; k < D; k += 32) xi[k] = F.cf[(size_t)k * Ns + i];
    __syncwarp();
    const double Ui = __longlong_as_double((long long)F.U[i]);
    const double ni = F.nrm2[i], ri = (double)F.rn[i];
    const int nt_row = i / kFT + 1;   // column tiles that hold some j < i
    for (int t0 = 0; t0 < nt_row; t0 += 32) {
        const int t = t0 + lane;
        const bool hit = t < nt_row && (double)F.tmin[(size_t)i * F.nt + t] <= Ui;
        unsigned mask = __ballot_sync(0xffffffffu, hit);
        while (mask) {
            const int tt = t0 + __ffs(mask) - 1;
            mask &= mask - 1;
            const int j0 = tt * kFT + lane, j1 = j0 + 32;   // this lane's two columns of the tile
            float a0 = 0.0f, a1 = 0.0f;
            const float *c0 = F.cf + j0, *c1 = F.cf + j1;   // (j < Ns always: Ns is a multiple of 32 >= N; zero beyond N)
            const bool in0 = j0 < Ns, in1 = j1 < Ns;
            for (int k = 0; k < D; ++k) {
                const float x = xi[k];
                if (in0) a0 = fmaf(x, c0[(size_t)k * Ns], a0);
                if (in1) a1 = fmaf(x, c1[(size_t)k * Ns], a1);
            }
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int j = h ? j1 : j0;
                if (j < i) {
                    const double nj = F.nrm2[j];
                    const double approx = (ni + nj) - 2.0 * (double)(h ? a1 : a0);
                    const double E = F.c1 * ri * (double)F.rn[j] + F.c2 * (ni + nj);
                    if (approx - E <= Ui) {
                        const int slot = atomicAdd(&F.counters[0], 1);
                        if (slot < F.cap) F.cand[slot] = make_int2(i, j);
                        else F.counters[2] = 1;
                    }
                }
            }
        }
    }
}

// the reference's chain for every candidate; its minimum per row as an integer atomic on the distance bits
__global__ void ahc_filter_exact_kernel(const double *__restrict__ cols, int D, int Ns, FilterBufs F) {
    const int slot = blockIdx.x * blockDim.x + threadIdx.x;
    const int count = min(F.counters[0], F.cap);
    if (slot >= count) return;
    const int2 c = F.cand[slot];
    double sum = 0.0;
    for (int k = 0; k < D; ++k) sum = sq_step(sum, cols[(size_t)k * Ns + c.x], cols[(size_t)k * Ns + c.y]);
    F.cand_d[slot] = sum;
    if (sum != sum) F.counters[1] = 1;
    else atomicMin(&F.best_d[c.x], (unsigned long long)__double_as_longlong(sum));
}
__global__ void ahc_filter_argmin_kernel(FilterBufs F) {
    const int slot = blockIdx.x * blockDim.x + threadIdx.x;
    const int count = min(F.counters[0], F.cap);
    if (slot >= count) return;
    const int2 c = F.cand[slot];
    if ((unsigned long long)__double_as_longlong(F.cand_d[slot]) == F.best_d[c.x]) atomicMin(&F.best_j[c.x], c.y);
}
__global__ void ahc_filter_finish_kernel(int N, FilterBufs F, double *key, int *nn, int *node_weight) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    node_weight[i] = 1;
    if (i < 1) {
        key[0] = INFINITY;
        nn[0] = 0;
        return;
    }
    if (F.best_j[i] == INT_MAX) {   // cannot happen with a valid bound: force the exact fall-back
        F.counters[2] = 1;
        return;
    }
    key[i] = __longlong_as_double((long long)F.best_d[i]);
    nn[i] = F.best_j[i];
}

// ------------------------------------------------------------------------------------------------ merge loop
constexpr int kMergeThreads = 128;
constexpr int kMaxRounds = 16;    // streamed mode only: slots per thread
enum { CMD_MERGE = 1, CMD_RESCAN = 2, CMD_EXIT = 3 };
typedef unsigned long long u64;

__device__ __forceinline__ u64 ld_acquire_u64(const u64 *p) {
    u64 v;
    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ u64 ld_relaxed_u64(const u64 *p) {
    u64 v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void ld_relaxed_v2(const u64 *p, u64 &x, u64 &y) {   // p 16-byte aligned
    asm volatile("ld.relaxed.gpu.global.v2.u64 {%0, %1}, [%2];" : "=l"(x), "=l"(y) : "l"(p) : "memory");
}
__device__ __forceinline__ void st_release_u64(u64 *p, u64 v) {
    asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void st_relaxed_u64(u64 *p, u64 v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void fence_acq_rel_gpu() { asm volatile("fence.acq_rel.gpu;" ::: "memory"); }
__device__ __forceinline__ u64 global_ns() {
    u64 t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
#define FA_TRACE(slot)                                                                         \
    do {                                                                                       \
        if ((P.flags & 4) && trace_step >= 0 && trace_step < kTraceSteps) P.trace[trace_step * 16 + (slot)] = global_ns(); \
    } while (0)

__device__ __forceinline__ u64 pack_cmd(int type, unsigned counter, int a, int b) {
    return ((u64)type << 62) | ((u64)(counter & 0x3fffu) << 48) | ((u64)(unsigned)a << 24) | (u64)(unsigned)b;
}

__device__ __forceinline__ void cand_min(double &d, int &id, double od, int oid) {
    if (cand_less(od, oid, d, id)) {
        d = od;
        id = oid;
    }
}

// Lexicographic (distance, id) minimum over a warp in three REDUX instructions instead of a five-step shuffle tree
// (~0.2 us per use, twice per merge step).  Squared distances are sums of squares starting from +0, so they are
// non-negative and their IEEE bit patterns order like unsigned integers; NaNs never get here (`bad` flags).
__device__ __forceinline__ void warp_cand_min(double &d, int &id) {
    const unsigned full = 0xffffffffu;
    const unsigned hi = (unsigned)__double2hiint(d), lo = (unsigned)__double2loint(d);
    const unsigned mh = __reduce_min_sync(full, hi);
    const unsigned ml = __reduce_min_sync(full, hi == mh ? lo : 0xffffffffu);
    const unsigned mi = __reduce_min_sync(full, (hi == mh && lo == ml) ? (unsigned)id : 0xffffffffu);
    d = __hiloint2double((int)mh, (int)ml);
    id = (int)mi;
}

// One polling snapshot: both words of up to Q slots per lane plus (optionally) the threshold words.
template <int Q> struct PollSnap {
    u64 a0[Q], a1[Q], t0, t1;
    __device__ __forceinline__ void issue(const ResultSlot *results, int shift, int W, int lane, unsigned tag,
                                          const u64 *thr) {
#pragma unroll
        for (int q = 0; q < Q; ++q) {
            const int w = lane + 32 * q;
            a0[q] = (u64)(tag & 0xffu);
            a1[q] = (u64)tag;
            if (w < W) ld_relaxed_v2(&results[(size_t)w << shift].w0, a0[q], a1[q]);   // one 16-byte request per slot
        }
        t0 = t1 = (u64)tag;
        if (thr) ld_relaxed_v2(thr, t0, t1);
    }
    __device__ __forceinline__ bool complete(unsigned tag) const {   // warp-uniform
        bool pending = (unsigned)t0 != tag || (unsigned)t1 != tag;
#pragma unroll
        for (int q = 0; q < Q; ++q)
            pending = pending || ((unsigned)(a0[q] & 0xffu) != (tag & 0xffu)) || ((unsigned)a1[q] != tag);
        return !__any_sync(0xffffffffu, pending);
    }
    __device__ __forceinline__ void reduce(int W, int lane, double &d, int &id, bool &bad, double *T) const {
        if (T) *T = __longlong_as_double((long long)((t0 & 0xffffffff00000000ull) | (t1 >> 32)));
        d = INFINITY;
        id = INT_MAX;
        bad = false;
#pragma unroll
        for (int q = 0; q < Q; ++q) {
            const int w = lane + 32 * q;
            if (w < W) {
                const unsigned oid = (unsigned)(a0[q] >> 8) & 0xffffffu;
                const u64 bits = (a0[q] & 0xffffffff00000000ull) | (a1[q] >> 32);
                if (oid == 0xfffffeu) bad = true;
                else if (oid != 0xffffffu) cand_min(d, id, __longlong_as_double((long long)bits), (int)oid);
            }
        }
    }
};

// One warp gathers the candidates of ALL worker CTAs for scan round `tag` (used by the master warp and by the
// service warp of every worker CTA: the exchange is all-to-all) and, optionally, the round's threshold words in the
// same polling loop.  Each lane owns slots lane, lane+32, ...; all words are self-validating, all loads relaxed.
// ~90 CTAs poll the same few lines, so the polling traffic itself sets the latency of the exchange: one 16-byte
// request per candidate, one snapshot in flight, and every candidate in its own 128-byte line (slot_shift = 3)
// measured 1.1 us from the last candidate's store to the decision, against 1.9 us with two 8-byte loads per
// packed slot, and three staggered snapshots in flight were slower than one (profiles/r01c_ahc_trace.md).
// Returns the lexicographic (distance, id) minimum in every lane; `bad` = a NaN seen by any CTA.
__device__ __forceinline__ void gather_candidates(const ResultSlot *results, int shift, int W, int lane, unsigned tag,
                                                  double &d, int &id, bool &bad, const u64 *thr = nullptr,
                                                  double *T = nullptr) {
    const unsigned full = 0xffffffffu;
    if (W <= 96) {
        PollSnap<3> s0;
        do {
            s0.issue(results, shift, W, lane, tag, thr);
        } while (!s0.complete(tag));
        s0.reduce(W, lane, d, id, bad, T);
    } else {
        PollSnap<8> s0;   // W <= 255 worker CTAs
        do {
            s0.issue(results, shift, W, lane, tag, thr);
        } while (!s0.complete(tag));
        s0.reduce(W, lane, d, id, bad, T);
    }
    warp_cand_min(d, id);
    bad = __any_sync(full, bad);
}

// Threshold of a scan round: the key of the root's smaller child in the master's heap (after the round's erase).
// If the new node's nearest-neighbour distance d satisfies d <= T the new node stays at the heap top and the next
// merge is (new node, its nearest neighbour) — every CTA can conclude that by itself.  Two self-validating words.
__device__ __forceinline__ void publish_threshold(u64 *thr, double T, unsigned tag) {
    const u64 bits = (u64)__double_as_longlong(T);
    st_relaxed_u64(&thr[0], (bits & 0xffffffff00000000ull) | (u64)tag);
    st_release_u64(&thr[1], (bits << 32) | (u64)tag);
}
// Master: one warp of CTA 0.  Lane 0 runs the reference's control flow (fastcluster_internal.hpp:1685-1799); the
// other lanes help gathering.  Heap, nearest-neighbour table, slot->node table and live bitmap sit in shared memory:
// every acquire of a polling loop invalidates this SM's L1, and a sift through L2-resident arrays would cost ~100
// dependent 300-cycle loads per step.
//
// The master is OFF the critical path in the common case.  Per scanned merge it (1) does the bookkeeping and the
// reference's erase(), (2) pre-computes the root's descent path and publishes the round's threshold T, (3) gathers
// the candidates like everybody else and finishes replace_key() as one parallel rotation.  If d <= T the workers
// have already started the next merge on their own ("self-issued"); only otherwise (and for lazy nearest-neighbour
// repairs, and for the very first merge) do they wait for an explicit command word.
template <typename Idx>
__device__ void ahc_master(const Problem &P, int W, unsigned char *sm) {
    const int lane = threadIdx.x;
    const unsigned full = 0xffffffffu;
    const int N = P.N;
    const int words = (2 * N - 1 + 31) >> 5;
    double *key = P.key;
    Idx *at = static_cast<Idx *>(P.heap_at), *where = static_cast<Idx *>(P.heap_where);
    int *nn = P.nn, *node_of = P.node_of;
    unsigned *bits = P.live_bits;
    if (P.smem_level >= 1) {
        size_t off = 0;
        auto take = [&](size_t bytes) {
            unsigned char *p = sm + off;
            off = (off + bytes + 15) & ~size_t(15);
            return p;
        };
        double *s_key = reinterpret_cast<double *>(take(sizeof(double) * N));
        Idx *s_at = reinterpret_cast<Idx *>(take(sizeof(Idx) * N));
        Idx *s_where = reinterpret_cast<Idx *>(take(sizeof(Idx) * N));
        unsigned *s_bits = reinterpret_cast<unsigned *>(take(sizeof(unsigned) * words));
        for (int i = lane; i < N; i += 32) {
            s_key[i] = key[i];
            s_where[i] = where[i];
            if (i < N - 1) s_at[i] = at[i];
        }
        for (int i = lane; i < words; i += 32) s_bits[i] = 0xffffffffu;
        key = s_key;
        at = s_at;
        where = s_where;
        bits = s_bits;
        if (P.smem_level >= 2) {
            int *s_nn = reinterpret_cast<int *>(take(sizeof(int) * N));
            for (int i = lane; i < N; i += 32) s_nn[i] = nn[i];
            nn = s_nn;
        }
        if (P.smem_level >= 3) {
            int *s_node = reinterpret_cast<int *>(take(sizeof(int) * N));
            for (int i = lane; i < N; i += 32) s_node[i] = i;
            node_of = s_node;
        }
    } else {
        for (int i = lane; i < words; i += 32) bits[i] = 0xffffffffu;
    }
    if (P.smem_level < 3)
        for (int i = lane; i < N; i += 32) node_of[i] = i;
    for (int i = lane; i < N; i += 32) P.slot_of[i] = i;
    __syncwarp();

    NnHeapT<Idx> heap{key, at, where, P.heap_size};
    LiveSet live{bits, 2 * N - 1, 0};
    unsigned cmd_counter = 0, round = 0;
    bool failed = false;
    __shared__ int path_pos[40], path_slot[40], path_depth;
    __shared__ double path_key[40];
    const bool allow_self = (P.flags & 8) == 0;

    auto publish = [&](int type, int a, int b) {   // lane 0
        st_release_u64(P.cmd, pack_cmd(type, ++cmd_counter, a, b));
    };

    int sa = 0;               // slot at the heap top (lane 0)
    bool self_issued = false; // the workers already know the pair of this step
    for (int step = 0; step < N - 1 && !failed; ++step) {
        const int fresh = N + step;
        const int trace_step = step - N / 2;   // trace a window in the middle of the run
        if (!self_issued) {
            for (;;) {    // lazy repair of a stale nearest neighbour (:1706-1734)
                int stale = 0;
                if (lane == 0) {
                    sa = heap.top();
                    stale = live.dead(nn[sa]) ? 1 : 0;
                    if (stale) publish(CMD_RESCAN, node_of[sa], 0);
                }
                stale = __shfl_sync(full, stale, 0);
                if (!stale) break;
                ++round;
                double d;
                int id;
                bool bad;
                gather_candidates(P.results + (round & 1u) * P.result_stride, P.slot_shift, W, lane, round, d, id, bad);
                if (bad) {
                    failed = true;
                    break;
                }
                if (lane == 0) {
                    nn[sa] = id;
                    heap.raise_key(sa, d);
                }
                __syncwarp();
            }
            if (failed) break;
        }
        int a = 0, b = 0;
        double T = INFINITY;
        if (lane == 0) {
            a = node_of[sa];
            b = nn[sa];
            if (step < N - 2 && !self_issued) publish(CMD_MERGE, a, b);
            FA_TRACE(0);
            live.drop(a);
            live.drop(b);
            P.merge_a[step] = a;
            P.merge_b[step] = b;
            P.merge_d[step] = key[sa];
            if (step < N - 2) {
                const int sb = P.slot_of[b];
                node_of[sa] = fresh;
                node_of[sb] = -1;
                P.slot_of[fresh] = sa;
                // Heap maintenance that does not depend on the scan result, in the reference's order (erase first,
                // :1792-1796).  sa stays at the root: the element moved by erase() can only rise while strictly
                // smaller than its parent, never past the minimum.
                if (b < live.head) heap.erase(P.slot_of[live.head]); else heap.erase(sb);
                // Descent path the root would take in replace_key (:1797 -> update_geq_): at every level the smaller
                // child, the left one on ties.  sift_down(root, d) swaps along exactly this path while the child's
                // key is < d, so once d is known the whole sift is one parallel rotation, and d <= path_key[1]
                // means the new node stays on top.
                int pos = 0, depth = 0;
                path_pos[0] = 0;
                for (;;) {
                    int child = 2 * pos + 1;
                    if (child >= heap.size) break;
                    if (child + 1 < heap.size && heap.val(child + 1) < heap.val(child)) ++child;
                    ++depth;
                    path_pos[depth] = child;
                    path_slot[depth] = (int)at[child];
                    path_key[depth] = heap.val(child);
                    pos = child;
                }
                path_depth = depth;
                T = depth >= 1 ? path_key[1] : INFINITY;
                if (!allow_self) T = -1.0;   // tuning hook: never self-issue
                publish_threshold(P.threshold + 2 * ((round + 1) & 1u), T, round + 1);
            }
            FA_TRACE(1);
        }
        if (step < N - 2) {
            ++round;
            double d;
            int id;
            bool bad;
            gather_candidates(P.results + (round & 1u) * P.result_stride, P.slot_shift, W, lane, round, d, id, bad);
            if (lane == 0) FA_TRACE(2);
            if (bad) {
                failed = true;
                break;
            }
            __syncwarp();
            const int depth = path_depth;
            T = __shfl_sync(full, T, 0);
            // lane 0 alone touches the root's key (it rewrites it below): read once, broadcast
            const double old_key = __shfl_sync(full, lane == 0 ? key[sa] : 0.0, 0);
            // levels 1..m move up one position, the root element lands at level m
            const bool goes_below = lane >= 1 && lane <= depth && path_key[lane] < d;
            const unsigned below = __ballot_sync(full, goes_below) | 1u;   // bit 0 set so that ffs(~below) = m + 2
            const int m = (d <= old_key) ? 0 : (__ffs(~below) - 2);        // lower_key at the root never moves
            if (lane >= 1 && lane <= m) {
                const int slot = path_slot[lane], to = path_pos[lane - 1];
                at[to] = (Idx)slot;
                where[slot] = (Idx)to;
            }
            if (lane == 0) {
                const int to = path_pos[m];
                at[to] = (Idx)sa;
                where[sa] = (Idx)to;
                key[sa] = d;
                nn[sa] = id;
                FA_TRACE(3);
            }
            __syncwarp();
            self_issued = d <= T;   // same doubles, same comparison as in every worker CTA
        } else {
            self_issued = false;
        }
    }
    if (lane == 0) {
        if (failed) *P.error = 1;
        publish(CMD_EXIT, 0, 0);
    }
}

// Worker CTAs: kMergeThreads scan threads (one resident node each) plus one SERVICE warp that owns all cross-CTA
// traffic of the CTA: it waits for command words, publishes the CTA's candidate, gathers everybody's candidates and
// the round's threshold, decides the next pair, and executes the CTA's only gpu-scope fence.
//
// Memory ordering without a fence on the critical path.  The only worker-written data other CTAs read are the node
// store rows[fresh] / node_weight[fresh] of a merge.  Candidate slots and threshold words are self-validating and
// relaxed.  At the END of every round the service warp executes one fence.acq_rel.gpu:
//   * as a release it orders the CTA's row writes of round q (made visible to it by the round's block barriers)
//     before its slot store of round q+1;
//   * as an acquire it orders the slots it gathered in round q+1 before everything after the next block barrier it
//     joins, i.e. before the row loads of round q+3 (a self-issued round q+2 starts its loads concurrently with it).
// So rows[fresh_q] must not be read before round q+3 — and it is not: the vectors and weights of the two newest
// nodes (fresh_{q+2}, fresh_{q+1}) are kept in shared memory by every CTA and used from there.  Explicit commands
// are stronger still (release/acquire on the command word through the master, which gathered the same slots).
constexpr int kWorkerThreads = kMergeThreads + 32;

__global__ void __launch_bounds__(kWorkerThreads, 1) ahc_merge_kernel(const Problem *pp) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const Problem P = *pp;
    const int W = (int)gridDim.x - 1;
    if (blockIdx.x == 0) {
        if (threadIdx.x < 32) {
            if (P.idx16) ahc_master<uint16_t>(P, W, smem_raw); else ahc_master<int>(P, W, smem_raw);
        }
        return;
    }
    const int wb = (int)blockIdx.x - 1;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const bool svc = warp == kMergeThreads / 32;   // the service warp
    const int N = P.N, D = P.D, Ns = P.Ns;
    const int Dp = (D + 1) & ~1;
    double *vbuf0 = reinterpret_cast<double *>(smem_raw);   // three vector buffers: the two newest nodes + scratch
    double *vbuf1 = vbuf0 + Dp;
    double *vbuf2 = vbuf1 + Dp;
    double *red_d = vbuf2 + Dp;                             // [scan warps]
    int *red_id = reinterpret_cast<int *>(red_d + kMergeThreads / 32);
    double *sv = red_d + kMergeThreads / 32 + kMergeThreads / 32;   // resident node vectors [D x SP], k-major
    __shared__ u64 s_cmd;
    __shared__ int s_owner, s_next_b, s_have_pair;
    __shared__ double s_wnew, s_wprev;

    const bool resident = P.resident != 0;
    const int SP = P.slots_per_cta;
    const int rounds_per_thread = resident ? 1 : (Ns + W * kMergeThreads - 1) / (W * kMergeThreads);
    int ids[kMaxRounds];
#pragma unroll
    for (int r = 0; r < kMaxRounds; ++r) ids[r] = -1;
    if (!svc) {
        if (resident) {
            const int s = wb * SP + t;
            if (t < SP && s < N) {
                ids[0] = s;
                for (int k = 0; k < D; ++k) sv[k * SP + t] = P.cols[(size_t)k * Ns + s];   // coalesced over t
            }
        } else {
#pragma unroll
            for (int r = 0; r < kMaxRounds; ++r) {
                const int s = (r * W + wb) * kMergeThreads + t;
                ids[r] = (r < rounds_per_thread && s < N) ? s : -1;
            }
        }
    }
    unsigned cmd_expect = 0, round = 0;
    int merges = 0;
    int prev_fresh = -1, prev_prev = -1;   // nodes whose vectors vcur / vprev hold
    double *vcur = vbuf0, *vprev = vbuf1, *valt = vbuf2;
    bool have_pair = false;
    int a = 0, b = 0;
    if (t == kMergeThreads) s_owner = -1;
    for (;;) {
        int type = CMD_MERGE;
        if (!have_pair) {          // wait for an explicit command word
            ++cmd_expect;
            if (t == kMergeThreads) {
                u64 c;
                do {
                    c = ld_acquire_u64(P.cmd);
                } while ((unsigned)((c >> 48) & 0x3fffu) != (cmd_expect & 0x3fffu));
                s_cmd = c;
            }
            __syncthreads();
            const u64 c = s_cmd;
            type = (int)(c >> 62);
            a = (int)((c >> 24) & 0xffffffu);
            b = (int)(c & 0xffffffu);
            if (type == CMD_EXIT) break;
        }
        ++round;
        const int trace_step = (wb == 0 && lane == 0 && type == CMD_MERGE) ? merges - N / 2 : -1;
        if (t == 0) FA_TRACE(4);
        const int all_step = (lane == 0 && type == CMD_MERGE) ? merges - N / 2 : -1;   // any CTA (trace of the slowest)
        if ((P.flags & 4) && t == 0 && all_step >= 0 && all_step < kTraceSteps) atomicMax(&P.trace[all_step * 16 + 12], global_ns());
        int limit;
        const double *v;
        if (type == CMD_MERGE) {
            const int fresh = N + merges;
            ++merges;
            // operands: the two newest nodes live on chip (see the ordering note above), older ones in the node store
            const double *la = a == prev_fresh ? vcur : (a == prev_prev ? vprev : nullptr);
            const double *lb = b == prev_fresh ? vcur : (b == prev_prev ? vprev : nullptr);
            double wa = 0.0, wbv = 0.0;
            if (!svc) {
                wa = a == prev_fresh ? s_wnew : (a == prev_prev ? s_wprev : (double)__ldcg(P.node_weight + a));
                wbv = b == prev_fresh ? s_wnew : (b == prev_prev ? s_wprev : (double)__ldcg(P.node_weight + b));
                const double *ra = P.rows + (size_t)a * D, *rb = P.rows + (size_t)b * D;
                const double den = __dadd_rn(wa, wbv);
                for (int k = t; k < D; k += kMergeThreads) {
                    const double xa = la ? la[k] : __ldcg(ra + k);
                    const double xb = lb ? lb[k] : __ldcg(rb + k);
                    valt[k] = __ddiv_rn(__dadd_rn(__dmul_rn(xa, wa), __dmul_rn(xb, wbv)), den);
                }
                // the thread holding a turns into `fresh`, the one holding b goes idle
#pragma unroll
                for (int r = 0; r < kMaxRounds; ++r) {
                    if (r < rounds_per_thread) {
                        if (ids[r] == a) {
                            ids[r] = fresh;
                            s_owner = resident ? t : (r * W + wb) * kMergeThreads + t;
                        } else if (ids[r] == b) {
                            ids[r] = -1;
                        }
                    }
                }
            }
            __syncthreads();   // valt complete, s_owner set; all reads of s_wnew / s_wprev / vcur / vprev done
            {
                double *tmp = vprev;
                vprev = vcur;
                vcur = valt;
                valt = tmp;
            }
            if (t == 0) {
                s_wprev = s_wnew;   // weight of the node vprev now holds
                s_wnew = __dadd_rn(wa, wbv);
            }
            const int os = s_owner;
            if (os >= 0 && !svc) {   // this CTA holds the slot: store the new node (scan copy + node-store row + weight)
                double *row = P.rows + (size_t)fresh * D;
                for (int k = t; k < D; k += kMergeThreads) {
                    if (resident) sv[k * SP + os] = vcur[k]; else P.cols[(size_t)k * Ns + os] = vcur[k];
                    row[k] = vcur[k];
                }
                if (t == 0) P.node_weight[fresh] = (int)(wa + wbv);
            }
            prev_prev = prev_fresh;
            prev_fresh = fresh;
            limit = fresh;
            v = vcur;
        } else {
            const double *lt = a == prev_fresh ? vcur : (a == prev_prev ? vprev : nullptr);
            if (lt) {
                v = lt;
            } else {
                const double *rt = P.rows + (size_t)a * D;
                if (!svc)
                    for (int k = t; k < D; k += kMergeThreads) valt[k] = __ldcg(rt + k);
                v = valt;
            }
            __syncthreads();
            limit = a;
        }
        if (t == 0) FA_TRACE(5);
        __syncwarp();   // lane 0's single-thread work above must not leave the warp split across the scan chain
        // ---- scan: one sequential chain per owned live node with id < limit ------------------------------
        if (!svc) {
            double best = INFINITY;
            int best_id = INT_MAX;
            bool bad = false;
            if (resident) {
                const int id = ids[0];
                if (id >= 0 && id < limit) {
                    const double *col = sv + t;
                    double sum = 0.0;
                    int k = 0;
                    for (; k + 8 <= D; k += 8) {
                        double x[8];
#pragma unroll
                        for (int u = 0; u < 8; ++u) x[u] = col[(k + u) * SP];
#pragma unroll
                        for (int u = 0; u < 8; ++u) sum = sq_step(sum, x[u], v[k + u]);
                    }
                    for (; k < D; ++k) sum = sq_step(sum, col[k * SP], v[k]);
                    if (sum != sum) bad = true;
                    best = sum;
                    best_id = id;
                }
            } else {
#pragma unroll
                for (int r = 0; r < kMaxRounds; ++r) {
                    if (r < rounds_per_thread) {
                        const int id = ids[r];
                        if (id >= 0 && id < limit) {
                            const int s = (r * W + wb) * kMergeThreads + t;
                            const double *col = P.cols + s;
                            double sum = 0.0;
                            int k = 0;
                            for (; k + 16 <= D; k += 16) {
                                double x[16];
#pragma unroll
                                for (int u = 0; u < 16; ++u) x[u] = __ldcg(col + (size_t)(k + u) * Ns);
#pragma unroll
                                for (int u = 0; u < 16; ++u) sum = sq_step(sum, x[u], v[k + u]);
                            }
                            for (; k < D; ++k) sum = sq_step(sum, __ldcg(col + (size_t)k * Ns), v[k]);
                            if (sum != sum) bad = true;
                            cand_min(best, best_id, sum, id);
                        }
                    }
                }
            }
            if (t == 0) FA_TRACE(6);
            if (bad) best = INFINITY, best_id = INT_MAX;   // keep NaN bit patterns out of the integer-ordered reduction
            warp_cand_min(best, best_id);
            const bool warp_bad = __any_sync(0xffffffffu, bad);
            if (lane == 0) {
                red_d[warp] = best;
                red_id[warp] = warp_bad ? -2 : best_id;
            }
            if (t == 0) FA_TRACE(11);
        }
        if (t == kMergeThreads) FA_TRACE(13);
        __syncthreads();
        if (t == 0) FA_TRACE(15);
        const bool last_scan = type == CMD_MERGE && merges >= N - 2;   // the master finishes the dendrogram alone
        if (svc) {
            if (lane == 0) {
                FA_TRACE(8);
                double best = INFINITY;
                int best_id = INT_MAX;
                bool any_bad = false;
                for (int w2 = 0; w2 < kMergeThreads / 32; ++w2) {
                    if (red_id[w2] == -2) any_bad = true; else cand_min(best, best_id, red_d[w2], red_id[w2]);
                }
                const u64 bits = (u64)__double_as_longlong(best);
                const unsigned oid = any_bad ? 0xfffffeu : (best_id == INT_MAX ? 0xffffffu : (unsigned)best_id);
                ResultSlot *slot = P.results + (round & 1u) * P.result_stride + ((size_t)wb << P.slot_shift);   // double-buffered by round parity:
                // a CTA reuses a slot two rounds later, which it can only reach after every reader finished this round
                st_relaxed_u64(&slot->w0, (bits & 0xffffffff00000000ull) | ((u64)oid << 8) | (u64)(round & 0xffu));
                st_relaxed_u64(&slot->w1, (bits << 32) | (u64)round);
                FA_TRACE(7);
                if ((P.flags & 4) && all_step >= 0 && all_step < kTraceSteps) atomicMax(&P.trace[all_step * 16 + 14], global_ns());
                s_owner = -1;
            }
            __syncwarp();   // lane 0 publishes before anybody starts polling
            // all-to-all: every CTA learns the new node's nearest neighbour and decides what comes next
            if (type == CMD_MERGE && !last_scan) {
                double d;
                int id;
                bool any_bad;
                double T;
                gather_candidates(P.results + (round & 1u) * P.result_stride, P.slot_shift, W, lane, round, d, id, any_bad,
                                  P.threshold + 2 * (round & 1u), &T);
                if (lane == 0) {
                    FA_TRACE(9);
                    s_have_pair = (!any_bad && d <= T) ? 1 : 0;
                    s_next_b = id;
                }
            }
        }
        if (type != CMD_MERGE) {      // lazy repair round: the master alone consumes the result
            have_pair = false;
            if (svc) fence_acq_rel_gpu();
            continue;
        }
        if (last_scan) break;
        __syncthreads();
        have_pair = s_have_pair != 0;
        a = prev_fresh;
        b = s_next_b;
        if (svc) {
            fence_acq_rel_gpu();   // the CTA's one fence per round, off the critical path (see above)
            if (lane == 0) FA_TRACE(10);
        }
    }
}

// ------------------------------------------------------------------------------------------------ small kernels
// Row-wise L2 normalisation with the oracle's (= AHCClustering.normalizeFeatures') operation order:
// s = sum_k x*x sequentially, scale = s > 0 ? 1/sqrt(s) : 0, out = x*scale.
// zero_scale: what a zero-norm row is multiplied by — 0 for AHCClustering.normalizeFeatures (:70-105), 1 for
// OfflineDiarizerManager.normalize (:824-860, the row is kept).
__global__ void ahc_normalize_rows_kernel(const double *__restrict__ in, double *__restrict__ out, int rows, int dim,
                                          double zero_scale) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= rows) return;
    const double *x = in + (size_t)r * dim;
    double s = 0.0;
    for (int k = 0; k < dim; ++k) s = __dadd_rn(s, __dmul_rn(x[k], x[k]));
    const double scale = s > 0.0 ? __ddiv_rn(1.0, __dsqrt_rn(s)) : zero_scale;
    double *o = out + (size_t)r * dim;
    for (int k = 0; k < dim; ++k) o[k] = __dmul_rn(x[k], scale);
}

__global__ void ahc_widen_kernel(const float *__restrict__ in, double *__restrict__ out, long long count) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) out[i] = (double)in[i];
}

int launch_normalize_rows(const double *d_in, double *d_out, int rows, int dim, cudaStream_t s) {
    if (rows <= 0) return FA_OK;
    ahc_normalize_rows_kernel<<<(rows + 127) / 128, 128, 0, s>>>(d_in, d_out, rows, dim, 0.0);
    FA_CUDA_TRY(cudaGetLastError());
    return FA_OK;
}

int launch_normalize_rows_keep(const double *d_in, double *d_out, int rows, int dim, cudaStream_t s) {
    if (rows <= 0) return FA_OK;
    ahc_normalize_rows_kernel<<<(rows + 127) / 128, 128, 0, s>>>(d_in, d_out, rows, dim, 1.0);
    FA_CUDA_TRY(cudaGetLastError());
    return FA_OK;
}

int launch_widen_rows(const float *d_in, double *d_out, long long count, cudaStream_t s) {
    if (count <= 0) return FA_OK;
    ahc_widen_kernel<<<(unsigned)((count + 255) / 256), 256, 0, s>>>(d_in, d_out, count);
    FA_CUDA_TRY(cudaGetLastError());
    return FA_OK;
}

// ------------------------------------------------------------------------------------------------ host solver
thread_local float g_last_ms[4] = {0, 0, 0, 0};
const float *last_stage_ms() { return g_last_ms; }
thread_local int g_placement[6] = {0, 0, 0, 0, 0, 0};
const int *last_placement() { return g_placement; }

Solver::~Solver() { release(); }

void Solver::release() {
    if (d_pool) cudaFree(d_pool);
    if (d_input) cudaFree(d_input);
    if (h_pool) cudaFreeHost(h_pool);
    d_pool = nullptr;
    d_input = nullptr;
    h_pool = nullptr;
    pool_bytes = h_pool_bytes = input_cap = 0;
}

int Solver::init(cudaStream_t s, int worker_limit) {
    stream = s;
    int dev = 0;
    FA_CUDA_TRY(cudaGetDevice(&dev));
    cudaDeviceProp prop;
    FA_CUDA_TRY(cudaGetDeviceProperties(&prop, dev));
    if (prop.major != 10) {
        fa::set_error("fluidaudio_b200 requires an sm_100a device, found sm_%d%d", prop.major, prop.minor);
        return FA_NO_DEVICE;
    }
    int coop = 0;
    FA_CUDA_TRY(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev));
    if (!coop) {
        fa::set_error("device does not support cooperative launch");
        return FA_UNSUPPORTED;
    }
    num_sms = prop.multiProcessorCount;
    max_workers = std::max(1, std::min(num_sms - 1, worker_limit > 0 ? worker_limit : num_sms - 1));
    return FA_OK;
}

namespace {
struct Carver {
    size_t off = 0;
    template <typename T> size_t take(size_t count) {
        off = (off + 255) & ~size_t(255);
        const size_t at = off;
        off += count * sizeof(T);
        return at;
    }
};
struct Layout {
    size_t rows, cols, node_weight, key, nn, heap_at, heap_where, node_of, slot_of, live_bits, merge_a, merge_b, merge_d,
        cmd, threshold, results, error, trace, init_partial, problem, total;
    size_t f_cf, f_nrm2, f_rn, f_U, f_best_d, f_best_j, f_cand, f_cand_d, f_counters, f_tmin;
    bool f_keep_tmin;
    int ranges, filter_cap;
};
Layout make_layout(int N, int D, int Ns, int workers) {
    Layout L{};
    Carver c;
    L.rows = c.take<double>((size_t)(2 * N - 1) * D);
    L.cols = c.take<double>((size_t)D * Ns);
    L.node_weight = c.take<int>((size_t)2 * N);
    L.key = c.take<double>((size_t)N + 2);
    L.nn = c.take<int>((size_t)N + 2);
    L.heap_at = c.take<int>((size_t)N + 2);
    L.heap_where = c.take<int>((size_t)N + 2);
    L.node_of = c.take<int>((size_t)N + 2);
    L.slot_of = c.take<int>((size_t)2 * N);
    L.live_bits = c.take<unsigned>((size_t)(2 * N + 31) / 32 + 2);
    L.merge_a = c.take<int>((size_t)N);
    L.merge_b = c.take<int>((size_t)N);
    L.merge_d = c.take<double>((size_t)N);
    L.cmd = c.take<unsigned long long>(32);         // own 256-byte line
    L.threshold = c.take<unsigned long long>(32);   // own 256-byte line
    L.results = c.take<ResultSlot>(2 * 8 * ((size_t)workers + 1));
    L.error = c.take<int>(64);
    L.trace = c.take<unsigned long long>((size_t)kTraceSteps * 16);
    L.ranges = (N + kJR - 1) / kJR;
    L.init_partial = c.take<Cand>((size_t)L.ranges * N);
    L.problem = c.take<Problem>(1);
    // float32 filter of the initial nearest-neighbour pass (N >= kFilterMinN only, but sized unconditionally: small)
    L.filter_cap = (int)std::min<long long>(64LL * N, 1 << 24);
    L.f_cf = c.take<float>((size_t)((D + 7) & ~7) * Ns);   // rows rounded up to the GEMM's k-chunk (zero rows)
    L.f_nrm2 = c.take<double>((size_t)N);
    L.f_rn = c.take<float>((size_t)N);
    L.f_U = c.take<unsigned long long>((size_t)N);
    L.f_best_d = c.take<unsigned long long>((size_t)N);
    L.f_best_j = c.take<int>((size_t)N);
    L.f_cand = c.take<int2>((size_t)L.filter_cap);
    L.f_cand_d = c.take<double>((size_t)L.filter_cap);
    L.f_counters = c.take<int>(64);
    {
        const long long nt = (N + 63) / 64;
        L.f_keep_tmin = (long long)N * nt <= (16LL << 20);   // <= 64 MB
        L.f_tmin = c.take<float>(L.f_keep_tmin ? (size_t)((long long)N * nt) : 1);
    }
    L.total = (c.off + 255) & ~size_t(255);
    return L;
}
// bytes of master state staged in shared memory at each level (must mirror ahc_master's carving)
size_t master_smem_bytes(int N, int level) {
    auto up = [](size_t b) { return (b + 15) & ~size_t(15); };
    const size_t words = (size_t)(2 * N - 1 + 31) >> 5;
    size_t b = up(sizeof(double) * N) + 2 * up(sizeof(uint16_t) * N) + up(sizeof(unsigned) * words);
    if (level >= 2) b += up(sizeof(int) * N);
    if (level >= 3) b += up(sizeof(int) * N);
    return b;
}
} // namespace

// Worker CTAs a problem needs to keep every node vector in shared memory (the fast placement), or 0 if a single CTA
// cannot hold even one vector.  Mirrors the sizing in linkage_device.
int resident_workers_needed(int N, int D) {
    const size_t smem_cap = 227 * 1024 - 2048;
    const size_t worker_fixed = 3 * sizeof(double) * (size_t)((D + 1) & ~1) + 2 * sizeof(double) * (kMergeThreads / 32) + 64;
    if (worker_fixed + sizeof(double) * D > smem_cap) return 0;
    const int cap_slots = (int)std::min<size_t>(kMergeThreads, (smem_cap - worker_fixed) / (sizeof(double) * (size_t)D));
    if (cap_slots < 1) return 0;
    return (N + cap_slots - 1) / cap_slots;
}

int Solver::ensure_pool(int N, int D) {
    const int Ns = (N + 31) & ~31;
    const Layout L = make_layout(N, D, Ns, max_workers);
    if (L.total > pool_bytes) {
        if (d_pool) cudaFree(d_pool);
        d_pool = nullptr;
        pool_bytes = 0;
        FA_CUDA_TRY(cudaMalloc(&d_pool, L.total));
        pool_bytes = L.total;
    }
    const size_t hneed = sizeof(double) * (size_t)(2 * N + 16) + sizeof(int) * (size_t)(4 * N + 64);
    if (hneed > h_pool_bytes) {
        if (h_pool) cudaFreeHost(h_pool);
        h_pool = nullptr;
        h_pool_bytes = 0;
        FA_CUDA_TRY(cudaMallocHost(&h_pool, hneed));
        h_pool_bytes = hneed;
    }
    return FA_OK;
}

// FA_AHC_* environment hooks (test / tuning only: fall-back placements at small N, trace, candidate spacing), read once.
struct Hooks {
    bool force_global = false, force_stream = false;
    int slot_shift = 3, flags = 0;
    int filter_min_n = 2048;   // FA_AHC_FILTER_MIN_N: problems at least this large take the float32 filter (0 = never)
    int filter_impl = 0;       // FA_AHC_FILTER_IMPL: bit 0 = 64 x 64 tiles in pass 1, bit 1 = dense pass 2 (A/B measurements)
};
static const Hooks &hooks() {
    static const Hooks h = [] {
        Hooks x;
        const char *g = std::getenv("FA_AHC_FORCE_GLOBAL_MASTER"), *s = std::getenv("FA_AHC_FORCE_STREAMED");
        const char *sh = std::getenv("FA_AHC_SLOT_SHIFT"), *f = std::getenv("FA_AHC_FLAGS");
        x.force_global = g && g[0] == '1';
        x.force_stream = s && s[0] == '1';
        if (sh) x.slot_shift = std::min(3, std::max(0, std::atoi(sh)));
        if (f) x.flags = std::atoi(f);
        if (const char *m = std::getenv("FA_AHC_FILTER_MIN_N")) x.filter_min_n = std::atoi(m);
        if (const char *m = std::getenv("FA_AHC_FILTER_IMPL")) x.filter_impl = std::atoi(m);
        return x;
    }();
    return h;
}

int Solver::linkage_device(const double *d_rows, int N, int D, double *Z) {
    if (N < 2) return FA_OK;
    const int Ns = (N + 31) & ~31;
    // master placement: slot-indexed heap (+ nn, + node_of) in shared memory when it fits
    const size_t smem_cap = 227 * 1024 - 2048;   // leaves room for the kernel's static shared memory
    int level = 0;
    if (N <= 65535)
        for (int l = 1; l <= 3; ++l)
            if (master_smem_bytes(N, l) <= smem_cap) level = l;
    // test hooks: exercise the fall-back placements at small N (tests/test_gpu_parity.py)
    // (all FA_AHC_* hooks are read ONCE per process, see hooks(): stray variables cannot change behaviour mid-run)
    const Hooks &hk = hooks();
    const bool force_global = hk.force_global, force_stream = hk.force_stream;
    if (force_global) level = 0;
    const bool idx16 = level >= 1;
    // worker placement: resident (each CTA keeps <= 128 node vectors in shared memory) when the whole problem fits
    // into max_workers CTAs, else streamed from the k-major global copy
    const size_t worker_fixed = 3 * sizeof(double) * (size_t)((D + 1) & ~1) + 2 * sizeof(double) * (kMergeThreads / 32) + 64;
    if (worker_fixed + sizeof(double) * D > smem_cap) {
        fa::set_error("dimension %d too large for the merge kernel's shared-memory target vector", D);
        return FA_RUNTIME_ERROR;
    }
    const int cap_slots = (int)std::min<size_t>(kMergeThreads, (smem_cap - worker_fixed) / (sizeof(double) * (size_t)D));
    bool resident = cap_slots >= 1 && (long long)cap_slots * max_workers >= N;
    if (force_stream) resident = false;
    int workers, slots_per_cta = 0;
    size_t worker_smem = worker_fixed;
    if (resident) {
        // enough CTAs to hold every node, but no more than needed: the per-step barrier cost grows with CTA count
        workers = std::min(max_workers, std::max(1, (N + cap_slots - 1) / cap_slots));
        slots_per_cta = (N + workers - 1) / workers;
        worker_smem += sizeof(double) * (size_t)D * slots_per_cta;
    } else {
        workers = std::max(1, std::min(max_workers, (Ns + kMergeThreads - 1) / kMergeThreads));
        if ((long long)workers * kMergeThreads * kMaxRounds < Ns) {
            fa::set_error("point count %d exceeds the capacity of the merge kernel (%lld)", N,
                          (long long)workers * kMergeThreads * kMaxRounds);
            return FA_RUNTIME_ERROR;
        }
    }
    const size_t smem = std::max(worker_smem, level ? master_smem_bytes(N, level) : (size_t)0);
    g_placement[0] = level;
    g_placement[1] = resident ? 1 : 0;
    g_placement[2] = workers;
    g_placement[3] = slots_per_cta;
    g_placement[4] = kInitExact;
    g_placement[5] = num_sms;
    int st = ensure_pool(N, D);
    if (st != FA_OK) return st;
    const Layout L = make_layout(N, D, Ns, max_workers);
    char *base = static_cast<char *>(d_pool);
    Problem P{};
    P.N = N;
    P.D = D;
    P.Ns = Ns;
    P.rows = reinterpret_cast<double *>(base + L.rows);
    P.cols = reinterpret_cast<double *>(base + L.cols);
    P.node_weight = reinterpret_cast<int *>(base + L.node_weight);
    P.key = reinterpret_cast<double *>(base + L.key);
    P.nn = reinterpret_cast<int *>(base + L.nn);
    P.heap_at = base + L.heap_at;
    P.heap_where = base + L.heap_where;
    P.node_of = reinterpret_cast<int *>(base + L.node_of);
    P.slot_of = reinterpret_cast<int *>(base + L.slot_of);
    P.live_bits = reinterpret_cast<unsigned *>(base + L.live_bits);
    P.merge_a = reinterpret_cast<int *>(base + L.merge_a);
    P.merge_b = reinterpret_cast<int *>(base + L.merge_b);
    P.merge_d = reinterpret_cast<double *>(base + L.merge_d);
    P.cmd = reinterpret_cast<unsigned long long *>(base + L.cmd);
    P.threshold = reinterpret_cast<unsigned long long *>(base + L.threshold);
    P.results = reinterpret_cast<ResultSlot *>(base + L.results);
    P.slot_shift = hk.slot_shift;   // tuning hook: 0 = packed, 1 = 32 B, 3 = 128 B per candidate (default)
    P.result_stride = (max_workers + 1) << P.slot_shift;
    P.error = reinterpret_cast<int *>(base + L.error);
    P.trace = reinterpret_cast<unsigned long long *>(base + L.trace);
    P.resident = resident ? 1 : 0;
    P.slots_per_cta = slots_per_cta;
    P.idx16 = idx16 ? 1 : 0;
    P.smem_level = level;
    P.flags = hk.flags;             // tuning hooks: 4 = globaltimer trace, 8 = never self-issue
    Cand *init_partial = reinterpret_cast<Cand *>(base + L.init_partial);
    Problem *d_prob = reinterpret_cast<Problem *>(base + L.problem);

    // pinned host mirrors
    char *hb = static_cast<char *>(h_pool);
    double *h_key = reinterpret_cast<double *>(hb);
    double *h_md = h_key + N + 4;
    int *h_at = reinterpret_cast<int *>(h_md + N + 4);   // N ints (reused as uint16 when idx16)
    int *h_where = h_at + N + 2;
    int *h_ma = h_where + N + 2;
    int *h_mb = h_ma + N;
    int *h_err = h_mb + N;

    // timing events live in a guard: every early return below (FA_CUDA_TRY) releases them
    struct Events {
        cudaEvent_t e[4] = {nullptr, nullptr, nullptr, nullptr};
        ~Events() {
            for (auto x : e)
                if (x) cudaEventDestroy(x);
        }
        cudaEvent_t &operator[](int i) { return e[i]; }
    } ev;
    for (int i = 0; i < 4; ++i) FA_CUDA_TRY(cudaEventCreate(&ev.e[i]));
    auto drop_events = [&]() {};

    FA_CUDA_TRY(cudaMemsetAsync(base + L.cmd, 0, 256, stream));
    FA_CUDA_TRY(cudaMemsetAsync(base + L.threshold, 0, 256, stream));
    FA_CUDA_TRY(cudaMemsetAsync(base + L.results, 0, 2 * 8 * sizeof(ResultSlot) * (size_t)(max_workers + 1), stream));
    FA_CUDA_TRY(cudaMemsetAsync(base + L.error, 0, 256, stream));
    FA_CUDA_TRY(cudaMemsetAsync(base + L.trace, 0, sizeof(unsigned long long) * kTraceSteps * 16, stream));
    FA_CUDA_TRY(cudaEventRecord(ev[0], stream));
    {
        dim3 grid((Ns + 31) / 32, (D + 31) / 32), block(32, 8);
        ahc_stage_kernel<<<grid, block, 0, stream>>>(d_rows, P.rows, P.cols, N, D, Ns);
        FA_CUDA_TRY(cudaGetLastError());
        launches += 1;
    }
    auto exact_init = [&]() -> int {
        dim3 g2((N + kTI - 1) / kTI, L.ranges);
        ahc_init_nn_kernel<<<g2, kTI, 0, stream>>>(P.cols, N, D, Ns, init_partial, P.error);
        FA_CUDA_TRY(cudaGetLastError());
        ahc_init_reduce_kernel<<<(N + 127) / 128, 128, 0, stream>>>(init_partial, N, L.ranges, P.key, P.nn,
                                                                     P.node_weight);
        FA_CUDA_TRY(cudaGetLastError());
        launches += 2;
        return FA_OK;
    };
    const bool use_filter = hk.filter_min_n > 0 && N >= hk.filter_min_n;
    int *h_fc = h_err + 1;   // [3] filter counters (pinned)
    if (use_filter) {
        FilterBufs F{};
        F.cf = reinterpret_cast<float *>(base + L.f_cf);
        F.nrm2 = reinterpret_cast<double *>(base + L.f_nrm2);
        F.rn = reinterpret_cast<float *>(base + L.f_rn);
        F.U = reinterpret_cast<unsigned long long *>(base + L.f_U);
        F.best_d = reinterpret_cast<unsigned long long *>(base + L.f_best_d);
        F.best_j = reinterpret_cast<int *>(base + L.f_best_j);
        F.cand = reinterpret_cast<int2 *>(base + L.f_cand);
        F.cand_d = reinterpret_cast<double *>(base + L.f_cand_d);
        F.counters = reinterpret_cast<int *>(base + L.f_counters);
        F.cap = L.filter_cap;
        F.nt = (N + kFT - 1) / kFT;
        F.tmin = L.f_keep_tmin ? reinterpret_cast<float *>(base + L.f_tmin) : nullptr;
        F.c1 = 2.02 * (double)(D + 3) * 5.9604644775390625e-08;   // 2^-24
        F.c2 = 2e-12;
        FA_CUDA_TRY(cudaMemsetAsync(F.counters, 0, 64 * sizeof(int), stream));
        ahc_filter_prep_kernel<<<(Ns + 127) / 128, 128, 0, stream>>>(P.cols, N, D, Ns, F);
        const int nt = (N + kFT - 1) / kFT;
        const unsigned tiles = (unsigned)((long long)nt * (nt + 1) / 2);
        if (hk.filter_impl & 1) {
            ahc_filter_tile_kernel<false><<<tiles, 256, 0, stream>>>(N, D, Ns, F);
        } else {
            const int nt2 = (N + kGT - 1) / kGT;
            ahc_filter_tile128_kernel<<<(unsigned)((long long)nt2 * (nt2 + 1) / 2), 256, 0, stream>>>(N, D, Ns, F);
        }
        if (!(hk.filter_impl & 2) && F.tmin && (size_t)8 * D * sizeof(float) <= 48 * 1024) {
            ahc_filter_rows_kernel<<<(N + 7) / 8, 256, (size_t)8 * D * sizeof(float), stream>>>(N, D, Ns, F);
            g_placement[4] = kInitFilterRows;
        } else {
            ahc_filter_tile_kernel<true><<<tiles, 256, 0, stream>>>(N, D, Ns, F);
            g_placement[4] = kInitFilterTiles;
        }
        const unsigned cgrid = (unsigned)((F.cap + 255) / 256);
        ahc_filter_exact_kernel<<<cgrid, 256, 0, stream>>>(P.cols, D, Ns, F);
        ahc_filter_argmin_kernel<<<cgrid, 256, 0, stream>>>(F);
        ahc_filter_finish_kernel<<<(N + 127) / 128, 128, 0, stream>>>(N, F, P.key, P.nn, P.node_weight);
        FA_CUDA_TRY(cudaGetLastError());
        launches += 6;
        FA_CUDA_TRY(cudaMemcpyAsync(h_fc, F.counters, 3 * sizeof(int), cudaMemcpyDeviceToHost, stream));
        FA_CUDA_TRY(cudaStreamSynchronize(stream));
        if (h_fc[1] || h_fc[2]) {   // non-finite / huge input, or more candidates than the list holds: the exact pass decides
            g_placement[4] = kInitFilterFellBack;
            const int st2 = exact_init();
            if (st2 != FA_OK) return st2;
        }
    } else {
        const int st2 = exact_init();
        if (st2 != FA_OK) return st2;
    }
    FA_CUDA_TRY(cudaEventRecord(ev[1], stream));
    FA_CUDA_TRY(cudaMemcpyAsync(h_key, P.key, sizeof(double) * N, cudaMemcpyDeviceToHost, stream));
    FA_CUDA_TRY(cudaMemcpyAsync(h_err, P.error, sizeof(int), cudaMemcpyDeviceToHost, stream));
    FA_CUDA_TRY(cudaStreamSynchronize(stream));
    if (*h_err != 0) {
        drop_events();
        fa::set_error("NaN distance between input vectors");
        return FA_RUNTIME_ERROR;   // reference: nan_error -> FASTCLUSTER_WRAPPER_RUNTIME_ERROR
    }
    // heapify on the host (fastcluster_internal.hpp:1682): O(N), ~50 us, avoids ~1 ms of serial device work
    size_t idx_bytes;
    if (idx16) {
        NnHeapT<uint16_t> heap{h_key, reinterpret_cast<uint16_t *>(h_at), reinterpret_cast<uint16_t *>(h_where), 0};
        heap.where[0] = 0;
        heap.build(N - 1, 1);
        P.heap_size = heap.size;
        idx_bytes = sizeof(uint16_t);
    } else {
        NnHeapT<int> heap{h_key, h_at, h_where, 0};
        heap.where[0] = 0;
        heap.build(N - 1, 1);
        P.heap_size = heap.size;
        idx_bytes = sizeof(int);
    }
    FA_CUDA_TRY(cudaMemcpyAsync(P.heap_at, h_at, idx_bytes * (N - 1), cudaMemcpyHostToDevice, stream));
    FA_CUDA_TRY(cudaMemcpyAsync(P.heap_where, h_where, idx_bytes * N, cudaMemcpyHostToDevice, stream));
    FA_CUDA_TRY(cudaMemcpyAsync(d_prob, &P, sizeof(Problem), cudaMemcpyHostToDevice, stream));
    FA_CUDA_TRY(cudaEventRecord(ev[2], stream));
    {
        static std::once_flag once;   // a per-function attribute: set it once to the maximum, solvers run concurrently
        static cudaError_t attr_err = cudaSuccess;
        std::call_once(once, [&]() {
            attr_err = cudaFuncSetAttribute(ahc_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_cap);
        });
        FA_CUDA_TRY(attr_err);
        void *args[] = {&d_prob};
        FA_CUDA_TRY(cudaLaunchCooperativeKernel((void *)ahc_merge_kernel, dim3(workers + 1), dim3(kWorkerThreads), args,
                                                smem, stream));
        ++launches;
    }
    FA_CUDA_TRY(cudaEventRecord(ev[3], stream));
    FA_CUDA_TRY(cudaMemcpyAsync(h_ma, P.merge_a, sizeof(int) * (N - 1), cudaMemcpyDeviceToHost, stream));
    FA_CUDA_TRY(cudaMemcpyAsync(h_mb, P.merge_b, sizeof(int) * (N - 1), cudaMemcpyDeviceToHost, stream));
    FA_CUDA_TRY(cudaMemcpyAsync(h_md, P.merge_d, sizeof(double) * (N - 1), cudaMemcpyDeviceToHost, stream));
    FA_CUDA_TRY(cudaMemcpyAsync(h_err, P.error, sizeof(int), cudaMemcpyDeviceToHost, stream));
    FA_CUDA_TRY(cudaStreamSynchronize(stream));
    cudaEventElapsedTime(&last_ms[0], ev[0], ev[1]);
    cudaEventElapsedTime(&last_ms[1], ev[1], ev[2]);
    cudaEventElapsedTime(&last_ms[2], ev[2], ev[3]);
    cudaEventElapsedTime(&last_ms[3], ev[0], ev[3]);
    for (int q = 0; q < 4; ++q) g_last_ms[q] = last_ms[q];
    if ((P.flags & 4) && N > 2 * kTraceSteps + 8) {
        std::vector<unsigned long long> tr((size_t)kTraceSteps * 16);
        cudaMemcpy(tr.data(), P.trace, tr.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost);
        double acc[16] = {0};
        int used = 0;
        for (int i = 1; i + 1 < kTraceSteps; ++i) {
            const unsigned long long t0 = tr[(size_t)i * 16];
            if (!t0) continue;
            for (int q = 0; q < 16; ++q)
                if (tr[(size_t)i * 16 + q]) acc[q] += (double)((long long)(tr[(size_t)i * 16 + q] - t0));
            acc[0] += (double)((long long)(tr[(size_t)(i + 1) * 16] - t0));   // slot 0: step period
            ++used;
        }
        for (int q = 0; q < 8; ++q) trace_avg_ns[q] = used ? acc[q] / used : 0.0;
        const auto avg = [&](int q) { return used ? acc[q] / used : 0.0; };
        std::fprintf(stderr,
                     "[ahc trace] ns from the master's step start, mean of %d steps | period %.0f | master: bookkeeping+erase+"
                     "path %.0f, candidates gathered %.0f, heap rotated %.0f | worker 0: round start %.0f, centroid built %.0f, "
                     "scan done %.0f, warp reduce done %.0f, service warp at barrier %.0f / released %.0f, candidate published "
                     "%.0f, all gathered %.0f, fence retired %.0f | slowest CTA: round start %.0f, candidate published %.0f",
                     used, avg(0), avg(1), avg(2), avg(3), avg(4), avg(5), avg(6), avg(11), avg(13), avg(8), avg(7), avg(9),
                     avg(10), avg(12), avg(14));
        std::fprintf(stderr, "\n");
    }
    drop_events();
    if (*h_err != 0) {
        fa::set_error("NaN distance during merging");
        return FA_RUNTIME_ERROR;
    }
    // SciPy rows in merge order (FastClusterWrapper.cpp:128-130,169-192): sqrt of the squared distance,
    // smaller id first, size = sum of the children's sizes
    for (int s = 0; s < N - 1; ++s) {
        const int lo = std::min(h_ma[s], h_mb[s]), hi = std::max(h_ma[s], h_mb[s]);
        const double sz = (lo < N ? 1.0 : Z[(size_t)(lo - N) * 4 + 3]) + (hi < N ? 1.0 : Z[(size_t)(hi - N) * 4 + 3]);
        Z[(size_t)s * 4 + 0] = (double)lo;
        Z[(size_t)s * 4 + 1] = (double)hi;
        Z[(size_t)s * 4 + 2] = std::sqrt(h_md[s]);
        Z[(size_t)s * 4 + 3] = sz;
    }
    return FA_OK;
}

int Solver::linkage_host(const double *rows_host, size_t N, size_t D, double *Z, size_t z_len) {
    // argument contract of FastClusterWrapper.cpp:203-223
    if (!rows_host || !Z) return FA_INVALID_ARGUMENT;
    if (N == 0) return FA_OK;
    if (D == 0) return FA_INVALID_ARGUMENT;
    if (N > 0x7fffffffull || D > 0x7fffffffull) return FA_INDEX_OVERFLOW;
    if (z_len < (N > 1 ? (N - 1) * 4 : 0)) return FA_OUTPUT_TOO_SMALL;
    if (N == 1) return FA_OK;
    const size_t count = N * D;
    if (count > input_cap) {
        if (d_input) cudaFree(d_input);
        d_input = nullptr;
        input_cap = 0;
        FA_CUDA_TRY(cudaMalloc(&d_input, count * sizeof(double)));
        input_cap = count;
    }
    FA_CUDA_TRY(cudaMemcpyAsync(d_input, rows_host, count * sizeof(double), cudaMemcpyHostToDevice, stream));
    return linkage_device(d_input, (int)N, (int)D, Z);
}

// Swift-side cut (AHCClustering.swift:112-121 clamp, :124-197 traversal, :200-210 relabel)
void dendrogram_cut(const double *Z, long long count, double threshold, int32_t *labels) {
    if (count <= 0) return;
    if (count == 1) {
        labels[0] = 0;
        return;
    }
    const double thr = (threshold != threshold) ? 0.0 : std::max(0.0, std::min(2.0, threshold));
    const long long total = 2 * count - 1;
    std::vector<long long> lc(total, -1), rc(total, -1);
    std::vector<double> nd(total, 0.0);
    for (long long m = 0; m + 1 < count; ++m) {
        // children of row m must be earlier nodes (0 <= id < count + m): anything else in a caller-supplied Z (NaN, a
        // negative or forward reference) is dropped, which also rules out cycles; the leaves it orphans get fresh labels
        const double za = Z[m * 4], zb = Z[m * 4 + 1];
        const double hi = (double)(count + m);
        lc[count + m] = (za >= 0.0 && za < hi) ? (long long)za : -1;
        rc[count + m] = (zb >= 0.0 && zb < hi) ? (long long)zb : -1;
        nd[count + m] = Z[m * 4 + 2];
    }
    std::vector<long long> lab(count, -1), todo, sub;
    todo.push_back(total - 1);
    long long next = 0;
    while (!todo.empty()) {
        const long long node = todo.back();
        todo.pop_back();
        if (node < 0) continue;
        if (node < count) {
            if (lab[node] < 0) lab[node] = next++;
            continue;
        }
        if (nd[node] <= thr) {          // whole subtree is one cluster
            const long long id = next++;
            sub.assign(1, node);
            while (!sub.empty()) {
                const long long cur = sub.back();
                sub.pop_back();
                if (cur < count) lab[cur] = id;
                else {
                    if (lc[cur] >= 0) sub.push_back(lc[cur]);
                    if (rc[cur] >= 0) sub.push_back(rc[cur]);
                }
            }
        } else {                        // split: left pushed first, so the right child is visited first
            if (lc[node] >= 0) todo.push_back(lc[node]);
            if (rc[node] >= 0) todo.push_back(rc[node]);
        }
    }
    for (long long i = 0; i < count; ++i)
        if (lab[i] < 0) lab[i] = next++;
    std::vector<int32_t> canon((size_t)next, -1);
    int32_t fresh = 0;
    for (long long i = 0; i < count; ++i) {
        if (canon[lab[i]] < 0) canon[lab[i]] = fresh++;
        labels[i] = canon[lab[i]];
    }
}

} // namespace ahc
} // namespace fa
