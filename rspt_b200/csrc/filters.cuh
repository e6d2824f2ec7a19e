// Pre-filter step in front of the packers for sm_100a: the IIR / FIR filtering the reference's
// pipeline applies to a frame before packing it (lib_rspt_test/rspt_test.cpp:116-136) with
// i_filter (lib_rspt/filter.h:23-89, lib_filter/iir_filter.cpp:46-116, fir_filter.cpp:26-68),
// batched over frames.  Results are bit-identical to the reference's: the same double-precision
// operations in the same order, each rounded separately (__dmul_rn / __dadd_rn keep the compiler
// from contracting them into FMAs, which the reference's x86-64 build does not use).
//
// IIR: the reference walks ONE filter object over the channels of a frame and only re-settles it
// with init_history_values (4 * nr_samples steps on the channel's first sample) -- the state of
// the previous channel is not cleared and has not fully decayed after that many steps (the
// 0.4 Hz high-pass pole of the test's band-pass keeps ~0.7 % of it).  Reproducing the output
// bit for bit therefore means running the frame's channels in sequence: one thread per frame, a
// serial chain of ch * (4 * nr_samples + ns) steps.  The kernel is latency-bound by that chain
// (8 dependent FP64 adds per step); frames are the parallel axis.
// FIR: after init_history_values the ring holds kernel_size copies of the channel's first sample
// whatever it held before, so channels and samples are independent: one thread per output sample.
#pragma once

#include "common.cuh"

namespace rspt {

struct IirCoef {
    double n[5], d[5];
    int nc;          // 2..5 coefficients
    int init_calls;  // 4 * nr_samples (iir_filter.cpp:105-109)
};

// One warp per 32 frames, lane = frame.  The words of the 32 frames are moved through a 32 x 32
// shared-memory tile (row = frame, padded to 33) so that global loads and stores are coalesced
// 128-byte rows; the next tile is fetched into registers while the current one is filtered, so the
// memory latency hides behind the serial chain.
template <int NC>
__global__ void __launch_bounds__(32) k_iir_frames(int32_t* __restrict__ words, Shape s, uint32_t n_frames, IirCoef c)
{
    __shared__ int32_t tile[32][33];
    const uint32_t lane = threadIdx.x, f0 = blockIdx.x * 32u;
    const uint32_t nf = min(32u, n_frames - f0);  // frames of this warp
    const bool live = lane < nf;
    int32_t* w0 = words + (size_t)f0 * s.N;
    const uint32_t ns = (uint32_t)s.ns;
    double x[NC], y[NC];
#pragma unroll
    for (int i = 0; i < NC; ++i) x[i] = y[i] = 0.0;
    auto fetch = [&](int32_t (&v)[32], uint32_t j, uint32_t i0) {
#pragma unroll
        for (uint32_t r = 0; r < 32; ++r)
            v[r] = (r < nf && i0 + lane < ns) ? w0[(size_t)r * s.N + (size_t)j * ns + i0 + lane] : 0;
    };
    int32_t nxt[32];
    fetch(nxt, 0, 0);
    for (uint32_t j = 0; j < (uint32_t)s.ch; ++j) {
        for (uint32_t i0 = 0; i0 < ns; i0 += 32) {
#pragma unroll
            for (uint32_t r = 0; r < 32; ++r) tile[r][lane] = nxt[r];
            __syncwarp();
            // the tile after this one (same channel, or the start of the next channel)
            {
                const uint32_t ni = i0 + 32 < ns ? i0 + 32 : 0u, nj = i0 + 32 < ns ? j : j + 1;
                if (nj < (uint32_t)s.ch) fetch(nxt, nj, ni);
            }
            if (i0 == 0 && live) {
                // init_history_values: iir_filter::filter (iir_filter.cpp:58-73), d and n terms alternating
                const double x0 = (double)tile[lane][0];
                for (int it = 0; it < c.init_calls; ++it) {
#pragma unroll
                    for (int i = NC - 1; i > 0; --i) {
                        x[i] = x[i - 1];
                        y[i] = y[i - 1];
                    }
                    x[0] = x0;
                    double acc = __dmul_rn(c.d[0], x[0]);
#pragma unroll
                    for (int i = 1; i < NC; ++i) {
                        acc = __dadd_rn(acc, __dmul_rn(c.d[i], x[i]));
                        acc = __dsub_rn(acc, __dmul_rn(c.n[i], y[i]));
                    }
                    y[0] = acc;
                }
            }
            // filter_opt (iir_filter.cpp:75-103, rolling_iir_filter_N_ :26-44): d terms, then n terms
            const uint32_t cnt = min(32u, ns - i0);
            if (live) {
                for (uint32_t k = 0; k < cnt; ++k) {
#pragma unroll
                    for (int i = NC - 1; i > 0; --i) {
                        x[i] = x[i - 1];
                        y[i] = y[i - 1];
                    }
                    x[0] = (double)tile[lane][k];
                    double acc = __dmul_rn(c.d[0], x[0]);
#pragma unroll
                    for (int i = 1; i < NC; ++i) acc = __dadd_rn(acc, __dmul_rn(c.d[i], x[i]));
#pragma unroll
                    for (int i = 1; i < NC; ++i) acc = __dsub_rn(acc, __dmul_rn(c.n[i], y[i]));
                    y[0] = acc;
                    tile[lane][k] = to_i32_x86(acc);  // rspt_test.cpp:132: double -> int32, toward zero
                }
            }
            __syncwarp();
#pragma unroll
            for (uint32_t r = 0; r < 32; ++r)
                if (r < nf && i0 + lane < ns) w0[(size_t)r * s.N + (size_t)j * ns + i0 + lane] = tile[r][lane];
            __syncwarp();
        }
    }
}

// FIR over the int32 words ([frame][channel][sample], from k_raw_to_words): one CTA per 256 samples
// of one channel, the tile and its kernel_size - 1 predecessors staged in shared memory as doubles,
// the coefficients too; one thread per output sample.  Out of place (a tile's halo is its
// neighbour's data).
constexpr int kFirTile = 256;

__global__ void __launch_bounds__(kFirTile) k_fir_words(const int32_t* __restrict__ in, Shape s, uint32_t tiles,
                                                        const double* __restrict__ kernel, int K, int32_t* __restrict__ out)
{
    extern __shared__ __align__(16) double fir_sm[];  // [K] coefficients, then [kFirTile + K - 1] samples
    double* kc = fir_sm;
    double* xs = fir_sm + K;
    const uint32_t t = blockIdx.x % tiles, row = blockIdx.x / tiles;  // row = frame * ch + channel
    const int32_t* src = in + (size_t)row * s.ns;
    const int i0 = (int)(t * kFirTile);
    for (int q = (int)threadIdx.x; q < K; q += kFirTile) kc[q] = kernel[q];
    for (int q = (int)threadIdx.x; q < kFirTile + K - 1; q += kFirTile) {
        int src_i = i0 - (K - 1) + q;  // samples before the channel start = its first sample
        src_i = src_i < 0 ? 0 : (src_i >= s.ns ? s.ns - 1 : src_i);
        xs[q] = (double)src[src_i];
    }
    __syncthreads();
    const int i = i0 + (int)threadIdx.x;
    if (i >= s.ns) return;
    double acc = 0.0;
    for (int q = 0; q < K; ++q)
        acc = __dadd_rn(acc, __dmul_rn(xs[threadIdx.x + q], kc[q]));  // fir_filter.cpp:52-54, oldest first
    out[(size_t)row * s.ns + i] = to_i32_x86(acc);
}

}  // namespace rspt
