// Lossy packers: integer fast Walsh-Hadamard transform and DCT-II / DCT-III with the reference's
// uniform quantisation.  Replaces lib_fwht/fwht.c (fwht_transform :4-28, fwht_normalize :30-34),
// signal_packer_hadamard.cpp:57-104 and signal_packer_dct.cpp:60-153.
//
// hadamard is pure integer arithmetic mod 2^32 (butterfly order is irrelevant) and therefore
// bit-exact.  dct: the reference evaluates the O(n^2) sum with FLOAT products accumulated in
// double (dct.cpp:83,96).  Two paths are provided:
//   * fast (default, ns a power of two): FP64 FFT-based DCT (Makhoul reordering through one
//     n-point complex FFT in shared memory).  Its result is the exactly-rounded-ish value; it
//     differs from the reference only where a coefficient lies within ~1e-5 of an integer.
//   * direct (any ns; RSPT_DCT_DIRECT=1 forces it): the same float-product / double-accumulate
//     sum in the same order over the same float cosine table, built on the host with the
//     reference's expression -- bit-exact, O(n^2).
#pragma once

#include <math.h>
#include <stdlib.h>

#include <vector>

#include "packer.cuh"
#include "transforms.cuh"

namespace rspt {

constexpr uint32_t kFwhtMaxN = 32768;  // ns * 4 bytes of shared memory per channel
constexpr uint32_t kDctMaxN = 8192;    // ns * 16 bytes of shared memory per channel (fast path)

// floor-mean of a channel exactly as average_32 computes it (utils.cpp:30-40): the int64 sum is
// divided as UNSIGNED 64-bit by the length and narrowed to int32.
__device__ __forceinline__ int32_t reference_mean(long long sum, uint32_t len)
{
    return (int32_t)(long long)((unsigned long long)sum / (unsigned long long)len);
}

__device__ __forceinline__ void store_mean24(uint8_t* hdr, int32_t m)
{
    hdr[0] = (uint8_t)m; hdr[1] = (uint8_t)((uint32_t)m >> 8); hdr[2] = (uint8_t)((uint32_t)m >> 16);
}

__device__ __forceinline__ int32_t load_mean24(const uint8_t* hdr)
{
    const uint32_t v = (uint32_t)hdr[0] | ((uint32_t)hdr[1] << 8) | ((uint32_t)hdr[2] << 16);
    return (int32_t)(v << 8) >> 8;  // hadamard.cpp:99, dct.cpp:148
}

// in-place natural-order FWHT of a[0..n) in shared memory, wrap-around int32 (fwht.c:15-25)
__device__ __forceinline__ void fwht_smem(uint32_t* a, uint32_t n)
{
    for (uint32_t h = n >> 1; h > 0; h >>= 1) {
        for (uint32_t t = threadIdx.x; t < (n >> 1); t += blockDim.x) {
            const uint32_t i = ((t & ~(h - 1)) << 1) | (t & (h - 1));
            const uint32_t u = a[i], v = a[i + h];
            a[i] = u + v;
            a[i + h] = u - v;
        }
        __syncthreads();
    }
}

// one CTA per (frame, channel): mean removal, FWHT, q = trunc(X / n), three byte planes
__global__ void __launch_bounds__(256) k_fwht_fwd(const int32_t* __restrict__ words, const long long* __restrict__ sums,
                                                   Shape s, uint8_t* __restrict__ planes, uint8_t* __restrict__ headers)
{
    extern __shared__ __align__(16) uint32_t a[];
    const uint32_t f = blockIdx.x / s.ch, c = blockIdx.x % s.ch, n = (uint32_t)s.ns;
    const int32_t mean = reference_mean(sums[(size_t)f * s.ch + c], n);
    const int32_t* w = words + (size_t)f * s.N + (size_t)c * n;
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) a[i] = (uint32_t)w[i] - (uint32_t)mean;
    if (threadIdx.x == 0) store_mean24(headers + (size_t)f * s.hdr_bytes + 3 * c, mean);
    __syncthreads();
    fwht_smem(a, n);
    const int lg = 31 - __clz((int)n);
    uint8_t* out = planes + (size_t)f * s.nb_alloc * s.plane_stride + (size_t)c * n;
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
        const int32_t X = (int32_t)a[i];
        // (int)(X / (double)(n / 1.0)) -- truncation toward zero of an exact power-of-two quotient
        const int32_t q = (X + ((X >> 31) & (int32_t)(n - 1))) >> lg;
        for (uint32_t k = 0; k < s.nb_alloc; ++k) out[(size_t)k * s.plane_stride + i] = (uint8_t)((uint32_t)q >> (8 * k));
    }
}

// the float output of a hadamard sample word w (the full 32-bit sum): sign-extended from 8 * bps bits as
// k_words_sext does, then dequantized
template <class OutT>
__device__ __forceinline__ OutT fwht_out(uint32_t w, int sh, const ChanDq& d)
{
    return out_elem<OutT>((int32_t)(w << sh) >> sh, d);
}

// one CTA per (frame, channel): planes -> q (sign-extended from 24 bits) -> FWHT -> + mean24.  The body of
// k_fwht_inv (OutT = int32_t: the full words) and k_dq_fwht_inv (float / __nv_bfloat16: the samples, dequantized
// with dq).
template <class OutT>
__device__ __forceinline__ void fwht_inv(const uint8_t* __restrict__ planes, const uint8_t* __restrict__ headers,
                                         const uint8_t* __restrict__ dec_nb, Shape s, OutT* __restrict__ words, Dequant dq)
{
    extern __shared__ __align__(16) uint32_t a[];
    const uint32_t f = blockIdx.x / s.ch, c = blockIdx.x % s.ch, n = (uint32_t)s.ns;
    const uint32_t nb = dec_nb[f];
    const int sh = 32 - 8 * (int)nb;
    const uint8_t* in = planes + (size_t)f * s.nb_alloc * s.plane_stride + (size_t)c * n;
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
        uint32_t v = 0;
        for (uint32_t k = 0; k < nb; ++k) v |= (uint32_t)in[(size_t)k * s.plane_stride + i] << (8 * k);
        a[i] = (uint32_t)((int32_t)(v << sh) >> sh);
    }
    __syncthreads();
    fwht_smem(a, n);
    const int32_t mean = load_mean24(headers + (size_t)f * s.hdr_bytes + 3 * c);
    OutT* w = words + (size_t)f * s.N + (size_t)c * n;
    if constexpr (std::is_same_v<OutT, int32_t>) {
        for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) w[i] = (int32_t)(a[i] + (uint32_t)mean);
    } else {
        const ChanDq d = chan_dq(dq, c);
        const int osh = 32 - 8 * s.bps;
        for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) w[i] = fwht_out<OutT>(a[i] + (uint32_t)mean, osh, d);
    }
}

__global__ void __launch_bounds__(256) k_fwht_inv(const uint8_t* __restrict__ planes, const uint8_t* __restrict__ headers,
                                                   const uint8_t* __restrict__ dec_nb, Shape s, int32_t* __restrict__ words)
{
    fwht_inv(planes, headers, dec_nb, s, words, Dequant{});
}

template <class OutT>
__global__ void __launch_bounds__(256) k_dq_fwht_inv(const uint8_t* __restrict__ planes, const uint8_t* __restrict__ headers,
                                                      const uint8_t* __restrict__ dec_nb, Shape s, OutT* __restrict__ dst,
                                                      Dequant dq)
{
    fwht_inv(planes, headers, dec_nb, s, dst, dq);
}

// ---- n = 4096 / 8192 fast path: three radix-16 passes in registers ---------------------------
// n/16 threads x 16 elements.  Pass 1 takes the top four index bits (elements t + (n/16) j, read
// straight from global memory), pass 2 the next four, pass 3 bits 0..3 (elements 16 t + j, so a
// thread ends up with 16 consecutive coefficients and writes one 128-bit word per plane); for
// n = 8192 the thirteenth bit (bit 4) is a butterfly between neighbouring lanes (one shuffle per
// element).  Between passes the data sits in shared memory at i + (i >> 5) (one pad word per 32),
// which keeps the stride-16 accesses of pass 3 conflict-free.  Butterfly order is irrelevant mod
// 2^32, so the result is the reference's natural-order transform (fwht.c:15-25).
__device__ __forceinline__ uint32_t fwht_phys(uint32_t i) { return i + (i >> 5); }

__device__ __forceinline__ void radix16(uint32_t (&r)[16])
{
#pragma unroll
    for (int h = 1; h < 16; h <<= 1)
#pragma unroll
        for (int j = 0; j < 16; ++j)
            if ((j & h) == 0) {
                const uint32_t u = r[j], v = r[j + h];
                r[j] = u + v;
                r[j + h] = u - v;
            }
}

// butterfly on index bit 4 = bit 0 of the thread index (elements 16 t + j and 16 (t ^ 1) + j)
__device__ __forceinline__ void lane_pair_butterfly(uint32_t (&r)[16])
{
    const bool upper = threadIdx.x & 1u;
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        const uint32_t o = __shfl_xor_sync(0xFFFFFFFFu, r[j], 1);
        r[j] = upper ? o - r[j] : r[j] + o;
    }
}

template <int LG>
__global__ void __launch_bounds__((1 << LG) / 16) k_fwht_fast_fwd(const int32_t* __restrict__ words, const long long* __restrict__ sums,
                                                                   Shape s, uint8_t* __restrict__ planes, uint8_t* __restrict__ headers)
{
    constexpr uint32_t N = 1u << LG, T = N / 16, S2 = N / 256;  // threads; element stride of pass 2
    __shared__ uint32_t a[N + N / 32];
    const uint32_t f = blockIdx.x / s.ch, c = blockIdx.x % s.ch, t = threadIdx.x;
    const int32_t mean = reference_mean(sums[(size_t)f * s.ch + c], N);
    const uint32_t* w = reinterpret_cast<const uint32_t*>(words) + (size_t)f * s.N + (size_t)c * N;
    if (t == 0) store_mean24(headers + (size_t)f * s.hdr_bytes + 3 * c, mean);
    uint32_t r[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) r[j] = __ldg(w + t + T * j);
    radix16(r);
#pragma unroll
    for (int j = 0; j < 16; ++j) a[fwht_phys(t + T * j)] = r[j];
    __syncthreads();
    const uint32_t b2 = (t / S2) * (16 * S2) + (t % S2);
#pragma unroll
    for (int j = 0; j < 16; ++j) r[j] = a[fwht_phys(b2 + S2 * j)];
    radix16(r);
#pragma unroll
    for (int j = 0; j < 16; ++j) a[fwht_phys(b2 + S2 * j)] = r[j];
    __syncthreads();
#pragma unroll
    for (int j = 0; j < 16; ++j) r[j] = a[fwht_phys(16 * t + j)];
    radix16(r);
    if (LG == 13) lane_pair_butterfly(r);
    // the per-channel mean is removed before the transform (hadamard.cpp:60-65); by linearity mod
    // 2^32 that only changes the DC coefficient
    if (t == 0) r[0] -= N * (uint32_t)mean;
    uint32_t pl[4][4];
#pragma unroll
    for (int g = 0; g < 4; ++g) {
        uint32_t q[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int32_t X = (int32_t)r[4 * g + i];
            // (int)(X / (double)n): truncation toward zero of an exact power-of-two quotient (fwht.c:33)
            q[i] = (uint32_t)((X + ((X >> 31) & (int32_t)(N - 1))) >> LG);
        }
        const uint32_t t01 = prmt(q[0], q[1], 0x5140u), t23 = prmt(q[2], q[3], 0x5140u);
        const uint32_t u01 = prmt(q[0], q[1], 0x7362u), u23 = prmt(q[2], q[3], 0x7362u);
        pl[0][g] = prmt(t01, t23, 0x5410u);
        pl[1][g] = prmt(t01, t23, 0x7632u);
        pl[2][g] = prmt(u01, u23, 0x5410u);
        pl[3][g] = prmt(u01, u23, 0x7632u);
    }
    uint8_t* out = planes + (size_t)f * s.nb_alloc * s.plane_stride + (size_t)c * N + 16 * t;
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if ((uint32_t)k < s.nb_alloc)
            *reinterpret_cast<uint4*>(out + (size_t)k * s.plane_stride) = make_uint4(pl[k][0], pl[k][1], pl[k][2], pl[k][3]);
}

// the body of k_fwht_fast_inv and k_dq_fwht_fast_inv; OutT as for fwht_inv.  t = threadIdx.x, read by the kernel:
// there the compiler knows from __launch_bounds__ that t < N / 16 and keeps the index terms' disjoint bits as
// ORs and narrow masks, which a read inside this inlined body loses.
template <int LG, class OutT>
__device__ __forceinline__ void fwht_fast_inv(const uint8_t* __restrict__ planes, const uint8_t* __restrict__ headers,
                                              const uint8_t* __restrict__ dec_nb, Shape s, OutT* __restrict__ words, Dequant dq,
                                              uint32_t t)
{
    constexpr uint32_t N = 1u << LG, T = N / 16, S2 = N / 256;
    __shared__ uint32_t a[N + N / 32];
    const uint32_t f = blockIdx.x / s.ch, c = blockIdx.x % s.ch;
    const uint32_t nb = dec_nb[f];
    const uint8_t* in = planes + (size_t)f * s.nb_alloc * s.plane_stride + (size_t)c * N + 16 * t;
    uint4 pv[4];
#pragma unroll
    for (int k = 0; k < 4; ++k)
        pv[k] = (uint32_t)k < s.nb_alloc ? __ldg(reinterpret_cast<const uint4*>(in + (size_t)k * s.plane_stride)) : make_uint4(0, 0, 0, 0);
    uint32_t r[16];
    {
        uint32_t y[4];
        planes_to_words(pv[0].x, pv[1].x, pv[2].x, pv[3].x, nb, y);
        r[0] = y[0]; r[1] = y[1]; r[2] = y[2]; r[3] = y[3];
        planes_to_words(pv[0].y, pv[1].y, pv[2].y, pv[3].y, nb, y);
        r[4] = y[0]; r[5] = y[1]; r[6] = y[2]; r[7] = y[3];
        planes_to_words(pv[0].z, pv[1].z, pv[2].z, pv[3].z, nb, y);
        r[8] = y[0]; r[9] = y[1]; r[10] = y[2]; r[11] = y[3];
        planes_to_words(pv[0].w, pv[1].w, pv[2].w, pv[3].w, nb, y);
        r[12] = y[0]; r[13] = y[1]; r[14] = y[2]; r[15] = y[3];
    }
    radix16(r);
    if (LG == 13) lane_pair_butterfly(r);
#pragma unroll
    for (int j = 0; j < 16; ++j) a[fwht_phys(16 * t + j)] = r[j];
    __syncthreads();
    const uint32_t b2 = (t / S2) * (16 * S2) + (t % S2);
#pragma unroll
    for (int j = 0; j < 16; ++j) r[j] = a[fwht_phys(b2 + S2 * j)];
    radix16(r);
#pragma unroll
    for (int j = 0; j < 16; ++j) a[fwht_phys(b2 + S2 * j)] = r[j];
    __syncthreads();
#pragma unroll
    for (int j = 0; j < 16; ++j) r[j] = a[fwht_phys(t + T * j)];
    radix16(r);
    const uint32_t mean = (uint32_t)load_mean24(headers + (size_t)f * s.hdr_bytes + 3 * c);
    if constexpr (std::is_same_v<OutT, int32_t>) {
        uint32_t* w = reinterpret_cast<uint32_t*>(words) + (size_t)f * s.N + (size_t)c * N;
#pragma unroll
        for (int j = 0; j < 16; ++j) w[t + T * j] = r[j] + mean;
    } else {
        const ChanDq d = chan_dq(dq, c);
        const int osh = 32 - 8 * s.bps;
        OutT* w = words + (size_t)f * s.N + (size_t)c * N;
#pragma unroll
        for (int j = 0; j < 16; ++j) w[t + T * j] = fwht_out<OutT>(r[j] + mean, osh, d);
    }
}

template <int LG>
__global__ void __launch_bounds__((1 << LG) / 16) k_fwht_fast_inv(const uint8_t* __restrict__ planes, const uint8_t* __restrict__ headers,
                                                                   const uint8_t* __restrict__ dec_nb, Shape s, int32_t* __restrict__ words)
{
    fwht_fast_inv<LG>(planes, headers, dec_nb, s, words, Dequant{}, threadIdx.x);
}

template <int LG, class OutT>
__global__ void __launch_bounds__((1 << LG) / 16) k_dq_fwht_fast_inv(const uint8_t* __restrict__ planes, const uint8_t* __restrict__ headers,
                                                                      const uint8_t* __restrict__ dec_nb, Shape s, OutT* __restrict__ dst,
                                                                      Dequant dq)
{
    fwht_fast_inv<LG>(planes, headers, dec_nb, s, dst, dq, threadIdx.x);
}

// ---- fused fast path: interleaved samples <-> planes without the int32 word matrix ------------
// ch % 4 == 0: a CTA takes FOUR channels of one frame.  The 4 x BPS bytes of a sample row that belong
// to them are contiguous in the interleaved input, so thread t reads them for its 16 samples
// t + T j (one 128-bit load per sample for 4-byte samples; the other channel groups of the frame
// read the neighbouring bytes of the same lines at the same time and find them in L2), unpacks them
// with PRMT and runs the three radix-16 passes of k_fwht_fast_* on four shared-memory buffers.
// k_raw_to_words / k_words_to_raw and the word matrix (2 x 4 bytes of traffic per sample) drop out.
// The channel mean needs the 64-bit sum (average_32, utils.cpp:30-40): its low 32 bits are the DC
// coefficient X[0] of the transform itself, the rest follows from the sum of the samples' upper
// halves (one warp reduction per channel): sum = 65536 * S_hi + ((X[0] - 65536 * S_hi) mod 2^32).
template <int LG, int BPS>
__global__ void __launch_bounds__((1 << LG) / 16) k_fwht_raw_fwd(const uint8_t* __restrict__ src, Shape s,
                                                                  uint8_t* __restrict__ planes, uint8_t* __restrict__ headers)
{
    constexpr uint32_t N = 1u << LG, T = N / 16, S2 = N / 256, A = N + N / 32;
    extern __shared__ __align__(16) uint32_t a4[];  // [4][A]
    __shared__ int s_hi[4];
    const uint32_t G = (uint32_t)s.ch >> 2, f = blockIdx.x / G, g = blockIdx.x % G, t = threadIdx.x;
    const uint32_t roww = ((uint32_t)s.ch * BPS) >> 2;  // words per sample row
    const uint32_t* base = reinterpret_cast<const uint32_t*>(src + (size_t)f * s.frame_bytes) + g * BPS;
    if (t < 4) s_hi[t] = 0;
    uint32_t v[4][16];
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        const uint32_t* p = base + (size_t)(t + T * j) * roww;
        uint32_t w[4], x[4];
        if (BPS == 4) {
            const uint4 q = __ldg(reinterpret_cast<const uint4*>(p));
            w[0] = q.x; w[1] = q.y; w[2] = q.z; w[3] = q.w;
        } else {
#pragma unroll
            for (int i = 0; i < BPS; ++i) w[i] = __ldg(p + i);
        }
        unpack4<BPS>(w, x);
#pragma unroll
        for (int cc = 0; cc < 4; ++cc) v[cc][j] = x[cc];
    }
    __syncthreads();  // s_hi cleared
#pragma unroll
    for (int cc = 0; cc < 4; ++cc) {
        int hi = 0;
#pragma unroll
        for (int j = 0; j < 16; ++j) hi += (int32_t)v[cc][j] >> 16;
        hi = __reduce_add_sync(0xFFFFFFFFu, hi);
        if ((t & 31u) == 0) atomicAdd(&s_hi[cc], hi);
        radix16(v[cc]);
#pragma unroll
        for (int j = 0; j < 16; ++j) a4[cc * A + fwht_phys(t + T * j)] = v[cc][j];
    }
    __syncthreads();
    const uint32_t b2 = (t / S2) * (16 * S2) + (t % S2);
#pragma unroll
    for (int cc = 0; cc < 4; ++cc) {
        uint32_t r[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) r[j] = a4[cc * A + fwht_phys(b2 + S2 * j)];
        radix16(r);
#pragma unroll
        for (int j = 0; j < 16; ++j) a4[cc * A + fwht_phys(b2 + S2 * j)] = r[j];
    }
    __syncthreads();
#pragma unroll
    for (int cc = 0; cc < 4; ++cc) {
        const uint32_t c = 4 * g + cc;
        uint32_t r[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) r[j] = a4[cc * A + fwht_phys(16 * t + j)];
        radix16(r);
        if (LG == 13) lane_pair_butterfly(r);
        if (t == 0) {
            const int shi = s_hi[cc];
            const uint32_t lo = r[0] - ((uint32_t)shi << 16);  // sum of the samples' lower halves (< 2^29)
            const int32_t mean = reference_mean((long long)shi * 65536ll + (long long)lo, N);
            store_mean24(headers + (size_t)f * s.hdr_bytes + 3 * c, mean);
            // the mean is removed before the transform (hadamard.cpp:60-65): only the DC coefficient changes
            r[0] -= N * (uint32_t)mean;
        }
        uint32_t pl[4][4];
#pragma unroll
        for (int gq = 0; gq < 4; ++gq) {
            uint32_t q[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int32_t X = (int32_t)r[4 * gq + i];
                q[i] = (uint32_t)((X + ((X >> 31) & (int32_t)(N - 1))) >> LG);  // trunc(X / n), fwht.c:33
            }
            const uint32_t t01 = prmt(q[0], q[1], 0x5140u), t23 = prmt(q[2], q[3], 0x5140u);
            const uint32_t u01 = prmt(q[0], q[1], 0x7362u), u23 = prmt(q[2], q[3], 0x7362u);
            pl[0][gq] = prmt(t01, t23, 0x5410u);
            pl[1][gq] = prmt(t01, t23, 0x7632u);
            pl[2][gq] = prmt(u01, u23, 0x5410u);
            pl[3][gq] = prmt(u01, u23, 0x7632u);
        }
        uint8_t* out = planes + (size_t)f * s.nb_alloc * s.plane_stride + (size_t)c * N + 16 * t;
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if ((uint32_t)k < s.nb_alloc)
                *reinterpret_cast<uint4*>(out + (size_t)k * s.plane_stride) = make_uint4(pl[k][0], pl[k][1], pl[k][2], pl[k][3]);
    }
}

template <int LG, int BPS>
__global__ void __launch_bounds__((1 << LG) / 16) k_fwht_raw_inv(const uint8_t* __restrict__ planes, const uint8_t* __restrict__ headers,
                                                                  const uint8_t* __restrict__ dec_nb, Shape s, uint8_t* __restrict__ dst)
{
    constexpr uint32_t N = 1u << LG, T = N / 16, S2 = N / 256, A = N + N / 32;
    extern __shared__ __align__(16) uint32_t a4[];  // [4][A]
    const uint32_t G = (uint32_t)s.ch >> 2, f = blockIdx.x / G, g = blockIdx.x % G, t = threadIdx.x;
    const uint32_t nb = dec_nb[f];
    uint4 pv[4][4];
#pragma unroll
    for (int cc = 0; cc < 4; ++cc) {
        const uint8_t* in = planes + (size_t)f * s.nb_alloc * s.plane_stride + (size_t)(4 * g + cc) * N + 16 * t;
#pragma unroll
        for (int k = 0; k < 4; ++k)
            pv[cc][k] = (uint32_t)k < s.nb_alloc ? __ldg(reinterpret_cast<const uint4*>(in + (size_t)k * s.plane_stride)) : make_uint4(0, 0, 0, 0);
    }
#pragma unroll
    for (int cc = 0; cc < 4; ++cc) {
        uint32_t r[16], y[4];
        planes_to_words(pv[cc][0].x, pv[cc][1].x, pv[cc][2].x, pv[cc][3].x, nb, y);
        r[0] = y[0]; r[1] = y[1]; r[2] = y[2]; r[3] = y[3];
        planes_to_words(pv[cc][0].y, pv[cc][1].y, pv[cc][2].y, pv[cc][3].y, nb, y);
        r[4] = y[0]; r[5] = y[1]; r[6] = y[2]; r[7] = y[3];
        planes_to_words(pv[cc][0].z, pv[cc][1].z, pv[cc][2].z, pv[cc][3].z, nb, y);
        r[8] = y[0]; r[9] = y[1]; r[10] = y[2]; r[11] = y[3];
        planes_to_words(pv[cc][0].w, pv[cc][1].w, pv[cc][2].w, pv[cc][3].w, nb, y);
        r[12] = y[0]; r[13] = y[1]; r[14] = y[2]; r[15] = y[3];
        radix16(r);
        if (LG == 13) lane_pair_butterfly(r);
#pragma unroll
        for (int j = 0; j < 16; ++j) a4[cc * A + fwht_phys(16 * t + j)] = r[j];
    }
    __syncthreads();
    const uint32_t b2 = (t / S2) * (16 * S2) + (t % S2);
#pragma unroll
    for (int cc = 0; cc < 4; ++cc) {
        uint32_t r[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) r[j] = a4[cc * A + fwht_phys(b2 + S2 * j)];
        radix16(r);
#pragma unroll
        for (int j = 0; j < 16; ++j) a4[cc * A + fwht_phys(b2 + S2 * j)] = r[j];
    }
    __syncthreads();
    uint32_t x[4][16];
#pragma unroll
    for (int cc = 0; cc < 4; ++cc) {
#pragma unroll
        for (int j = 0; j < 16; ++j) x[cc][j] = a4[cc * A + fwht_phys(t + T * j)];
        radix16(x[cc]);
        const uint32_t mean = (uint32_t)load_mean24(headers + (size_t)f * s.hdr_bytes + 3 * (4 * g + cc));
#pragma unroll
        for (int j = 0; j < 16; ++j) x[cc][j] += mean;
    }
    // the 4 channels of a sample row, low BPS bytes each (convert_i32_to_native, utils.cpp:51-121)
    const uint32_t roww = ((uint32_t)s.ch * BPS) >> 2;
    uint32_t* base = reinterpret_cast<uint32_t*>(dst + (size_t)f * s.frame_bytes) + g * BPS;
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        uint32_t* p = base + (size_t)(t + T * j) * roww;
        const uint32_t a = x[0][j], b = x[1][j], c2 = x[2][j], d = x[3][j];
        if (BPS == 4) {
            *reinterpret_cast<uint4*>(p) = make_uint4(a, b, c2, d);
        } else if (BPS == 3) {
            p[0] = prmt(a, b, 0x4210u);
            p[1] = prmt(b, c2, 0x5421u);
            p[2] = prmt(c2, d, 0x6542u);
        } else if (BPS == 2) {
            p[0] = prmt(a, b, 0x5410u);
            p[1] = prmt(c2, d, 0x5410u);
        } else {
            p[0] = prmt(prmt(a, b, 0x0040u), prmt(c2, d, 0x0040u), 0x5410u);
        }
    }
}

// ---- FP64 complex FFT in shared memory ------------------------------------------------------
// x[0..n) complex, n = 2^lg.  Input must already be in bit-reversed order.  tw[j] = e^{-2 pi i j/n}
// for j < n/2; INVERSE conjugates it.  Radix-2 decimation in time.
template <bool INVERSE>
__device__ __forceinline__ void fft_smem(double2* x, uint32_t n, const double2* __restrict__ tw)
{
    uint32_t stage_shift = 31 - __clz((int)n);  // twiddle stride = n / (2*half) = n >> s
    for (uint32_t half = 1; half < n; half <<= 1) {
        --stage_shift;
        for (uint32_t t = threadIdx.x; t < (n >> 1); t += blockDim.x) {
            const uint32_t jj = t & (half - 1);
            const uint32_t i = ((t & ~(half - 1)) << 1) | jj;
            double2 w = __ldg(tw + ((size_t)jj << stage_shift));
            if (INVERSE) w.y = -w.y;
            const double2 u = x[i], v = x[i + half];
            const double2 m = make_double2(v.x * w.x - v.y * w.y, v.x * w.y + v.y * w.x);
            x[i] = make_double2(u.x + m.x, u.y + m.y);
            x[i + half] = make_double2(u.x - m.x, u.y - m.y);
        }
        __syncthreads();
    }
}

// forward DCT of one channel, fast path.  post[k] = e^{-i pi k / (2n)}.
__global__ void __launch_bounds__(256) k_dct_fwd_fast(int32_t* __restrict__ words, const long long* __restrict__ sums, Shape s,
                                                       const double2* __restrict__ tw, const double2* __restrict__ post,
                                                       uint8_t* __restrict__ headers)
{
    extern __shared__ __align__(16) double2 xs[];
    const uint32_t f = blockIdx.x / s.ch, c = blockIdx.x % s.ch, n = (uint32_t)s.ns;
    const int lg = 31 - __clz((int)n);
    const int32_t mean = reference_mean(sums[(size_t)f * s.ch + c], n);
    int32_t* w = words + (size_t)f * s.N + (size_t)c * n;
    if (threadIdx.x == 0) store_mean24(headers + (size_t)f * s.hdr_bytes + 3 * c, mean);
    // v[m] = x[2m], v[n-1-m] = x[2m+1]; stored at the bit-reversed index for the DIT FFT
    for (uint32_t j = threadIdx.x; j < n; j += blockDim.x) {
        const int32_t xv = (int32_t)((uint32_t)w[j] - (uint32_t)mean);
        const uint32_t m = (j & 1u) ? n - 1 - (j >> 1) : (j >> 1);
        xs[__brev(m) >> (32 - lg)] = make_double2((double)xv, 0.0);
    }
    __syncthreads();
    fft_smem<false>(xs, n, tw);
    const double ratio1 = sqrt(2.0 / (double)(int)n);
    for (uint32_t k = threadIdx.x; k < n; k += blockDim.x) {
        const double2 V = xs[k], p = __ldg(post + k);
        double sum = V.x * p.x - V.y * p.y;
        const float cs = k ? 1.0f : (float)(1 / sqrt(2.0));
        sum *= (double)cs * ratio1 / 128.0;  // dct.cpp:84 (quality = 128)
        w[k] = (int32_t)sum;                 // truncation toward zero, dct.cpp:85
    }
}

// ---- half-size FFT path (n a power of two >= 16) ---------------------------------------------
// The Makhoul sequence v is real, so its n-point spectrum comes from ONE complex FFT of half the
// length over z[p] = v[2p] + i v[2p+1] (M = n/2 points) and a butterfly of Z[k] with Z[M-k]; the
// inverse runs the same steps backwards.  The FFT itself is the radix-2 decimation-in-time
// network on bit-reversed input, but three stages at a time: a thread keeps 8 points in
// registers, so the data passes through shared memory ceil(lg M / 3) times instead of lg M
// times.  Shared memory is padded by one point per 8 and one more per 64 (16-byte points: 8 cover
// all 32 banks), which keeps the stride-8 accesses of the first pass and the stride-M/32 stores
// of the bit-reversed load conflict-free.
__device__ __forceinline__ uint32_t fpad(uint32_t i) { return i + (i >> 3) + (i >> 6); }

// R fused radix-2 DIT stages starting at butterfly half-width h.  tw = e^{-2 pi i j / n}, j < n/2.
template <int R, bool INVERSE>
__device__ __forceinline__ void fft_pass(double2* x, uint32_t M, uint32_t h, uint32_t lgn, const double2* __restrict__ tw)
{
    constexpr int Q = 1 << R;
    const uint32_t lgh = 31 - __clz((int)h);
    for (uint32_t t = threadIdx.x; t < (M >> R); t += blockDim.x) {
        const uint32_t jj0 = t & (h - 1);
        const uint32_t base = ((t & ~(h - 1)) << R) | jj0;
        double2 a[Q];
#pragma unroll
        for (int q = 0; q < Q; ++q) a[q] = x[fpad(base + (uint32_t)q * h)];
#pragma unroll
        for (int st = 0; st < R; ++st) {
            // stage half-width h << st: the twiddle of position pos = jj0 + r h is
            // e^{-2 pi i pos / (2 (h << st))} = w0 * e^{-i pi r / 2^st}: one table look-up per stage,
            // the other positions by exact rotations (multiples of pi/4)
            const uint32_t sh = lgn - 1u - lgh - (uint32_t)st;
            const double2 w0 = __ldg(tw + ((size_t)jj0 << sh));
#pragma unroll
            for (int q = 0; q < Q; ++q) {
                if (q & (1 << st)) continue;
                const int r8 = (q & ((1 << st) - 1)) * (4 >> st);  // rotation in units of pi/4 (st <= 2)
                constexpr double kS = 0.70710678118654752440;
                double2 w = w0;
                if (r8 == 1) w = make_double2((w0.x + w0.y) * kS, (w0.y - w0.x) * kS);
                if (r8 == 2) w = make_double2(w0.y, -w0.x);
                if (r8 == 3) w = make_double2((w0.y - w0.x) * kS, -(w0.x + w0.y) * kS);
                if (INVERSE) w.y = -w.y;
                const double2 u = a[q], v = a[q + (1 << st)];
                const double2 m = make_double2(v.x * w.x - v.y * w.y, v.x * w.y + v.y * w.x);
                a[q] = make_double2(u.x + m.x, u.y + m.y);
                a[q + (1 << st)] = make_double2(u.x - m.x, u.y - m.y);
            }
        }
#pragma unroll
        for (int q = 0; q < Q; ++q) x[fpad(base + (uint32_t)q * h)] = a[q];
    }
}

// First three stages (half-widths 1, 2, 4) with the input taken straight from `load(p)` (natural
// index p) instead of a bit-reversed copy in shared memory: thread t owns the butterfly whose 8
// inputs are p = t + q M/8, so consecutive lanes load consecutive p; all twiddles of these stages
// are multiples of pi/4.  Results land at the bit-reversed-order positions 8 brev(t) + q.
template <bool INVERSE, class Load>
__device__ __forceinline__ void fft_first_pass(double2* x, uint32_t lgm, Load load)
{
    const uint32_t G = 1u << (lgm - 3);
    constexpr double kS = 0.70710678118654752440;
    for (uint32_t t = threadIdx.x; t < G; t += blockDim.x) {
        double2 a[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) a[q] = load(t + (uint32_t)(((q & 1) << 2) | (q & 2) | (q >> 2)) * G);
#pragma unroll
        for (int st = 0; st < 3; ++st) {
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                if (q & (1 << st)) continue;
                const int r8 = (q & ((1 << st) - 1)) * (4 >> st);  // twiddle e^{-+ i pi r8 / 4}
                const double2 u = a[q], v = a[q + (1 << st)];
                double2 m = v;
                if (!INVERSE) {
                    if (r8 == 1) m = make_double2((v.x + v.y) * kS, (v.y - v.x) * kS);
                    if (r8 == 2) m = make_double2(v.y, -v.x);
                    if (r8 == 3) m = make_double2((v.y - v.x) * kS, -(v.x + v.y) * kS);
                } else {
                    if (r8 == 1) m = make_double2((v.x - v.y) * kS, (v.x + v.y) * kS);
                    if (r8 == 2) m = make_double2(-v.y, v.x);
                    if (r8 == 3) m = make_double2(-(v.x + v.y) * kS, (v.x - v.y) * kS);
                }
                a[q] = make_double2(u.x + m.x, u.y + m.y);
                a[q + (1 << st)] = make_double2(u.x - m.x, u.y - m.y);
            }
        }
        const uint32_t base = lgm > 3 ? (__brev(t) >> (32 - (lgm - 3))) << 3 : 0u;
#pragma unroll
        for (int q = 0; q < 8; ++q) x[fpad(base + (uint32_t)q)] = a[q];
    }
    __syncthreads();
}

// M-point FFT (M = 2^lgm >= 8): input through `load(p)`, natural-order output in x at padded indices
template <bool INVERSE, class Load>
__device__ __forceinline__ void fft_fused(double2* x, uint32_t lgm, uint32_t lgn, const double2* __restrict__ tw, Load load)
{
    const uint32_t M = 1u << lgm;
    fft_first_pass<INVERSE>(x, lgm, load);
    uint32_t h = 8, left = lgm - 3;
    while (left >= 3) {
        fft_pass<3, INVERSE>(x, M, h, lgn, tw);
        __syncthreads();
        h <<= 3;
        left -= 3;
    }
    if (left == 2) {
        fft_pass<2, INVERSE>(x, M, h, lgn, tw);
        __syncthreads();
    } else if (left == 1) {
        fft_pass<1, INVERSE>(x, M, h, lgn, tw);
        __syncthreads();
    }
}

// index of v[m] in the channel's sample row: v[m] = x[2m] (m < n/2), v[n-1-m] = x[2m+1]
__device__ __forceinline__ uint32_t makhoul_src(uint32_t m, uint32_t n) { return m < (n >> 1) ? 2u * m : 2u * (n - 1u - m) + 1u; }

// forward DCT of one channel.  post[k] = e^{-i pi k / (2n)}.
__global__ void __launch_bounds__(256, 4) k_dct_fwd_half(int32_t* __restrict__ words, const long long* __restrict__ sums, Shape s,
                                                       const double2* __restrict__ tw, const double2* __restrict__ post,
                                                       uint8_t* __restrict__ headers)
{
    extern __shared__ __align__(16) double2 xs[];
    const uint32_t f = blockIdx.x / s.ch, c = blockIdx.x % s.ch, n = (uint32_t)s.ns, M = n >> 1;
    const uint32_t lgn = 31 - __clz((int)n), lgm = lgn - 1;
    const int32_t mean = reference_mean(sums[(size_t)f * s.ch + c], n);
    int32_t* w = words + (size_t)f * s.N + (size_t)c * n;
    if (threadIdx.x == 0) store_mean24(headers + (size_t)f * s.hdr_bytes + 3 * c, mean);
    fft_fused<false>(xs, lgm, lgn, tw, [&](uint32_t p) {
        const int32_t re = (int32_t)((uint32_t)w[makhoul_src(2u * p, n)] - (uint32_t)mean);
        const int32_t im = (int32_t)((uint32_t)w[makhoul_src(2u * p + 1u, n)] - (uint32_t)mean);
        return make_double2((double)re, (double)im);
    });
    // V[k] = E[k] + e^{-2 pi i k/n} O[k], E = (Z[k] + conj Z[M-k]) / 2, O = (Z[k] - conj Z[M-k]) / 2i;
    // V[n-k] = conj V[k];  X[k] = Re(post[k] V[k])
    const double ratio1 = sqrt(2.0 / (double)(int)n) / 128.0;  // dct.cpp:84 (quality = 128)
    for (uint32_t k = threadIdx.x; k <= M; k += blockDim.x) {
        const double2 Zk = xs[fpad(k & (M - 1))], Zm = xs[fpad((M - k) & (M - 1))];
        const double ex = 0.5 * (Zk.x + Zm.x), ey = 0.5 * (Zk.y - Zm.y);
        const double ox = 0.5 * (Zk.y + Zm.y), oy = -0.5 * (Zk.x - Zm.x);
        const double2 t = k < M ? __ldg(tw + k) : make_double2(-1.0, 0.0);
        const double vx = ex + (t.x * ox - t.y * oy), vy = ey + (t.x * oy + t.y * ox);
        const double2 pk = __ldg(post + (k < n ? k : 0));
        double sum = vx * pk.x - vy * pk.y;
        const float cs = k ? 1.0f : (float)(1 / sqrt(2.0));
        sum *= (double)cs * ratio1;
        w[k] = (int32_t)sum;  // truncation toward zero, dct.cpp:85
        if (k > 0 && k < M) {
            const double2 pn = __ldg(post + (n - k));
            w[n - k] = (int32_t)((vx * pn.x + vy * pn.y) * ratio1);
        }
    }
}

// inverse DCT of one channel: U[0] = T[0], U[k] = conj(post[k]) (T[k] - i T[n-k]) / 2 (Hermitian),
// Zin[k] = (U[k] + conj U[M-k]) + i (U[k] - conj U[M-k]) e^{+2 pi i k/n}, z = M-point inverse FFT,
// v[2p] = Re z[p], v[2p+1] = Im z[p]; T[k] = Cs[k] * coef[k].
__global__ void __launch_bounds__(256, 4) k_dct_inv_half(int32_t* __restrict__ words, const uint8_t* __restrict__ headers, Shape s,
                                                       const double2* __restrict__ tw, const double2* __restrict__ post)
{
    extern __shared__ __align__(16) double2 xs[];
    const uint32_t f = blockIdx.x / s.ch, c = blockIdx.x % s.ch, n = (uint32_t)s.ns, M = n >> 1;
    const uint32_t lgn = 31 - __clz((int)n), lgm = lgn - 1;
    int32_t* w = words + (size_t)f * s.N + (size_t)c * n;
    const double cs0 = (double)(float)(1 / sqrt(2.0));
    auto U = [&](uint32_t k) {
        if (k == 0) return make_double2(cs0 * (double)w[0], 0.0);
        const double a = (double)w[k], b = (double)w[n - k];
        const double2 p = __ldg(post + k);  // conj(p) * (a - i b) / 2
        return make_double2(0.5 * (p.x * a - p.y * b), -0.5 * (p.x * b + p.y * a));
    };
    fft_fused<true>(xs, lgm, lgn, tw, [&](uint32_t k) {
        const double2 Uk = U(k), Um = U(M - k);
        const double ax = Uk.x + Um.x, ay = Uk.y - Um.y;   // U[k] + conj U[M-k]
        const double dx = Uk.x - Um.x, dy = Uk.y + Um.y;   // U[k] - conj U[M-k]
        const double2 t = __ldg(tw + k);                    // times conj(t)
        const double bx = dx * t.x + dy * t.y, by = dy * t.x - dx * t.y;
        return make_double2(ax - by, ay + bx);
    });
    const int32_t mean = load_mean24(headers + (size_t)f * s.hdr_bytes + 3 * c);
    const double scale = sqrt(2.0 / (double)(int)n) * 128.0;  // dct.cpp:97
    for (uint32_t p = threadIdx.x; p < M; p += blockDim.x) {
        const double2 z = xs[fpad(p)];
        w[makhoul_src(2u * p, n)] = (int32_t)((uint32_t)to_i32_x86(z.x * scale) + (uint32_t)mean);
        w[makhoul_src(2u * p + 1u, n)] = (int32_t)((uint32_t)to_i32_x86(z.y * scale) + (uint32_t)mean);
    }
}

// forward DCT, direct path: dct.cpp:76-87 verbatim arithmetic.  cosT[x][i] is the float table.
__global__ void __launch_bounds__(256) k_dct_fwd_direct(int32_t* __restrict__ words, const long long* __restrict__ sums, Shape s,
                                                         const float* __restrict__ cosT, uint8_t* __restrict__ headers)
{
    extern __shared__ __align__(16) float xf[];
    const uint32_t f = blockIdx.x / s.ch, c = blockIdx.x % s.ch, n = (uint32_t)s.ns;
    const int32_t mean = reference_mean(sums[(size_t)f * s.ch + c], n);
    int32_t* w = words + (size_t)f * s.N + (size_t)c * n;
    if (threadIdx.x == 0) store_mean24(headers + (size_t)f * s.hdr_bytes + 3 * c, mean);
    for (uint32_t j = threadIdx.x; j < n; j += blockDim.x) xf[j] = (float)(int32_t)((uint32_t)w[j] - (uint32_t)mean);
    __syncthreads();
    const double ratio1 = sqrt(2.0 / (double)(int)n);
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
        double sum = 0;
        for (uint32_t x = 0; x < n; ++x) sum += (double)__fmul_rn(xf[x], __ldg(cosT + (size_t)x * n + i));
        const float cs = i ? 1.0f : (float)(1 / sqrt(2.0));
        sum *= (double)cs * ratio1 / 128.0;
        w[i] = (int32_t)sum;
    }
}

// inverse DCT, fast path: U[0] = T[0], U[k] = conj(post[k]) (T[k] - i T[n-k]) / 2, v = n-point
// inverse FFT, x[2m] = v[m], x[2m+1] = v[n-1-m]; T[k] = Cs[k] * coef[k].
__global__ void __launch_bounds__(256) k_dct_inv_fast(int32_t* __restrict__ words, const uint8_t* __restrict__ headers, Shape s,
                                                       const double2* __restrict__ tw, const double2* __restrict__ post)
{
    extern __shared__ __align__(16) double2 xs[];
    const uint32_t f = blockIdx.x / s.ch, c = blockIdx.x % s.ch, n = (uint32_t)s.ns;
    const int lg = 31 - __clz((int)n);
    int32_t* w = words + (size_t)f * s.N + (size_t)c * n;
    const double cs0 = (double)(float)(1 / sqrt(2.0));
    for (uint32_t k = threadIdx.x; k < n; k += blockDim.x) {
        double2 U;
        if (k == 0) {
            U = make_double2(cs0 * (double)w[0], 0.0);
        } else {
            const double a = (double)w[k], b = (double)w[n - k];
            const double2 p = __ldg(post + k);  // conj(p) * (a - i b) / 2
            U = make_double2(0.5 * (p.x * a - p.y * b), -0.5 * (p.x * b + p.y * a));
        }
        xs[__brev(k) >> (32 - lg)] = U;
    }
    __syncthreads();
    fft_smem<true>(xs, n, tw);
    const int32_t mean = load_mean24(headers + (size_t)f * s.hdr_bytes + 3 * c);
    const double scale = sqrt(2.0 / (double)(int)n) * 128.0;  // dct.cpp:97
    for (uint32_t m = threadIdx.x; m < n; m += blockDim.x) {
        const uint32_t j = m < (n >> 1) ? 2 * m : 2 * (n - 1 - m) + 1;
        const double sum = xs[m].x * scale;
        w[j] = (int32_t)((uint32_t)to_i32_x86(sum) + (uint32_t)mean);
    }
}

// inverse DCT, direct path: dct.cpp:89-100 verbatim arithmetic (cosT[i][x])
__global__ void __launch_bounds__(256) k_dct_inv_direct(int32_t* __restrict__ words, const uint8_t* __restrict__ headers, Shape s,
                                                         const float* __restrict__ cosT)
{
    extern __shared__ __align__(16) float tf[];
    const uint32_t f = blockIdx.x / s.ch, c = blockIdx.x % s.ch, n = (uint32_t)s.ns;
    int32_t* w = words + (size_t)f * s.N + (size_t)c * n;
    const float cs0 = (float)(1 / sqrt(2.0));
    for (uint32_t k = threadIdx.x; k < n; k += blockDim.x) tf[k] = __fmul_rn(k ? 1.0f : cs0, (float)w[k]);
    __syncthreads();
    const int32_t mean = load_mean24(headers + (size_t)f * s.hdr_bytes + 3 * c);
    const double scale = sqrt(2.0 / (double)(int)n) * 128.0;
    // each thread owns output samples i; the table row i is contiguous in x
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
        double sum = 0;
        const float* rowp = cosT + (size_t)i * n;
        for (uint32_t x = 0; x < n; ++x) sum += (double)__fmul_rn(tf[x], __ldg(rowp + x));
        sum *= scale;
        w[i] = (int32_t)((uint32_t)to_i32_x86(sum) + (uint32_t)mean);  // out of int32 range: 0x80000000 + mean
    }
}

// ---- dct tables (host) ----------------------------------------------------------------------------

// the path a handle starts on: non-power-of-two lengths need the direct path, RSPT_DCT_DIRECT=1 requests it
inline bool dct_choose_direct(uint32_t n)
{
    const char* e = getenv("RSPT_DCT_DIRECT");
    return (n & (n - 1)) != 0 || (e && e[0] == '1');
}

// FFT path (power-of-two n): n/2 twiddles in a buffer of n/2 + 1, and n post-rotations, uploaded on p->stream
inline cudaError_t dct_build_fft_tables(rspt_gpu_packer* p)
{
    const uint32_t n = (uint32_t)p->s.ns;
    std::vector<double2> tw(n / 2), post(n);
    for (uint32_t j = 0; j < n / 2; ++j) {
        const long double a = -2.0L * 3.14159265358979323846264338327950288L * j / n;
        tw[j] = make_double2((double)cosl(a), (double)sinl(a));
    }
    for (uint32_t k = 0; k < n; ++k) {
        const long double a = -3.14159265358979323846264338327950288L * k / (2.0L * n);
        post[k] = make_double2((double)cosl(a), (double)sinl(a));
    }
    cudaError_t e = dalloc(p->d_twiddle, n / 2 + 1, 0);
    if (e == cudaSuccess) e = dalloc(p->d_post, n, 0);
    if (e == cudaSuccess) e = cudaMemcpyAsync(p->d_twiddle, tw.data(), sizeof(double2) * (n / 2), cudaMemcpyHostToDevice, p->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(p->d_post, post.data(), sizeof(double2) * n, cudaMemcpyHostToDevice, p->stream);
    return e;
}

// direct path: the n x n cosine table, uploaded on p->stream; p->d_cos is set only once the upload is enqueued
inline cudaError_t dct_build_cos_table(rspt_gpu_packer* p)
{
    const uint32_t n = (uint32_t)p->s.ns;
    // COSINES[i][j] = (float)cos(((i << 1) * j + j) * PI / (2n))  (dct.cpp:60-68); the same
    // symmetric-in-role table serves the forward ([x][i]) and inverse ([i][x]) sums
    std::vector<float> t((size_t)n * n);
    const double pi_n_2 = 3.14159265358979323846 / (n * 2.0);
    for (uint32_t i = 0; i < n; ++i)
        for (uint32_t j = 0; j < n; ++j) t[(size_t)i * n + j] = (float)cos((double)(int)(((int)i << 1) * (int)j + (int)j) * pi_n_2);
    DeviceBuf<float> c;
    cudaError_t e = dalloc(c, t.size(), 0);
    if (e == cudaSuccess) e = cudaMemcpyAsync(c, t.data(), sizeof(float) * t.size(), cudaMemcpyHostToDevice, p->stream);
    if (e == cudaSuccess) p->d_cos = std::move(c);
    return e;
}

}  // namespace rspt
