// Sample-domain kernels: de-interleave / sign-extend, the delta - offset - xor chain, byte-plane
// split and their inverses.  Replaces lib_signalpacker/utils.cpp (convert_native_to_i32 :123-191,
// convert_i32_to_native :51-121, delta_encode :193, offset_32 :215, xor_encode_32 :221,
// xor_decode_32 :232, delta_decode :204) and the plane split / reassembly of
// signal_packer_base.cpp:40-68 and :122-138.
#pragma once

#include "common.cuh"
#include "hzr_encode.cuh"

namespace rspt {

// cooperative copy of the global byte range [g, g + len) into shared memory at sm + (g & 15):
// 16-byte vector loads for the aligned interior, byte loads for the ragged ends
__device__ __forceinline__ uint32_t tile_load(uint8_t* sm, const uint8_t* __restrict__ g, uint32_t len)
{
    const uint32_t phase = (uint32_t)((uintptr_t)g & 15u);
    const uint32_t head = phase ? min(len, 16u - phase) : 0u;
    for (uint32_t i = threadIdx.x; i < head; i += blockDim.x) sm[phase + i] = g[i];
    const uint32_t nvec = (len - head) >> 4;
    const uint4* gv = reinterpret_cast<const uint4*>(g + head);
    uint4* sv = reinterpret_cast<uint4*>(sm + phase + head);
    for (uint32_t i = threadIdx.x; i < nvec; i += blockDim.x) sv[i] = __ldg(gv + i);
    const uint32_t done = head + (nvec << 4);
    for (uint32_t i = done + threadIdx.x; i < len; i += blockDim.x) sm[phase + i] = g[i];
    return phase;
}

template <int BPS>
__device__ __forceinline__ int32_t load_sample(const uint8_t* p)
{
    uint32_t v = p[0];
    if (BPS > 1) v |= (uint32_t)p[1] << 8;
    if (BPS > 2) v |= (uint32_t)p[2] << 16;
    if (BPS > 3) v |= (uint32_t)p[3] << 24;
    return (int32_t)(v << (32 - 8 * BPS)) >> (32 - 8 * BPS);  // sign extension (utils.cpp:141,158,174,189)
}

// x at flat (channel-major) index i of a frame, 0 for i < 0: the predecessor convention of
// delta_encode / xor_encode_32, whose chains run over the flat [ch*ns] array and therefore
// cross channel rows (signal_packer_xdelta_hzr.cpp:55-57)
template <int BPS>
__device__ __forceinline__ int32_t frame_sample_flat(const uint8_t* __restrict__ frame, const Shape& s, int64_t i)
{
    if (i < 0) return 0;
    const uint32_t c = (uint32_t)(i / s.ns), smp = (uint32_t)(i % s.ns);
    return load_sample<BPS>(frame + ((size_t)smp * s.ch + c) * BPS);
}

// planes required to represent y losslessly when only 8*bps bits matter: the smallest nb such
// that bits [8nb-1 .. 8bps-1] of y agree (equivalent to the reference's decode-and-memcmp test,
// signal_packer_xdelta_hzr.cpp:59-69)
__device__ __forceinline__ uint32_t planes_needed(uint32_t y, int bps)
{
    uint32_t z = (y ^ (y << 1)) & 0xFFFFFF00u;
    if (bps < 4) z &= (1u << (8 * bps)) - 1u;
    return z ? (31u - (uint32_t)__clz((int)z)) / 8u + 1u : 1u;
}

// raw frame tile -> byte planes.  One CTA handles `ts` consecutive samples of every channel of
// one frame: the tile is contiguous in the interleaved input, so every input byte is read
// exactly once, coalesced.  STENCIL = xdelta_hzr (y = ((x-x1)-128) ^ ((x1-x2)-128)), else the
// plain hzr packer (y = x).
template <int BPS, bool STENCIL>
__global__ void __launch_bounds__(256) k_xdelta_planes(const uint8_t* __restrict__ src, Shape s, uint32_t ts,
                                                        uint32_t tiles_per_frame, uint8_t* __restrict__ planes,
                                                        uint32_t* __restrict__ need)
{
    extern __shared__ __align__(16) uint8_t sm[];
    const uint32_t f = blockIdx.x / tiles_per_frame, tile = blockIdx.x % tiles_per_frame;
    const uint32_t s0 = tile * ts;
    const uint32_t tsv = min(ts, (uint32_t)s.ns - s0);
    const uint8_t* frame = src + (size_t)f * s.frame_bytes;
    const uint32_t row = (uint32_t)s.ch * BPS;
    // shared layout: [raw tile (+15 phase) | xw[ch][ts + 2]]
    int32_t* xw = reinterpret_cast<int32_t*>(sm + ((ts * row + 31u) & ~15u));
    const uint32_t xs = ts + 2;
    const uint32_t phase = tile_load(sm, frame + (size_t)s0 * row, tsv * row);
    __syncthreads();
    // de-interleave: lanes run along samples so the strided byte reads spread over banks
    for (uint32_t e = threadIdx.x; e < tsv * s.ch; e += blockDim.x) {
        const uint32_t c = e / tsv, j = e % tsv;
        xw[c * xs + 2 + j] = load_sample<BPS>(sm + phase + (j * s.ch + c) * BPS);
    }
    if (STENCIL) {
        // two predecessors of the first sample of every channel row of this tile
        for (uint32_t e = threadIdx.x; e < 2u * s.ch; e += blockDim.x) {
            const uint32_t c = e >> 1, back = 2 - (e & 1);  // back = 2 -> slot 0, back = 1 -> slot 1
            const int64_t flat = (int64_t)c * s.ns + s0 - back;
            xw[c * xs + (2 - back)] = frame_sample_flat<BPS>(frame, s, flat);
        }
    }
    __syncthreads();
    uint32_t my_need = 1;
    for (uint32_t e = threadIdx.x; e < tsv * s.ch; e += blockDim.x) {
        const uint32_t c = e / tsv, j = e % tsv;
        const int32_t* px = xw + c * xs + 2 + j;
        uint32_t y = (uint32_t)px[0];
        if (STENCIL) {
            const uint32_t x0 = (uint32_t)px[0], x1 = (uint32_t)px[-1], x2 = (uint32_t)px[-2];
            uint32_t d0 = x0 - x1 - 128u, d1 = x1 - x2 - 128u;
            // the very first word of the frame has no predecessor delta: y[0] = x[0] - 128
            if (c == 0 && s0 + j == 0) d1 = 0;
            y = d0 ^ d1;
            if (need) my_need = max(my_need, planes_needed(y, BPS));
        }
        uint8_t* out = planes + (size_t)f * s.nb_alloc * s.plane_stride + (size_t)c * s.ns + s0 + j;
        for (uint32_t k = 0; k < s.nb_alloc; ++k) out[(size_t)k * s.plane_stride] = (uint8_t)(y >> (8 * k));
    }
    if (STENCIL && need) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) my_need = max(my_need, __shfl_xor_sync(0xFFFFFFFFu, my_need, o));
        if (lane_id() == 0 && my_need > 1) atomicMax(&need[f], my_need);
    }
}


// ------------------------------------------------------------------------------------------
// Fast path of the forward sample transform (ch % 4 == 0, ns % 4 == 0): same results as
// k_xdelta_planes with ~2.5 instructions per raw byte.
//
// A CTA owns `tsq` sample QUADS (4 consecutive samples of every channel; 4*row bytes, contiguous
// and 16-byte aligned in the interleaved input) plus one halo quad in front (the two predecessor
// samples of the stencil).  Quads are staged in shared memory at a stride of row + 1 words -- an
// odd stride, so that 32 lanes reading the same word of 32 consecutive quads hit 32 banks.
// A work item is (channel group g of 4 channels, quad jq): 6 rows x BPS words are read, the
// 4 x BPS bytes of a row are unpacked with one PRMT per sample (sign replication in the
// selector), the 3-tap stencil runs in registers, and a 4 x 4 byte transpose (8 PRMT) turns four
// consecutive y words into one 32-bit word per plane, stored coalesced (lanes run along jq).
// ------------------------------------------------------------------------------------------

// the 4 sign-extended samples packed in BPS consecutive words
template <int BPS>
__device__ __forceinline__ void unpack4(const uint32_t* w, uint32_t (&x)[4])
{
    if (BPS == 4) {
        x[0] = w[0]; x[1] = w[1]; x[2] = w[2]; x[3] = w[3];
    } else if (BPS == 3) {
        x[0] = prmt(w[0], w[0], 0xA210u);
        x[1] = prmt(w[0], w[1], 0xD543u);
        x[2] = prmt(w[1], w[2], 0xC432u);
        x[3] = prmt(w[2], w[2], 0xB321u);
    } else if (BPS == 2) {
        x[0] = prmt(w[0], w[0], 0x9910u);
        x[1] = prmt(w[0], w[0], 0xBB32u);
        x[2] = prmt(w[1], w[1], 0x9910u);
        x[3] = prmt(w[1], w[1], 0xBB32u);
    } else {
        x[0] = prmt(w[0], w[0], 0x8880u);
        x[1] = prmt(w[0], w[0], 0x9991u);
        x[2] = prmt(w[0], w[0], 0xAAA2u);
        x[3] = prmt(w[0], w[0], 0xBBB3u);
    }
}

template <int BPS, bool STENCIL>
__global__ void __launch_bounds__(128) k_xdelta_planes_fast(const uint8_t* __restrict__ src, Shape s, uint32_t tsq,
                                                             uint32_t tiles_per_frame, uint8_t* __restrict__ planes,
                                                             uint32_t* __restrict__ need)
{
    extern __shared__ __align__(16) uint32_t smw[];
    const uint32_t f = blockIdx.x / tiles_per_frame, tile = blockIdx.x % tiles_per_frame;
    const uint32_t row = (uint32_t)s.ch * BPS;       // bytes per sample row == words per quad
    const uint32_t qstride = row + 1;                // words
    const uint32_t cpq = row >> 2;                   // 16-byte chunks per quad
    const uint32_t nq = (uint32_t)s.ns >> 2;         // quads per frame
    const uint32_t q0 = tile * tsq;
    const uint32_t tq = min(tsq, nq - q0);           // quads of this tile
    const uint8_t* frame = src + (size_t)f * s.frame_bytes;
    const uint32_t halo = (STENCIL && q0 > 0) ? 1u : 0u;
    // stage quads [q0 - halo, q0 + tq) at slots [1 - halo, 1 + tq)
    {
        const uint4* g4 = reinterpret_cast<const uint4*>(frame + (size_t)(q0 - halo) * 4u * row);
        const uint32_t nchunks = (tq + halo) * cpq;
        uint32_t q = threadIdx.x / cpq, r = threadIdx.x % cpq;
        const uint32_t dq = blockDim.x / cpq, dr = blockDim.x % cpq;
        for (uint32_t c = threadIdx.x; c < nchunks; c += blockDim.x) {
            const uint4 v = __ldg(g4 + c);
            uint32_t* d = smw + (q + 1 - halo) * qstride + 4u * r;
            d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
            q += dq; r += dr;
            if (r >= cpq) { r -= cpq; ++q; }
        }
    }
    __syncthreads();
    const uint32_t G = (uint32_t)s.ch >> 2;
    const uint32_t rw = row >> 2;                    // words per row
    uint32_t my_need = 1;
    for (uint32_t item = threadIdx.x; item < G * tq; item += blockDim.x) {
        const uint32_t g = item / tq, jq = item - g * tq;
        const uint32_t* base = smw + (jq + 1) * qstride + g * BPS;
        uint32_t x[6][4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            uint32_t w[4];
#pragma unroll
            for (int t = 0; t < BPS; ++t) w[t] = base[i * rw + t];
            unpack4<BPS>(w, x[i + 2]);
        }
        if (STENCIL) {
            if (q0 + jq > 0) {
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    uint32_t w[4];
#pragma unroll
                    for (int t = 0; t < BPS; ++t) w[t] = base[(int)(i + 2) * (int)rw - (int)qstride + t];
                    unpack4<BPS>(w, x[i]);
                }
            } else {
                // first quad of the frame: the flat chain continues from the end of the previous
                // channel row (signal_packer_xdelta_hzr.cpp:55-57 run over the flat [ch*ns] array)
#pragma unroll
                for (int cc = 0; cc < 4; ++cc) {
                    const int64_t flat = (int64_t)(4 * g + cc) * s.ns;
                    x[0][cc] = (uint32_t)frame_sample_flat<BPS>(frame, s, flat - 2);
                    x[1][cc] = (uint32_t)frame_sample_flat<BPS>(frame, s, flat - 1);
                }
            }
        }
        const uint32_t s_first = (q0 + jq) << 2;
#pragma unroll
        for (int cc = 0; cc < 4; ++cc) {
            uint32_t y[4];
            if (STENCIL) {
                uint32_t d[5];
#pragma unroll
                for (int i = 0; i < 5; ++i) d[i] = x[i + 1][cc] - x[i][cc] - 128u;
                // the very first word of the frame has no predecessor delta: y[0] = x[0] - 128
                if (s_first == 0 && g == 0 && cc == 0) d[0] = 0;
#pragma unroll
                for (int i = 0; i < 4; ++i) y[i] = d[i + 1] ^ d[i];
                if (need) {
#pragma unroll
                    for (int i = 0; i < 4; ++i) my_need = max(my_need, planes_needed(y[i], BPS));
                }
            } else {
#pragma unroll
                for (int i = 0; i < 4; ++i) y[i] = x[i + 2][cc];
            }
            const uint32_t t01 = prmt(y[0], y[1], 0x5140u), t23 = prmt(y[2], y[3], 0x5140u);
            const uint32_t u01 = prmt(y[0], y[1], 0x7362u), u23 = prmt(y[2], y[3], 0x7362u);
            uint32_t* out = reinterpret_cast<uint32_t*>(planes + (size_t)f * s.nb_alloc * s.plane_stride +
                                                        (size_t)(4 * g + cc) * s.ns + s_first);
            const uint32_t ps = s.plane_stride >> 2;
            out[0] = prmt(t01, t23, 0x5410u);
            if (s.nb_alloc > 1) out[ps] = prmt(t01, t23, 0x7632u);
            if (s.nb_alloc > 2) out[2 * ps] = prmt(u01, u23, 0x5410u);
            if (s.nb_alloc > 3) out[3 * ps] = prmt(u01, u23, 0x7632u);
        }
    }
    if (STENCIL && need) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) my_need = max(my_need, __shfl_xor_sync(0xFFFFFFFFu, my_need, o));
        if (lane_id() == 0 && my_need > 1) atomicMax(&need[f], my_need);
    }
}

// ------------------------------------------------------------------------------------------
// planes -> samples.  One CTA per frame.  The decode-side chains are two scans over the flat
// [ch*ns] order that cross channel rows: d = prefix-xor(y) (xor_decode_32, utils.cpp:232-236),
// x = prefix-sum(d + 128) (offset_32(+128) and delta_decode, :204-219).  The frame is cut into
// PIECES of 256 consecutive samples of one channel (one warp, 8 samples per lane); piece totals
// are scanned in shared memory: pass 1 xor totals, pass 2 sums of d + 128, pass 3 the samples.
// OUT_RAW: pass 3 walks sample tiles, transposes through shared memory and stores interleaved
// little-endian samples (convert_i32_to_native, utils.cpp:51-121) with coalesced writes;
// otherwise the int32 words are stored in flat order (input of the inverse DCT).
// ------------------------------------------------------------------------------------------
constexpr int kPiece = 256;

// y[0..7] for flat elements [e0, e0 + cnt) of one frame, sign-extended from 8*nb bits
// (signal_packer_base.cpp:126-138)
__device__ __forceinline__ void load_y8(const uint8_t* __restrict__ fplanes, uint32_t stride, uint32_t nb, uint32_t e0,
                                        uint32_t cnt, uint32_t (&y)[8])
{
#pragma unroll
    for (int i = 0; i < 8; ++i) y[i] = 0;
    const bool vec = cnt == 8 && ((e0 & 7u) == 0);
    for (uint32_t k = 0; k < nb; ++k) {
        const uint8_t* row = fplanes + (size_t)k * stride + e0;
        if (vec) {
            const uint2 v = __ldg(reinterpret_cast<const uint2*>(row));
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                y[i] |= ((v.x >> (8 * i)) & 0xFFu) << (8 * k);
                y[4 + i] |= ((v.y >> (8 * i)) & 0xFFu) << (8 * k);
            }
        } else {
#pragma unroll
            for (int i = 0; i < 8; ++i)
                if ((uint32_t)i < cnt) y[i] |= (uint32_t)row[i] << (8 * k);
        }
    }
    const int sh = 32 - 8 * (int)nb;
#pragma unroll
    for (int i = 0; i < 8; ++i) y[i] = (uint32_t)((int32_t)(y[i] << sh) >> sh);
}

// exclusive scan (xor or add) of a shared array by warp 0
template <bool XOR>
__device__ __forceinline__ void smem_exclusive_scan(uint32_t* a, uint32_t n)
{
    if (warp_id() == 0) {
        uint32_t carry = 0;
        for (uint32_t base = 0; base < n; base += 32) {
            const uint32_t i = base + lane_id();
            const uint32_t v = i < n ? a[i] : 0u;
            uint32_t inc = v;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, inc, o);
                if (lane_id() >= (uint32_t)o) inc = XOR ? (inc ^ t) : (inc + t);
            }
            if (i < n) a[i] = XOR ? (carry ^ inc ^ v) : (carry + inc - v);
            const uint32_t tot = __shfl_sync(0xFFFFFFFFu, inc, 31);
            carry = XOR ? (carry ^ tot) : (carry + tot);
        }
    }
}

template <int BPS, bool SCAN, bool OUT_RAW>
__global__ void __launch_bounds__(512) k_planes_to_samples(const uint8_t* __restrict__ planes, Shape s,
                                                            const uint8_t* __restrict__ dec_nb,
                                                            uint8_t* __restrict__ dst_raw, int32_t* __restrict__ dst_words)
{
    extern __shared__ __align__(16) uint32_t sm32[];
    const uint32_t f = blockIdx.x;
    const uint32_t nb = dec_nb[f];
    const uint32_t ns = (uint32_t)s.ns, ch = (uint32_t)s.ch;
    const uint32_t ppc = (ns + kPiece - 1) / kPiece, np = ppc * ch;
    uint32_t* pxor = sm32;          // [np]
    uint32_t* psum = sm32 + np;     // [np]
    uint32_t* tile = sm32 + 2 * np; // OUT_RAW: [kPiece * ch * BPS bytes] (+4 words slack)
    const uint8_t* fpl = planes + (size_t)f * s.nb_alloc * s.plane_stride;
    const uint32_t lane = lane_id(), wid = warp_id(), nwarps = blockDim.x >> 5;
    uint32_t y[8];

    if (SCAN) {
        for (uint32_t p = wid; p < np; p += nwarps) {
            const uint32_t c = p / ppc, j = p % ppc;
            const uint32_t s0 = j * kPiece + lane * 8;
            const uint32_t cnt = s0 < ns ? min(8u, ns - s0) : 0u;
            load_y8(fpl, s.plane_stride, nb, c * ns + s0, cnt, y);
            uint32_t x = 0;
#pragma unroll
            for (int i = 0; i < 8; ++i) x ^= (uint32_t)i < cnt ? y[i] : 0u;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) x ^= __shfl_xor_sync(0xFFFFFFFFu, x, o);
            if (lane == 0) pxor[p] = x;
        }
        __syncthreads();
        smem_exclusive_scan<true>(pxor, np);
        __syncthreads();
        for (uint32_t p = wid; p < np; p += nwarps) {
            const uint32_t c = p / ppc, j = p % ppc;
            const uint32_t s0 = j * kPiece + lane * 8;
            const uint32_t cnt = s0 < ns ? min(8u, ns - s0) : 0u;
            load_y8(fpl, s.plane_stride, nb, c * ns + s0, cnt, y);
            // lane-local inclusive xor prefix, then the lanes before me
            uint32_t run = 0;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                run ^= (uint32_t)i < cnt ? y[i] : 0u;
                y[i] = run;
            }
            uint32_t inc = run;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, inc, o);
                if (lane >= (uint32_t)o) inc ^= t;
            }
            const uint32_t before = pxor[p] ^ inc ^ run;
            uint32_t sum = 0;
#pragma unroll
            for (int i = 0; i < 8; ++i)
                if ((uint32_t)i < cnt) sum += (y[i] ^ before) + 128u;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xFFFFFFFFu, sum, o);
            if (lane == 0) psum[p] = sum;
        }
        __syncthreads();
        smem_exclusive_scan<false>(psum, np);
        __syncthreads();
    }

    const uint32_t row = ch * BPS;
    uint8_t* tb = reinterpret_cast<uint8_t*>(tile);
    // pass 3: tile j = samples [j*256, j*256+256) of every channel
    for (uint32_t j = 0; j < ppc; ++j) {
        const uint32_t tsv = min((uint32_t)kPiece, ns - j * kPiece);
        for (uint32_t c = wid; c < ch; c += nwarps) {
            const uint32_t p = c * ppc + j;
            const uint32_t s0 = j * kPiece + lane * 8;
            const uint32_t cnt = s0 < ns ? min(8u, ns - s0) : 0u;
            load_y8(fpl, s.plane_stride, nb, c * ns + s0, cnt, y);
            if (SCAN) {
                uint32_t run = 0;
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    run ^= (uint32_t)i < cnt ? y[i] : 0u;
                    y[i] = run;
                }
                uint32_t inc = run;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, inc, o);
                    if (lane >= (uint32_t)o) inc ^= t;
                }
                const uint32_t before = pxor[p] ^ inc ^ run;
                uint32_t acc = 0;
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    acc += (uint32_t)i < cnt ? (y[i] ^ before) + 128u : 0u;
                    y[i] = acc;
                }
                uint32_t sinc = acc;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, sinc, o);
                    if (lane >= (uint32_t)o) sinc += t;
                }
                const uint32_t base = psum[p] + sinc - acc;
#pragma unroll
                for (int i = 0; i < 8; ++i) y[i] += base;
            }
            if (OUT_RAW) {
#pragma unroll
                for (int i = 0; i < 8; ++i)
                    if ((uint32_t)i < cnt) {
                        uint8_t* q = tb + ((lane * 8 + i) * ch + c) * BPS;
#pragma unroll
                        for (int bb = 0; bb < BPS; ++bb) q[bb] = (uint8_t)(y[i] >> (8 * bb));
                    }
            } else {
                int32_t* w = dst_words + (size_t)f * s.N + (size_t)c * ns + s0;
#pragma unroll
                for (int i = 0; i < 8; ++i)
                    if ((uint32_t)i < cnt) w[i] = (int32_t)y[i];
            }
        }
        if (OUT_RAW) {
            __syncthreads();
            copy_smem_to_global(dst_raw + (size_t)f * s.frame_bytes + (size_t)j * kPiece * row, tile, 0, tsv * row);
            __syncthreads();
        }
    }
}

// ------------------------------------------------------------------------------------------
// Fast path of planes -> samples (ch % 4 == 0, ns % 128 == 0): one CTA of 8 warps per frame.
// A PIECE is 128 consecutive flat elements (one warp, 4 per lane, one 32-bit word per plane).
//   pass 1  xor of every piece (plane words folded byte-wise; no transpose needed)
//   pass 2  sum of (prefix-xor + 128) of every piece
//   pass 3  a warp takes (4 channels x 128 samples): per channel the 4 x 4 byte transpose back to
//           sign-extended words, lane-local + warp xor scan, +128, lane-local + warp add scan;
//           the four channels' samples are packed row-wise with PRMT into a shared-memory tile
//           (quad stride row + 1 words, conflict-free) that the CTA then copies out coalesced.
// SCAN = false is the plain hzr packer (no chain).  WORDS = true stops after the scans and stores
// the int32 words in flat order (the coefficient words of the inverse DCT): pass 3 then walks the
// pieces like pass 2 and every lane writes its 4 consecutive words with one 128-bit store.
// ------------------------------------------------------------------------------------------
constexpr int kInvThreads = 256;
constexpr uint32_t kInvPiece = 128;

// plane words (4 consecutive elements each) -> the 4 sign-extended 32-bit words
__device__ __forceinline__ void planes_to_words(uint32_t q0, uint32_t q1, uint32_t q2, uint32_t q3, uint32_t nb, uint32_t (&y)[4])
{
    // missing planes = sign bytes of the highest stored plane (signal_packer_base.cpp:126-138)
    if (nb == 1) q1 = prmt(q0, q0, 0xBA98u);
    if (nb <= 2) q2 = prmt(q1, q1, 0xBA98u);
    if (nb <= 3) q3 = prmt(q2, q2, 0xBA98u);
    const uint32_t t01 = prmt(q0, q1, 0x5140u), t23 = prmt(q2, q3, 0x5140u);
    const uint32_t u01 = prmt(q0, q1, 0x7362u), u23 = prmt(q2, q3, 0x7362u);
    y[0] = prmt(t01, t23, 0x5410u);
    y[1] = prmt(t01, t23, 0x7632u);
    y[2] = prmt(u01, u23, 0x5410u);
    y[3] = prmt(u01, u23, 0x7632u);
}

__device__ __forceinline__ uint32_t warp_xor_inclusive(uint32_t v)
{
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, v, o);
        if (lane_id() >= (uint32_t)o) v ^= t;
    }
    return v;
}

__device__ __forceinline__ uint32_t warp_add_inclusive(uint32_t v)
{
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, v, o);
        if (lane_id() >= (uint32_t)o) v += t;
    }
    return v;
}

template <int BPS, bool SCAN, bool WORDS = false>
__global__ void __launch_bounds__(1024, 1) k_planes_to_samples_fast(const uint8_t* __restrict__ planes, Shape s,
                                                                            const uint8_t* __restrict__ dec_nb,
                                                                            uint32_t tiles_per_group,
                                                                            uint8_t* __restrict__ dst_raw,
                                                                            int32_t* __restrict__ dst_words = nullptr)
{
    extern __shared__ __align__(16) uint32_t sm32[];
    const uint32_t f = blockIdx.x;
    const uint32_t nb = dec_nb[f];
    const uint32_t ns = (uint32_t)s.ns, ch = (uint32_t)s.ch;
    const uint32_t ppc = ns / kInvPiece, np = ppc * ch;      // pieces per channel row / per frame
    uint32_t* pxor = sm32;           // [np] exclusive xor carry of every piece
    uint32_t* psum = sm32 + np;      // [np] exclusive sum carry
    uint32_t* tile = sm32 + 2 * np;  // output tile: quads of 4 sample rows at a stride of row + 1 words
    const uint32_t* fpl = reinterpret_cast<const uint32_t*>(planes + (size_t)f * s.nb_alloc * s.plane_stride);
    const uint32_t pstride = s.plane_stride >> 2;
    const uint32_t lane = lane_id(), wid = warp_id(), nwarps = blockDim.x >> 5;
    const int sext = 32 - 8 * (int)nb;

    // plane words of piece p for this lane; planes >= nb are replaced by sign bytes later, so
    // every allocated plane is simply loaded (independent loads, all in flight together)
    const uint32_t nba = s.nb_alloc;
    auto load_piece = [&](uint32_t p, uint32_t (&q)[4]) {
        const uint32_t* a = fpl + p * 32u + lane;
        q[0] = __ldg(a);
        q[1] = nba > 1 ? __ldg(a + pstride) : 0u;
        q[2] = nba > 2 ? __ldg(a + 2 * pstride) : 0u;
        q[3] = nba > 3 ? __ldg(a + 3 * pstride) : 0u;
    };
    constexpr int U = 4;  // pieces in flight per warp
    // four pieces at a time (np is a multiple of 4 because ch is): 16 consecutive elements per lane
    const uint4* fpl4 = reinterpret_cast<const uint4*>(fpl);
    const uint32_t pstride4 = s.plane_stride >> 4, nbig = np >> 2;
    constexpr int UB = 2;
    auto load_big = [&](uint32_t P, uint4 (&q)[4]) {
        const uint4* a = fpl4 + P * 32u + lane;
        q[0] = __ldg(a);
        q[1] = nba > 1 ? __ldg(a + pstride4) : make_uint4(0, 0, 0, 0);
        q[2] = nba > 2 ? __ldg(a + 2 * pstride4) : make_uint4(0, 0, 0, 0);
        q[3] = nba > 3 ? __ldg(a + 3 * pstride4) : make_uint4(0, 0, 0, 0);
    };
    if (SCAN) {
        // pass 1: xor of all words of a piece = byte-wise fold of the plane words
        // (passes 1 and 2 walk the planes in runs of four pieces: a lane takes 16 consecutive elements with one
        // 128-bit load per plane, eight lanes make a piece, and the warp-level steps are shared by four pieces)
        for (uint32_t P0 = wid * UB; P0 < nbig; P0 += nwarps * UB) {
            uint4 q[UB][4];
#pragma unroll
            for (int u = 0; u < UB; ++u)
                if (P0 + u < nbig) load_big(P0 + u, q[u]);
#pragma unroll
            for (int u = 0; u < UB; ++u) {
                if (P0 + u >= nbig) break;
                uint32_t x = 0;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    uint32_t w = (uint32_t)k < nb ? q[u][k].x ^ q[u][k].y ^ q[u][k].z ^ q[u][k].w : 0u;
                    w ^= w >> 16;
                    w ^= w >> 8;
                    x |= (w & 0xFFu) << (8 * k);
                }
                x = (uint32_t)((int32_t)(x << sext) >> sext);
#pragma unroll
                for (int o = 4; o > 0; o >>= 1) x ^= __shfl_xor_sync(0xFFFFFFFFu, x, o);
                if ((lane & 7u) == 0u) pxor[4u * (P0 + u) + (lane >> 3)] = x;
            }
        }
        __syncthreads();
        smem_exclusive_scan<true>(pxor, np);
        __syncthreads();
        // pass 2: sum of (prefix-xor + 128) over every piece
        for (uint32_t P0 = wid * UB; P0 < nbig; P0 += nwarps * UB) {
            uint4 q[UB][4];
#pragma unroll
            for (int u = 0; u < UB; ++u)
                if (P0 + u < nbig) load_big(P0 + u, q[u]);
#pragma unroll
            for (int u = 0; u < UB; ++u) {
                if (P0 + u >= nbig) break;
                uint32_t y[16];
                {
                    uint32_t t[4];
                    planes_to_words(q[u][0].x, q[u][1].x, q[u][2].x, q[u][3].x, nb, t);
                    y[0] = t[0]; y[1] = t[1]; y[2] = t[2]; y[3] = t[3];
                    planes_to_words(q[u][0].y, q[u][1].y, q[u][2].y, q[u][3].y, nb, t);
                    y[4] = t[0]; y[5] = t[1]; y[6] = t[2]; y[7] = t[3];
                    planes_to_words(q[u][0].z, q[u][1].z, q[u][2].z, q[u][3].z, nb, t);
                    y[8] = t[0]; y[9] = t[1]; y[10] = t[2]; y[11] = t[3];
                    planes_to_words(q[u][0].w, q[u][1].w, q[u][2].w, q[u][3].w, nb, t);
                    y[12] = t[0]; y[13] = t[1]; y[14] = t[2]; y[15] = t[3];
                }
#pragma unroll
                for (int i = 1; i < 16; ++i) y[i] ^= y[i - 1];
                uint32_t inc = y[15];   // inclusive xor over the lanes of my piece (8 lanes)
#pragma unroll
                for (int o = 1; o < 8; o <<= 1) {
                    const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, inc, o);
                    if ((lane & 7u) >= (uint32_t)o) inc ^= t;
                }
                const uint32_t before = pxor[4u * (P0 + u) + (lane >> 3)] ^ inc ^ y[15];
                uint32_t sum = 16u * 128u;
#pragma unroll
                for (int i = 0; i < 16; ++i) sum += y[i] ^ before;
#pragma unroll
                for (int o = 4; o > 0; o >>= 1) sum += __shfl_xor_sync(0xFFFFFFFFu, sum, o);
                if ((lane & 7u) == 0u) psum[4u * (P0 + u) + (lane >> 3)] = sum;
            }
        }
        __syncthreads();
        smem_exclusive_scan<false>(psum, np);
        __syncthreads();
    }

    if (WORDS) {
        // pass 3, word output: two pieces at a time, 8 consecutive words per lane (one 64-bit load per plane, 16 lanes
        // make a piece; np is even because ch is a multiple of 4)
        uint4* wout = reinterpret_cast<uint4*>(dst_words + (size_t)f * s.N);
        const uint2* fpl2 = reinterpret_cast<const uint2*>(fpl);
        const uint32_t pstride2 = s.plane_stride >> 3, half = lane >> 4;
        for (uint32_t P0 = wid * U; P0 < (np >> 1); P0 += nwarps * U) {
            uint2 q[U][4];
#pragma unroll
            for (int u = 0; u < U; ++u)
                if (P0 + u < (np >> 1)) {
                    const uint2* a = fpl2 + (P0 + u) * 32u + lane;
                    q[u][0] = __ldg(a);
                    q[u][1] = nba > 1 ? __ldg(a + pstride2) : make_uint2(0, 0);
                    q[u][2] = nba > 2 ? __ldg(a + 2 * pstride2) : make_uint2(0, 0);
                    q[u][3] = nba > 3 ? __ldg(a + 3 * pstride2) : make_uint2(0, 0);
                }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                if (P0 + u >= (np >> 1)) break;
                const uint32_t pp = 2u * (P0 + u) + half;
                uint32_t y[8];
                {
                    uint32_t tq[4];
                    planes_to_words(q[u][0].x, q[u][1].x, q[u][2].x, q[u][3].x, nb, tq);
                    y[0] = tq[0]; y[1] = tq[1]; y[2] = tq[2]; y[3] = tq[3];
                    planes_to_words(q[u][0].y, q[u][1].y, q[u][2].y, q[u][3].y, nb, tq);
                    y[4] = tq[0]; y[5] = tq[1]; y[6] = tq[2]; y[7] = tq[3];
                }
                if (SCAN) {
#pragma unroll
                    for (int i = 1; i < 8; ++i) y[i] ^= y[i - 1];
                    uint32_t inc = y[7];
#pragma unroll
                    for (int o = 1; o < 16; o <<= 1) {
                        const uint32_t tt = __shfl_up_sync(0xFFFFFFFFu, inc, o);
                        if ((lane & 15u) >= (uint32_t)o) inc ^= tt;
                    }
                    const uint32_t before = pxor[pp] ^ inc ^ y[7];
                    y[0] = (y[0] ^ before) + 128u;
#pragma unroll
                    for (int i = 1; i < 8; ++i) y[i] = (y[i] ^ before) + 128u + y[i - 1];
                    uint32_t acc = y[7];
#pragma unroll
                    for (int o = 1; o < 16; o <<= 1) {
                        const uint32_t tt = __shfl_up_sync(0xFFFFFFFFu, acc, o);
                        if ((lane & 15u) >= (uint32_t)o) acc += tt;
                    }
                    const uint32_t base = psum[pp] + acc - y[7];
#pragma unroll
                    for (int i = 0; i < 8; ++i) y[i] += base;
                }
                uint4* w2 = wout + (size_t)(P0 + u) * 64u + 2u * lane;
                w2[0] = make_uint4(y[0], y[1], y[2], y[3]);
                w2[1] = make_uint4(y[4], y[5], y[6], y[7]);
            }
        }
        return;
    }

    // pass 3: groups of `tiles_per_group` sample tiles (128 samples each); work item = (tile, channel group)
    const uint32_t row = ch * BPS, rw = row >> 2, qstride = row + 1, G = ch >> 2, cpq = row >> 2;
    if (((ppc | tiles_per_group) & 1u) == 0u) {
        // Two tiles per item: a lane takes 8 consecutive samples of each of the 4 channels (one 64-bit load per
        // plane), 16 lanes make a piece, so the warp-level scan steps are shared by two pieces.  The lane's two
        // quads lie 2 * qstride words apart: with one pad word per 32 quads the 32 lanes hit 32 banks.
        const uint2* fpl2 = reinterpret_cast<const uint2*>(fpl);
        const uint32_t pstride2 = s.plane_stride >> 3, half = lane >> 4;
        for (uint32_t t0 = 0; t0 < ppc; t0 += tiles_per_group) {
            const uint32_t nt = min(tiles_per_group, ppc - t0);
            for (uint32_t item = wid; item < (nt >> 1) * G; item += nwarps) {
                const uint32_t tl2 = item / G, g = item - tl2 * G, t = t0 + 2u * tl2;
                uint2 q[4][4];
#pragma unroll
                for (int cc = 0; cc < 4; ++cc) {
                    const uint2* a = fpl2 + ((4 * g + cc) * ppc + t) * 16u + lane;
                    q[cc][0] = __ldg(a);
                    q[cc][1] = nba > 1 ? __ldg(a + pstride2) : make_uint2(0, 0);
                    q[cc][2] = nba > 2 ? __ldg(a + 2 * pstride2) : make_uint2(0, 0);
                    q[cc][3] = nba > 3 ? __ldg(a + 3 * pstride2) : make_uint2(0, 0);
                }
                uint32_t x[4][8];
#pragma unroll
                for (int cc = 0; cc < 4; ++cc) {
                    const uint32_t pp = (4 * g + cc) * ppc + t + half;   // my piece
                    uint32_t* y = x[cc];
                    {
                        uint32_t tq[4];
                        planes_to_words(q[cc][0].x, q[cc][1].x, q[cc][2].x, q[cc][3].x, nb, tq);
                        y[0] = tq[0]; y[1] = tq[1]; y[2] = tq[2]; y[3] = tq[3];
                        planes_to_words(q[cc][0].y, q[cc][1].y, q[cc][2].y, q[cc][3].y, nb, tq);
                        y[4] = tq[0]; y[5] = tq[1]; y[6] = tq[2]; y[7] = tq[3];
                    }
                    if (SCAN) {
#pragma unroll
                        for (int i = 1; i < 8; ++i) y[i] ^= y[i - 1];
                        uint32_t inc = y[7];
#pragma unroll
                        for (int o = 1; o < 16; o <<= 1) {
                            const uint32_t tt = __shfl_up_sync(0xFFFFFFFFu, inc, o);
                            if ((lane & 15u) >= (uint32_t)o) inc ^= tt;
                        }
                        const uint32_t before = pxor[pp] ^ inc ^ y[7];
                        y[0] = (y[0] ^ before) + 128u;
#pragma unroll
                        for (int i = 1; i < 8; ++i) y[i] = (y[i] ^ before) + 128u + y[i - 1];
                        uint32_t acc = y[7];
#pragma unroll
                        for (int o = 1; o < 16; o <<= 1) {
                            const uint32_t tt = __shfl_up_sync(0xFFFFFFFFu, acc, o);
                            if ((lane & 15u) >= (uint32_t)o) acc += tt;
                        }
                        const uint32_t base = psum[pp] + acc - y[7];
#pragma unroll
                        for (int i = 0; i < 8; ++i) y[i] += base;
                    }
                }
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const uint32_t Q = tl2 * 64u + 2u * lane + h;
                    uint32_t* out = tile + Q * qstride + (Q >> 5) + g * BPS;
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const uint32_t a = x[0][4 * h + i], b = x[1][4 * h + i], c2 = x[2][4 * h + i], d = x[3][4 * h + i];
                        if (BPS == 4) {
                            out[i * rw + 0] = a; out[i * rw + 1] = b; out[i * rw + 2] = c2; out[i * rw + 3] = d;
                        } else if (BPS == 3) {
                            out[i * rw + 0] = prmt(a, b, 0x4210u);
                            out[i * rw + 1] = prmt(b, c2, 0x5421u);
                            out[i * rw + 2] = prmt(c2, d, 0x6542u);
                        } else if (BPS == 2) {
                            out[i * rw + 0] = prmt(a, b, 0x5410u);
                            out[i * rw + 1] = prmt(c2, d, 0x5410u);
                        } else {
                            out[i * rw + 0] = prmt(prmt(a, b, 0x0040u), prmt(c2, d, 0x0040u), 0x5410u);
                        }
                    }
                }
            }
            __syncthreads();
            {
                uint4* g4 = reinterpret_cast<uint4*>(dst_raw + (size_t)f * s.frame_bytes + (size_t)t0 * kInvPiece * row);
                const uint32_t nchunks = nt * 32u * cpq;
                uint32_t q = threadIdx.x / cpq, r = threadIdx.x % cpq;
                const uint32_t dq = blockDim.x / cpq, dr = blockDim.x % cpq;
                for (uint32_t c = threadIdx.x; c < nchunks; c += blockDim.x) {
                    const uint32_t* sp = tile + q * qstride + (q >> 5) + 4u * r;
                    g4[c] = make_uint4(sp[0], sp[1], sp[2], sp[3]);
                    q += dq; r += dr;
                    if (r >= cpq) { r -= cpq; ++q; }
                }
            }
            __syncthreads();
        }
        return;
    }
    for (uint32_t t0 = 0; t0 < ppc; t0 += tiles_per_group) {
        const uint32_t nt = min(tiles_per_group, ppc - t0);
        for (uint32_t item = wid; item < nt * G; item += nwarps) {
            const uint32_t tl = item / G, g = item - tl * G, t = t0 + tl;
            uint32_t x[4][4];
#pragma unroll
            for (int cc = 0; cc < 4; ++cc) load_piece((4 * g + cc) * ppc + t, x[cc]);
#pragma unroll
            for (int cc = 0; cc < 4; ++cc) {
                const uint32_t c = 4 * g + cc, p = c * ppc + t;
                planes_to_words(x[cc][0], x[cc][1], x[cc][2], x[cc][3], nb, x[cc]);
                if (SCAN) {
                    uint32_t* y = x[cc];
                    y[1] ^= y[0]; y[2] ^= y[1]; y[3] ^= y[2];
                    const uint32_t before = pxor[p] ^ warp_xor_inclusive(y[3]) ^ y[3];
                    y[0] = (y[0] ^ before) + 128u;
                    y[1] = (y[1] ^ before) + 128u + y[0];
                    y[2] = (y[2] ^ before) + 128u + y[1];
                    y[3] = (y[3] ^ before) + 128u + y[2];
                    const uint32_t base = psum[p] + warp_add_inclusive(y[3]) - y[3];
                    y[0] += base; y[1] += base; y[2] += base; y[3] += base;
                }
            }
            // pack the 4 channels of every sample row into BPS words (convert_i32_to_native, utils.cpp:51-121)
            uint32_t* out = tile + (tl * 32u + lane) * qstride + g * BPS;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const uint32_t a = x[0][i], b = x[1][i], c2 = x[2][i], d = x[3][i];
                if (BPS == 4) {
                    out[i * rw + 0] = a; out[i * rw + 1] = b; out[i * rw + 2] = c2; out[i * rw + 3] = d;
                } else if (BPS == 3) {
                    out[i * rw + 0] = prmt(a, b, 0x4210u);
                    out[i * rw + 1] = prmt(b, c2, 0x5421u);
                    out[i * rw + 2] = prmt(c2, d, 0x6542u);
                } else if (BPS == 2) {
                    out[i * rw + 0] = prmt(a, b, 0x5410u);
                    out[i * rw + 1] = prmt(c2, d, 0x5410u);
                } else {
                    out[i * rw + 0] = prmt(prmt(a, b, 0x0040u), prmt(c2, d, 0x0040u), 0x5410u);
                }
            }
        }
        __syncthreads();
        // coalesced copy of the group's rows (contiguous in the interleaved output); drops the pad word
        {
            uint4* g4 = reinterpret_cast<uint4*>(dst_raw + (size_t)f * s.frame_bytes + (size_t)t0 * kInvPiece * row);
            const uint32_t nchunks = nt * 32u * cpq;
            uint32_t q = threadIdx.x / cpq, r = threadIdx.x % cpq;
            const uint32_t dq = blockDim.x / cpq, dr = blockDim.x % cpq;
            for (uint32_t c = threadIdx.x; c < nchunks; c += blockDim.x) {
                const uint32_t* sp = tile + q * qstride + 4u * r;
                g4[c] = make_uint4(sp[0], sp[1], sp[2], sp[3]);
                q += dq; r += dr;
                if (r >= cpq) { r -= cpq; ++q; }
            }
        }
        __syncthreads();
    }
}

// int32 words [ch][ns] -> interleaved little-endian samples; one CTA per (frame, 256-sample tile)
template <int BPS>
__global__ void __launch_bounds__(256) k_words_to_raw(const int32_t* __restrict__ words, Shape s, uint32_t tiles,
                                                       uint8_t* __restrict__ dst)
{
    extern __shared__ __align__(16) uint32_t sm32[];
    uint8_t* tb = reinterpret_cast<uint8_t*>(sm32);
    const uint32_t f = blockIdx.x / tiles, j = blockIdx.x % tiles;
    const uint32_t ns = (uint32_t)s.ns, ch = (uint32_t)s.ch, row = ch * BPS;
    const uint32_t s0 = j * kPiece, tsv = min((uint32_t)kPiece, ns - s0);
    const int32_t* w = words + (size_t)f * s.N;
    for (uint32_t e = threadIdx.x; e < tsv * ch; e += blockDim.x) {
        const uint32_t c = e / tsv, i = e % tsv;
        const uint32_t v = (uint32_t)w[(size_t)c * ns + s0 + i];
        uint8_t* q = tb + (i * ch + c) * BPS;
#pragma unroll
        for (int bb = 0; bb < BPS; ++bb) q[bb] = (uint8_t)(v >> (8 * bb));
    }
    __syncthreads();
    copy_smem_to_global(dst + (size_t)f * s.frame_bytes + (size_t)s0 * row, sm32, 0, tsv * row);
}

// interleaved samples -> int32 words [ch][ns] (+ per-channel sums for the mean); one CTA per
// (frame, sample tile)
template <int BPS>
__global__ void __launch_bounds__(256) k_raw_to_words(const uint8_t* __restrict__ src, Shape s, uint32_t tiles,
                                                       int32_t* __restrict__ words, long long* __restrict__ sums)
{
    extern __shared__ __align__(16) uint8_t sm[];
    const uint32_t f = blockIdx.x / tiles, j = blockIdx.x % tiles;
    const uint32_t ns = (uint32_t)s.ns, ch = (uint32_t)s.ch, row = ch * BPS;
    const uint32_t s0 = j * kPiece, tsv = min((uint32_t)kPiece, ns - s0);
    const uint32_t phase = tile_load(sm, src + (size_t)f * s.frame_bytes + (size_t)s0 * row, tsv * row);
    __syncthreads();
    int32_t* w = words + (size_t)f * s.N;
    // a warp takes one channel at a time so that its partial sum needs one atomic
    for (uint32_t c = warp_id(); c < ch; c += (blockDim.x >> 5)) {
        long long acc = 0;
        for (uint32_t i = lane_id(); i < tsv; i += 32) {
            const int32_t v = load_sample<BPS>(sm + phase + (i * ch + c) * BPS);
            w[(size_t)c * ns + s0 + i] = v;
            acc += v;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xFFFFFFFFu, acc, o);
        if (lane_id() == 0) atomicAdd(reinterpret_cast<unsigned long long*>(sums + (size_t)f * ch + c), (unsigned long long)acc);
    }
}

// ---- four-channel-group variants (ch % 4 == 0, ns % 4 == 0, 16-byte aligned frames) -------------
// The 4 x BPS bytes that four neighbouring channels contribute to a sample row are contiguous, so a
// thread that owns 4 consecutive samples of a channel group moves them between the interleaved frame
// (BPS words per sample, at the row stride) and the word matrix (one 128-bit access per channel,
// lanes along the samples) in registers -- no shared-memory tile.  The other channel groups touch the
// neighbouring bytes of the same lines at the same time; the L2 merges them.
template <int BPS>
__global__ void __launch_bounds__(256) k_words_to_raw_g4(const int32_t* __restrict__ words, Shape s, uint8_t* __restrict__ dst)
{
    const uint32_t nq = (uint32_t)s.ns >> 2, G = (uint32_t)s.ch >> 2;
    const size_t item = (size_t)blockIdx.x * blockDim.x + threadIdx.x;  // (frame, group, sample quad)
    const uint32_t jq = (uint32_t)(item % nq), g = (uint32_t)((item / nq) % G);
    const size_t f = item / ((size_t)nq * G);
    const uint32_t* w = reinterpret_cast<const uint32_t*>(words) + f * s.N + (size_t)(4 * g) * s.ns + 4 * jq;
    uint4 x[4];
#pragma unroll
    for (int cc = 0; cc < 4; ++cc) x[cc] = __ldg(reinterpret_cast<const uint4*>(w + (size_t)cc * s.ns));
    const uint32_t roww = ((uint32_t)s.ch * BPS) >> 2;
    uint32_t* base = reinterpret_cast<uint32_t*>(dst + f * s.frame_bytes) + (size_t)(4 * jq) * roww + g * BPS;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const uint32_t a = i == 0 ? x[0].x : i == 1 ? x[0].y : i == 2 ? x[0].z : x[0].w;
        const uint32_t b = i == 0 ? x[1].x : i == 1 ? x[1].y : i == 2 ? x[1].z : x[1].w;
        const uint32_t c2 = i == 0 ? x[2].x : i == 1 ? x[2].y : i == 2 ? x[2].z : x[2].w;
        const uint32_t d = i == 0 ? x[3].x : i == 1 ? x[3].y : i == 2 ? x[3].z : x[3].w;
        uint32_t* p = base + (size_t)i * roww;
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

// nq % 32 == 0 (a warp stays inside one frame and channel group), so the per-channel sums of a warp's
// 128 samples go out with one 64-bit atomic per channel
template <int BPS>
__global__ void __launch_bounds__(256) k_raw_to_words_g4(const uint8_t* __restrict__ src, Shape s, int32_t* __restrict__ words,
                                                          long long* __restrict__ sums)
{
    const uint32_t nq = (uint32_t)s.ns >> 2, G = (uint32_t)s.ch >> 2;
    const size_t item = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t jq = (uint32_t)(item % nq), g = (uint32_t)((item / nq) % G);
    const size_t f = item / ((size_t)nq * G);
    const uint32_t roww = ((uint32_t)s.ch * BPS) >> 2;
    const uint32_t* base = reinterpret_cast<const uint32_t*>(src + f * s.frame_bytes) + (size_t)(4 * jq) * roww + g * BPS;
    uint32_t x[4][4];  // [sample][channel]
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const uint32_t* p = base + (size_t)i * roww;
        uint32_t w[4];
        if (BPS == 4) {
            const uint4 q = __ldg(reinterpret_cast<const uint4*>(p));
            w[0] = q.x; w[1] = q.y; w[2] = q.z; w[3] = q.w;
        } else {
#pragma unroll
            for (int t = 0; t < BPS; ++t) w[t] = __ldg(p + t);
        }
        unpack4<BPS>(w, x[i]);
    }
    uint32_t* wout = reinterpret_cast<uint32_t*>(words) + f * s.N + (size_t)(4 * g) * s.ns + 4 * jq;
#pragma unroll
    for (int cc = 0; cc < 4; ++cc) {
        *reinterpret_cast<uint4*>(wout + (size_t)cc * s.ns) = make_uint4(x[0][cc], x[1][cc], x[2][cc], x[3][cc]);
        // 64-bit channel sum from two 32-bit warp reductions: upper halves (signed) and lower halves
        int hi = 0;
        uint32_t lo = 0;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            hi += (int32_t)x[i][cc] >> 16;
            lo += x[i][cc] & 0xFFFFu;
        }
        hi = __reduce_add_sync(0xFFFFFFFFu, hi);
        lo = __reduce_add_sync(0xFFFFFFFFu, lo);
        if (lane_id() == 0)
            atomicAdd(reinterpret_cast<unsigned long long*>(sums + f * s.ch + 4 * g + cc),
                      (unsigned long long)((long long)hi * 65536ll + (long long)lo));
    }
}

// flat int32 words -> byte planes with the delta / offset / xor stencil (dct coefficients,
// signal_packer_dct.cpp:117-119); one CTA per (frame, 1024-element chunk)
__global__ void __launch_bounds__(256) k_words_stencil_planes(const int32_t* __restrict__ words, Shape s, uint32_t chunks,
                                                               uint8_t* __restrict__ planes)
{
    const uint32_t f = blockIdx.x / chunks, cidx = blockIdx.x % chunks;
    const int32_t* w = words + (size_t)f * s.N;
    uint8_t* out = planes + (size_t)f * s.nb_alloc * s.plane_stride;
    if ((s.N & 3u) == 0u) {
        // four consecutive elements per thread: one 128-bit load, the stencil in registers, a 4x4
        // byte transpose (PRMT) and one 32-bit store per plane
        const uint32_t i = cidx * 1024u + threadIdx.x * 4u;
        if (i >= s.N) return;
        const uint4 v = __ldg(reinterpret_cast<const uint4*>(w + i));
        const uint32_t xm1 = i ? (uint32_t)__ldg(w + i - 1) : 0u, xm2 = i ? (uint32_t)__ldg(w + i - 2) : 0u;
        const uint32_t dm = i ? xm1 - xm2 - 128u : 0u;
        const uint32_t d0 = v.x - xm1 - 128u, d1 = v.y - v.x - 128u, d2 = v.z - v.y - 128u, d3 = v.w - v.z - 128u;
        const uint32_t y0 = d0 ^ dm, y1 = d1 ^ d0, y2 = d2 ^ d1, y3 = d3 ^ d2;
        const uint32_t a = __byte_perm(y0, y1, 0x5140), b = __byte_perm(y2, y3, 0x5140);
        *reinterpret_cast<uint32_t*>(out + i) = __byte_perm(a, b, 0x5410);
        if (s.nb_alloc > 1) *reinterpret_cast<uint32_t*>(out + (size_t)s.plane_stride + i) = __byte_perm(a, b, 0x7632);
        if (s.nb_alloc > 2) {
            const uint32_t c = __byte_perm(y0, y1, 0x7362), d = __byte_perm(y2, y3, 0x7362);
            *reinterpret_cast<uint32_t*>(out + 2 * (size_t)s.plane_stride + i) = __byte_perm(c, d, 0x5410);
            if (s.nb_alloc > 3) *reinterpret_cast<uint32_t*>(out + 3 * (size_t)s.plane_stride + i) = __byte_perm(c, d, 0x7632);
        }
        return;
    }
    for (uint32_t i = cidx * 1024u + threadIdx.x; i < min(s.N, (cidx + 1) * 1024u); i += blockDim.x) {
        const uint32_t x0 = (uint32_t)w[i], x1 = i >= 1 ? (uint32_t)w[i - 1] : 0u, x2 = i >= 2 ? (uint32_t)w[i - 2] : 0u;
        const uint32_t d0 = x0 - x1 - 128u, d1 = i >= 1 ? x1 - x2 - 128u : 0u;
        const uint32_t y = d0 ^ d1;
        for (uint32_t k = 0; k < s.nb_alloc; ++k) out[(size_t)k * s.plane_stride + i] = (uint8_t)(y >> (8 * k));
    }
}

}  // namespace rspt
