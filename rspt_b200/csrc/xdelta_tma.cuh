// Forward sample transform of the xdelta_hzr / hzr packers for sm_100a, fed by the TMA unit: one bulk
// asynchronous copy global -> shared per tile of raw samples, completion on an mbarrier, then de-interleave +
// sign-extend (convert_native_to_i32, utils.cpp:123-191), the delta / offset / xor stencil (utils.cpp:193-230,
// flat chain crossing channel rows) and the byte-plane split (signal_packer_base.cpp:40-68).
// Compiled for ch in {4, 8, 12} (RSPT_TMA_SHAPES in rspt_gpu.cu); k_xdelta_planes_fast serves the other shapes.
#pragma once

#include <type_traits>
#include <utility>

#include "bulk.cuh"
#include "common.cuh"

namespace rspt {

constexpr int kTmaThreads = 128;
constexpr int kTmaQuads = 128;                   // sample quads per tile: 512 samples = one 512-byte step per channel and plane

template <class F, int... I>
__device__ __forceinline__ void static_for_impl(F&& f, std::integer_sequence<int, I...>)
{
    (f(std::integral_constant<int, I>{}), ...);
}
template <int N, class F>
__device__ __forceinline__ void static_for(F&& f)
{
    static_for_impl(f, std::make_integer_sequence<int, N>{});
}

// sign-extended sample whose BPS bytes start at the compile-time byte offset OFF of the word array w
template <int BPS, int OFF>
__device__ __forceinline__ uint32_t unpack_at(const uint32_t* w)
{
    constexpr int k = OFF / 4, s = OFF % 4;
    if constexpr (BPS == 4) {
        return w[k];
    } else if constexpr (BPS == 3) {
        if constexpr (s == 0) return prmt(w[k], w[k], 0xA210u);
        else if constexpr (s == 1) return prmt(w[k], w[k], 0xB321u);
        else if constexpr (s == 2) return prmt(w[k], w[k + 1], 0xC432u);
        else return prmt(w[k], w[k + 1], 0xD543u);
    } else {
        static_assert(BPS == 2, "unpack_at: 2, 3 or 4 bytes per sample");
        if constexpr (s == 0) return prmt(w[k], w[k], 0x9910u);
        else return prmt(w[k], w[k], 0xBB32u);
    }
}

// ------------------------------------------------------------------------------------------
// Forward sample transform, TMA-fed (default for the eligible shapes; k_xdelta_planes_fast for the others).
// One CTA (128 threads) per tile of 128 sample quads of one frame.  The raw tile (+ the quad in front of it, whose
// last two sample rows are the stencil's predecessors) arrives with ONE bulk asynchronous copy global -> shared,
// completion on an mbarrier; it lies UNPADDED in shared memory and thread t reads the whole quad t + 1 with 128-bit
// loads (lanes are 4 * ROW bytes apart: 144 bytes for 12 ch x 3 B, conflict-free for 128-bit accesses), so that all
// CH channels of its four samples are in registers at once: one PRMT per sample to unpack, the stencil, the 4 x 4
// byte transpose (8 PRMT), one 32-bit store per plane and channel (lanes run along the samples: coalesced).
// About 9 instructions per sample against 25 in k_xdelta_planes_fast (whose staging loop, padded layout and 32-bit
// shared-memory loads are gone).  Same bytes as k_xdelta_planes (tests: STREAM_CASES, test_transform_planes_bit_exact).
// ------------------------------------------------------------------------------------------
template <int BPS, int CH, bool STENCIL>
__global__ void __launch_bounds__(kTmaThreads, 4) k_xdelta_planes_tma(const uint8_t* __restrict__ src, Shape s, uint32_t tiles_per_frame,
                                                                        uint8_t* __restrict__ planes)
{
    constexpr int ROW = CH * BPS;          // bytes per sample row == words per quad
    constexpr int QB = 4 * ROW;            // bytes per quad
    constexpr int QW = ROW;                // words per quad
    constexpr int HSTART = (QW / 2) & ~3;  // first word of the 16-byte chunks that hold rows 2, 3 of a quad
    constexpr int HW = QW - HSTART;
    extern __shared__ __align__(128) uint8_t smem[];   // quads t*128 - 1 .. t*128 + 127, then the frame's last quad
    __shared__ __align__(8) uint64_t s_full;
    const uint32_t f = blockIdx.x / tiles_per_frame, t = blockIdx.x % tiles_per_frame, tid = threadIdx.x;
    const uint32_t nb = s.nb_alloc, ns = (uint32_t)s.ns, nq = ns >> 2;
    const uint8_t* frame = src + (size_t)f * s.frame_bytes;
    uint8_t* raw = smem;
    uint8_t* tail = smem + (size_t)(kTmaQuads + 1) * QB;
    if (tid == 0) {
        mbar_init(&s_full, 1);
        mbar_fence_init();
        if (t == 0) {
            mbar_arrive_expect_tx(&s_full, (uint32_t)(kTmaQuads * QB + (STENCIL ? QB : 0)));
            bulk_g2s(raw + QB, frame, (uint32_t)(kTmaQuads * QB), &s_full);
            if (STENCIL) bulk_g2s(tail, frame + (size_t)(nq - 1) * QB, (uint32_t)QB, &s_full);
        } else {
            mbar_arrive_expect_tx(&s_full, (uint32_t)((kTmaQuads + 1) * QB));
            bulk_g2s(raw, frame + ((size_t)t * kTmaQuads - 1) * QB, (uint32_t)((kTmaQuads + 1) * QB), &s_full);
        }
    }
    __syncthreads();   // the barrier is initialised before anyone waits on it
    mbar_wait(&s_full, 0);
    if (STENCIL && t == 0) {
        // the flat chain crosses channel rows (signal_packer_xdelta_hzr.cpp:55-57): the two predecessors of channel
        // c's first sample are the last two samples of channel c - 1 (zero for channel 0): rows 2, 3 of the halo quad
        for (uint32_t i = tid; i < 2u * ROW; i += kTmaThreads) {
            const uint32_t r = 2u + i / ROW, bb = i % ROW;
            raw[r * ROW + bb] = bb < (uint32_t)BPS ? (uint8_t)0 : tail[r * ROW + bb - BPS];
        }
        __syncthreads();
    }
    uint32_t w[QW];
    const uint4* q4 = reinterpret_cast<const uint4*>(raw + (size_t)(tid + 1) * QB);
#pragma unroll
    for (int i = 0; i < QW / 4; ++i) {
        const uint4 v = q4[i];
        w[4 * i] = v.x; w[4 * i + 1] = v.y; w[4 * i + 2] = v.z; w[4 * i + 3] = v.w;
    }
    uint32_t hw[STENCIL ? HW : 4];
    if (STENCIL) {
        const uint4* h4 = reinterpret_cast<const uint4*>(raw + (size_t)tid * QB + HSTART * 4);
#pragma unroll
        for (int i = 0; i < HW / 4; ++i) {
            const uint4 v = h4[i];
            hw[4 * i] = v.x; hw[4 * i + 1] = v.y; hw[4 * i + 2] = v.z; hw[4 * i + 3] = v.w;
        }
    }
    const bool first = t == 0 && tid == 0;
    const uint32_t ps = s.plane_stride >> 2;
    uint32_t* out0 = reinterpret_cast<uint32_t*>(planes + (size_t)f * nb * s.plane_stride) + (t * (uint32_t)kTmaQuads + tid);
    static_for<CH>([&](auto cc) {
        constexpr int c = decltype(cc)::value;
        uint32_t y[4];
        const uint32_t x0 = unpack_at<BPS, 0 * ROW + c * BPS>(w), x1 = unpack_at<BPS, 1 * ROW + c * BPS>(w);
        const uint32_t x2 = unpack_at<BPS, 2 * ROW + c * BPS>(w), x3 = unpack_at<BPS, 3 * ROW + c * BPS>(w);
        if constexpr (STENCIL) {
            constexpr int HB = (QW / 2 - HSTART) * 4;  // byte offset of row 2 inside hw
            const uint32_t xm2 = unpack_at<BPS, HB + c * BPS>(hw), xm1 = unpack_at<BPS, HB + ROW + c * BPS>(hw);
            uint32_t d0 = xm1 - xm2 - 128u;
            // the very first word of the frame has no predecessor delta: y[0] = x[0] - 128
            if (c == 0 && first) d0 = 0;
            const uint32_t d1 = x0 - xm1 - 128u, d2 = x1 - x0 - 128u, d3 = x2 - x1 - 128u, d4 = x3 - x2 - 128u;
            y[0] = d1 ^ d0; y[1] = d2 ^ d1; y[2] = d3 ^ d2; y[3] = d4 ^ d3;
        } else {
            y[0] = x0; y[1] = x1; y[2] = x2; y[3] = x3;
        }
        const uint32_t t01 = prmt(y[0], y[1], 0x5140u), t23 = prmt(y[2], y[3], 0x5140u);
        uint32_t* out = out0 + (size_t)c * (ns >> 2);
        out[0] = prmt(t01, t23, 0x5410u);
        if (nb > 1) out[ps] = prmt(t01, t23, 0x7632u);
        if (nb > 2) {
            const uint32_t u01 = prmt(y[0], y[1], 0x7362u), u23 = prmt(y[2], y[3], 0x7362u);
            out[2 * ps] = prmt(u01, u23, 0x5410u);
            if (nb > 3) out[3 * ps] = prmt(u01, u23, 0x7632u);
        }
    });
}

}  // namespace rspt
