// Shared definitions for the sm_100a signal-packer kernels.
//
// Vocabulary (follows the reference): a FRAME is one compress() call's input,
// [ns][ch][bps] interleaved little-endian samples; its N = ch*ns sample words are split into
// `nb` byte PLANES (signal_packer_base.cpp:40-68); each plane is an hzr stream cut into BLOCKS
// of <= 65536 bytes (hzr_encode.c:528-539).  Inside a block a warp processes a STEP of 512 bytes
// at a time, 16 bytes per lane.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace rspt {

constexpr int kNumSymbols = 261;       // hzr_internal.h:114
constexpr int kSymStride = 264;        // padded row for per-block tables
constexpr int kTreeWords = 92;         // >= ceil((11*261-1)/32)
constexpr uint32_t kBlock = 65536;     // HZR_MAX_BLOCK_SIZE, hzr_internal.h:109
constexpr uint32_t kRunCap = 16662;    // hzr_encode.c:149
// Decode index (out of band, never part of the stream): 32-bit entries, one per INTERVAL of a HUFF block's
// payload bits.  The interval length follows from the payload length alone (both sides know it): 512 bits,
// or as many as it takes to cut the payload into at most 512 intervals -- one decoder thread each, so a
// full-size block keeps a whole CTA busy and a sparse block gets a handful of short intervals.  Entry k
// names a token boundary at or shortly after bit k * interval:
//   bits 0..11  start bit of that token minus k * interval     bits 12..  output byte the token starts at
// A decoder thread takes the tokens from its entry's boundary up to the next entry's.  The entries of a
// block sit at slot (payload byte offset in the batch's stream >> 6) + block ordinal + k, so the index of
// a batch lies in a prefix of the sidecar buffer whose length follows the compressed size.
constexpr uint32_t kIdxMinBits = 512;
constexpr uint32_t kIdxPosShift = 12;
constexpr int kMaxSegs = 512;             // intervals per block at most: one decoder thread each
struct IdxGeom {
    uint32_t bits;   // interval length
    uint32_t inv;    // ceil(2^32 / bits): x / bits == __umulhi(x, inv) for x < 2^19
    uint32_t n;      // intervals of the block
};
__host__ __device__ __forceinline__ IdxGeom idx_geom(uint32_t payload_len)
{
    IdxGeom g;
    const uint32_t total = payload_len * 8u;
    g.bits = (total + (uint32_t)kMaxSegs - 1u) / (uint32_t)kMaxSegs;
    if (g.bits < kIdxMinBits) g.bits = kIdxMinBits;
    g.inv = 0xFFFFFFFFu / g.bits + 1u;
    g.n = (total + g.bits - 1u) / g.bits;
    return g;
}
__device__ __forceinline__ uint32_t idx_interval_of(const IdxGeom& g, uint32_t bit) { return __umulhi(bit, g.inv); }
__host__ __device__ __forceinline__ size_t idx_slot_base(unsigned long long payload_rel, uint32_t blk)
{
    return (size_t)(payload_rel >> 6) + blk;
}

enum : uint32_t { MODE_COPY = 0, MODE_HUFF = 1, MODE_FILL = 2 };  // hzr_internal.h:98-101

// Per-block plan written by the tree kernel and consumed by layout + encode.
struct BlkInfo {
    uint32_t payload_len;  // bytes after the 7-byte block header
    uint32_t total_bits;   // tree bits + token bits (HUFF)
    uint16_t tree_nbits;
    uint8_t mode;
    uint8_t fill;
    uint16_t n_used;       // symbols with a non-zero count
    uint16_t n_tokens;     // tokens of the block, saturated at 65535 (selects the encoder path)
};

constexpr uint32_t kNoList = 0xFFFFFFFFu;           // list_n value of a block that has no sparse list
// which encoder writes a block: the list-based one iff there is a list, the block is HUFF and its payload
// fits that kernel's staging; both encoders evaluate this same predicate, so they need no hand-shake
__device__ __forceinline__ bool sparse_block_is_packed_from_list(uint32_t list_m, const BlkInfo& bi, uint32_t stage_bytes)
{
    return list_m != kNoList && bi.mode == MODE_HUFF && bi.payload_len <= stage_bytes;
}

struct Shape {
    int kind;
    int bps, ch, ns;
    uint32_t N;             // ch * ns
    uint32_t nblk;          // hzr blocks per plane
    uint32_t nb_init;       // planes the instance starts with
    uint32_t nb_alloc;      // planes reserved per frame in scratch (max reachable)
    uint32_t hdr_bytes;     // 3*ch for hadamard/dct
    uint32_t plane_stride;  // N rounded up to 16
    uint32_t frame_bytes;   // bps * N
    uint32_t method;        // frame method byte (0 hzr/xdelta, 1 dct, 2 hadamard)
};

__host__ __device__ __forceinline__ uint32_t blk_len(const Shape& s, uint32_t b)
{
    uint32_t off = b * kBlock;
    return s.N - off < kBlock ? s.N - off : kBlock;
}

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31; }
__device__ __forceinline__ uint32_t warp_id() { return threadIdx.x >> 5; }

// Shared-memory accesses through a 32-bit shared-window address taken once (__cvta_generic_to_shared).
// ptxas otherwise re-derives the address of a __shared__ array at every use inside a loop whose
// registers are tight (S2R SR_CgaCtaId + MOV + LEA in front of each LDS / ATOMS on sm_100).
__device__ __forceinline__ uint32_t smem_addr(const void* p)
{
    uint32_t a = (uint32_t)__cvta_generic_to_shared(p);
    asm volatile("" : "+r"(a));  // opaque, so that the address stays in its register instead of being re-derived
    return a;
}
__device__ __forceinline__ uint32_t lds_u16(uint32_t a)
{
    uint32_t v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t a)
{
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel)
{
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
    return d;
}
__device__ __forceinline__ void reds_or(uint32_t a, uint32_t v) { asm volatile("red.shared.or.b32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }

// double -> int32 as the reference's x86-64 build does it (cvttsd2si): toward zero, and the
// "integer indefinite" 0x80000000 for NaN and for values outside the int32 range (CUDA's own
// conversion would saturate instead).
__device__ __forceinline__ int32_t to_i32_x86(double v)
{
    return (v >= 2147483648.0 || v <= -2147483649.0 || v != v) ? (int32_t)0x80000000 : (int32_t)v;
}

// Extra bits carried by the zero-run symbols 256..260 (hzr_internal.h:117-121).
__device__ __forceinline__ uint32_t sym_extra_bits(uint32_t sym)
{
    // 256:0 257:2 258:4 259:8 260:14
    return sym < 257 ? 0u : (sym == 257 ? 2u : (sym == 258 ? 4u : (sym == 259 ? 8u : 14u)));
}

// Classify a zero-run chunk z in [1, 16662] -> (symbol, extra value, extra bits); hzr_encode.c:152-166.
// Branch-free: class index 0..5 for 1 | 2 | 3-6 | 7-22 | 23-278 | 279-16662.
__device__ __forceinline__ void run_token(uint32_t z, uint32_t& sym, uint32_t& ev, uint32_t& eb)
{
    const uint32_t idx = (z >= 2u) + (z >= 3u) + (z >= 7u) + (z >= 23u) + (z >= 279u);
    sym = idx ? 255u + idx : 0u;
    eb = (0xE84200u >> (4u * idx)) & 0xFu;                      // 0 0 2 4 8 14
    const uint32_t base = idx == 5u ? 279u : (0x17070300u >> (8u * (idx < 2u ? 0u : idx - 1u))) & 0xFFu;  // 3 7 23
    ev = idx < 2u ? 0u : z - base;
}

// ---- zero runs ---------------------------------------------------------------------------
// Tokens of one maximal zero run of z bytes inside a block: greedy chunks of <= 16662
// (hzr_encode.c:146-166 and :415-452); every chunk goes to sink.token(symbol, extra, extra bits).
template <class Sink>
__device__ __forceinline__ void emit_run(uint32_t z, Sink& sink)
{
    while (z > kRunCap) {
        sink.token(260u, kRunCap - 279u, 14u);
        z -= kRunCap;
    }
    uint32_t sym, ev, eb;
    run_token(z, sym, ev, eb);
    sink.token(sym, ev, eb);
}

#define RSPT_CUDA_CHECK(call)                                      \
    do {                                                           \
        cudaError_t e_ = (call);                                   \
        if (e_ != cudaSuccess) return rspt::fail_cuda(p, e_, #call); \
    } while (0)

}  // namespace rspt
