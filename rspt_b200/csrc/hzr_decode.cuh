// hzr decoder for sm_100a.  Replaces decompress_i32's chunk walk
// (lib_signalpacker/signal_packer_base.cpp:98-121) and lib_hzr/hzr_decode.c (hzr_decode :626-674,
// DecodeSingleBlock :335-567, RecoverTree :263-333).  Like the reference, the block CRC is not
// checked on decode (hzr_decode.c:343).
//
// Parallelism: frames and hzr blocks are located by a cheap header walk (one thread per frame);
// the code table of every HUFF block is recovered from the tree bits in its payload (one warp per
// block, k_hzr_recover_codes); each block is decoded by one CTA.  Inside a block the token stream
// has no sync points, so the decoder is seeded from the out-of-band decode index (common.cuh: one
// token boundary and its output position per 1024 payload bits; rspt_gpu_compress_batch's
// d_sidecar) and every thread decodes the tokens between two boundaries through a 12-bit look-up
// table.  Streams without an index (produced by the CPU reference) get one from
// k_hzr_build_index first.
#pragma once

#include <type_traits>

#include "bulk.cuh"
#include "common.cuh"
#include "hzr_encode.cuh"

namespace rspt {

constexpr int kDecodeThreads = kMaxSegs;  // one thread per decode segment
// decode classes: HUFF payloads up to kSmallPayload / kMediumPayload bytes are decoded by CTAs with one thread per
// index interval of the largest such payload; class 0 takes everything else (longer payloads, COPY / FILL blocks)
constexpr uint32_t kSmallPayload = 4096, kMediumPayload = 16384;
__host__ __device__ constexpr int decode_class_threads(uint32_t payload) { return (int)(payload * 8 / kIdxMinBits); }
__host__ __device__ constexpr size_t decode_class_smem(uint32_t payload) { return payload + 64; }
constexpr int kLutBits = 12;
constexpr int kPairBits = 11;  // index width of the pair table (32-bit entries in the same 8 KB)
constexpr uint32_t kModeZero = 3;      // frame failed to parse: emit zeros
constexpr uint32_t kModeInactive = 255;

struct DecBlk {
    unsigned long long payload_off;  // byte offset of the payload in the stream buffer
    uint32_t payload_len;
    uint32_t out_n;
    uint32_t mode;
    uint32_t pad;
};

__device__ __forceinline__ uint32_t decode_class(const DecBlk& d)
{
    if (d.mode != MODE_HUFF) return 0u;
    return d.payload_len <= kSmallPayload ? 1u : (d.payload_len <= kMediumPayload ? 2u : 0u);
}

__device__ __forceinline__ uint32_t ld_le32(const uint8_t* p)
{
    return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
}

// one thread per frame: method byte, header, nb chunks, block headers
__global__ void __launch_bounds__(128) k_frame_parse(const uint8_t* __restrict__ src, const uint64_t* __restrict__ offsets,
                                                      Shape s, const uint8_t* __restrict__ frame_nb_in,
                                                      const uint32_t* __restrict__ nb_state, uint32_t n_frames,
                                                      DecBlk* __restrict__ dec, uint8_t* __restrict__ headers,
                                                      uint8_t* __restrict__ dec_nb, int32_t* __restrict__ status,
                                                      Counters* __restrict__ ctr)
{
    const uint32_t f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f == 0) atomicAdd(&ctr->frames_decompressed, (unsigned long long)n_frames);
    if (f >= n_frames) return;
    const unsigned long long base = offsets[f], end = offsets[f + 1];
    uint32_t nb = frame_nb_in ? frame_nb_in[f] : *nb_state;
    int err = 0;
    if (nb < 1 || nb > s.nb_alloc) {
        err = 1;
        nb = nb < 1 ? 1 : s.nb_alloc;
    }
    unsigned long long pos = base;
    if (end < base + 1 + s.hdr_bytes) err = 1;
    if (!err) {
        // "ERROR: compression method unsupported." in the reference (e.g. xdelta.cpp:78-79)
        if (src[pos] != s.method) err = 1;
        ++pos;
        for (uint32_t i = 0; i < s.hdr_bytes; ++i) headers[(size_t)f * s.hdr_bytes + i] = src[pos + i];
        pos += s.hdr_bytes;
    }
    DecBlk* row = dec + (size_t)f * s.nb_alloc * s.nblk;
    for (uint32_t k = 0; k < s.nb_alloc; ++k) {
        for (uint32_t b = 0; b < s.nblk; ++b) {
            DecBlk d;
            d.payload_off = 0; d.payload_len = 0; d.out_n = blk_len(s, b); d.pad = 0;
            d.mode = k < nb ? kModeZero : kModeInactive;
            row[k * s.nblk + b] = d;
        }
    }
    for (uint32_t k = 0; k < nb && !err; ++k) {
        if (pos + 8 > end) { err = 1; break; }
        const uint32_t len = ld_le32(src + pos);            // chunk length (base.cpp:103)
        const unsigned long long cend = pos + 4 + len;
        if (cend > end || len < 4) { err = 1; break; }
        if (ld_le32(src + pos + 4) != s.N) { err = 1; break; }  // hzr master header (dec:644)
        unsigned long long q = pos + 8;
        for (uint32_t b = 0; b < s.nblk; ++b) {
            if (q + 7 > cend) { err = 1; break; }
            const uint32_t plen = ((uint32_t)src[q] | ((uint32_t)src[q + 1] << 8)) + 1u;  // dec:342
            const uint32_t mode = src[q + 6];
            if (mode > MODE_FILL || q + 7 + plen > cend) { err = 1; break; }
            // A legitimate block stream is capped at header + in_size (hzr_encode.c:377-382), COPY carries
            // exactly the block (:307-339) and FILL one byte (:352-364).  Anything else is rejected here:
            // the decode / index / verify kernels stage payload_len bytes in shared memory sized for the
            // largest legitimate payload.
            const uint32_t bl = blk_len(s, b);
            if ((mode == MODE_HUFF && plen > bl) || (mode == MODE_COPY && plen != bl) || (mode == MODE_FILL && plen != 1u)) { err = 1; break; }
            DecBlk& d = row[k * s.nblk + b];
            d.payload_off = q + 7;
            d.payload_len = plen;
            d.mode = mode;
            q += 7 + plen;
        }
        if (!err && q != cend) err = 1;
        pos = cend;
    }
    if (!err && pos != end) err = 1;
    if (err) {
        for (uint32_t k = 0; k < nb; ++k)
            for (uint32_t b = 0; b < s.nblk; ++b) row[k * s.nblk + b].mode = kModeZero;
    }
    dec_nb[f] = (uint8_t)nb;
    status[f] = err ? -4 : 0;
}

// sequential bit reader over the payload staged in shared memory (word 0 = payload bytes 0..3),
// LSB-first, 32-bit refills into a 64-bit window
struct BitReader {
    const uint32_t* words;
    uint32_t widx;
    unsigned long long buf;
    uint32_t cnt;
    __device__ __forceinline__ void init(const uint32_t* pay_words, uint32_t bitpos)
    {
        words = pay_words;
        widx = bitpos >> 5;
        buf = (unsigned long long)words[widx] | ((unsigned long long)words[widx + 1] << 32);
        widx += 2;
        const uint32_t drop = bitpos & 31u;
        buf >>= drop;
        cnt = 64u - drop;
    }
    __device__ __forceinline__ void refill()
    {
        if (cnt <= 32u) {
            buf |= (unsigned long long)words[widx] << cnt;
            cnt += 32u;
            ++widx;
        }
    }
    __device__ __forceinline__ uint32_t peek(uint32_t n) const { return (uint32_t)buf & ((1u << n) - 1u); }
    __device__ __forceinline__ void skip(uint32_t n)
    {
        buf >>= n;
        cnt -= n;
    }
    __device__ __forceinline__ uint32_t take(uint32_t n)
    {
        const uint32_t v = peek(n);
        skip(n);
        return v;
    }
};

constexpr uint32_t kDecPayWords = kBlock / 4 + 16;  // cap of the payload staging: 16-byte chunks at any alignment + slack
constexpr size_t kDecodeSmem = (size_t)kDecPayWords * 4;
constexpr uint32_t kLongFlag = 0x8000u;
constexpr uint32_t kLongEnd = 0x1FFu;  // flagged table entries: index of the first long symbol of the chain, kLongEnd = none

// RecoverTree (dec:263-333) by ONE thread: the tree bits are pre-order, 0 = branch, 1 + 9-bit symbol =
// leaf, and only the code word of every leaf is needed.  One step per LEAF: the zeros in front of a leaf
// are that many descents to the left; after a leaf the walk resumes at the right child of the deepest
// ancestor that was entered to the left, which is the highest zero bit of the path (code words are
// LSB-first: bit i of the code is the turn taken at depth i).  cw[sym] = code | len << 27 (must be
// zeroed by the caller; global or shared memory).  `words` / `bit0`: the word that holds the tree's first bit and
// that bit's position in it.  Returns the number of tree bits (11 per leaf - 1), or 0xFFFFFFFF on a malformed tree.
__device__ __forceinline__ uint32_t recover_tree(const uint32_t* words, uint32_t bit0, uint32_t plen, uint32_t* cw)
{
    BitReader r;
    r.init(words, bit0);
    uint32_t leaves = 0, bits_used = 0, code = 0, depth = 0;
    const uint32_t limit = plen * 8u;
    for (;;) {
        r.refill();
        const uint32_t w = (uint32_t)r.buf;
        if (w == 0u) return 0xFFFFFFFFu;                  // 32 branches in a row: deeper than any code word
        const uint32_t z = (uint32_t)__ffs(w) - 1u;
        depth += z;
        if (depth > 27u) return 0xFFFFFFFFu;
        r.skip(z + 1u);
        r.refill();
        const uint32_t sym = r.take(9);
        bits_used += z + 10u;
        if (bits_used > limit || sym >= (uint32_t)kNumSymbols || leaves >= (uint32_t)kNumSymbols) return 0xFFFFFFFFu;
        cw[sym] = code | (max(depth, 1u) << 27);          // lone leaf: 1-bit code (dec:306 `hzr_max(bits, 1)`)
        ++leaves;
        const uint32_t m = ~code & ((1u << depth) - 1u);  // levels entered to the left
        if (m == 0u) break;                               // the tree is complete
        const uint32_t i = 31u - (uint32_t)__clz((int)m);
        code = (code & ((1u << i) - 1u)) | (1u << i);
        depth = i + 1u;
    }
    return bits_used;
}

// One THREAD per block: the code table of every HUFF block from its in-stream tree, read straight from the
// stream (k_hzr_decode and k_hzr_build_index read the tables from `codes`, which the host zeroes beforehand).
// The walk is serial and latency-bound; with a thread per block a whole batch is in flight at once (a warp
// takes as long as its block with the most leaves).  status[f] = -4 on a malformed tree; the block then
// decodes to zeros.  A symbol named by two leaves keeps the later code (no memory safety issue: the table is
// only ever indexed by symbol).
constexpr int kRecoverThreads = 64;
__global__ void __launch_bounds__(kRecoverThreads) k_hzr_recover_codes(const uint8_t* __restrict__ src, uint32_t total_blocks,
                                                                       DecBlk* __restrict__ dec, uint32_t* __restrict__ codes,
                                                                       Shape s, int32_t* __restrict__ status)
{
    const uint32_t blk = blockIdx.x * kRecoverThreads + threadIdx.x;
    if (blk >= total_blocks) return;
    const DecBlk d = dec[blk];
    if (d.mode != MODE_HUFF) return;
    const uintptr_t pa = (uintptr_t)(src + d.payload_off);
    const uint32_t tb = recover_tree(reinterpret_cast<const uint32_t*>(pa & ~(uintptr_t)3), (uint32_t)(pa & 3u) * 8u, d.payload_len,
                                     codes + (size_t)blk * kSymStride);
    if (tb == 0xFFFFFFFFu) {
        uint32_t f, k, b;
        blk_decode(s, blk, f, k, b);
        status[f] = -4;
        dec[blk].mode = kModeZero;
    }
}

// look-up table on the next kLutBits bits (whole CTA): a warp per symbol, lanes over the
// 2^(12 - len) entries that end in its code; symbols with longer codes go to the list `longs`
// (*nlong must be 0 on entry).  The caller initialises lut to kLongFlag and synchronises after.
template <class T, int BITS = kLutBits>
__device__ __forceinline__ void build_lut(const uint32_t* cw_tab, T* lut, uint16_t* longs, uint32_t* nlong)
{
    const uint32_t lane = lane_id();
    // A symbol's entries lie 2^len apart.  Short codes (len <= 5, at most 32 of them): a warp per symbol, lanes over
    // the entries (neighbouring lanes are <= 64 bytes apart: at most two per bank).  Longer codes would put all 32
    // lanes into ONE bank that way (entries >= 128 bytes apart), so they get a thread per symbol instead: the 32
    // lanes then write into 32 unrelated places, and neighbouring symbols have similar lengths (<= 64 entries each).
    for (uint32_t sym = warp_id(); sym < (uint32_t)kNumSymbols; sym += (blockDim.x >> 5)) {
        const uint32_t cw = cw_tab[sym];
        const uint32_t len = cw >> 27, code = cw & 0x07FFFFFFu;
        if (cw == 0u || len > 5u) continue;
        const T e = (T)(sym | (len << 9));
        for (uint32_t i = lane; i < (1u << (BITS - len)); i += 32) lut[(i << len) | code] = e;
    }
    for (uint32_t sym = threadIdx.x; sym < (uint32_t)kNumSymbols; sym += blockDim.x) {
        const uint32_t cw = cw_tab[sym];
        const uint32_t len = cw >> 27, code = cw & 0x07FFFFFFu;
        if (cw == 0u || len <= 5u) continue;
        if (len <= (uint32_t)BITS) {
            const T e = (T)(sym | (len << 9));
            for (uint32_t i = 0; i < (1u << (BITS - len)); ++i) lut[(i << len) | code] = e;
        } else {
            longs[atomicAdd(nlong, 1u)] = (uint16_t)sym;
        }
    }
}

// Long codes: the table entry of their first kLutBits bits (kLongFlag | index) heads a chain through
// `next` of the long symbols that share those bits, so a long code costs a compare or two instead of
// a scan of all long symbols (a lane on this path stalls its whole warp).  Whole CTA; the table must have
// been initialised to kLongFlag | kLongEnd; synchronise after.
template <class T, int BITS = kLutBits>
__device__ __forceinline__ void chain_long_codes(const uint32_t* cw_tab, T* lut, const uint16_t* longs, uint16_t* next,
                                                 uint32_t nlong)
{
    for (uint32_t j = threadIdx.x; j < nlong; j += blockDim.x) {
        const uint32_t prefix = cw_tab[longs[j]] & ((1u << BITS) - 1u);
        if (sizeof(T) == 4) {  // 32-bit entries: one exchange
            next[j] = (uint16_t)(atomicExch(reinterpret_cast<uint32_t*>(lut) + prefix, kLongFlag | j) & kLongEnd);
            continue;
        }
        uint32_t* word = reinterpret_cast<uint32_t*>(lut) + (prefix >> 1);
        const uint32_t shift = (prefix & 1u) * 16u;
        uint32_t old = *word, seen;
        do {
            seen = old;
            old = atomicCAS(word, seen, (seen & ~(0xFFFFu << shift)) | ((kLongFlag | j) << shift));
        } while (old != seen);
        next[j] = (uint16_t)((seen >> shift) & kLongEnd);
    }
}

// One CTA per hzr block.  The payload is staged in shared memory with ONE bulk asynchronous copy (the
// 16-byte chunks of the stream that hold it, unshifted; the bit reader starts 8 * (address mod 16) bits
// later) that lands while the tables are built; the code table comes from k_hzr_recover_codes; a 12-bit
// look-up table maps the next bits to (symbol, length), longer codes are matched against the short list
// of long code words.  Thread k decodes the tokens between the k-th and the (k + 1)-th boundary of the
// decode index (common.cuh) and writes the bytes they produce.
__global__ void __launch_bounds__(kDecodeThreads, 3) k_hzr_decode(const uint8_t* __restrict__ src, Shape s,
                                                                   const DecBlk* __restrict__ dec,
                                                                   const uint64_t* __restrict__ offsets,
                                                                   const uint32_t* __restrict__ sidecar,
                                                                   const uint32_t* __restrict__ codes,
                                                                   uint8_t* __restrict__ planes, int32_t* __restrict__ status,
                                                                   uint32_t pair_max_bits, uint32_t small_class)
{
    extern __shared__ __align__(16) uint32_t payw[];  // payload words (+ zero slack)
    // 8 KB of look-up table in one of two shapes, chosen per block:
    //   kLutBits bits -> 16-bit entries: sym | len << 9, or kLongFlag | chain head
    //   kPairBits bits -> 32-bit entries: the same in the low half; high half: a second literal whose whole
    //   code the same bits also hold -- bit 31, both lengths << 24, its byte << 16
    __shared__ __align__(16) uint16_t s_lut[1 << kLutBits];
    uint32_t* s_lut32 = reinterpret_cast<uint32_t*>(s_lut);
    __shared__ uint32_t s_cw[kSymStride];            // code | len << 27 per symbol, 0 = unused
    __shared__ uint16_t s_long[kSymStride];          // symbols whose code is longer than the table
    __shared__ uint16_t s_next[kSymStride];          // chains of the long symbols that share their first kLutBits bits
    __shared__ uint32_t s_meta[4];                   // -, error, long count
    __shared__ __align__(8) uint64_t s_bar;

    const uint32_t blk = blockIdx.x, tid = threadIdx.x;
    const DecBlk d = dec[blk];
    if (d.mode == kModeInactive) return;
    // three launches share the blocks by payload size (decode_class): a CTA has as many threads as its class has
    // index intervals and stages no more than its class's payload, so that short payloads (the sparse planes: a
    // handful of busy threads) and half-size blocks do not hold a full-size CTA's shared memory
    if (decode_class(d) != small_class) return;
    uint32_t f, k, b;
    blk_decode(s, blk, f, k, b);
    uint8_t* out = planes + ((size_t)f * s.nb_alloc + k) * s.plane_stride + (size_t)b * kBlock;
    uint4* out4 = reinterpret_cast<uint4*>(out);
    const uint32_t n = d.out_n, nq = (n + 15u) >> 4;
    const uint8_t* pay = src + d.payload_off;

    if (d.mode == MODE_FILL || d.mode == kModeZero) {
        const uint32_t v = d.mode == MODE_FILL ? pay[0] * 0x01010101u : 0u;  // memset (dec:362-370)
        for (uint32_t i = tid; i < nq; i += blockDim.x) out4[i] = make_uint4(v, v, v, v);
        return;
    }
    const uintptr_t pa = (uintptr_t)pay;
    if (d.mode == MODE_COPY) {
        if (d.payload_len != n) {  // "Encoded / decoded size mismatch (COPY)" dec:351-355
            if (tid == 0) status[f] = -4;
            for (uint32_t i = tid; i < nq; i += blockDim.x) out4[i] = make_uint4(0, 0, 0, 0);
            return;
        }
        const uint32_t* aw = reinterpret_cast<const uint32_t*>(pa & ~(uintptr_t)3);
        const uint32_t lead = (uint32_t)(pa & 3u), sh = lead * 8u;
        const uint32_t naw = (lead + n + 3u) >> 2, nw = (n + 3u) >> 2;
        uint32_t* out32 = reinterpret_cast<uint32_t*>(out);
        for (uint32_t i = tid; i < nw; i += blockDim.x) {
            const uint32_t lo = __ldg(aw + i), hi = (i + 1 < naw) ? __ldg(aw + i + 1) : 0u;
            out32[i] = __funnelshift_r(lo, hi, sh);
        }
        return;
    }

    // ---- MODE_HUFF
    const uint32_t plen = d.payload_len;   // <= n (k_frame_parse), so it fits the staging sized for the largest block
    const uint32_t lead16 = (uint32_t)(pa & 15u), n16 = (lead16 + plen + 15u) >> 4;
    if (tid == 0) {
        mbar_init(&s_bar, 1);
        mbar_fence_init();
        mbar_arrive_expect_tx(&s_bar, 16u * n16);
        bulk_g2s(payw, reinterpret_cast<const void*>(pa & ~(uintptr_t)15), 16u * n16, &s_bar);
        s_meta[0] = 0; s_meta[1] = 0; s_meta[2] = 0;
    }
    // Pairs are worth it where codes are short and tokens many (1/2 .. pair_max_bits payload bits per output byte):
    // quantised coefficient planes, smooth upper planes.  Sparse blocks would only pay for the extra pass, and
    // planes with ~6-bit codes rarely hold two codes in the window and want the longer single-symbol table.
    // pair_max_bits bit 8: after a pair, look up once more in the same window (hzr decode 1.95 -> 1.80 ms per 4096 frames;
    // on the coefficient planes of hadamard and dct, where single literals sit between short runs, it costs 4 %)
    const bool chain_pairs = (pair_max_bits >> 8) & 1u;
    const bool use_pairs = plen * 16u >= d.out_n && plen * 8u <= (pair_max_bits & 255u) * d.out_n;
    for (uint32_t i = tid; i < kSymStride; i += blockDim.x) s_cw[i] = i < (uint32_t)kNumSymbols ? codes[(size_t)blk * kSymStride + i] : 0u;
    if (!use_pairs) {
        for (uint32_t i = tid; i < (1u << kLutBits) / 2; i += blockDim.x) s_lut32[i] = (kLongFlag | kLongEnd) * 0x00010001u;
        __syncthreads();
        build_lut(s_cw, s_lut, s_long, &s_meta[2]);
        __syncthreads();
        chain_long_codes(s_cw, s_lut, s_long, s_next, s_meta[2]);
    } else {
        for (uint32_t i = tid; i < (1u << kPairBits); i += blockDim.x) s_lut32[i] = kLongFlag | kLongEnd;
        __syncthreads();
        build_lut<uint32_t, kPairBits>(s_cw, s_lut32, s_long, &s_meta[2]);
        __syncthreads();
        chain_long_codes<uint32_t, kPairBits>(s_cw, s_lut32, s_long, s_next, s_meta[2]);
        __syncthreads();
        // pair pass: only the high half of an entry changes, so the look-ups of the other threads into the
        // low halves stay valid while it runs
        for (uint32_t i = tid; i < (1u << kPairBits); i += blockDim.x) {
            const uint32_t e1 = s_lut32[i], len1 = (e1 >> 9) & 15u;
            if (!(e1 & kLongFlag) && (e1 & 511u) < 256u && len1 < (uint32_t)kPairBits) {
                const uint32_t e2 = s_lut32[i >> len1] & 0xFFFFu, len2 = (e2 >> 9) & 15u;
                if (!(e2 & kLongFlag) && (e2 & 511u) < 256u && len1 + len2 <= (uint32_t)kPairBits)
                    s_lut32[i] = e1 | 0x80000000u | ((len1 + len2) << 24) | ((e2 & 255u) << 16);
            }
        }
    }
    // The whole output block is cleared first (coalesced 128-bit stores that the L2 merges with the word
    // stores below), so a zero run only advances the write position and the token loop is the same
    // straight-line code for literals and runs.
    for (uint32_t i = tid; i < nq; i += blockDim.x) out4[i] = make_uint4(0, 0, 0, 0);
    __syncthreads();
    mbar_wait(&s_bar, 0);
    // the bit reader looks two words past the payload: keep what follows it in the stream out of the window
    if (tid < 8u) {
        const uint32_t endb = lead16 + plen;                      // first byte behind the payload
        uint8_t* pb = reinterpret_cast<uint8_t*>(payw);
        if (tid == 0)
            for (uint32_t i = endb; i < 16u * n16; ++i) pb[i] = 0;
        payw[4u * n16 + tid] = 0u;
    }
    __syncthreads();

    const IdxGeom ig = idx_geom(plen);
    const uint32_t limit = plen * 8u, nint = ig.n;
    const uint32_t* my_idx = sidecar + idx_slot_base(d.payload_off - offsets[0], blk);
    uint32_t my_err = 0;
    if (tid < nint) {
        const uint32_t e0 = my_idx[tid];
        uint32_t bitpos = tid * ig.bits + (e0 & ((1u << kIdxPosShift) - 1u)), pos = e0 >> kIdxPosShift;
        uint32_t end_bit = limit;
        if (tid + 1 < nint) end_bit = min(limit, (tid + 1u) * ig.bits + (my_idx[tid + 1] & ((1u << kIdxPosShift) - 1u)));
        if (bitpos > limit || pos > n) { my_err = 1; bitpos = end_bit; }   // an index that does not belong to this stream
        if (bitpos < end_bit && pos < n) {
            // the thread's bytes are gathered into the open word w (bytes of the word at and beyond pos are
            // zero); a word goes out when the position leaves it, unless it is empty.  The first word may be
            // shared with the thread before (it is OR-ed in), and so may the last one.
            const uint32_t first_w = (pos & 3u) ? pos >> 2 : 0xFFFFFFFFu;
            uint32_t w = 0;
            // The reader keeps no window between tokens: the 32 bits at the bit position are fetched anew for
            // every token (two LDS and one funnel shift, no refill branch, no 64-bit state).  bp counts from
            // the start of the staging (payload bit 0 is bit 8 * lead16).
            const uint32_t lut_s = smem_addr(s_lut), pay_s = smem_addr(payw), cw_s = smem_addr(s_cw);
            const uint32_t base_bits = 8u * lead16;
            uint32_t bp = bitpos + base_bits;
            const uint32_t end_bp = end_bit + base_bits;
            auto window = [&](uint32_t at) {
                const uint32_t a = pay_s + ((at >> 3) & ~3u);
                return __funnelshift_r(lds_u32(a), lds_u32(a + 4u), at);   // the shift uses the low 5 bits of `at`
            };
            auto token_loop = [&](auto pairs_t, auto chain_t) {
            // PAIRS: pair table; CHAIN: further look-ups into the same window (pair table: one more after a pair;
            // single-symbol table: up to three more literals)
            constexpr bool PAIRS = decltype(pairs_t)::value, CHAIN = decltype(chain_t)::value;
            while (bp < end_bp && pos < n) {
                uint32_t win = window(bp);
                uint32_t e = PAIRS ? lds_u32(lut_s + 4u * (win & ((1u << kPairBits) - 1u))) : lds_u16(lut_s + 2u * (win & ((1u << kLutBits) - 1u)));
                if (e & kLongFlag) {
                    // code longer than the table: match the few long code words (dec:418-431 walks the tree)
                    uint32_t j = e & kLongEnd;
                    e = 0;
                    while (j != kLongEnd) {
                        const uint32_t sym = s_long[j], cw = lds_u32(cw_s + 4u * sym), len = cw >> 27;
                        if ((win & ((1u << len) - 1u)) == (cw & 0x07FFFFFFu)) {
                            e = sym | 0x10000u;
                            bp += len;
                            break;
                        }
                        j = s_next[j];
                    }
                    if (e == 0u) { my_err = 1; break; }
                    // consumed here (length field 0 below); the window is taken again so that the extra bits of a run are in it
                    e &= 511u;
                    win = window(bp);
                }
                // two literals at once when both belong to this thread: with the pair table the entry has them;
                // with the single-symbol table the second one comes from a second look-up into the same
                // window (<= kLutBits bits are gone, >= 20 are left)
                bool two = PAIRS && (e >> 31) != 0u && pos + 2u <= n && bp + ((e >> 24) & 15u) <= end_bp;
                uint32_t len = (two ? e >> 24 : e >> 9) & 15u, more = 0u;
                const uint32_t sym = e & 511u;
                uint32_t val = two ? sym | ((e >> 8) & 0xFF00u) : sym;  // the literal byte(s)
                const bool run = sym >= 256u;  // symbol 0 (a zero run of one) is handled as a literal
                if (!PAIRS && CHAIN && !run) {
                    // up to three more literals from the same window, as long as kLutBits unread bits are left in it
                    const uint32_t e2 = lds_u16(lut_s + 2u * ((win >> len) & ((1u << kLutBits) - 1u)));
                    const uint32_t len2 = len + (e2 >> 9);
                    if (!(e2 & (kLongFlag | 0x100u)) && pos + 2u <= n && bp + len2 <= end_bp) {
                        two = true;
                        len = len2;
                        val |= (e2 & 255u) << 8;
                        if (len <= 32u - kLutBits) {
                            const uint32_t e3 = lds_u16(lut_s + 2u * ((win >> len) & ((1u << kLutBits) - 1u)));
                            const uint32_t len3 = len + (e3 >> 9);
                            if (!(e3 & (kLongFlag | 0x100u)) && pos + 3u <= n && bp + len3 <= end_bp) {
                                more = 1u;
                                len = len3;
                                val |= (e3 & 255u) << 16;
                                if (len <= 32u - kLutBits) {
                                    const uint32_t e4 = lds_u16(lut_s + 2u * ((win >> len) & ((1u << kLutBits) - 1u)));
                                    const uint32_t len4 = len + (e4 >> 9);
                                    if (!(e4 & (kLongFlag | 0x100u)) && pos + 4u <= n && bp + len4 <= end_bp) {
                                        more = 2u;
                                        len = len4;
                                        val |= e4 << 24;
                                    }
                                }
                            }
                        }
                    }
                }
                if (PAIRS && CHAIN && two) {
                    // (planes of plain samples) a pair is usually inside a burst of literals: one more look-up into the same window
                    // (<= 11 bits are gone) for a third and fourth byte
                    const uint32_t e2 = lds_u32(lut_s + 4u * ((win >> len) & ((1u << kPairBits) - 1u)));
                    if (!(e2 & (kLongFlag | 0x100u))) {
                        const uint32_t l2 = (e2 >> 24) & 15u, l1 = (e2 >> 9) & 15u;
                        if ((e2 >> 31) != 0u && pos + 4u <= n && bp + len + l2 <= end_bp) {
                            val |= ((e2 & 255u) | ((e2 >> 8) & 0xFF00u)) << 16;
                            more = 2u;
                            len += l2;
                        } else if (pos + 3u <= n && bp + len + l1 <= end_bp) {
                            val |= (e2 & 255u) << 16;
                            more = 1u;
                            len += l1;
                        }
                    }
                }
                bp += len;   // a run's code is <= kLutBits bits: at least 20 of the window are left for its extra bits
                uint32_t adv = (two ? 2u : 1u) + more;
                if (run) {
                    const uint32_t kk = sym - 256u;                              // run class 0..4 (hzr_internal.h:117-121)
                    const uint32_t eb = (0xE8420u >> (4u * kk)) & 15u;             // 0, 2, 4, 8, 14 extra bits
                    const uint32_t ev = (win >> len) & ((1u << eb) - 1u);
                    bp += eb;
                    adv = ev + (kk == 4u ? 279u : (0x17070302u >> (8u * kk)) & 255u);
                    if (pos + adv > n) { my_err = 1; break; }  // "Output buffer full" dec:473-476
                    val = 0u;
                }
                const uint32_t np = pos + adv, sh = (pos & 3u) * 8u;
                const uint32_t wv = w | (val << sh);
                const bool cross = (np ^ pos) > 3u;
                w = wv;
                if (cross) {
                    if (wv) {
                        uint32_t* q = reinterpret_cast<uint32_t*>(out + (pos & ~3u));
                        if ((pos >> 2) == first_w) atomicOr(q, wv);
                        else *q = wv;
                    }
                    // a pair that starts in a word's last byte leaves its second byte in the next word
                    w = __funnelshift_l(val, 0u, sh);   // 0 unless the token is a pair
                }
                pos = np;
            }
            };
            if (!use_pairs) token_loop(std::false_type{}, std::true_type{});
            else if (chain_pairs) token_loop(std::true_type{}, std::true_type{});
            else token_loop(std::true_type{}, std::false_type{});
            bitpos = bp - base_bits;
            if (bitpos > limit) my_err = 1;
            if (w) atomicOr(reinterpret_cast<uint32_t*>(out + (pos & ~3u)), w);
        }
    }
    if (my_err) status[f] = -4;
}

// ------------------------------------------------------------------------------------------
// Decode index for streams that arrive without one (written by the CPU reference): one CTA per
// HUFF block.  The token stream has no sync points, but a prefix code re-synchronises by itself
// after a few tokens, so thread k decodes from a guessed start -- the first bit of index interval k
// (the first thread that has tokens from the true start behind the tree) -- to the first token
// boundary inside the next interval, which becomes that neighbour's start.  Threads whose start
// moved decode again; the starts are exact once nothing moves (each round fixes at least one more
// interval, in practice two or three rounds do).  A scan of the bytes every interval produces
// gives the output position of its first token: together the entry of the decode index
// (common.cuh).  (hzr_decode.c has no counterpart: DecodeSingleBlock :335-567 is a sequential walk.)
// ------------------------------------------------------------------------------------------
constexpr int kIndexThreads = kMaxSegs;

struct TokenDecoder {
    const uint16_t* lut;
    const uint32_t* cw;
    const uint16_t* longs;
    const uint16_t* chain;
    // one token at the reader's position: bits consumed (0 = no code word matches) and bytes produced
    __device__ __forceinline__ uint32_t next(BitReader& r, uint32_t& out_bytes) const
    {
        r.refill();
        uint32_t e = lut[r.peek(kLutBits)];
        if (e & kLongFlag) {
            uint32_t j = e & kLongEnd;
            e = 0;
            while (j != kLongEnd) {
                const uint32_t sym = longs[j], c = cw[sym], len = c >> 27;
                if (((uint32_t)r.buf & ((1u << len) - 1u)) == (c & 0x07FFFFFFu)) {
                    e = sym | (len << 9);
                    break;
                }
                j = chain[j];
            }
            if (e == 0u) return 0u;
        }
        uint32_t len = e >> 9;
        const uint32_t sym = e & 511u;
        r.skip(len);
        out_bytes = 1u;
        if (sym >= 256u) {
            out_bytes = 2u;
            if (sym > 256u) {
                const uint32_t eb = sym_extra_bits(sym);
                r.refill();
                out_bytes = r.take(eb) + (sym == 257u ? 3u : sym == 258u ? 7u : sym == 259u ? 23u : 279u);
                len += eb;
            }
        }
        return len;
    }
};

__global__ void __launch_bounds__(kIndexThreads, 2) k_hzr_build_index(const uint8_t* __restrict__ src, Shape s,
                                                                       const DecBlk* __restrict__ dec,
                                                                       const uint64_t* __restrict__ offsets,
                                                                       const uint32_t* __restrict__ codes,
                                                                       uint32_t* __restrict__ sidecar,
                                                                       int32_t* __restrict__ status)
{
    extern __shared__ __align__(16) uint32_t payw[];  // payload words (+ zero slack)
    __shared__ __align__(16) uint16_t s_lut[1 << kLutBits];
    __shared__ uint32_t s_cw[kSymStride];
    __shared__ uint16_t s_long[kSymStride];
    __shared__ uint16_t s_next[kSymStride];
    __shared__ uint32_t s_meta[4];                    // -, -, long count
    __shared__ uint32_t s_start[kIndexThreads + 1];   // first token boundary of every interval
    __shared__ uint32_t s_wsum[kIndexThreads / 32];

    const uint32_t blk = blockIdx.x, tid = threadIdx.x, lane = lane_id(), wid = warp_id();
    const DecBlk d = dec[blk];
    if (d.mode != MODE_HUFF) return;  // COPY / FILL / unparsed frames need no index
    uint32_t f, k, b;
    blk_decode(s, blk, f, k, b);
    const uint32_t n = d.out_n;
    uint32_t* my_idx = sidecar + idx_slot_base(d.payload_off - offsets[0], blk);
    const uint8_t* pay = src + d.payload_off;
    const uintptr_t pa = (uintptr_t)pay;
    const uint32_t* aw = reinterpret_cast<const uint32_t*>(pa & ~(uintptr_t)3);
    const uint32_t lead = (uint32_t)(pa & 3u), sh = lead * 8u;
    const uint32_t plen = d.payload_len, pwords = (plen + 3u) >> 2, naw = (lead + plen + 3u) >> 2;
    for (uint32_t i = tid; i < pwords + 4u; i += blockDim.x) {
        uint32_t v = 0;
        if (i < pwords) {
            const uint32_t lo = __ldg(aw + i), hi = (i + 1 < naw) ? __ldg(aw + i + 1) : 0u;
            v = __funnelshift_r(lo, hi, sh);
            if (4u * i + 4u > plen) v &= (1u << (8u * (plen - 4u * i))) - 1u;  // bytes behind the payload
        }
        payw[i] = v;
    }
    for (uint32_t i = tid; i < (1u << kLutBits) / 2; i += blockDim.x) reinterpret_cast<uint32_t*>(s_lut)[i] = (kLongFlag | kLongEnd) * 0x00010001u;
    uint32_t mytb = 0;  // tree bits: 11 per leaf - 1 (StoreTree, hzr_encode.c:177-219)
    for (uint32_t i = tid; i < kSymStride; i += blockDim.x) {
        const uint32_t c = i < (uint32_t)kNumSymbols ? codes[(size_t)blk * kSymStride + i] : 0u;
        s_cw[i] = c;
        mytb += c ? 11u : 0u;
    }
    if (tid == 0) s_meta[2] = 0;
    mytb = __reduce_add_sync(0xFFFFFFFFu, mytb);
    if (lane == 0) s_wsum[wid] = mytb;
    __syncthreads();
    uint32_t t0 = 0;
    for (uint32_t w = 0; w < (blockDim.x >> 5); ++w) t0 += s_wsum[w];
    t0 = t0 ? t0 - 1u : 0u;
    __syncthreads();
    build_lut(s_cw, s_lut, s_long, &s_meta[2]);
    __syncthreads();
    chain_long_codes(s_cw, s_lut, s_long, s_next, s_meta[2]);
    __syncthreads();
    const IdxGeom ig = idx_geom(plen);
    const uint32_t limit = plen * 8u, nint = ig.n;
    bool bad = t0 > limit;
    // interval k: tokens that START in [lo, hi); the intervals in front of the first token have none
    const uint32_t lo = max(tid * ig.bits, t0), hi = min(limit, (tid + 1u) * ig.bits);
    const bool live = !bad && tid < nint && lo < hi;
    const TokenDecoder td{s_lut, s_cw, s_long, s_next};
    if (tid <= nint) s_start[tid] = min(lo, limit);
    __syncthreads();
    uint32_t my_start = 0xFFFFFFFFu, land = 0, cnt = 0;
    if (!bad) {
        for (;;) {
            const uint32_t st = live ? s_start[tid] : 0u;
            const bool redo = live && st != my_start;
            if (redo) {
                my_start = st;
                BitReader r;
                uint32_t pos = st;
                cnt = 0;
                if (pos < hi) r.init(payw, pos);
                while (pos < hi) {
                    uint32_t ob = 0;
                    uint32_t l = td.next(r, ob);
                    if (l == 0u) {  // no code word here (only from a wrong start, or a corrupt stream): slip one bit
                        l = 1u;
                        ob = 0u;
                        r.skip(1);
                    }
                    pos += l;
                    cnt += ob;
                }
                land = min(pos, limit);
            }
            __syncthreads();
            bool moved = false;
            if (redo && tid + 1 < nint && s_start[tid + 1] != land) {
                s_start[tid + 1] = land;
                moved = true;
            }
            if (!__syncthreads_or(moved)) break;
        }
    }
    // output position of every interval: exclusive scan of the byte counts
    uint32_t v = live ? cnt : 0u, inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, inc, o);
        if (lane >= (uint32_t)o) inc += y;
    }
    __syncthreads();
    if (lane == 31) s_wsum[wid] = inc;
    __syncthreads();
    uint32_t opos = inc - v, total = 0;
    for (uint32_t w = 0; w < (blockDim.x >> 5); ++w) {
        const uint32_t t = s_wsum[w];
        if (w < wid) opos += t;
        total += t;
    }
    // the tokens must produce at least n bytes (zero padding of the last byte may decode into a
    // few more: they are ignored, like the reference stops at the output size, dec:440)
    if (total < n) bad = true;
    if (bad) {
        if (tid < nint) my_idx[tid] = 0xFFFFFFFFu;  // k_hzr_decode reports the frame and writes zeros
        if (tid == 0) status[f] = -4;
        return;
    }
    if (tid < nint) {
        const uint32_t st = min(max(s_start[tid], lo), limit);
        my_idx[tid] = (st - tid * ig.bits) | (min(opos, n) << kIdxPosShift);
    }
}

// ------------------------------------------------------------------------------------------
// Integrity check without decoding: hzr_verify (lib_hzr/hzr_decode.c:569-624) for every hzr
// stream of every frame.  The header walk is k_frame_parse's; here one CTA per block stages the
// payload in shared memory and compares its CRC-32C with the block header's
// (hzr_decode.c:606-611: "CRC32 check failed").  status[f] = RSPT_E_CRC (-6) on a mismatch.
// ------------------------------------------------------------------------------------------
constexpr int kVerifyThreads = 256;
constexpr int kVerifyZtSel = 1;  // log2(kVerifyThreads / 128)

__global__ void __launch_bounds__(kVerifyThreads) k_hzr_verify(const uint8_t* __restrict__ src, Shape s,
                                                                const DecBlk* __restrict__ dec,
                                                                const CrcConst* __restrict__ cc,
                                                                int32_t* __restrict__ status, Counters* __restrict__ ctr)
{
    extern __shared__ __align__(16) uint32_t payw[];
    __shared__ __align__(16) uint32_t s_zt[1024];
    __shared__ uint32_t s_red[33];
    const uint32_t blk = blockIdx.x, tid = threadIdx.x;
    const DecBlk d = dec[blk];
    if (d.mode == kModeInactive || d.mode == kModeZero) return;  // not there / frame already flagged
    for (uint32_t i = tid; i < 256; i += blockDim.x)
        reinterpret_cast<uint4*>(s_zt)[i] = __ldg(reinterpret_cast<const uint4*>(&cc->zt[kVerifyZtSel][0][0]) + i);
    const uint8_t* pay = src + d.payload_off;
    const uintptr_t pa = (uintptr_t)pay;
    const uint32_t* aw = reinterpret_cast<const uint32_t*>(pa & ~(uintptr_t)3);
    const uint32_t lead = (uint32_t)(pa & 3u), sh = lead * 8u;
    const uint32_t plen = d.payload_len, pwords = (plen + 3u) >> 2, naw = (lead + plen + 3u) >> 2;
    for (uint32_t i = tid; i < pwords; i += blockDim.x) {
        const uint32_t lo = __ldg(aw + i), hi = (i + 1 < naw) ? __ldg(aw + i + 1) : 0u;
        payw[i] = __funnelshift_r(lo, hi, sh);
    }
    __syncthreads();
    const uint32_t crc = block_crc32c(payw, plen, s_zt, cc, s_red);
    if (tid == 0) {
        const uint32_t want = ld_le32(pay - 5);  // block header: size u16, crc u32, mode u8
        if (crc != want) {
            uint32_t f, k, b;
            blk_decode(s, blk, f, k, b);
            status[f] = -6;
            atomicAdd(&ctr->crc_failures, 1ull);
        }
    }
}

}  // namespace rspt
