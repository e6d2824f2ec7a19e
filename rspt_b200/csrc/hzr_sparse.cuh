// Sparse hzr blocks for sm_100a, packed from the sorted list of non-zero bytes that k_hzr_hist
// left (position | value << 16): one CTA per block, the plane is not read again.  Replaces, for
// these blocks, the encode loop and WriteBits of lib_hzr/hzr_encode.c:410-457, :94-113 and the
// block header + CRC of :463-484.  Runs after the layout kernels, so the block (7-byte header +
// payload) goes straight to its place in the output stream; k_hzr_encode skips it.  The decode
// index of such a block is written here too.
#pragma once

#include "common.cuh"
#include "hzr_tree.cuh"
#include "hzr_hist.cuh"
#include "hzr_pack.cuh"

namespace rspt {

constexpr int kSpThreads = 256;
constexpr uint32_t kSpStageBytes = 12288;                // largest payload packed here
constexpr uint32_t kSpStageWords = kSpStageBytes / 4 + 8;
constexpr size_t kSparseSmem = (size_t)(kListCap + 4 + kSpStageWords) * 4;

// frame / chunk framing, written by the CTA that owns the chunk's first block (whichever encoder that is):
// chunk length and hzr decoded size in front of the block, method byte and header at the frame start
// (signal_packer_base.cpp:78,83-95; hzr_encode.c:521)
__device__ __forceinline__ void write_chunk_framing(const Shape& s, const BlkInfo* __restrict__ info, uint32_t f, uint32_t k,
                                                    uint8_t* __restrict__ dst, unsigned long long frame_off, uint8_t* out,
                                                    const uint8_t* __restrict__ headers)
{
    if (threadIdx.x == 0) {
        uint32_t clen = 4;
        const size_t row = ((size_t)f * s.nb_alloc + k) * s.nblk;
        for (uint32_t bb = 0; bb < s.nblk; ++bb) clen += 7u + info[row + bb].payload_len;
        uint8_t* q = out - 8;
        q[0] = (uint8_t)clen; q[1] = (uint8_t)(clen >> 8); q[2] = (uint8_t)(clen >> 16); q[3] = (uint8_t)(clen >> 24);
        q[4] = (uint8_t)s.N; q[5] = (uint8_t)(s.N >> 8); q[6] = (uint8_t)(s.N >> 16); q[7] = (uint8_t)(s.N >> 24);
        if (k == 0) dst[frame_off] = (uint8_t)s.method;
    }
    if (k == 0)
        for (uint32_t i = threadIdx.x; i < s.hdr_bytes; i += blockDim.x) dst[frame_off + 1 + i] = headers[(size_t)f * s.hdr_bytes + i];
}

struct SparseOut {
    uint8_t* dst;         // output stream
    const uint64_t* offsets;   // byte offset of every frame in dst
    const uint32_t* blk_off;   // per block: offset of its header from the frame start
    uint32_t stage_bytes;      // largest payload packed here (<= kSpStageBytes; smaller values only in tests)
    const uint8_t* headers;    // per frame: the packer's header bytes (hadamard / dct means)
    uint32_t* sidecar;    // decode index (may be null), see common.cuh
};

// Every entry i <= m of the list stands for the tokens between the previous non-zero byte and this
// one: the zero run (if any), its extra bits, then the literal (entry m: the run up to the block end).
// The entries' bit offsets are a prefix sum of their bit lengths: the CTA takes the entries 256 at a
// time, one per thread, and places each with a warp scan plus the warp totals of that round (one
// barrier per round), so every entry is classified and looked up once.
__global__ void __launch_bounds__(kSpThreads, 6) k_hzr_encode_sparse(Shape s, const uint8_t* __restrict__ frame_nb,
                                                                     const BlkInfo* __restrict__ info,
                                                                     const uint32_t* __restrict__ codes,
                                                                     const uint32_t* __restrict__ tree,
                                                                     const uint32_t* __restrict__ lists,
                                                                     const uint32_t* __restrict__ list_n,
                                                                     const CrcConst* __restrict__ cc, SparseOut so)
{
    extern __shared__ __align__(16) uint32_t s_dyn[];  // the list, then the payload staging
    __shared__ uint32_t s_codes[kSymStride];
    __shared__ uint32_t s_wtot[2][kSpThreads / 32];
    uint32_t f, k, b;
    const uint32_t blk = blockIdx.x;
    const uint32_t m = list_n[blk];
    const BlkInfo bi = info[blk];
    if (!sparse_block_is_packed_from_list(m, bi, so.stage_bytes)) return;  // k_hzr_encode packs it from the plane
    blk_decode(s, blk, f, k, b);
    if (k >= frame_nb[f]) return;
    const uint32_t tid = threadIdx.x, lane = lane_id(), wid = warp_id();
    const uint32_t n = blk_len(s, b);
    const uint32_t* glist = lists + (size_t)blk * kListCap;
    uint32_t* list = s_dyn;
    uint32_t* stg = s_dyn + kListCap;  // block header at bytes 9..15, payload from byte 16
    uint32_t* pay = stg + 4;
    const uint32_t plen = bi.payload_len, tw = (bi.tree_nbits + 31u) >> 5, pw = (plen + 3u) >> 2;
    // the list arrives asynchronously (16-byte chunks; its slot in d_lists is kListCap entries, a multiple of 4)
    // while the code table, the tree bits and the zeroed staging are set up
    {
        const uint32_t list_s = smem_addr(list);
        const uint4* g4 = reinterpret_cast<const uint4*>(glist);
        for (uint32_t i = tid; i < (m + 3u) / 4u; i += blockDim.x)
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(list_s + 16u * i), "l"(g4 + i) : "memory");
        asm volatile("cp.async.commit_group;" ::: "memory");
    }
    for (uint32_t i = tid; i < kSymStride; i += blockDim.x) s_codes[i] = __ldg(codes + (size_t)blk * kSymStride + i);
    // decode index: where this block's entries go (common.cuh); the first token starts behind the tree bits
    const unsigned long long frame_off = so.offsets[f];
    uint32_t* my_idx = so.sidecar ? so.sidecar + idx_slot_base(frame_off + so.blk_off[blk] + 7u, blk) : nullptr;
    const IdxGeom ig = idx_geom(bi.payload_len);
    if (my_idx && tid <= idx_interval_of(ig, bi.tree_nbits)) my_idx[tid] = bi.tree_nbits - tid * ig.bits;
    // staging: tree words, then zeros (the code words are OR-ed in)
    for (uint32_t i = tid; i < pw + 2u; i += blockDim.x) pay[i] = i < tw ? __ldg(tree + (size_t)blk * kTreeWords + i) : 0u;
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();

    // bit packing: every entry's <= 3 slots (run code, run extra bits, literal) are placed with a warp
    // scan of the entry bit lengths
    uint32_t base = bi.tree_nbits;
    const uint32_t ne = m + 1u;  // entries, the run up to the block end included
    // the trip count depends on m alone, so every warp reaches the barrier of every round
    for (uint32_t i0 = 0, r = 0; i0 < ne; i0 += blockDim.x, r ^= 1u) {
        const uint32_t i = i0 + tid;
        const bool live = i < ne;
        uint32_t bits = 0, gap = 0, cur = 0, rs = 0, c_run = 0, c_ext = 0, c_lit = 0;
        if (live) {
            const uint32_t e = i < m ? list[i] : n;
            cur = i < m ? e & 0xFFFFu : n;
            rs = i ? (list[i - 1] & 0xFFFFu) + 1u : 0u;
            gap = cur - rs;
            if (i < m) c_lit = s_codes[e >> 16];
            if (gap > kRunCap) {
                bits = run_bits(gap, s_codes);
            } else if (gap) {
                uint32_t sym, ev, eb;
                run_token(gap, sym, ev, eb);
                c_run = s_codes[sym];
                c_ext = ev | (eb << 27);
                bits = slot_bits(c_run) + eb;
            }
            bits += slot_bits(c_lit);
        }
        uint32_t inc = bits;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, inc, o);
            if (lane >= (uint32_t)o) inc += y;
        }
        // warp totals of this round (double-buffered: a warp may start the next round before the
        // others have read this one)
        if (lane == 31) s_wtot[r][wid] = inc;
        __syncthreads();
        const uint32_t t = lane < (blockDim.x >> 5) ? s_wtot[r][lane] : 0u;
        const uint32_t o0 = base + __reduce_add_sync(0xFFFFFFFFu, lane < wid ? t : 0u) + inc - bits;
        base += __reduce_add_sync(0xFFFFFFFFu, t);
        if (live) {
            if (bits > 64u || gap > kRunCap) {
                EmitSink es{s_codes, pay, 0ull, o0 & 31u, o0 >> 5, true};
                if (gap) emit_run(gap, es);
                if (i < m) es.append(c_lit & 0x07FFFFFFu, slot_bits(c_lit));
                es.finish();
            } else if (bits) {
                // concatenate the slots last-first, shift to the bit offset, OR into <= 3 words
                uint32_t lo = c_lit & 0x07FFFFFFu, hi = 0, l = slot_bits(c_ext);
                hi = __funnelshift_l(lo, hi, l);
                lo = (lo << l) | (c_ext & 0x07FFFFFFu);
                l = slot_bits(c_run);
                hi = __funnelshift_l(lo, hi, l);
                lo = (lo << l) | (c_run & 0x07FFFFFFu);
                const uint32_t sh = o0 & 31u;
                uint32_t* w = pay + (o0 >> 5);
                const uint32_t v0 = lo << sh, v1 = __funnelshift_l(lo, hi, sh), v2 = __funnelshift_l(hi, 0u, sh);
                atomicOr(w, v0);
                if (v1) atomicOr(w + 1, v1);
                if (v2) atomicOr(w + 2, v2);
            }
        }
        // decode index: the entry whose tokens cover the last bit before an interval boundary names the
        // token behind them (the next entry's run, or nothing after the last one)
        if (my_idx && live) {
            const uint32_t e = o0 + bits;
            const uint32_t kk = idx_interval_of(ig, e);
            if (kk != idx_interval_of(ig, o0)) my_idx[kk] = (e - kk * ig.bits) | ((i < m ? cur + 1u : n) << kIdxPosShift);
        }
    }
    __syncthreads();

    // the payload goes out while warp 0 takes its CRC-32C and then writes the 7-byte block header
    uint8_t* out = so.dst + frame_off + so.blk_off[blk];
    if (b == 0) write_chunk_framing(s, info, f, k, so.dst, frame_off, out, so.headers);
    copy_smem_to_global(out + 7, stg, 16, plen);
    if (wid != 0) return;
    const uint32_t crc = warp_crc32c(pay, plen, cc);
    if (lane < 7) {
        const uint32_t lo = (plen - 1u) | (crc << 16), hi = (crc >> 16) | ((uint32_t)MODE_HUFF << 16);
        out[lane] = (uint8_t)((lane < 4 ? lo : hi) >> (8u * (lane & 3u)));
    }
}

}  // namespace rspt
