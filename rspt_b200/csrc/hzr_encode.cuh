// hzr encoder for sm_100a: per-block histogram -> batched tree build -> sized layout -> bit
// packing with CRC-32C.  Replaces lib_hzr/hzr_encode.c (Histogram :133-173, MakeTree :222-283,
// StoreTree :177-219, OnlySingleCode :285-305, EncodeSingleBlock :369-487, PlainCopy :307-339,
// EncodeFill :341-367, hzr_encode :499-544) and the framing half of compress_i32
// (lib_signalpacker/signal_packer_base.cpp:69-95).  The output is byte-identical to the
// reference's.
#pragma once

#include "common.cuh"
#include "hzr_tree.cuh"
#include "hzr_hist.cuh"
#include "hzr_pack.cuh"
#include "hzr_sparse.cuh"

namespace rspt {

// ------------------------------------------------------------------------------------------
// 3. layout: per-frame plane count (prefix max of `need`, the reference's sticky
// nr_bytes_to_compress_++), frame sizes, exclusive scan -> byte offset of every frame.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) k_frame_nb(const uint32_t* __restrict__ need, uint32_t n_frames,
                                                    uint32_t* __restrict__ nb_state, uint8_t* __restrict__ frame_nb,
                                                    Counters* __restrict__ ctr)
{
    __shared__ uint32_t s_w[33];
    uint32_t carry = *nb_state;
    const uint32_t start_nb = carry;
    for (uint32_t base = 0; base < n_frames; base += blockDim.x) {
        const uint32_t f = base + threadIdx.x;
        uint32_t v = f < n_frames ? need[f] : 0u;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t y = __shfl_up_sync(0xFFFFFFFFu, v, o);
            if (lane_id() >= (uint32_t)o) v = max(v, y);
        }
        if (lane_id() == 31) s_w[warp_id()] = v;
        __syncthreads();
        uint32_t pre = carry;
        for (uint32_t w = 0; w < warp_id(); ++w) pre = max(pre, s_w[w]);
        v = max(v, pre);
        if (f < n_frames) frame_nb[f] = (uint8_t)v;
        uint32_t all = carry;
        for (uint32_t w = 0; w < (blockDim.x >> 5); ++w) all = max(all, s_w[w]);
        carry = all;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        *nb_state = carry;
        if (carry > start_nb) atomicAdd(&ctr->escalations, (unsigned long long)(carry - start_nb));
    }
}

// per frame: total size and the byte offset (from the frame start) of every block's 7-byte header
__global__ void k_frame_sizes(const BlkInfo* __restrict__ info, Shape s, const uint8_t* __restrict__ frame_nb,
                              uint32_t n_frames, uint32_t* __restrict__ sizes, uint32_t* __restrict__ blk_off)
{
    const uint32_t f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= n_frames) return;
    uint32_t sz = 1 + s.hdr_bytes;  // method byte + header (signal_packer_base.cpp:83-91)
    const uint32_t nb = frame_nb[f];
    for (uint32_t k = 0; k < nb; ++k) {
        sz += 8;  // chunk len:u32 (:78) + hzr decoded size:u32 (hzr_encode.c:521)
        const size_t row = ((size_t)f * s.nb_alloc + k) * s.nblk;
        for (uint32_t b = 0; b < s.nblk; ++b) {
            blk_off[row + b] = sz;
            sz += 7u + info[row + b].payload_len;
        }
    }
    sizes[f] = sz;
}

// offsets[f] = base + the sizes of frames 0 .. f - 1 (base: where the batch starts in the stored batch it extends)
__global__ void __launch_bounds__(1024) k_scan_offsets(const uint32_t* __restrict__ sizes, uint32_t n_frames,
                                                        unsigned long long base, uint64_t* __restrict__ offsets,
                                                        Counters* __restrict__ ctr, uint32_t frame_bytes)
{
    __shared__ unsigned long long s_w[33];
    const uint32_t per = (n_frames + blockDim.x - 1) / blockDim.x;
    const uint32_t lo = min(n_frames, threadIdx.x * per), hi = min(n_frames, lo + per);
    unsigned long long sum = 0;
    for (uint32_t f = lo; f < hi; ++f) sum += sizes[f];
    unsigned long long inc = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        unsigned long long y = __shfl_up_sync(0xFFFFFFFFu, inc, o);
        if (lane_id() >= (uint32_t)o) inc += y;
    }
    if (lane_id() == 31) s_w[warp_id()] = inc;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long run = 0;
        for (uint32_t w = 0; w < (blockDim.x >> 5); ++w) {
            unsigned long long t = s_w[w];
            s_w[w] = run;
            run += t;
        }
        s_w[32] = run;
    }
    __syncthreads();
    unsigned long long off = base + s_w[warp_id()] + inc - sum;
    for (uint32_t f = lo; f < hi; ++f) {
        offsets[f] = off;
        off += sizes[f];
    }
    if (threadIdx.x == 0) {
        offsets[n_frames] = base + s_w[32];
        atomicAdd(&ctr->frames_compressed, (unsigned long long)n_frames);
        atomicAdd(&ctr->raw_bytes_in, (unsigned long long)n_frames * frame_bytes);
        atomicAdd(&ctr->compressed_bytes_out, s_w[32]);
    }
}

// ------------------------------------------------------------------------------------------
// 4. encode: one CTA of 16 warps per block.  The block is walked in GROUPS of 16 warp-steps
// (8 KiB); in a group every lane owns 16 consecutive bytes and the tokens that START in them:
// its literals and the zero runs whose first zero lies in the chunk (a run that continues into
// later chunks is measured with the lane's forward zero count: stop bits of the following lanes,
// then the per-step leading-zero counts left by the histogram pass).
//
// Every byte becomes one look-up in a per-block table of (value, bit length):
//   entries 0..255   the byte's code word (entry 0: symbol 0, a zero run of one)
//   entry 256        nothing -- zeros inside a run, bytes beyond the block end
//   entries 257..383 the whole token of a zero run of 2..128: run symbol + extra bits
// so the per-byte work is the same straight line for literals and runs: a lane with zero runs only
// rewrites the index bytes of the affected positions first (rare per lane).  The four slots of a
// word are concatenated last-first into 64 bits; lane bit lengths -> warp scan + one
// __syncthreads per group -> each word is shifted to its bit offset and OR-ed into <= 3 staging
// words.  Words that do not fit (> 64 bits, runs > 128) take a generic token walker.
// The block's bytes [7-byte header | payload] are staged in shared memory starting at byte 9
// (payload 16-byte aligned at byte 16); the CRC-32C is taken from the staged payload and the
// whole thing is copied to its final, arbitrarily aligned position in the output stream
// (hzr_encode.c:410-484, WriteBits :94-113).
// ------------------------------------------------------------------------------------------
constexpr int kEncThreads = 512;
constexpr int kEncWarps = kEncThreads / 32;
constexpr int kEncZtSel = 2;  // log2(kEncThreads / 128)
constexpr uint32_t kTabNull = 256;       // table entry that contributes no bits
constexpr uint32_t kTabMaxRun = 128;     // longest zero run that has a table entry (257 + L - 2)
constexpr uint32_t kTabSize = 256 + kTabMaxRun;
constexpr uint32_t kTabSlow = 255;       // bit length of an entry that cannot be used (forces the generic path)

// tokens that start in one 4-byte word, in stream order (general path: any run length)
template <class Sink>
__device__ __forceinline__ void walk_word(uint32_t x, uint32_t nz, uint32_t starts, uint32_t stop, uint32_t fwd, Sink& sink)
{
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        if ((nz >> j) & 1u) {
            sink.token((x >> (8 * j)) & 0xFFu, 0u, 0u);
        } else if ((starts >> j) & 1u) {
            const uint32_t sb = (stop >> j) & 0xFu;
            emit_run(sb ? (uint32_t)__ffs(sb) - 1u : 4u - j + fwd, sink);
        }
    }
}

__device__ __forceinline__ uint2 lds_v2(uint32_t a)
{
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a));
    return v;
}
// shifts whose amount may reach 32 (PTX clamps, C++ does not define them)
__device__ __forceinline__ uint32_t shl_c(uint32_t a, uint32_t n)
{
    uint32_t d;
    asm("shl.b32 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(n));
    return d;
}
__device__ __forceinline__ uint32_t shf_l_c(uint32_t lo, uint32_t hi, uint32_t n)
{
    uint32_t d;
    asm("shf.l.clamp.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(lo), "r"(hi), "r"(n));
    return d;
}

constexpr uint32_t kStgWords = 12 + kBlock / 4 + 8;   // header + payload at an offset of 16 .. 31 + 7 bytes, + slack
constexpr size_t kEncodeSmem = (size_t)kStgWords * 4;

// MINB = CTAs per SM the register allocation aims at: 2 (63 registers) or 3 (40 registers, 36 bytes of spills);
// which one is faster depends on the planes (rspt_gpu.cu: encode_ctas_per_sm)
template <int MINB>
__global__ void __launch_bounds__(kEncThreads, MINB) k_hzr_encode(const uint8_t* __restrict__ planes, Shape s,
                                                                const uint8_t* __restrict__ frame_nb,
                                                                const BlkInfo* __restrict__ info,
                                                                const uint32_t* __restrict__ blk_off,
                                                                const uint32_t* __restrict__ codes,
                                                                const uint32_t* __restrict__ tree,
                                                                const uint16_t* __restrict__ step_lz,
                                                                const uint32_t* __restrict__ lists,
                                                                const uint32_t* __restrict__ list_n, uint32_t sparse_stage,
                                                                const uint64_t* __restrict__ offsets,
                                                                const uint8_t* __restrict__ headers,
                                                                const CrcConst* __restrict__ cc,
                                                                uint8_t* __restrict__ dst,
                                                                uint32_t* __restrict__ sidecar)
{
    // The block (7 header bytes + payload) is staged at an offset CONGRUENT to its address in the output stream mod 16,
    // so that it leaves with one bulk asynchronous store: header at byte hoff = 16 + (address & 15), payload at
    // poff = hoff + 7, i.e. `lead` = poff & 3 bytes into the word array `pay`; every bit offset below counts from pay[0].
    extern __shared__ __align__(16) uint32_t stg[];
    __shared__ uint32_t s_codes[kSymStride];
    __shared__ __align__(8) uint2 s_tab[kTabSize];
    __shared__ __align__(16) uint32_t s_zt[1024];
    __shared__ uint32_t s_after[kMaxSteps];          // zeros that follow the end of every step
    __shared__ uint32_t s_tot[2][kEncWarps];
    __shared__ uint32_t s_red[33];

    uint32_t f, k, b;
    const uint32_t blk = blockIdx.x;
    // a block with a list is k_hzr_encode_sparse's (framing included), unless its payload does not fit that
    // kernel's staging: those CTAs (2/3 of the grid on delta-coded signals) leave at once
    const BlkInfo bi = info[blk];
    const uint32_t list_m = list_n[blk];
    if (sparse_block_is_packed_from_list(list_m, bi, sparse_stage)) return;
    blk_decode(s, blk, f, k, b);
    const uint32_t nb = frame_nb[f];
    if (k >= nb) return;
    const uint32_t n = blk_len(s, b);
    const uint32_t tid = threadIdx.x, lane = lane_id(), wid = warp_id();
    const unsigned long long frame_off = offsets[f];
    uint8_t* out = dst + frame_off + blk_off[blk];
    if (b == 0) write_chunk_framing(s, info, f, k, dst, frame_off, out, headers);
    if (bi.mode == MODE_FILL) {
        if (tid == 0) {
            const uint32_t crc = ~(0x00FFFFFFu ^ __ldg(&cc->byte_tab[0xFFu ^ bi.fill]));
            out[0] = 0; out[1] = 0;
            out[2] = (uint8_t)crc; out[3] = (uint8_t)(crc >> 8); out[4] = (uint8_t)(crc >> 16); out[5] = (uint8_t)(crc >> 24);
            out[6] = MODE_FILL;
            out[7] = bi.fill;
        }
        return;
    }

    uint8_t* sbytes = reinterpret_cast<uint8_t*>(stg);
    const uint32_t plen = bi.payload_len;
    const uint32_t hoff = 16u + (uint32_t)((uintptr_t)out & 15u), poff = hoff + 7u;
    const uint32_t lead = poff & 3u, lead_bits = 8u * lead, pw0 = poff >> 2;
    uint32_t* pay = stg + pw0;
    for (uint32_t i = tid; i < 256; i += blockDim.x)
        reinterpret_cast<uint4*>(s_zt)[i] = __ldg(reinterpret_cast<const uint4*>(&cc->zt[kEncZtSel][0][0]) + i);
    const uint8_t* src = blk_ptr(planes, s, f, k, b);

    if (bi.mode == MODE_COPY) {
        // raw plane bytes are the payload (PlainCopy); rows are 16-byte aligned
        // (moved `lead` bytes up: word w of the staging = bytes 4w - lead .. 4w - lead + 3 of the plane)
        const uint32_t* s32 = reinterpret_cast<const uint32_t*>(src);
        const uint4* s4 = reinterpret_cast<const uint4*>(src);
        const uint32_t nq = (n + 15u) >> 4;   // 16-byte chunks of the plane row (rows are padded to 16 bytes)
        for (uint32_t i = tid; i <= nq; i += blockDim.x) {
            const uint32_t prev = i ? __ldg(s32 + 4u * i - 1u) : 0u;
            const uint4 v = i < nq ? __ldg(s4 + i) : make_uint4(0, 0, 0, 0);
            uint32_t* d = pay + 4u * i;
            d[0] = __funnelshift_l(prev, v.x, lead_bits);
            if (i < nq) {
                d[1] = __funnelshift_l(v.x, v.y, lead_bits);
                d[2] = __funnelshift_l(v.y, v.z, lead_bits);
                d[3] = __funnelshift_l(v.z, v.w, lead_bits);
            }
        }
        for (uint32_t w = tid; w < pw0; w += blockDim.x) stg[w] = 0;   // header bytes: zero until the CRC is taken
        __syncthreads();
    } else {
        const uint32_t nsteps = (n + kStepBytes - 1) / kStepBytes;
        const uint32_t* gc = codes + (size_t)blk * kSymStride;
        for (uint32_t i = tid; i < kTabSize; i += blockDim.x) {
            if (i < (uint32_t)kSymStride) s_codes[i] = __ldg(gc + i);
            uint2 e;
            if (i < 256u) {
                const uint32_t cw = __ldg(gc + i);
                e = make_uint2(cw & 0x07FFFFFFu, cw >> 27);
            } else if (i == kTabNull) {
                e = make_uint2(0u, 0u);
            } else {
                uint32_t sym, ev, eb;
                run_token(i - 255u, sym, ev, eb);
                const uint32_t cw = __ldg(gc + sym), len = cw >> 27;
                e = len + eb <= 32u ? make_uint2((cw & 0x07FFFFFFu) | (ev << len), len + eb) : make_uint2(0u, kTabSlow);
            }
            s_tab[i] = e;
        }
        const uint32_t tw = (bi.tree_nbits + 31u) >> 5, pw = (plen + 3u) >> 2;
        // staging: tree words, then zeros (the code words are OR-ed in)
        // (stg words 0 .. pw0 - 1 are zero: the header is written after the CRC has been taken; the tree words
        // are moved up by `lead` bytes and spill into one more word)
        const uint32_t tw4 = (pw0 + tw + 1u + 3u) & ~3u;
        const uint32_t* gt = tree + (size_t)blk * kTreeWords;
        for (uint32_t i = tid; i < tw4; i += blockDim.x) {
            uint32_t v = 0;
            if (i >= pw0 && i <= pw0 + tw) {
                const uint32_t j = i - pw0;
                v = __funnelshift_l(j ? __ldg(gt + j - 1) : 0u, j < tw ? __ldg(gt + j) : 0u, lead_bits);
            }
            stg[i] = v;
        }
        for (uint32_t i = (tw4 >> 2) + tid; i < ((pw0 + pw + 3u + 3u) >> 2); i += blockDim.x) reinterpret_cast<uint4*>(stg)[i] = make_uint4(0, 0, 0, 0);
        // decode index: where this block's entries go (common.cuh); offsets are store-relative and `sidecar`
        // starts at the batch's first block ordinal, so an appended batch lands where one long batch would
        uint32_t* my_idx = sidecar ? sidecar + idx_slot_base(frame_off + blk_off[blk] + 7u, blk) : nullptr;
        const IdxGeom ig = idx_geom(plen);
        if (my_idx && tid <= idx_interval_of(ig, bi.tree_nbits)) my_idx[tid] = bi.tree_nbits - tid * ig.bits;  // first token, output byte 0
        if (wid == kEncWarps - 1) {
            // s_after[st] = zeros between the end of step st and the next stop byte (or the block
            // end): suffix chain over the per-step leading-zero counts, 4 steps per lane
            const uint16_t* lzp = step_lz + (size_t)blk * kMaxSteps;
            uint32_t lz[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const uint32_t st = 4u * lane + j;
                lz[j] = st < nsteps ? (uint32_t)lzp[st] : 0u;  // beyond the block: a stop at once
                if (list_m != kNoList && st < nsteps) {
                    // listed block handed over by the sparse encoder (payload beyond its staging, rare):
                    // it never went through the dense scan, so its leading-zero counts come from the list
                    const uint32_t* gl = lists + (size_t)blk * kListCap;
                    uint32_t lo = 0, hi = list_m;  // first entry at or after the step start
                    while (lo < hi) {
                        const uint32_t mid = (lo + hi) >> 1;
                        if ((__ldg(gl + mid) & 0xFFFFu) < st * kStepBytes) lo = mid + 1u;
                        else hi = mid;
                    }
                    const uint32_t pos = lo < list_m ? __ldg(gl + lo) & 0xFFFFu : n;
                    lz[j] = min(min(pos, n) - st * kStepBytes, (uint32_t)kStepBytes);
                }
            }
            // leading zeros counted from the start of my 4 steps, and whether all 4 are zero
            uint32_t mine = 0;
            bool open = true;
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (open) {
                    mine += lz[j];
                    open = lz[j] == kStepAllZero;
                }
            const uint32_t openm = __ballot_sync(0xFFFFFFFFu, open);
            const uint32_t above = lane < 31 ? ~openm & ~((2u << lane) - 1u) : 0u;  // closed lanes after me
            const uint32_t q = above ? (uint32_t)__ffs(above) - 1u : 31u;
            const uint32_t mq = __shfl_sync(0xFFFFFFFFu, mine, q);
            // zeros that follow the end of my 4 steps
            uint32_t carry = above ? 4u * kStepBytes * (q - lane - 1u) + mq : 4u * kStepBytes * (31u - lane);
#pragma unroll
            for (int j = 3; j >= 0; --j) {
                const uint32_t st = 4u * lane + j;
                if (st < kMaxSteps) s_after[st] = carry;
                carry = lz[j] == kStepAllZero ? carry + kStepBytes : lz[j];
            }
        }
        __syncthreads();

        uint32_t base = bi.tree_nbits + lead_bits;  // bit offset of the group from pay[0] (same in every thread)
        const uint32_t ngroups = (nsteps + kEncWarps - 1) / kEncWarps;
        const uint32_t tab_s = smem_addr(s_tab), pay_s = smem_addr(pay);  // see common.cuh
        // the chunk of the next group and the byte before its step are fetched one group ahead, so
        // their latency hides behind the current group's work
        uint4 v_next = make_uint4(0, 0, 0, 0);
        uint32_t pstep_next = 1;
        {
            const uint32_t sb0 = wid * kStepBytes;
            if (lane == 0 && sb0 > 0 && sb0 <= n) pstep_next = src[sb0 - 1];
            if (sb0 + kStepBytes <= n) v_next = __ldg(reinterpret_cast<const uint4*>(src + sb0 + lane * 16u));
        }
        for (uint32_t g = 0; g < ngroups; ++g) {
            const uint32_t st = g * kEncWarps + wid;
            const uint32_t sbase = st * kStepBytes, off = sbase + lane * 16u;
            uint32_t x[4], NZ, INV = 0;
            const uint32_t pstep = pstep_next;  // the byte before the step (lane 0 only)
            const uint4 v = v_next;
            {
                const uint32_t sbn = sbase + kEncWarps * kStepBytes;
                pstep_next = 1;
                if (lane == 0 && sbn <= n) pstep_next = src[sbn - 1];
                if (sbn + kStepBytes <= n) v_next = __ldg(reinterpret_cast<const uint4*>(src + sbn + lane * 16u));
            }
            if (sbase + kStepBytes <= n) {
                x[0] = v.x; x[1] = v.y; x[2] = v.z; x[3] = v.w;
                NZ = nz_mask16(v);
            } else {
                const Chunk c = load_chunk(src, n, off);
                x[0] = c.v.x; x[1] = c.v.y; x[2] = c.v.z; x[3] = c.v.w;
                NZ = c.nz;
                INV = c.stop & ~c.nz;
                // bytes beyond the block end: no token, and nothing in the index byte
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    const uint32_t iv = (INV >> (4 * r)) & 0xFu;
                    if (iv) x[r] &= ~(((iv * 0x00204081u) & 0x01010101u) * 0xFFu);
                }
            }
            const uint32_t STOP = NZ | INV, Z = ~STOP & 0xFFFFu;
            const uint32_t after = st < nsteps ? s_after[st] : 0u;  // zeros that follow the step
            const uint32_t z_up = __shfl_up_sync(0xFFFFFFFFu, Z, 1), z_dn = __shfl_down_sync(0xFFFFFFFFu, Z, 1);
            const uint32_t pz = lane > 0 ? z_up >> 15 : (pstep == 0u ? 1u : 0u);          // the byte before my chunk is a zero
            const uint32_t nzx = lane < 31 ? z_dn & 1u : (after ? 1u : 0u);              // the byte after my chunk is a zero
            const uint32_t starts = Z & ~((Z << 1) | pz);                  // first zero of a run
            const uint32_t run2 = starts & ((Z >> 1) | (nzx << 15));      // ... of a run of >= 2
            const uint32_t special = (Z & ~starts) | run2 | INV;          // positions that are not "one byte, one code"
            // zeros between the end of my chunk and the next stop byte: when a run leaves its chunk
            const bool leaves = ((Z >> 15) & nzx) != 0u;
            uint32_t fwd = 0;
            if (__any_sync(0xFFFFFFFFu, leaves)) {
                const uint32_t sm = __ballot_sync(0xFFFFFFFFu, STOP != 0u);
                const uint32_t fs = STOP ? (uint32_t)__ffs(STOP) - 1u : 16u;
                const uint32_t above = lane < 31 ? sm & ~((2u << lane) - 1u) : 0u;
                const uint32_t q = above ? (uint32_t)__ffs(above) - 1u : 0u;
                const uint32_t fq = __shfl_sync(0xFFFFFFFFu, fs, q);
                fwd = above ? 16u * (q - lane - 1u) + fq : 16u * (31u - lane) + after;
            }
            // ---- index bytes of the special positions: high byte 1, low byte 0 (nothing) or run length - 1
            uint32_t G[4] = {0, 0, 0, 0}, slow = 0;
            if (special) {
#pragma unroll
                for (int r = 0; r < 4; ++r) G[r] = (((special >> (4 * r)) & 0xFu) * 0x00204081u) & 0x01010101u;
                uint32_t rs = run2;
                while (rs) {
                    const uint32_t j = __ffs(rs) - 1u;
                    rs &= rs - 1u;
                    const uint32_t sb = STOP >> j;
                    const uint32_t len = sb ? (uint32_t)__ffs(sb) - 1u : 16u - j + fwd;
                    const uint32_t r = j >> 2;
                    const uint32_t cb = len <= kTabMaxRun ? (len - 1u) << (8u * (j & 3u)) : 0u;
                    if (len > kTabMaxRun) slow |= 1u << r;  // generic path (also: several tokens beyond 16662)
#pragma unroll
                    for (int rr = 0; rr < 4; ++rr)
                        if (r == (uint32_t)rr) x[rr] |= cb;  // (the slow path masks the byte out again)
                }
            }
            // ---- look-ups and slot concatenation, word by word (last slot first)
            uint32_t lo[4], hi[4], bits[4];
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const uint2 e0 = lds_v2(tab_s + 8u * prmt(x[r], G[r], 0xCC40u)), e1 = lds_v2(tab_s + 8u * prmt(x[r], G[r], 0xDD51u));
                const uint2 e2 = lds_v2(tab_s + 8u * prmt(x[r], G[r], 0xEE62u)), e3 = lds_v2(tab_s + 8u * prmt(x[r], G[r], 0xFF73u));
                uint32_t l = e3.x, h = 0;
                h = shf_l_c(l, h, e2.y); l = shl_c(l, e2.y) | e2.x;
                h = shf_l_c(l, h, e1.y); l = shl_c(l, e1.y) | e1.x;
                h = shf_l_c(l, h, e0.y); l = shl_c(l, e0.y) | e0.x;
                lo[r] = l; hi[r] = h;
                bits[r] = e0.y + e1.y + e2.y + e3.y;
                if (bits[r] > 64u) slow |= 1u << r;
            }
            if (__any_sync(0xFFFFFFFFu, slow != 0u)) {
                // undo the run-length bytes, then measure the slow words with the generic walker
                if (slow) {
#pragma unroll
                    for (int r = 0; r < 4; ++r)
                        if ((slow >> r) & 1u) {
                            const uint32_t zb = (((Z >> (4 * r)) & 0xFu) * 0x00204081u) & 0x01010101u;
                            x[r] &= ~(zb * 0xFFu);
                            const uint32_t sb = r < 3 ? STOP >> (4 * r + 4) : 0u;
                            const uint32_t fw = sb ? (uint32_t)__ffs(sb) - 1u : 12u - 4u * r + fwd;
                            LenSink ls{s_codes, 0};
                            walk_word(x[r], (NZ >> (4 * r)) & 0xFu, (starts >> (4 * r)) & 0xFu, (STOP >> (4 * r)) & 0xFu, fw, ls);
                            bits[r] = ls.bits;
                        }
                }
            }
            // ---- bit offsets
            const uint32_t lbits = bits[0] + bits[1] + bits[2] + bits[3];
            uint32_t inc = lbits;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, inc, o);
                if (lane >= (uint32_t)o) inc += y;
            }
            if (lane == 31) s_tot[g & 1][wid] = inc;
            __syncthreads();
            uint32_t tw2 = lane < kEncWarps ? s_tot[g & 1][lane] : 0u;
#pragma unroll
            for (int o = 1; o < kEncWarps; o <<= 1) {
                const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, tw2, o);
                if (lane >= (uint32_t)o) tw2 += y;
            }
            uint32_t o = base + (wid ? __shfl_sync(0xFFFFFFFFu, tw2, wid - 1) : 0u) + inc - lbits;
            base += __shfl_sync(0xFFFFFFFFu, tw2, kEncWarps - 1);
            // ---- decode index: the lane whose tokens cover the last bit before an interval boundary names the
            // boundary behind its chunk: the next token starts at its end bit, at the first byte that follows
            // the zeros running out of the chunk
            if (my_idx) {
                const uint32_t e = o + lbits - lead_bits;   // payload bit offsets
                const uint32_t kk = idx_interval_of(ig, e);
                if (kk != idx_interval_of(ig, o - lead_bits)) {
                    const uint32_t P = min(off + 16u + (leaves ? fwd : 0u), n);
                    my_idx[kk] = (e - kk * ig.bits) | (P << kIdxPosShift);
                }
            }
            // ---- emit
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                if (bits[r]) {
                    if ((slow >> r) & 1u) {
                        const uint32_t sb = r < 3 ? STOP >> (4 * r + 4) : 0u;
                        const uint32_t fw = sb ? (uint32_t)__ffs(sb) - 1u : 12u - 4u * r + fwd;
                        EmitSink es{s_codes, pay, 0ull, o & 31u, o >> 5, true};
                        walk_word(x[r], (NZ >> (4 * r)) & 0xFu, (starts >> (4 * r)) & 0xFu, (STOP >> (4 * r)) & 0xFu, fw, es);
                        es.finish();
                    } else {
                        // <= 64 bits: shift to the bit offset, OR into <= 3 staging words
                        const uint32_t sh = o & 31u;
                        const uint32_t wa = pay_s + 4u * (o >> 5);
                        const uint32_t v0 = lo[r] << sh, v1 = __funnelshift_l(lo[r], hi[r], sh), v2 = __funnelshift_l(hi[r], 0u, sh);
                        reds_or(wa, v0);
                        if (v1) reds_or(wa + 4u, v1);
                        if (v2) reds_or(wa + 8u, v2);
                    }
                }
                o += bits[r];
            }
        }
        __syncthreads();
    }
    const uint32_t crc = block_crc32c(pay, plen, s_zt, cc, s_red, lead);
    if (tid == 0) {
        uint8_t* hb = sbytes + hoff;
        hb[0] = (uint8_t)(plen - 1); hb[1] = (uint8_t)((plen - 1) >> 8);
        hb[2] = (uint8_t)crc; hb[3] = (uint8_t)(crc >> 8); hb[4] = (uint8_t)(crc >> 16); hb[5] = (uint8_t)(crc >> 24);
        hb[6] = (uint8_t)bi.mode;
    }
    fence_async_smem();   // the staging was written by ordinary stores and reductions; the bulk store reads it
    __syncthreads();
    copy_smem_to_global_bulk(out, sbytes + hoff, 7u + plen);
}

// stand-alone CRC-32C of a global buffer of <= 65536 bytes (tests / rspt_gpu_crc32c)
__global__ void __launch_bounds__(1024) k_crc32c(const uint8_t* __restrict__ data, uint32_t n,
                                                  const CrcConst* __restrict__ cc, int zt_sel, uint32_t* out)
{
    extern __shared__ __align__(16) uint32_t stg[];
    __shared__ uint32_t s_zt[1024];
    __shared__ uint32_t s_red[33];
    uint8_t* sb = reinterpret_cast<uint8_t*>(stg);
    for (uint32_t i = threadIdx.x; i < ((n + 3) >> 2) + 1; i += blockDim.x) stg[i] = 0;
    for (uint32_t i = threadIdx.x; i < 1024; i += blockDim.x) s_zt[i] = __ldg(&cc->zt[zt_sel][0][0] + i);
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) sb[i] = data[i];
    __syncthreads();
    const uint32_t crc = block_crc32c(stg, n, s_zt, cc, s_red);
    if (threadIdx.x == 0) *out = crc;
}

}  // namespace rspt
