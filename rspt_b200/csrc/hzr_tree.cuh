// hzr tree build for sm_100a: one warp per hzr block.
//
// Replaces MakeTree (lib_hzr/hzr_encode.c:222-283), StoreTree (:177-219), OnlySingleCode
// (:285-305) and the size / mode decision of EncodeSingleBlock (:377-382, :399-405, :466-467).
// hzr's Huffman code is NOT canonical: code words follow the exact merge order of MakeTree, whose
// selection loop (:247-261) picks, every round, the two live nodes that are smallest under the key
// (count ascending, node index descending) -- leaves are indexed in ascending symbol order and
// internal nodes after them in creation order.  child_a = the smallest, child_b = the second;
// the code of child_b gets bit `depth` set (LSB-first codes); the tree is serialised pre-order,
// branch = 0, leaf = 1 + 9-bit symbol.
//
// Phases (all 32 lanes unless noted):
//   A  load the 261 counts, classify (FILL?), compact the used symbols into sort keys
//      count << 9 | (511 - symbol), sort ascending in registers (one key per lane and
//      shuffles for <= 32 symbols; otherwise K keys per lane over 32 * K >= L slots)
//   B  lane 0: two-queue merge (sorted leaves / internal nodes in creation order).  Internal
//      nodes win ties against leaves; inside a run of equal-weight internal nodes the most
//      recently created one is taken first -- exactly MakeTree's tie-break.  Also counts the
//      leaves below every internal node.
//   C  breadth-first top-down pass, one frontier node per lane: depth, code and pre-order bit
//      offset of every node.  A subtree with l leaves serialises to 11*l - 1 bits, which places
//      child_b without walking child_a.  Leaves are finished as they are reached: code table
//      entry, tree bits, payload bit total, maximum code length.
#pragma once

#include "common.cuh"

namespace rspt {

constexpr int kTreeWarps = 2;  // trees per CTA (5.6 KB of shared memory each: 40 trees per SM)
constexpr uint32_t kLeafSlots = 264;       // node[0, kLeafSlots): leaves by rank; internal node j is node[kLeafSlots + j]
constexpr uint32_t kNodeInf = 0x7FFFFFFFu; // an internal slot not filled yet: heavier than any leaf

struct TreeWarpSmem {
    // leaf r: its sort key (+inf from L on).  Internal node j, phase B: weight << 9 | leaves below;
    // phase C: its code.  A node's id is its slot.
    uint32_t node[kLeafSlots + 260];
    uint32_t child[260];       // internal node j: child_a id | child_b id << 10
    uint32_t ninfo[260];       // C: depth | pre-order bit offset << 8
    uint32_t tree[kTreeWords];
    uint16_t front[2][264];    // C: breadth-first frontiers (internal node indices)
    uint32_t pad;              // odd word stride between the warps' trees; part of the measured shared-memory footprint
};

struct Counters {
    unsigned long long frames_compressed, frames_decompressed, raw_bytes_in, compressed_bytes_out;
    unsigned long long blocks_copy, blocks_huff, blocks_fill, escalations;
    unsigned long long crc_failures;
};

// Block addressing: blk = (f * nb_alloc + k) * nblk + b
__device__ __forceinline__ void blk_decode(const Shape& s, uint32_t blk, uint32_t& f, uint32_t& k, uint32_t& b)
{
    b = blk % s.nblk;
    uint32_t fk = blk / s.nblk;
    k = fk % s.nb_alloc;
    f = fk / s.nb_alloc;
}

__device__ __forceinline__ const uint8_t* blk_ptr(const uint8_t* planes, const Shape& s, uint32_t f, uint32_t k, uint32_t b)
{
    return planes + ((size_t)f * s.nb_alloc + k) * s.plane_stride + (size_t)b * kBlock;
}

// The tree build of one block in three parts (several trees sharing a warp for the serial part was
// measured and is slower: 4 merges side by side in one warp's lanes diverge on every pick and leave
// too few warps to hide the latency of the cooperative parts).  h = the block's 261 token counts (global or shared memory), n = block length.
// tree_prepare and tree_assign are warp-cooperative; tree_merge is ONE thread's job.

// Bitonic sort of key[0..L), L <= 32 * K, with K keys per lane in registers: slot lane * K + r,
// slots from L on +inf.  The network is in its all-ascending form (the first step of every merge
// pairs slot i with its mirror image i ^ (kk - 1)), so no compare depends on a direction: strides
// below K are min/max pairs inside a lane, strides >= K one shuffle and one min-or-max per key.
// Writes every slot below kLeafSlots back (+inf from L on).
template <int K>
__device__ __forceinline__ void warp_sort_regs(uint32_t* key, const uint32_t L)
{
    const uint32_t lane = lane_id();
    uint32_t v[K];
#pragma unroll
    for (int r = 0; r < K; ++r) v[r] = lane * K + r < L ? key[lane * K + r] : 0xFFFFFFFFu;
    auto cas = [&](int r, int q) {  // r < q
        const uint32_t a = v[r], b = v[q];
        v[r] = min(a, b);
        v[q] = max(a, b);
    };
#pragma unroll
    for (int kk = 2; kk <= 32 * K; kk <<= 1) {
        if (kk <= K) {
#pragma unroll
            for (int r = 0; r < K; ++r)
                if (!(r & (kk >> 1))) cas(r, r ^ (kk - 1));
        } else {
            // mirror step across lanes: lane ^ (kk / K - 1), key K - 1 - r
            const bool lower = (lane & (kk / K / 2)) == 0;
#pragma unroll
            for (int r = 0; r < K / 2; ++r) {
                const uint32_t o0 = __shfl_xor_sync(0xFFFFFFFFu, v[K - 1 - r], kk / K - 1);
                const uint32_t o1 = __shfl_xor_sync(0xFFFFFFFFu, v[r], kk / K - 1);
                v[r] = lower ? min(v[r], o0) : max(v[r], o0);
                v[K - 1 - r] = lower ? min(v[K - 1 - r], o1) : max(v[K - 1 - r], o1);
            }
        }
#pragma unroll
        for (int j = kk >> 2; j > 0; j >>= 1) {
            if (j >= K) {
                const bool lower = (lane & (j / K)) == 0;
#pragma unroll
                for (int r = 0; r < K; ++r) {
                    const uint32_t o = __shfl_xor_sync(0xFFFFFFFFu, v[r], j / K);
                    v[r] = lower ? min(v[r], o) : max(v[r], o);
                }
            } else {
#pragma unroll
                for (int r = 0; r < K; ++r)
                    if (!(r & j)) cas(r, r | j);
            }
        }
    }
#pragma unroll
    for (int r = 0; r < K; ++r)
        if (lane * K + r < kLeafSlots) key[lane * K + r] = v[r];
}

// Part 1: classify (FILL?), compact the used symbols into sort keys, sort.  Returns true when the
// block is a FILL (bi is final then).  Unused symbols get code table entry 0.
__device__ __forceinline__ bool tree_prepare(TreeWarpSmem& S, const uint32_t* h, uint32_t* codes_out, uint32_t& L_out, BlkInfo& bi)
{
    const uint32_t lane = lane_id();
    // ---- phase A: classify and compact
    uint32_t L = 0, nz = 0, nzsym = 0, zero_class = 0;
    uint32_t mykey = 0xFFFFFFFFu;  // register copy for the <= 32 symbol network
#pragma unroll
    for (int r = 0; r < 9; ++r) {
        const uint32_t sym = r * 32 + lane;
        const uint32_t c = sym < kNumSymbols ? h[sym] : 0u;
        const bool used = c != 0;
        const uint32_t m = __ballot_sync(0xFFFFFFFFu, used);
        const uint32_t pos = L + __popc(m & ((1u << lane) - 1u));
        if (used) S.node[pos] = (c << 9) | (511u - sym);
        else if (sym < (uint32_t)kSymStride) codes_out[sym] = 0;  // 0 = symbol has no code
        L += __popc(m);
        if (r == 0) {
            zero_class |= m & 1u;
            const uint32_t mm = m & ~1u;
            nz += __popc(mm);
            if (mm) nzsym = __ffs(mm) - 1;
        } else if (r < 8) {
            nz += __popc(m);
            if (m && !nzsym) nzsym = r * 32 + __ffs(m) - 1;
        } else {
            zero_class |= m != 0;
        }
    }
    if (nz + (zero_class ? 1u : 0u) == 1u) {
        // single value class -> FILL (OnlySingleCode); payload is in[0]
        bi.payload_len = 1; bi.total_bits = 8; bi.tree_nbits = 0;
        bi.mode = MODE_FILL; bi.fill = (uint8_t)(nz ? nzsym : 0u); bi.n_used = (uint16_t)L; bi.n_tokens = 0;
        L_out = L;
        return true;
    }
    __syncwarp();
    if (L <= 32) {
        // one key per lane, bitonic network over the warp
        mykey = lane < L ? S.node[lane] : 0xFFFFFFFFu;
#pragma unroll
        for (uint32_t kk = 2; kk <= 32; kk <<= 1)
#pragma unroll
            for (uint32_t j = kk >> 1; j > 0; j >>= 1) {
                const uint32_t other = __shfl_xor_sync(0xFFFFFFFFu, mykey, j);
                const bool up = (lane & kk) == 0, lower = (lane & j) == 0;
                mykey = (lower == up) ? min(mykey, other) : max(mykey, other);
            }
        S.node[lane] = mykey;
    } else if (L <= 64) {
        warp_sort_regs<2>(S.node, L);
    } else if (L <= 128) {
        warp_sort_regs<4>(S.node, L);
    } else if (L <= 256) {
        warp_sort_regs<8>(S.node, L);
    } else {
        warp_sort_regs<16>(S.node, L);
    }
    for (uint32_t i = lane; i < kTreeWords; i += 32) S.tree[i] = 0;
    for (uint32_t i = lane; i < 260; i += 32) S.node[kLeafSlots + i] = kNodeInf;
    __syncwarp();

    L_out = L;
    return false;
}

// Part 2 (one thread): two-queue merge.  Internal nodes are kept in pick order: weights never
// decrease, and a run of equal weights goes latest first, so a node as heavy as the one before it
// takes the first slot of that run and the run moves up one slot.  A run is complete before its
// first node is taken (a node made later is heavier) and no node of it has a parent yet, so the
// move renames nothing.  Registers hold both queue heads: the leaf head as lc = key | 511 for the
// compare (an internal node of equal weight compares <= it: internal nodes win ties; its word is
// lc - 510), the internal head as ic = its word.  Words are weight << 9 | leaves below, so a new node's
// word is the sum of its children's.  A pick loads the next head of the queue it took from,
// node[id + 1]: +inf past the last leaf and in internal slots not filled yet.
__device__ __forceinline__ void tree_merge(TreeWarpSmem& S, const uint32_t L)
{
    uint32_t* node = S.node;
    node[L] = 0xFFFFFFFFu;  // the slot after the last leaf (the sorts leave it unwritten when L = 32 * K)
    uint32_t hl = 0, lc = node[0] | 511u;
    uint32_t hi = kLeafSlots, ic = kNodeInf;
    uint32_t last = 0, run = kLeafSlots;  // weight field of the newest node | 511; first slot of its run
    auto pick = [&](uint32_t& id, uint32_t& v) {
        const bool take = ic <= lc;
        id = take ? hi : hl;
        v = take ? ic : lc - 510u;  // a leaf's word: count << 9 | 1
        const uint32_t raw = node[id + 1];
        hi += take;
        hl += !take;
        if (take) ic = raw;
        else lc = raw | 511u;
    };
    for (uint32_t n = kLeafSlots; n < kLeafSlots + L - 1; ++n) {
        uint32_t a, b, va, vb;
        pick(a, va);
        pick(b, vb);
        const uint32_t w = va + vb, ch = a | (b << 10);
        uint32_t at = n;
        if (w <= last) {
#pragma unroll 1
            for (; at > run; --at) {
                node[at] = node[at - 1];
                S.child[at - kLeafSlots] = S.child[at - 1 - kLeafSlots];
            }
        } else {
            run = n;
        }
        node[at] = w;
        S.child[at - kLeafSlots] = ch;
        if (hi == at) ic = w;  // the new node is the internal head
        last = w | 511u;
    }
    // root = last internal node: depth 0, code 0, pre-order offset 0
    node[kLeafSlots + L - 2] = 0;
    S.ninfo[L - 2] = 0;
    S.front[0][0] = (uint16_t)(L - 2);
}

// Part 3: codes, tree bits and the block's plan (returned in every lane).
__device__ __forceinline__ BlkInfo tree_assign(TreeWarpSmem& S, const uint32_t L, uint32_t n, uint32_t* codes_out, uint32_t* tree_out)
{
    const uint32_t lane = lane_id();
    BlkInfo bi;
    // ---- phase C: breadth-first top-down pass, one frontier node per lane: depth, code and
    // pre-order bit offset of both children.  A leaf child is finished on the spot: code table
    // entry, its 10 tree bits (1 + 9-bit symbol), its share of the payload bit total.
    uint32_t token_bits = 0, maxlen = 0, ntok = 0;
    {
        auto leaf = [&](uint32_t rank, uint32_t code, uint32_t depth, uint32_t off) {
            const uint32_t kv = S.node[rank];
            const uint32_t sym = 511u - (kv & 511u), cnt = kv >> 9;
            codes_out[sym] = code | (depth << 27);
            token_bits += cnt * (depth + sym_extra_bits(sym));
            ntok += cnt;
            maxlen = max(maxlen, depth);
            const unsigned long long bits = (unsigned long long)(1u | (sym << 1)) << (off & 31u);
            atomicOr(&S.tree[off >> 5], (uint32_t)bits);
            if (bits >> 32) atomicOr(&S.tree[(off >> 5) + 1], (uint32_t)(bits >> 32));
        };
        uint32_t nf = 1, cur = 0;
        const uint32_t lt = (1u << lane) - 1u;
        while (nf) {
            uint32_t nn = 0;
            for (uint32_t fb = 0; fb < nf; fb += 32) {
                const uint32_t i = fb + lane;
                const bool act = i < nf;
                uint32_t a = 0, bb = 0;
                if (act) {
                    const uint32_t j = S.front[cur][i];
                    const uint32_t ch = S.child[j], code = S.node[kLeafSlots + j], inf = S.ninfo[j];
                    const uint32_t depth = inf & 255u, off = inf >> 8;
                    a = ch & 1023u;
                    bb = ch >> 10;
                    uint32_t bits_a = 10;
                    if (a < kLeafSlots) {
                        leaf(a, code, depth + 1u, off + 1u);
                    } else {
                        // node[a] still holds the merge's word: leaves below it in the low 9 bits
                        bits_a = 11u * (S.node[a] & 511u) - 1u;
                        S.node[a] = code;
                        S.ninfo[a - kLeafSlots] = (depth + 1u) | ((off + 1u) << 8);
                    }
                    const uint32_t code_b = code | (1u << depth), off_b = off + 1u + bits_a;
                    if (bb < kLeafSlots) {
                        leaf(bb, code_b, depth + 1u, off_b);
                    } else {
                        S.node[bb] = code_b;
                        S.ninfo[bb - kLeafSlots] = (depth + 1u) | (off_b << 8);
                    }
                }
                const bool ia = act && a >= kLeafSlots, ib = act && bb >= kLeafSlots;
                const uint32_t ma = __ballot_sync(0xFFFFFFFFu, ia), mb = __ballot_sync(0xFFFFFFFFu, ib);
                if (ia) S.front[cur ^ 1][nn + __popc(ma & lt)] = (uint16_t)(a - kLeafSlots);
                nn += __popc(ma);
                if (ib) S.front[cur ^ 1][nn + __popc(mb & lt)] = (uint16_t)(bb - kLeafSlots);
                nn += __popc(mb);
            }
            __syncwarp();
            cur ^= 1;
            nf = nn;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        token_bits += __shfl_xor_sync(0xFFFFFFFFu, token_bits, o);
        ntok += __shfl_xor_sync(0xFFFFFFFFu, ntok, o);
        maxlen = max(maxlen, __shfl_xor_sync(0xFFFFFFFFu, maxlen, o));
    }
    __syncwarp();
    const uint32_t tree_nbits = 11u * L - 1u;
    for (uint32_t i = lane; i < ((tree_nbits + 31u) >> 5); i += 32) tree_out[i] = S.tree[i];
    bi.tree_nbits = (uint16_t)tree_nbits;
    bi.total_bits = tree_nbits + token_bits;
    const uint32_t bytes = (bi.total_bits + 7u) >> 3;
    // capped block stream (hzr_encode.c:377-382), 16-bit size field (:466-467); codes longer
    // than 27 bits cannot occur for <= 65536 tokens (Fibonacci bound ~ 23)
    const bool copy = bytes > n || bytes >= kBlock || maxlen > 27u;
    bi.mode = copy ? MODE_COPY : MODE_HUFF;
    bi.payload_len = copy ? n : bytes;
    bi.fill = (uint8_t)maxlen;  // HUFF: longest code word (selects the encoder's merge width)
    bi.n_used = (uint16_t)L;
    bi.n_tokens = (uint16_t)min(ntok, 65535u);
    return bi;
}

// Build the tree of one block with one warp.  Writes the code table (code | length << 27, 0 = unused
// symbol) to codes_out[0..263] and the serialised tree to tree_out (global or shared memory).
// Returns the block's plan in every lane.  Touches no counters.
__device__ __forceinline__ BlkInfo warp_build_tree(TreeWarpSmem& S, const uint32_t* h, uint32_t n,
                                                   uint32_t* codes_out, uint32_t* tree_out)
{
    BlkInfo bi;
    uint32_t L;
    if (tree_prepare(S, h, codes_out, L, bi)) return bi;
    if (lane_id() == 0) tree_merge(S, L);
    __syncwarp();
    return tree_assign(S, L, n, codes_out, tree_out);
}

__device__ __forceinline__ void count_block_mode(Counters* ctr, uint32_t mode)
{
    atomicAdd(mode == MODE_FILL ? &ctr->blocks_fill : (mode == MODE_COPY ? &ctr->blocks_copy : &ctr->blocks_huff), 1ull);
}

// One warp per block of the class `cls` (blk_class is written by the histogram launches).  20 CTAs per SM
// keep 40 trees resident (as the shared memory allows), which caps the registers at 48.
__global__ void __launch_bounds__(kTreeWarps * 32, 20) k_hzr_tree(const uint32_t* __restrict__ hist, Shape s,
                                                               const uint8_t* __restrict__ frame_nb,
                                                               const uint8_t* __restrict__ blk_class, uint32_t cls,
                                                               uint32_t total_blocks,
                                                               uint32_t* __restrict__ codes,
                                                               uint32_t* __restrict__ tree,
                                                               BlkInfo* __restrict__ info,
                                                               Counters* __restrict__ ctr)
{
    __shared__ TreeWarpSmem s_all[kTreeWarps];
    TreeWarpSmem& S = s_all[warp_id()];
    const uint32_t blk = blockIdx.x * kTreeWarps + warp_id();
    if (blk >= total_blocks) return;
    uint32_t f, k, b;
    blk_decode(s, blk, f, k, b);
    if (k >= frame_nb[f] || blk_class[blk] != cls) return;
    const uint32_t n = blk_len(s, b);
    const BlkInfo bi = warp_build_tree(S, hist + (size_t)blk * kSymStride, n, codes + (size_t)blk * kSymStride, tree + (size_t)blk * kTreeWords);
    if (lane_id() == 0) {
        info[blk] = bi;
        count_block_mode(ctr, bi.mode);
    }
}

}  // namespace rspt
