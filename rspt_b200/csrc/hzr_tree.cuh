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
//      count << 9 | (511 - symbol), sort ascending (register bitonic network for <= 32 symbols,
//      shared-memory bitonic network otherwise)
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

struct TreeWarpSmem {
    uint32_t key[264];         // sorted leaf keys
    uint32_t icnt[260];        // B: internal node weight (| bit 31: next node has equal weight); C: node code
    uint32_t child[260];       // child_a | child_b << 10 | leaves below << 20; ids < 512 are leaf ranks, 512 + j internal node j
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
        if (used) S.key[pos] = (c << 9) | (511u - sym);
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
        mykey = lane < L ? S.key[lane] : 0xFFFFFFFFu;
#pragma unroll
        for (uint32_t kk = 2; kk <= 32; kk <<= 1)
#pragma unroll
            for (uint32_t j = kk >> 1; j > 0; j >>= 1) {
                const uint32_t other = __shfl_xor_sync(0xFFFFFFFFu, mykey, j);
                const bool up = (lane & kk) == 0, lower = (lane & j) == 0;
                mykey = (lower == up) ? min(mykey, other) : max(mykey, other);
            }
        S.key[lane] = mykey;
    } else {
        // bitonic network in its all-ascending form (the first step of every merge mirrors the
        // upper half), so the slots from L up to the next power of two are virtual +infinity
        // and need no storage: a compare whose upper partner is >= L is a no-op
        uint32_t P = 64;
        while (P < L) P <<= 1;
        for (uint32_t kk = 2; kk <= P; kk <<= 1) {
            for (uint32_t j = kk >> 1; j > 0; j >>= 1) {
                const bool mirror = j == (kk >> 1);
                for (uint32_t idx = lane; idx < (P >> 1); idx += 32) {
                    const uint32_t i = ((idx & ~(j - 1)) << 1) | (idx & (j - 1));
                    const uint32_t ixj = mirror ? i ^ (kk - 1u) : i | j;
                    if (ixj < L) {
                        const uint32_t a = S.key[i], c2 = S.key[ixj];
                        if (a > c2) {
                            S.key[i] = c2;
                            S.key[ixj] = a;
                        }
                    }
                }
                __syncwarp();
            }
        }
    }
    for (uint32_t i = lane; i < kTreeWords; i += 32) S.tree[i] = 0;
    __syncwarp();

    L_out = L;
    return false;
}

// Part 2 (one thread): two-queue merge.
// Phase B: two-queue merge.  Registers hold both queue heads; an internal node's
// weight word carries a flag "the node created right after me has the same weight", so the
// common pick (a run of one) needs no look-ahead load.
__device__ __forceinline__ void tree_merge(TreeWarpSmem& S, const uint32_t L)
{
    constexpr uint32_t kInf = 0x7FFFFFFFu, kEqNext = 0x80000000u;
    uint32_t li = 0, lc = S.key[0] >> 9;          // leaf queue head
    uint32_t fr = 0, ni = 0, ic = kInf;           // internal queue: head index, count, head weight
    uint32_t icf = 0;                             // head has an equal-weight successor (flag bit)
    uint32_t last_w = kInf;
    // one pick: the lighter head; ties go to the internal node.  Branch-free unless the
    // internal head starts a run of equal weights (then the latest of the run goes first).
    uint32_t top = 0, run_end = 0;
    bool in_run = false;
    auto pick = [&](uint32_t& id, uint32_t& wt, uint32_t& lv) {
        const bool take_int = ic <= lc;
        if (take_int && (in_run || icf)) {
            uint32_t pk;
            bool advance;
            if (!in_run) {
                top = fr + 1;
                while (top < ni && (S.icnt[top] & kInf) == ic) ++top;
                run_end = top;
                in_run = true;
                pk = --top;
                advance = false;  // a flagged run has >= 2 nodes
            } else {
                pk = --top;
                advance = top == fr;
            }
            id = 512u + pk;
            wt = ic;
            lv = S.child[pk] >> 20;
            if (advance) {
                in_run = false;
                fr = run_end;
                const uint32_t raw = fr < ni ? S.icnt[fr] : kInf;
                ic = raw & kInf;
                icf = raw & kEqNext;
            }
            return;
        }
        // heads after this pick, loaded unconditionally (indices stay inside the arrays)
        const uint32_t nfr = fr + (take_int ? 1u : 0u), nli = li + (take_int ? 0u : 1u);
        const uint32_t raw = S.icnt[nfr], nk = S.key[nli], ch = S.child[fr];
        id = take_int ? 512u + fr : li;
        wt = take_int ? ic : lc;
        lv = take_int ? ch >> 20 : 1u;
        if (take_int) {
            ic = nfr < ni ? raw & kInf : kInf;
            icf = nfr < ni ? raw & kEqNext : 0u;
        } else {
            lc = nli < L ? nk >> 9 : kInf;
        }
        fr = nfr;
        li = nli;
    };
    for (uint32_t round = 0; round + 1 < L; ++round) {
        uint32_t id0, id1, w0, w1, lv0, lv1;
        pick(id0, w0, lv0);
        pick(id1, w1, lv1);
        const uint32_t w = w0 + w1;
        if (w == last_w) {
            S.icnt[ni - 1] = w | kEqNext;
            if (ni - 1 == fr) icf = kEqNext;
        }
        if (fr == ni) {
            ic = w;
            icf = 0;
        }
        S.icnt[ni] = w;
        S.child[ni] = id0 | (id1 << 10) | ((lv0 + lv1) << 20);
        last_w = w;
        ++ni;
    }
    // root = last internal node: depth 0, code 0, pre-order offset 0
    S.icnt[L - 2] = 0;
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
            const uint32_t kv = S.key[rank];
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
                    const uint32_t ch = S.child[j], code = S.icnt[j], inf = S.ninfo[j];
                    const uint32_t depth = inf & 255u, off = inf >> 8;
                    a = ch & 1023u;
                    bb = (ch >> 10) & 1023u;
                    uint32_t bits_a = 10;
                    if (a < 512u) {
                        leaf(a, code, depth + 1u, off + 1u);
                    } else {
                        bits_a = 11u * (S.child[a - 512u] >> 20) - 1u;
                        S.icnt[a - 512u] = code;
                        S.ninfo[a - 512u] = (depth + 1u) | ((off + 1u) << 8);
                    }
                    const uint32_t code_b = code | (1u << depth), off_b = off + 1u + bits_a;
                    if (bb < 512u) {
                        leaf(bb, code_b, depth + 1u, off_b);
                    } else {
                        S.icnt[bb - 512u] = code_b;
                        S.ninfo[bb - 512u] = (depth + 1u) | (off_b << 8);
                    }
                }
                const bool ia = act && a >= 512u, ib = act && bb >= 512u;
                const uint32_t ma = __ballot_sync(0xFFFFFFFFu, ia), mb = __ballot_sync(0xFFFFFFFFu, ib);
                if (ia) S.front[cur ^ 1][nn + __popc(ma & lt)] = (uint16_t)(a - 512u);
                nn += __popc(ma);
                if (ib) S.front[cur ^ 1][nn + __popc(mb & lt)] = (uint16_t)(bb - 512u);
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

// One warp per block of the class `cls` (blk_class is written by the histogram launches).
__global__ void __launch_bounds__(kTreeWarps * 32) k_hzr_tree(const uint32_t* __restrict__ hist, Shape s,
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
