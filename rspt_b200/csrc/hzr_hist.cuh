// hzr token histogram for sm_100a: one CTA per hzr block, 16 bytes per lane, 512 bytes per
// warp-step.  Replaces Histogram (lib_hzr/hzr_encode.c:133-173).  Two launches (k_hzr_hist<3>,
// k_hzr_hist<2>) split the blocks by a density probe: sparse-looking blocks are tokenised from a
// sorted list of their non-zero bytes (described at the kernel), dense-looking ones by the scan
// described here.
//
// Tokens (hzr_encode.c:140-170): every non-zero byte is a literal; every maximal zero run inside
// the block is cut greedily into chunks of <= 16662 and each chunk becomes one of the symbols
// 0 (run of 1), 256 (run of 2), 257..260 (longer runs, with extra bits).  The literal counts are
// order-free; only the zero runs need structure (dense scan):
//   * a warp owns a CONTIGUOUS range of steps and walks it in order, so the zeros pending at the
//     end of one step are simply carried in a (warp-uniform) register to the next;
//   * inside a step every lane turns its 16 bytes into a 16-bit "stop" mask (non-zero or beyond
//     the block end).  Isolated zeros (both neighbours non-zero) are symbol 0 and are counted
//     with one popc; runs of >= 2 that start in a lane are measured against the lane's own stop
//     bits or, through one ballot + shuffle, against the next lane that has a stop bit;
//   * runs that touch the step start / end are not counted locally: the step reports its leading
//     and trailing zero counts, the warp chains them across its steps, and thread 0 chains the
//     (at most 8) warp ranges at the end.
// The per-step leading-zero counts are also written out (step_lz): k_hzr_encode uses them to
// measure runs that leave a step without re-reading the block.
#pragma once

#include "common.cuh"
#include "hzr_tree.cuh"

namespace rspt {

constexpr int kHistThreads = 256;
constexpr int kStepBytes = 512;                     // one warp-step: 32 lanes x 16 bytes
constexpr int kMaxSteps = kBlock / kStepBytes;      // 128 per block
constexpr uint32_t kStepAllZero = kStepBytes;       // step_lz value of a step without any stop byte

// 4-bit mask of the non-zero bytes of a word
__device__ __forceinline__ uint32_t nz_nibble(uint32_t x)
{
    const uint32_t t = (((x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | x) & 0x80808080u;
    return (t * 0x00204081u) >> 28;  // bits 7,15,23,31 -> bits 28..31
}

__device__ __forceinline__ uint32_t nz_mask16(const uint4& v)
{
    return nz_nibble(v.x) | (nz_nibble(v.y) << 4) | (nz_nibble(v.z) << 8) | (nz_nibble(v.w) << 12);
}

// One lane's view of a warp-step.
struct Chunk {
    uint4 v;         // the 16 bytes (garbage beyond `valid`)
    int valid;       // bytes of the block in this chunk, 0..16
    uint32_t nz;     // non-zero valid bytes
    uint32_t stop;   // nz | bytes beyond the block end: everything that terminates a zero run
    uint32_t z;      // valid zero bytes
};

__device__ __forceinline__ Chunk load_chunk(const uint8_t* __restrict__ blk, uint32_t n, uint32_t off)
{
    Chunk c;
    const int valid = (int)n - (int)off;
    c.valid = valid < 0 ? 0 : (valid > 16 ? 16 : valid);
    c.v = make_uint4(0, 0, 0, 0);
    if (c.valid > 0) c.v = __ldg(reinterpret_cast<const uint4*>(blk + off));
    const uint32_t vm = (1u << c.valid) - 1u;
    c.nz = ((c.v.x | c.v.y | c.v.z | c.v.w) == 0u) ? 0u : (nz_mask16(c.v) & vm);
    c.stop = c.nz | (0xFFFFu & ~vm);
    c.z = ~c.stop & 0xFFFFu;
    return c;
}

// zero flags of the neighbouring bytes inside the step; bytes outside the step count as zero so
// that runs touching the step boundary are never treated as closed
__device__ __forceinline__ void neighbour_zero(uint32_t z, uint32_t& prevz, uint32_t& nextz)
{
    const uint32_t up = __shfl_up_sync(0xFFFFFFFFu, z, 1), dn = __shfl_down_sync(0xFFFFFFFFu, z, 1);
    prevz = lane_id() > 0 ? (up >> 15) & 1u : 1u;
    nextz = lane_id() < 31 ? dn & 1u : 1u;
}

// count the tokens of one zero run of z >= 1 bytes; run[0] = symbol 0, run[1..5] = symbols 256..260
// (branch-free class: 1 | 2 | 3-6 | 7-22 | 23-278 | 279-16662, hzr_encode.c:152-166)
__device__ __forceinline__ void hist_run(uint32_t z, uint32_t* run)
{
    while (z > kRunCap) {
        atomicAdd(&run[5], 1u);
        z -= kRunCap;
    }
    const uint32_t idx = (z >= 2u) + (z >= 3u) + (z >= 7u) + (z >= 23u) + (z >= 279u);
    atomicAdd(&run[idx], 1u);
}

// ---- sparse blocks ---------------------------------------------------------------------------
// A block with few non-zero bytes (<= kListCap, i.e. mostly long zero runs: the upper byte planes
// of a delta-coded signal) is tokenised from a sorted list of its non-zero bytes.  Those bytes are
// clustered (~80 % of the steps hold some, ~4 of 32 chunks each), so the list is built in two light phases:
//   1. every warp only COUNTS the non-zero bytes of its contiguous range of <= 16 steps and notes, per
//      lane, which of its steps have a non-zero chunk (one bit each); one reduction per warp gives the
//      warp total;
//   2. after the block scan of the totals, the warp walks its steps that have a non-zero chunk: those
//      lanes reload their chunk into a 512-byte per-warp slot of shared memory, and the chunks are
//      served two at a time by half a warp each (lane p of the half reads byte p); a ballot of the
//      kept bytes gives their order, and a warp-uniform running count gives their list index
//      (position | value << 16, in shared memory);
//   3. token histogram from the list: a literal per entry, a zero run per gap.
// No per-step prefix scan and no per-step registers are needed, so the kernel fits 32 registers.
// The list goes to global memory for k_hzr_encode_sparse, which packs the block's payload without
// reading the plane again.  Blocks that are too dense for the list take the dense scan below.
constexpr uint32_t kListCap = 5120;                 // entries of a block's sparse list
constexpr uint8_t kClassSparse = 0, kClassDense = 1;  // blk_class: which histogram launch (and tree launch) owns the block
constexpr size_t kHistSmem = (size_t)kListCap * 4;
constexpr int kHistSteps = kMaxSteps / (kHistThreads / 32);      // steps per warp: 16
constexpr size_t kHistSmemList = kHistSmem + (size_t)(kHistThreads / 32) * kStepBytes;

// Two independent launches per batch, each over all blocks; the density probe (deterministic, the
// same in both) assigns every block to exactly one of them and is recorded in blk_class:
//   PART 3 takes the sparse-looking blocks (list + histogram; if the list overflows after all, the
//          dense scan runs here too -- rare);
//   PART 2 takes the dense-looking blocks (dense scan).
// They run on two streams: the tree build of the dense class (long, latency-bound) then overlaps
// with the sparse part.
template <int PART>
__global__ void __launch_bounds__(kHistThreads, 8) k_hzr_hist(const uint8_t* __restrict__ planes, Shape s,
                                                               const uint8_t* __restrict__ frame_nb,
                                                               uint32_t* __restrict__ hist,
                                                               uint16_t* __restrict__ step_lz,
                                                               uint32_t* __restrict__ lists, uint32_t* __restrict__ list_n,
                                                               uint8_t* __restrict__ blk_class)
{
    extern __shared__ __align__(16) uint32_t s_list[];  // sparse list under construction
    __shared__ uint32_t s_lit[256];  // raw byte counts; [0] is scratch (zeros are tokenised as runs)
    __shared__ uint32_t s_run[8];
    __shared__ uint32_t s_wsum[kHistThreads / 32][3];  // per warp range: seen, lead, trail
    __shared__ uint32_t s_wtot[kHistThreads / 32];
    uint32_t f, k, b;
    const uint32_t blk = blockIdx.x;
    blk_decode(s, blk, f, k, b);
    if (k >= frame_nb[f]) return;
    const uint32_t n = blk_len(s, b);
    const uint8_t* src = blk_ptr(planes, s, f, k, b);
    for (uint32_t i = threadIdx.x; i < 256; i += blockDim.x) s_lit[i] = 0;
    if (threadIdx.x < 8) s_run[threadIdx.x] = 0;

    const uint32_t tid = threadIdx.x, lane = lane_id(), wid = warp_id(), nwarps = blockDim.x >> 5;
    const uint32_t nsteps = (n + kStepBytes - 1) / kStepBytes;
    const uint32_t spw = (nsteps + nwarps - 1) / nwarps;
    const uint32_t s_lo = min(nsteps, wid * spw), s_hi = min(nsteps, s_lo + spw);

    // density probe: the first chunk of every warp range (spread over the block)
    {
        const Chunk probe = load_chunk(src, n, s_lo * kStepBytes + lane * 16u);
        const int dense_chunks = __syncthreads_count(__popc(probe.nz) >= 2);
        const int probed = __syncthreads_count(probe.valid > 0);
        const bool dense_class = dense_chunks * 4 > probed;
        if (tid == 0) blk_class[blk] = dense_class ? kClassDense : kClassSparse;  // both parts write the same value
        if (dense_class != (PART == 2)) return;  // the other launch owns this block
    }
    // ---- sparse path
    if (PART != 2) {
    do {
        uint32_t* list = s_list;
        uint32_t m = 0;
        // 1. count the non-zero bytes of my warp's range; bit j of smask: my chunk of step s_lo + j has some
        uint32_t cnt = 0, smask = 0;
#pragma unroll
        for (int j0 = 0; j0 < kHistSteps; j0 += 4) {
            uint4 v[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const uint32_t st = s_lo + j0 + j, off = st * kStepBytes + lane * 16u;
                v[j] = make_uint4(0, 0, 0, 0);
                if (st < s_hi && off < n) v[j] = __ldg(reinterpret_cast<const uint4*>(src + off));
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                if ((v[j].x | v[j].y | v[j].z | v[j].w) != 0u) {
                    const int valid = (int)n - (int)((s_lo + j0 + j) * kStepBytes + lane * 16u);  // > 0 here
                    const uint32_t c = __popc(nz_mask16(v[j]) & (valid >= 16 ? 0xFFFFu : (1u << valid) - 1u));
                    cnt += c;
                    smask |= (c != 0u ? 1u : 0u) << (j0 + j);
                }
            }
        }
        const uint32_t wtot = __reduce_add_sync(0xFFFFFFFFu, cnt);
        if (lane == 0) s_wtot[wid] = wtot;
        __syncthreads();
        uint32_t at = 0;  // list index of the next entry of my warp (warp-uniform)
        for (uint32_t w = 0; w < nwarps; ++w) {
            const uint32_t t = s_wtot[w];
            if (w < wid) at += t;
            m += t;
        }
        if (m > kListCap || m > n / 4u) break;

        // 2. scatter: chunks staged in my warp's slot, two per iteration, lane p of a half takes byte p
        uint4* slot = reinterpret_cast<uint4*>(s_list + kListCap) + wid * 32u;
        const uint8_t* slot_b = reinterpret_cast<const uint8_t*>(slot);
        const uint32_t p = lane & 15u, below = (1u << lane) - 1u;
        for (uint32_t steps = __reduce_or_sync(0xFFFFFFFFu, smask); steps; steps &= steps - 1u) {
            const uint32_t j = __ffs(steps) - 1u, st_off = (s_lo + j) * kStepBytes;
            const bool mine = (smask >> j) & 1u;
            if (mine) slot[lane] = __ldg(reinterpret_cast<const uint4*>(src + st_off + lane * 16u));
            uint32_t todo = __ballot_sync(0xFFFFFFFFu, mine);
            __syncwarp();
            while (todo) {
                const uint32_t la = __ffs(todo) - 1u;
                todo &= todo - 1u;
                uint32_t lb = la;  // odd count: the upper half reads the same chunk and keeps nothing
                if (todo) {
                    lb = __ffs(todo) - 1u;
                    todo &= todo - 1u;
                }
                const uint32_t sl = lane < 16 ? la : lb, pos = st_off + sl * 16u + p;
                const uint32_t x = slot_b[sl * 16u + p];
                const bool keep = x != 0u && pos < n && (lane < 16 || lb != la);
                const uint32_t kept = __ballot_sync(0xFFFFFFFFu, keep);
                if (keep) list[at + __popc(kept & below)] = pos | (x << 16);
                at += __popc(kept);
            }
            __syncwarp();  // the slot is read before the next step overwrites it
        }
        __syncthreads();

        // 3. token histogram: entry i < m = zeros (prev, cur) + the literal at cur; entry m = zeros up to n
        for (uint32_t i = tid; i <= m; i += blockDim.x) {
            const uint32_t rs = i ? (list[i - 1] & 0xFFFFu) + 1u : 0u;
            uint32_t cur = n;
            if (i < m) {
                const uint32_t e = list[i];
                cur = e & 0xFFFFu;
                atomicAdd(&s_lit[e >> 16], 1u);
            }
            if (cur > rs) hist_run(cur - rs, s_run);
        }
        __syncthreads();
        uint32_t* glist = lists + (size_t)blk * kListCap;
        for (uint32_t i = tid; i < m; i += blockDim.x) glist[i] = list[i];
        if (tid == 0) list_n[blk] = m;
        uint32_t* out = hist + (size_t)blk * kSymStride;
        for (uint32_t i = tid; i < kSymStride; i += blockDim.x)
            out[i] = i == 0 ? s_run[0] : (i < 256 ? s_lit[i] : (i < (uint32_t)kNumSymbols ? s_run[i - 255] : 0u));
        return;
    } while (0);
    // the list overflowed: undo the partial counts and take the dense scan
    __syncthreads();
    for (uint32_t i = tid; i < 256; i += blockDim.x) s_lit[i] = 0;
    if (tid < 8) s_run[tid] = 0;
    }
    if (tid == 0) list_n[blk] = kNoList;
    __syncthreads();

    // ---- dense blocks
    uint16_t* my_lz = step_lz + (size_t)blk * kMaxSteps;
    uint32_t pending = 0, lead = 0, cnt_a = 0, cnt_b = 0;  // packed per-thread counts of the short run classes
    bool seen = false;
    for (uint32_t st = s_lo; st < s_hi; ++st) {
        const Chunk c = load_chunk(src, n, st * kStepBytes + lane * 16u);
        const uint32_t anyt = __ballot_sync(0xFFFFFFFFu, c.stop != 0u);
        if (anyt == 0u) {
            if (lane == 0) my_lz[st] = (uint16_t)kStepAllZero;
            pending += kStepBytes;
            continue;
        }
        // literals: one shared-memory atomic per byte; zero bytes of a non-empty chunk land in the
        // scratch bin 0 (measured: ATOMS costs one issue slot + one cycle per bank-conflict way)
        if (c.nz) {
            const uint32_t w[4] = {c.v.x, c.v.y, c.v.z, c.v.w};
            if (c.valid == 16) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    atomicAdd(&s_lit[w[j] & 0xFFu], 1u);
                    atomicAdd(&s_lit[(w[j] >> 8) & 0xFFu], 1u);
                    atomicAdd(&s_lit[(w[j] >> 16) & 0xFFu], 1u);
                    atomicAdd(&s_lit[w[j] >> 24], 1u);
                }
            } else {
#pragma unroll
                for (int j = 0; j < 16; ++j)
                    if ((c.nz >> j) & 1u) atomicAdd(&s_lit[(w[j >> 2] >> (8 * (j & 3))) & 0xFFu], 1u);
            }
        }
        // zero runs closed inside the step
        uint32_t prevz, nextz;
        neighbour_zero(c.z, prevz, nextz);
        const uint32_t starts = c.z & ~((c.z << 1) | prevz);
        const uint32_t cont = (c.z >> 1) | (nextz << 15);  // the byte after is a zero too
        const uint32_t rs2 = starts & cont;                // first zero of a run of >= 2
        // runs that END inside the chunk are classified for all 16 positions at once: aK has bit p set when
        // the K bytes from p on are zeros of this chunk (hzr_encode.c:152-166; such a run is < 16 long)
        const uint32_t a2 = c.z & (c.z >> 1), a3 = a2 & (c.z >> 2), a4 = a2 & (a2 >> 2), a7 = a4 & (a3 >> 4);
        // the run that reaches the chunk's last byte (if any) is measured across lanes below
        const uint32_t top = c.stop ? 32u - (uint32_t)__clz((int)c.stop) : 0u;  // first byte after the last stop
        const uint32_t open_bit = (c.z >> 15) << top;
        const uint32_t closed = rs2 & ~open_bit;
        cnt_a += __popc(starts & ~cont) | (__popc(closed & ~a3) << 16);            // runs of 1 | runs of 2
        cnt_b += __popc(closed & a3 & ~a7) | (__popc(closed & a7) << 16);          // runs of 3-6 | 7-22
        // position of the first / last stop bit of every lane, for the neighbours
        const uint32_t first_stop = c.stop ? (uint32_t)__ffs(c.stop) - 1u : 16u;
        const bool open_run = (rs2 & open_bit) != 0u;
        if (__any_sync(0xFFFFFFFFu, open_run)) {
            const uint32_t above = lane < 31 ? anyt & ~((2u << lane) - 1u) : 0u;
            const uint32_t q = above ? (uint32_t)__ffs(above) - 1u : 0u;
            const uint32_t fq = __shfl_sync(0xFFFFFFFFu, first_stop, q);
            // zeros after my chunk up to the next stop; without one the run leaves the step and is part of
            // the step's trailing zeros
            if (open_run && above) hist_run(16u - top + 16u * (q - lane - 1u) + fq, s_run);
        }
        // chain the step's leading / trailing zeros along the warp's range
        const uint32_t qf = (uint32_t)__ffs(anyt) - 1u, ql = 31u - (uint32_t)__clz((int)anyt);
        const uint32_t lz = 16u * qf + __shfl_sync(0xFFFFFFFFu, first_stop, qf);
        const uint32_t last_stop = c.stop ? 31u - (uint32_t)__clz((int)c.stop) : 0u;
        const uint32_t tz = 16u * (31u - ql) + 15u - __shfl_sync(0xFFFFFFFFu, last_stop, ql);
        if (lane == 0) my_lz[st] = (uint16_t)lz;
        const uint32_t run = pending + lz;
        if (!seen) {
            lead = run;
            seen = true;
        } else if (run && lane == 0) {
            hist_run(run, s_run);
        }
        pending = tz;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        cnt_a += __shfl_xor_sync(0xFFFFFFFFu, cnt_a, o);  // <= 16 steps x 8 runs x 32 lanes per field
        cnt_b += __shfl_xor_sync(0xFFFFFFFFu, cnt_b, o);
    }
    if (lane == 0) {
        if (cnt_a & 0xFFFFu) atomicAdd(&s_run[0], cnt_a & 0xFFFFu);
        if (cnt_a >> 16) atomicAdd(&s_run[1], cnt_a >> 16);
        if (cnt_b & 0xFFFFu) atomicAdd(&s_run[2], cnt_b & 0xFFFFu);
        if (cnt_b >> 16) atomicAdd(&s_run[3], cnt_b >> 16);
        s_wsum[wid][0] = seen;
        s_wsum[wid][1] = lead;
        s_wsum[wid][2] = pending;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t pend = 0;
        for (uint32_t w = 0; w < nwarps; ++w) {
            if (!s_wsum[w][0]) {
                pend += s_wsum[w][2];
            } else {
                const uint32_t run = pend + s_wsum[w][1];
                if (run) hist_run(run, s_run);
                pend = s_wsum[w][2];
            }
        }
        if (pend) hist_run(pend, s_run);
    }
    __syncthreads();
    uint32_t* out = hist + (size_t)blk * kSymStride;
    for (uint32_t i = threadIdx.x; i < kSymStride; i += blockDim.x)
        out[i] = i == 0 ? s_run[0] : (i < 256 ? s_lit[i] : (i < (uint32_t)kNumSymbols ? s_run[i - 255] : 0u));
}

}  // namespace rspt
