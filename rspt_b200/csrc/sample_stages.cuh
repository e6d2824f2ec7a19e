// Host side of the sample stages: stage 1 of compress (samples -> byte planes + header), the last stage of
// decompress (byte planes -> samples) and the pre-filter's conversions between native samples and the int32
// word matrix, for both sample layouts (interleaved native bytes, int32 [ch][ns] words).  Which kernel runs is
// decided here, from the packer, the shape and the alignment of the caller's pointer, and so is its launch
// geometry.  The kernels are in transforms.cuh, xdelta_tma.cuh and spectral.cuh.
#pragma once

#include "../../include/rspt_gpu.h"
#include "packer.cuh"
#include "spectral.cuh"
#include "transforms.cuh"
#include "xdelta_tma.cuh"

namespace rspt {

// ---- shape limits: rspt_gpu_create refuses a shape that fails them, the launches are sized from them --------

constexpr size_t kTileSmemCap = 200 * 1024;  // dynamic shared memory the tile kernels are sized against

// the kPiece-sample tile of k_raw_to_words / k_words_to_raw; k_planes_to_samples stages native samples in one too
inline size_t piece_tile_bytes(const Shape& s) { return (size_t)kPiece * s.ch * s.bps + 48; }

// the carries of k_planes_to_samples: two words per kPiece-sample piece of every channel
inline size_t inv_carry_bytes(const Shape& s)
{
    const uint32_t np = (((uint32_t)s.ns + kPiece - 1) / kPiece) * (uint32_t)s.ch;
    return (size_t)2 * np * 4;
}

// tile height (samples) of k_xdelta_planes and the dynamic shared memory it needs; false = no tile fits
inline bool xdelta_tile(const Shape& s, uint32_t& ts, size_t& smem)
{
    const size_t row = (size_t)s.ch * s.bps, per = row + 4 * (size_t)s.ch;
    const size_t budget = 96 * 1024;
    size_t t = (budget - 64 - 8 * (size_t)s.ch) / per;
    t = t > 512 ? 512 : (t & ~(size_t)31);
    if (t < 32) return false;
    const size_t need_t = ((size_t)s.ns + 31) & ~(size_t)31;
    if (t > need_t) t = need_t;
    ts = (uint32_t)t;
    smem = ((t * row + 31) & ~(size_t)15) + (size_t)s.ch * (t + 2) * 4;
    return true;
}

// the generic tile kernels can stage the shape: the xdelta forward tile, the inverse's carries + sample tile
inline bool sample_tiles_fit(const Shape& s)
{
    uint32_t ts;
    size_t smem;
    if ((s.kind == RSPT_XDELTA_HZR || s.kind == RSPT_HZR) && !xdelta_tile(s, ts, smem)) return false;
    return inv_carry_bytes(s) + piece_tile_bytes(s) <= kTileSmemCap;
}

inline size_t fwht_smem(const Shape& s) { return (size_t)s.ns * 4; }  // k_fwht_fwd / _inv
inline size_t fwht_raw_smem(const Shape& s) { return (size_t)4 * ((size_t)s.ns + s.ns / 32) * 4; }  // k_fwht_raw_*

inline uint32_t fpad_host(uint32_t m) { return m + (m >> 3) + (m >> 6) + 2; }

// k_dct_*_direct: one float per sample; k_dct_*_half: the padded half-length FFT; k_dct_*_fast: ns points
inline size_t dct_smem(const rspt_gpu_packer* p)
{
    const Shape& s = p->s;
    if (p->dct_direct) return (size_t)s.ns * 4;
    return s.ns >= 16 ? (size_t)fpad_host((uint32_t)s.ns / 2) * 16 : (size_t)s.ns * 16;
}

// ---- eligibility of the specialised kernels ------------------------------------------------------------------

// k_xdelta_planes_tma: the shapes it is compiled for, whole tiles of 128 quads, 16-byte aligned input, no
// plane-count probe (that case keeps k_xdelta_planes_fast)
inline bool tma_transform_ok(const rspt_gpu_packer* p, const void* src)
{
    const Shape& s = p->s;
    bool compiled = false;
#define X(B, C) compiled |= s.bps == B && s.ch == C;
    RSPT_TMA_SHAPES(X)
#undef X
    return compiled && !p->can_escalate && ((uintptr_t)src & 15) == 0 && s.ns % (4 * kTmaQuads) == 0 &&
           s.ns >= 4 * kTmaQuads;
}

// quads per tile and dynamic shared memory of k_xdelta_planes_fast; false = shape or pointer not eligible
inline bool xdelta_fast_tile(const Shape& s, const void* src, uint32_t& tsq, size_t& smem)
{
    if ((s.ch & 3) || (s.ns & 3) || s.ns < 4 || ((uintptr_t)src & 15)) return false;
    const size_t row = (size_t)s.ch * s.bps;
    for (uint32_t t = 128; t >= 32; t >>= 1) {
        smem = (size_t)(t + 1) * (row + 1) * 4;
        if (smem <= 56 * 1024) {
            tsq = t;
            return true;
        }
    }
    return false;
}

inline bool fwht_fast_len(int ns) { return ns == 4096 || ns == 8192; }

// the fused hadamard kernels apply: four-channel groups, a transform length with a register path,
// 16-byte aligned frames
inline bool fwht_raw_ok(const Shape& s, const void* raw)
{
    return s.kind == RSPT_HADAMARD && (s.ch & 3) == 0 && fwht_fast_len(s.ns) && ((uintptr_t)raw & 15) == 0 &&
           (s.frame_bytes & 15) == 0;
}

// the four-channel-group word kernels apply (a warp's 32 sample quads stay inside one channel group)
inline bool words_g4_ok(const Shape& s, const void* raw)
{
    return (s.ch & 3) == 0 && (s.ns % 1024) == 0 && ((uintptr_t)raw & 15) == 0 && (s.frame_bytes & 15) == 0;
}

// sample tiles per output group and dynamic shared memory of k_planes_to_samples_fast writing native samples
// (4-channel groups, 128-sample pieces, PRMT packing), sized to keep 4 CTAs per SM; false = not eligible
inline bool inv_fast_tile(const Shape& s, const void* dst, uint32_t& tpg, size_t& smem)
{
    if ((s.ch & 3) || (s.ns % (int)kInvPiece) || ((uintptr_t)dst & 15)) return false;
    const size_t row = (size_t)s.ch * s.bps;
    const size_t npf = (size_t)((uint32_t)s.ns / kInvPiece) * s.ch;  // 128-element pieces per frame
    for (tpg = 8; tpg >= 1; tpg >>= 1) {
        smem = 2 * npf * 4 + (size_t)tpg * 32 * (row + 1) * 4 + (size_t)tpg * 4;  // + one pad word per 32 quads
        if (smem <= 54 * 1024) return true;
    }
    return false;
}

// k_planes_to_samples_fast writing words: the carries of its 128-element pieces
inline size_t inv_words_fast_smem(const Shape& s)
{
    const uint32_t npf = ((uint32_t)s.ns / kInvPiece) * (uint32_t)s.ch;
    return (size_t)2 * npf * 4;
}

// it walks a frame's 128-element pieces four at a time, so their number must be a multiple of 4, and it
// stores 128-bit words
inline bool inv_words_fast_ok(const Shape& s, const void* dst)
{
    const uint32_t npf = ((uint32_t)s.ns / kInvPiece) * (uint32_t)s.ch;
    return (s.ns % (int)kInvPiece) == 0 && (npf & 3u) == 0 && inv_words_fast_smem(s) <= kTileSmemCap &&
           ((uintptr_t)dst & 15) == 0;
}

// ---- native samples <-> the int32 word matrix (hadamard / dct, the pre-filter) --------------------------------

inline unsigned words_g4_grid(const Shape& s, size_t F) { return (unsigned)(F * (s.ch >> 2) * (size_t)(s.ns >> 2) / 256); }

// d_src -> p->d_words; each channel's samples are added to p->d_sums
inline int launch_raw_to_words(rspt_gpu_packer* p, const uint8_t* d_src, size_t F)
{
    const Shape& s = p->s;
    const uint32_t tiles = ((uint32_t)s.ns + kPiece - 1) / kPiece;
    return with_bps(s.bps, [&](auto B) {
        if (words_g4_ok(s, d_src))
            return launch(p, k_raw_to_words_g4<B>, words_g4_grid(s, F), 256, 0, d_src, s, p->d_words, p->d_sums);
        return launch(p, k_raw_to_words<B>, (unsigned)(F * tiles), 256, piece_tile_bytes(s), d_src, s, tiles,
                      p->d_words, p->d_sums);
    });
}

inline int launch_words_to_raw(rspt_gpu_packer* p, const int32_t* words, uint8_t* d_dst, size_t F)
{
    const Shape& s = p->s;
    const uint32_t tiles = ((uint32_t)s.ns + kPiece - 1) / kPiece;
    return with_bps(s.bps, [&](auto B) {
        if (words_g4_ok(s, d_dst)) return launch(p, k_words_to_raw_g4<B>, words_g4_grid(s, F), 256, 0, words, s, d_dst);
        return launch(p, k_words_to_raw<B>, (unsigned)(F * tiles), 256, piece_tile_bytes(s), words, s, tiles, d_dst);
    });
}

// ---- stage 1 of compress: samples -> byte planes (+ header, + need flags) -------------------------------------

// hadamard / dct: the word matrix in p->d_words (+ its per-channel sums in p->d_sums) -> planes + header
inline int spectral_words_forward(rspt_gpu_packer* p, size_t F)
{
    const Shape& s = p->s;
    const dim3 g2((unsigned)(F * s.ch));
    if (s.kind == RSPT_HADAMARD) {
        if (fwht_fast_len(s.ns))
            return with_flag(s.ns == 4096, [&](auto n4096) {
                constexpr int LG = n4096 ? 12 : 13;
                return launch(p, k_fwht_fast_fwd<LG>, g2, (1 << LG) / 16, 0, p->d_words, p->d_sums, s, p->d_planes,
                              p->d_headers);
            });
        return launch(p, k_fwht_fwd, g2, 256, fwht_smem(s), p->d_words, p->d_sums, s, p->d_planes, p->d_headers);
    }
    int rc;
    if (p->dct_direct)
        rc = launch(p, k_dct_fwd_direct, g2, 256, dct_smem(p), p->d_words, p->d_sums, s, p->d_cos, p->d_headers);
    else if (s.ns >= 16)
        rc = launch(p, k_dct_fwd_half, g2, 256, dct_smem(p), p->d_words, p->d_sums, s, p->d_twiddle, p->d_post,
                    p->d_headers);
    else
        rc = launch(p, k_dct_fwd_fast, g2, 256, dct_smem(p), p->d_words, p->d_sums, s, p->d_twiddle, p->d_post,
                    p->d_headers);
    if (rc) return rc;
    const uint32_t chunks = (s.N + 1023) / 1024;
    return launch(p, k_words_stencil_planes, (unsigned)(F * chunks), 256, 0, p->d_words, s, chunks, p->d_planes);
}

inline int launch_forward_transform(rspt_gpu_packer* p, const uint8_t* d_src, size_t F)
{
    const Shape& s = p->s;
    if (s.kind == RSPT_HADAMARD || s.kind == RSPT_DCT) {
        if (fwht_raw_ok(s, d_src))
            return with_flag(s.ns == 4096, [&](auto n4096) {
                constexpr int LG = n4096 ? 12 : 13;
                return with_bps(s.bps, [&](auto B) {
                    return launch(p, k_fwht_raw_fwd<LG, B>, (unsigned)(F * (s.ch >> 2)), (1 << LG) / 16,
                                  fwht_raw_smem(s), d_src, s, p->d_planes, p->d_headers);
                });
            });
        RSPT_CUDA_CHECK(cudaMemsetAsync(p->d_sums, 0, F * s.ch * sizeof(long long), p->stream));
        const int rc = launch_raw_to_words(p, d_src, F);
        return rc ? rc : spectral_words_forward(p, F);
    }
    uint32_t* need = p->can_escalate ? static_cast<uint32_t*>(p->d_need) : nullptr;
    if (need) RSPT_CUDA_CHECK(cudaMemsetAsync(need, 0, F * sizeof(uint32_t), p->stream));
    const bool st = s.kind == RSPT_XDELTA_HZR;
    if (tma_transform_ok(p, d_src)) {
        const uint32_t tiles = (uint32_t)s.ns / (4u * kTmaQuads);
        const size_t smem = (size_t)(kTmaQuads + 2) * 4u * s.ch * s.bps;
#define X(B, C)                                                                                                    \
    if (s.bps == B && s.ch == C)                                                                                   \
        return with_flag(st, [&](auto ST) {                                                                        \
            return launch(p, k_xdelta_planes_tma<B, C, ST>, (unsigned)(F * tiles), kTmaThreads, smem, d_src, s,    \
                          tiles, p->d_planes);                                                                     \
        });
        RSPT_TMA_SHAPES(X)
#undef X
    }
    uint32_t t;
    size_t smem;
    if (xdelta_fast_tile(s, d_src, t, smem)) {
        const uint32_t tiles = (((uint32_t)s.ns >> 2) + t - 1) / t;
        return with_bps(s.bps, [&](auto B) {
            return with_flag(st, [&](auto ST) {
                return launch(p, k_xdelta_planes_fast<B, ST>, (unsigned)(F * tiles), 128, smem, d_src, s, t, tiles,
                              p->d_planes, need);
            });
        });
    }
    xdelta_tile(s, t, smem);  // rspt_gpu_create refuses the shapes without one
    const uint32_t tiles = ((uint32_t)s.ns + t - 1) / t;
    return with_bps(s.bps, [&](auto B) {
        return with_flag(st, [&](auto ST) {
            return launch(p, k_xdelta_planes<B, ST>, (unsigned)(F * tiles), 256, smem, d_src, s, t, tiles, p->d_planes,
                          need);
        });
    });
}

// from int32 [ch][ns] words (rspt_gpu_compress_batch_i32): the same planes, header and need flags
inline int launch_forward_transform_i32(rspt_gpu_packer* p, const int32_t* d_src, size_t F)
{
    const Shape& s = p->s;
    if (s.kind == RSPT_HADAMARD || s.kind == RSPT_DCT) {
        const uint32_t tiles = ((uint32_t)s.ns + 1023) / 1024;
        RSPT_CUDA_CHECK(cudaMemsetAsync(p->d_sums, 0, F * s.ch * sizeof(long long), p->stream));
        const int rc = with_bps(s.bps, [&](auto B) {
            return launch(p, k_i32_to_words<B>, (unsigned)(F * s.ch * tiles), 256, 0, d_src, s, tiles, p->d_words,
                          p->d_sums);
        });
        return rc ? rc : spectral_words_forward(p, F);
    }
    uint32_t* need = p->can_escalate ? static_cast<uint32_t*>(p->d_need) : nullptr;
    if (need) RSPT_CUDA_CHECK(cudaMemsetAsync(need, 0, F * sizeof(uint32_t), p->stream));
    const uint32_t chunks = (s.N + kI32Chunk - 1) / kI32Chunk;
    return with_bps(s.bps, [&](auto B) {
        return with_flag(s.kind == RSPT_XDELTA_HZR, [&](auto ST) {
            return launch(p, k_xdelta_planes_i32<B, ST>, (unsigned)(F * chunks), 256, 0, d_src, s, chunks, p->d_planes,
                          need);
        });
    });
}

// ---- last stage of decompress: byte planes (decoded) -> samples ----------------------------------------------

// hadamard / dct: planes -> the samples as int32 words in `words`.  The dct kernels work in place on the
// coefficient words, so for dct `words` is also their scratch.
inline int spectral_inverse_words(rspt_gpu_packer* p, size_t F, int32_t* words)
{
    const Shape& s = p->s;
    const dim3 g2((unsigned)(F * s.ch));
    if (s.kind == RSPT_HADAMARD) {
        if (fwht_fast_len(s.ns))
            return with_flag(s.ns == 4096, [&](auto n4096) {
                constexpr int LG = n4096 ? 12 : 13;
                return launch(p, k_fwht_fast_inv<LG>, g2, (1 << LG) / 16, 0, p->d_planes, p->d_headers, p->d_dec_nb, s,
                              words);
            });
        return launch(p, k_fwht_inv, g2, 256, fwht_smem(s), p->d_planes, p->d_headers, p->d_dec_nb, s, words);
    }
    // the coefficient words (BPS unused for word output)
    const int rc = inv_words_fast_ok(s, words)
        ? launch(p, k_planes_to_samples_fast<4, true, true>, (unsigned)F, kInvThreads, inv_words_fast_smem(s),
                 p->d_planes, s, p->d_dec_nb, 1, nullptr, words)
        : launch(p, k_planes_to_samples<4, true, false>, (unsigned)F, 512, inv_carry_bytes(s) + piece_tile_bytes(s),
                 p->d_planes, s, p->d_dec_nb, nullptr, words);
    if (rc) return rc;
    if (p->dct_direct) return launch(p, k_dct_inv_direct, g2, 256, dct_smem(p), words, p->d_headers, s, p->d_cos);
    if (s.ns >= 16)
        return launch(p, k_dct_inv_half, g2, 256, dct_smem(p), words, p->d_headers, s, p->d_twiddle, p->d_post);
    return launch(p, k_dct_inv_fast, g2, 256, dct_smem(p), words, p->d_headers, s, p->d_twiddle, p->d_post);
}

inline int launch_inverse_transform(rspt_gpu_packer* p, uint8_t* d_dst, size_t F)
{
    const Shape& s = p->s;
    if (s.kind == RSPT_HADAMARD || s.kind == RSPT_DCT) {
        if (fwht_raw_ok(s, d_dst))
            return with_flag(s.ns == 4096, [&](auto n4096) {
                constexpr int LG = n4096 ? 12 : 13;
                return with_bps(s.bps, [&](auto B) {
                    return launch(p, k_fwht_raw_inv<LG, B>, (unsigned)(F * (s.ch >> 2)), (1 << LG) / 16,
                                  fwht_raw_smem(s), p->d_planes, p->d_headers, p->d_dec_nb, s, d_dst);
                });
            });
        const int rc = spectral_inverse_words(p, F, p->d_words);
        return rc ? rc : launch_words_to_raw(p, p->d_words, d_dst, F);
    }
    uint32_t tpg = 0;
    size_t smem = 0;
    const bool fast = inv_fast_tile(s, d_dst, tpg, smem);
    return with_bps(s.bps, [&](auto B) {
        return with_flag(s.kind == RSPT_XDELTA_HZR, [&](auto SC) {
            if (fast)
                return launch(p, k_planes_to_samples_fast<B, SC>, (unsigned)F, kInvThreads, smem, p->d_planes, s,
                              p->d_dec_nb, tpg, d_dst, nullptr);
            return launch(p, k_planes_to_samples<B, SC, true>, (unsigned)F, 512, inv_carry_bytes(s) + piece_tile_bytes(s),
                          p->d_planes, s, p->d_dec_nb, d_dst, p->d_words);
        });
    });
}

// to int32 [ch][ns] words, sign-extended from 8*bps bits (rspt_gpu_decompress_batch_i32).  d_dst only needs
// 4-byte alignment; 16 bytes let the fast sample kernel store it directly.
inline int launch_inverse_transform_i32(rspt_gpu_packer* p, int32_t* d_dst, size_t F)
{
    const Shape& s = p->s;
    if (s.kind == RSPT_HADAMARD || s.kind == RSPT_DCT) {
        // hadamard's inverse kernels only write their output, so 4-byte samples go straight to the caller;
        // dct transforms its coefficient words in place and keeps the handle's scratch
        int32_t* words = (s.kind == RSPT_HADAMARD && s.bps == 4) ? d_dst : p->d_words;
        const int rc = spectral_inverse_words(p, F, words);
        if (rc || words == d_dst) return rc;
        const size_t n = F * (size_t)s.N;
        return with_bps(s.bps, [&](auto B) {
            return launch(p, k_words_sext<B>, (unsigned)((n + 1023) / 1024), 256, 0, words, n, d_dst);
        });
    }
    const bool fast = inv_words_fast_ok(s, d_dst);
    return with_bps(s.bps, [&](auto B) {
        return with_flag(s.kind == RSPT_XDELTA_HZR, [&](auto SC) {
            if (fast)
                return launch(p, k_planes_to_samples_fast<B, SC, true>, (unsigned)F, kInvThreads, inv_words_fast_smem(s),
                              p->d_planes, s, p->d_dec_nb, 1, nullptr, d_dst);
            return launch(p, k_planes_to_samples<B, SC, false>, (unsigned)F, 512, inv_carry_bytes(s), p->d_planes, s,
                          p->d_dec_nb, nullptr, d_dst);
        });
    });
}

// to float32 / bfloat16 [ch][ns] (rspt_gpu_decompress_*_float, out_type RSPT_OUT_F32 / RSPT_OUT_BF16): the samples
// launch_inverse_transform_i32 writes, dequantized per channel by the kernel that produces them.  The same
// eligibility decides between the same kernels with a float store; hadamard needs no word scratch and no second
// kernel, dct ends in k_words_to_float instead of k_words_sext.  d_dst needs the alignment of its element; 16
// bytes let the fast sample kernel store it directly.
inline int launch_inverse_transform_float(rspt_gpu_packer* p, int out_type, void* d_dst, Dequant dq, size_t F)
{
    const Shape& s = p->s;
    auto run = [&](auto* dst) -> int {
        using OutT = std::remove_pointer_t<decltype(dst)>;
        const dim3 g2((unsigned)(F * s.ch));
        if (s.kind == RSPT_HADAMARD) {
            if (fwht_fast_len(s.ns))
                return with_flag(s.ns == 4096, [&](auto n4096) {
                    constexpr int LG = n4096 ? 12 : 13;
                    return launch(p, k_dq_fwht_fast_inv<LG, OutT>, g2, (1 << LG) / 16, 0, p->d_planes, p->d_headers,
                                  p->d_dec_nb, s, dst, dq);
                });
            return launch(p, k_dq_fwht_inv<OutT>, g2, 256, fwht_smem(s), p->d_planes, p->d_headers, p->d_dec_nb, s, dst, dq);
        }
        if (s.kind == RSPT_DCT) {
            const int rc = spectral_inverse_words(p, F, p->d_words);
            if (rc) return rc;
            const size_t n = F * (size_t)s.N;
            return with_bps(s.bps, [&](auto B) {
                return launch(p, k_words_to_float<B, OutT>, (unsigned)((n + 1023) / 1024), 256, 0, p->d_words, s, n, dst, dq);
            });
        }
        const bool fast = inv_words_fast_ok(s, dst);
        return with_bps(s.bps, [&](auto B) {
            return with_flag(s.kind == RSPT_XDELTA_HZR, [&](auto SC) {
                if (fast)
                    return launch(p, k_dq_planes_to_samples_fast<B, SC, OutT>, (unsigned)F, kInvThreads,
                                  inv_words_fast_smem(s), p->d_planes, s, p->d_dec_nb, dst, dq);
                return launch(p, k_dq_planes_to_samples<B, SC, OutT>, (unsigned)F, 512, inv_carry_bytes(s), p->d_planes,
                              s, p->d_dec_nb, dst, dq);
            });
        });
    };
    return out_type == RSPT_OUT_BF16 ? run(static_cast<__nv_bfloat16*>(d_dst)) : run(static_cast<float*>(d_dst));
}

}  // namespace rspt
