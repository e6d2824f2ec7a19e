// Host-side state behind an rspt_gpu_packer handle (one per reference packer instance).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <vector>

#include "common.cuh"
#include "hzr_encode.cuh"

// streams, events and double buffers of the pipelined host-buffer compress (rspt_gpu_compress_batch_host)
struct HostPipe {
    cudaStream_t s_in, s_out;
    cudaEvent_t ev_in[2], ev_comp[2], ev_off[2], ev_out[2];
    uint8_t* d_src[2];
    uint8_t* d_dst[2];
    uint64_t* d_off[2];
    uint64_t* h_off[2];
    size_t chunk;  // frames per chunk; 0 = not set up yet
};

struct rspt_gpu_packer {
    rspt::Shape s;
    int device;
    cudaStream_t stream;
    bool own_stream;
    size_t max_batch;
    size_t enc_smem;       // dynamic shared memory of k_hzr_encode (staging of the largest block)
    size_t dec_smem;       // dynamic shared memory of k_hzr_decode (payload of the largest block)
    bool can_escalate;     // xdelta_hzr with nb < bps
    bool dct_direct;       // dct: O(n^2) bit-exact path (fixed at create time)

    // compress scratch
    uint8_t* d_planes;
    uint32_t* d_hist;
    uint32_t* d_codes;
    uint32_t* d_tree;
    uint32_t* d_lists;     // per block: sorted non-zero bytes (position | value << 16) of sparse blocks, kListCap entries
    uint32_t* d_list_n;    // per block: entries in d_lists, kNoList = dense block
    uint8_t* d_blk_class;  // per block: kClassSparse / kClassDense (density probe of the histogram launches)
    cudaStream_t side;     // sparse-class histogram + trees run here, beside the dense class on `stream`
    cudaEvent_t ev_fork, ev_join, ev_fork2, ev_join2;
    cudaStream_t place;    // multi-GPU placement (all-gather of totals + offset rebase) runs here, off the compute stream
    cudaEvent_t ev_place;
    // placements possibly still in flight, by the offsets array they rewrite: a later compress into the same
    // array waits for its own entry only (rspt_gpu_place_offsets_async)
    static constexpr int kPlaceRing = 4;
    cudaEvent_t ev_placed[kPlaceRing];
    const void* placed_ptr[kPlaceRing];
    unsigned place_seq;
    uint64_t* d_all_totals;
    uint16_t* d_step_lz;   // per 512-byte step of every block: leading zero count (512 = all zero)
    rspt::BlkInfo* d_info;
    uint8_t* d_frame_nb;
    uint32_t* d_need;
    uint32_t* d_nb_state;
    uint32_t* d_sizes;
    uint32_t* d_blk_off;   // per block: offset of its header from the frame start
    uint8_t* d_headers;
    int32_t* d_words;      // hadamard / dct: de-interleaved samples, then coefficients
    long long* d_sums;     // hadamard / dct: per (frame, channel) sample sums
    rspt::Counters* d_ctr;
    const rspt::CrcConst* d_crc;
    // decompress scratch
    void* d_dec;           // block descriptors
    uint8_t* d_dec_nb;     // per-frame plane count used by the last decompress
    int32_t* d_status_tmp;
    void* d_auto_index;    // decode index built here for streams that came without one
    double* d_fir;         // FIR kernel coefficients of the last rspt_gpu_prefilter_fir call (lazy)
    size_t fir_cap;
    int32_t* d_words2;     // second word buffer (FIR is out of place), lazy
    uint32_t sp_stage;     // payload limit of k_hzr_encode_sparse (kSpStageBytes; lower only under RSPT_SPARSE_STAGE_BYTES)
    // transform constants (dct twiddles)
    double2* d_twiddle;
    double2* d_post;
    float* d_cos;          // dct direct path: the reference's float cosine table
    // single-frame host API staging
    uint8_t* d_one_src;
    uint8_t* d_one_dst;
    uint64_t* d_one_off;
    uint8_t* h_pin;
    size_t h_pin_bytes;
    // host batch API staging (grown on demand)
    uint8_t* d_hb_src;
    uint8_t* d_hb_dst;
    uint64_t* d_hb_off;
    size_t hb_frames;
    HostPipe pipe;

    unsigned long long launches;
    // stage timing
    bool timing;
    std::vector<cudaEvent_t>* ev_free;
    struct Pending { int stage; cudaEvent_t a, b; };
    std::vector<Pending>* ev_pending;
    double stage_ms[8];
    unsigned long long stage_calls[8];
    char err[256];
};

namespace rspt {

inline int fail_cuda(rspt_gpu_packer* p, cudaError_t e, const char* what)
{
    if (p) snprintf(p->err, sizeof(p->err), "CUDA error %d (%s) at %s", (int)e, cudaGetErrorString(e), what);
    return -2;  // RSPT_E_CUDA
}

inline int fail_arg(rspt_gpu_packer* p, const char* what)
{
    if (p) snprintf(p->err, sizeof(p->err), "%s", what);
    return -1;  // RSPT_E_ARG
}

}  // namespace rspt
