// Host-side state behind an rspt_gpu_packer handle (one per reference packer instance).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <mutex>
#include <type_traits>
#include <utility>
#include <vector>

#include "common.cuh"
#include "hzr_encode.cuh"

namespace rspt {

struct DecBlk;
struct DeviceFree { void operator()(void* q) const { cudaFree(q); } };
struct PinnedFree { void operator()(void* q) const { cudaFreeHost(q); } };
struct StreamDestroy { void operator()(cudaStream_t s) const { cudaStreamDestroy(s); } };
struct EventDestroy { void operator()(cudaEvent_t e) const { cudaEventDestroy(e); } };

// Sole owner of one CUDA resource, released by Release when the owner is destroyed or reset.  It converts to the
// raw handle, so that it is used where the handle is.
template <class H, class Release>
class Owned {
public:
    Owned() = default;
    Owned(Owned&& o) noexcept : h_(o.release()) {}
    Owned& operator=(Owned&& o) noexcept { reset(o.release()); return *this; }
    ~Owned() { reset(); }
    operator H() const { return h_; }
    void reset(H h = nullptr) { if (h_) Release()(h_); h_ = h; }
    H release() { return std::exchange(h_, nullptr); }
    // make_raw(&h) creates a resource; only if it succeeds does the owner take it, releasing the one it held
    template <class Make>
    cudaError_t make(Make&& make_raw)
    {
        H h = nullptr;
        const cudaError_t e = make_raw(&h);
        if (e == cudaSuccess) reset(h);
        return e;
    }

private:
    H h_ = nullptr;
};

template <class T> using DeviceBuf = Owned<T*, DeviceFree>;
template <class T> using PinnedBuf = Owned<T*, PinnedFree>;
using Stream = Owned<cudaStream_t, StreamDestroy>;
using Event = Owned<cudaEvent_t, EventDestroy>;

// count elements and `slack` bytes of device memory
template <class T>
cudaError_t dalloc(DeviceBuf<T>& b, size_t count, size_t slack = 64)
{
    return b.make([&](T** q) { return cudaMalloc(reinterpret_cast<void**>(q), count * sizeof(T) + slack); });
}

template <class T>
cudaError_t palloc(PinnedBuf<T>& b, size_t count)
{
    return b.make([&](T** q) { return cudaMallocHost(reinterpret_cast<void**>(q), count * sizeof(T)); });
}

inline cudaError_t create(Stream& s)
{
    return s.make([](cudaStream_t* h) { return cudaStreamCreateWithFlags(h, cudaStreamNonBlocking); });
}

inline cudaError_t create(Event& ev, unsigned flags = cudaEventDisableTiming)
{
    return ev.make([&](cudaEvent_t* h) { return cudaEventCreateWithFlags(h, flags); });
}

}  // namespace rspt

// streams, events and double buffers of the pipelined host-buffer compress (rspt_gpu_compress_batch_host)
struct HostPipe {
    rspt::Stream s_in, s_out;
    rspt::Event ev_in[2], ev_comp[2], ev_off[2], ev_out[2];
    rspt::DeviceBuf<uint8_t> d_src[2];
    rspt::DeviceBuf<uint8_t> d_dst[2];
    rspt::DeviceBuf<uint64_t> d_off[2];
    rspt::PinnedBuf<uint64_t> h_off[2];
    size_t chunk = 0;  // frames per chunk; 0 = not set up yet
};

struct rspt_gpu_packer {
    rspt::Shape s{};
    int device = 0;
    cudaStream_t stream = nullptr;          // the caller's
    size_t max_batch = 0;
    size_t enc_smem = 0;                    // dynamic shared memory of k_hzr_encode (staging of the largest block)
    size_t dec_smem = 0;                    // dynamic shared memory of k_hzr_decode (payload of the largest block)
    bool can_escalate = false;              // xdelta_hzr with nb < bps
    bool dct_direct = false;                // dct: O(n^2) bit-exact path; set only while d_cos holds the cosine table

    // compress scratch
    rspt::DeviceBuf<uint8_t> d_planes;
    rspt::DeviceBuf<uint32_t> d_hist;
    rspt::DeviceBuf<uint32_t> d_codes;
    rspt::DeviceBuf<uint32_t> d_tree;
    rspt::DeviceBuf<uint32_t> d_lists;      // per block: sorted non-zero bytes (position | value << 16) of sparse blocks, kListCap entries
    rspt::DeviceBuf<uint32_t> d_list_n;     // per block: entries in d_lists, kNoList = dense block
    rspt::DeviceBuf<uint8_t> d_blk_class;   // per block: kClassSparse / kClassDense (density probe of the histogram launches)
    rspt::Stream side;                      // sparse-class histogram + trees run here, beside the dense class on `stream`
    // fork_side / join_side: one pair serves every fork and join of a call, since cudaStreamWaitEvent waits for
    // the event's last record before the wait was enqueued
    rspt::Event ev_fork, ev_join;
    rspt::Stream place;                     // multi-GPU placement (all-gather of totals + offset rebase) runs here, off the compute stream
    rspt::Event ev_place;
    // placements possibly still in flight, by the offsets array they rewrite: a later compress into the same
    // array waits for its own entry only (rspt_gpu_place_offsets_async)
    static constexpr int kPlaceRing = 4;
    rspt::Event ev_placed[kPlaceRing];
    const void* placed_ptr[kPlaceRing] = {};
    unsigned place_seq = 0;
    rspt::DeviceBuf<uint64_t> d_all_totals;
    rspt::DeviceBuf<uint16_t> d_step_lz;    // per 512-byte step of every block: leading zero count (512 = all zero)
    rspt::DeviceBuf<rspt::BlkInfo> d_info;
    rspt::DeviceBuf<uint8_t> d_frame_nb;
    rspt::DeviceBuf<uint32_t> d_need;
    rspt::DeviceBuf<uint32_t> d_nb_state;
    rspt::DeviceBuf<uint32_t> d_sizes;
    rspt::DeviceBuf<uint32_t> d_blk_off;    // per block: offset of its header from the frame start
    rspt::DeviceBuf<uint8_t> d_headers;
    rspt::DeviceBuf<int32_t> d_words;       // hadamard / dct: de-interleaved samples, then coefficients
    rspt::DeviceBuf<long long> d_sums;      // hadamard / dct: per (frame, channel) sample sums
    rspt::DeviceBuf<rspt::Counters> d_ctr;
    const rspt::CrcConst* d_crc = nullptr;  // per device, for the life of the process
    // decompress scratch
    rspt::DeviceBuf<rspt::DecBlk> d_dec;    // block descriptors
    rspt::DeviceBuf<uint8_t> d_dec_nb;      // per-frame plane count used by the last decompress
    rspt::DeviceBuf<int32_t> d_status_tmp;
    rspt::DeviceBuf<uint32_t> d_auto_index; // decode index built here for streams that came without one
    rspt::DeviceBuf<double> d_fir;          // FIR kernel coefficients of the last rspt_gpu_prefilter_fir call (lazy)
    size_t fir_cap = 0;                     // coefficients d_fir holds room for
    rspt::DeviceBuf<int32_t> d_words2;      // second word buffer (FIR is out of place), lazy
    uint32_t sp_stage = 0;                  // payload limit of k_hzr_encode_sparse (kSpStageBytes; lower only under RSPT_SPARSE_STAGE_BYTES)
    // transform constants (dct twiddles)
    rspt::DeviceBuf<double2> d_twiddle;
    rspt::DeviceBuf<double2> d_post;
    rspt::DeviceBuf<float> d_cos;           // dct direct path: the reference's float cosine table
    // single-frame host API staging
    rspt::DeviceBuf<uint8_t> d_one_src;
    rspt::DeviceBuf<uint8_t> d_one_dst;
    rspt::DeviceBuf<uint64_t> d_one_off;
    rspt::PinnedBuf<uint8_t> h_pin;
    HostPipe pipe;

    unsigned long long launches = 0;
    // stage timing
    bool timing = false;
    std::vector<rspt::Event> ev_free;
    struct Pending { int stage; rspt::Event a, b; };
    std::vector<Pending> ev_pending;
    double stage_ms[8] = {};
    unsigned long long stage_calls[8] = {};
    char err[256] = {};
};

namespace rspt {

inline int fail_cuda(rspt_gpu_packer* p, cudaError_t e, const char* what)
{
    // the failed call's error is also the thread's last error: cleared, or the next launch reports it as its own
    cudaGetLastError();
    if (p) snprintf(p->err, sizeof(p->err), "CUDA error %d (%s) at %s", (int)e, cudaGetErrorString(e), what);
    return -2;  // RSPT_E_CUDA
}

inline int fail_arg(rspt_gpu_packer* p, const char* what)
{
    if (p) snprintf(p->err, sizeof(p->err), "%s", what);
    return -1;  // RSPT_E_ARG
}

// f(std::integral_constant<int, bps>{}) for bps 1..4 (anything above as 4): names a kernel template's
// instantiation from a run-time value.  f returns a status.  The return type is int, not deduced, so that
// the kernels f names are instantiated at the end of the translation unit: the order in which it first names
// its kernels orders their extern shared-memory declarations, which decides where k_hzr_hist<3>'s dynamic
// shared memory starts.
template <class F>
int with_bps(int bps, F&& f)
{
    switch (bps) {
    case 1: return f(std::integral_constant<int, 1>{});
    case 2: return f(std::integral_constant<int, 2>{});
    case 3: return f(std::integral_constant<int, 3>{});
    default: return f(std::integral_constant<int, 4>{});
    }
}

template <class F>
int with_flag(bool b, F&& f)
{
    return b ? f(std::true_type{}) : f(std::false_type{});
}

// The dynamic shared-memory limit belongs to the kernel, for the whole process and device, not to a handle.
// It only ever goes up, so that no handle can lower it under another handle's launch; the check and the raise
// hold one process mutex.
template <class K>
cudaError_t raise_smem_limit(K* kernel, size_t bytes)
{
    static std::mutex mu;
    std::lock_guard<std::mutex> lk(mu);
    cudaFuncAttributes a;
    cudaError_t e = cudaFuncGetAttributes(&a, kernel);
    if (e == cudaSuccess && (size_t)a.maxDynamicSharedSizeBytes < bytes)
        e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    return e;
}

// kernel<<<grid, block, smem, stream>>>(args...) and the launch's error.  A kernel's dynamic shared-memory limit
// starts at 48 KB minus its static shared memory.  Above 48 KB this raises the limit to smem.  Below, a kernel
// with static shared memory of its own can still need a raised limit: rspt_gpu_create raises the hzr kernels
// (up to 12 544 bytes of static shared memory) to the most any handle launches them with.
template <class... P, class... A>
cudaError_t launch(cudaStream_t stream, void (*kernel)(P...), dim3 grid, dim3 block, size_t smem, A&&... args)
{
    if (smem > 48 * 1024) {
        const cudaError_t e = raise_smem_limit(kernel, smem);
        if (e != cudaSuccess) return e;
    }
    kernel<<<grid, block, smem, stream>>>(std::forward<A>(args)...);
    return cudaGetLastError();
}

// the same on one of the handle's streams, counted in p->launches
template <class... P, class... A>
int launch(rspt_gpu_packer* p, cudaStream_t stream, void (*kernel)(P...), dim3 grid, dim3 block, size_t smem, A&&... args)
{
    p->launches += 1;
    RSPT_CUDA_CHECK(launch(stream, kernel, grid, block, smem, std::forward<A>(args)...));
    return 0;
}

template <class... P, class... A>
int launch(rspt_gpu_packer* p, void (*kernel)(P...), dim3 grid, dim3 block, size_t smem, A&&... args)
{
    return launch(p, p->stream, kernel, grid, block, smem, std::forward<A>(args)...);
}

// p->side starts behind the work enqueued on p->stream so far
inline int fork_side(rspt_gpu_packer* p)
{
    RSPT_CUDA_CHECK(cudaEventRecord(p->ev_fork, p->stream));
    RSPT_CUDA_CHECK(cudaStreamWaitEvent(p->side, p->ev_fork, 0));
    return 0;
}

// p->stream continues behind the work enqueued on p->side so far
inline int join_side(rspt_gpu_packer* p)
{
    RSPT_CUDA_CHECK(cudaEventRecord(p->ev_join, p->side));
    RSPT_CUDA_CHECK(cudaStreamWaitEvent(p->stream, p->ev_join, 0));
    return 0;
}

}  // namespace rspt
