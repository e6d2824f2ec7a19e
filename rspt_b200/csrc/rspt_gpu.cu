// librspt_gpu.so -- C ABI (include/rspt_gpu.h) over the sm_100a signal-packer kernels.
// Host code here only validates arguments, owns device scratch and launches kernels; there is
// no CPU implementation of any stage.
#include "../../include/rspt_gpu.h"
#include "../../include/rspt_synth.h"

#include <dlfcn.h>
#include <stdlib.h>

#include <atomic>
#include <mutex>
#include <new>
#include <vector>

#include "packer.cuh"
#include "transforms.cuh"
#include "xdelta_tma.cuh"
#include "hzr_decode.cuh"
#include "spectral.cuh"
#include "filters.cuh"

using namespace rspt;

// ---------------------------------------------------------------------------------------------
// per-device constants
// ---------------------------------------------------------------------------------------------
namespace {

constexpr int kMaxDevices = 64;
std::mutex g_mu;
CrcConst* g_crc[kMaxDevices] = {};
int32_t* g_synth_tab[kMaxDevices] = {};  // beat[1024] | sine[1024]
// 16-byte result slots of the synchronous helper calls (rspt_gpu_crc32c, rspt_gpu_prdn_terms): a ring per device,
// so that those calls allocate nothing (64 of them may be in flight from different host threads)
uint8_t* g_result_ring[kMaxDevices] = {};
std::atomic<unsigned> g_result_next{0};
void* result_slot(int dev) { return g_result_ring[dev] + 16u * (g_result_next.fetch_add(1) & 63u); }

uint32_t h_multmodp(uint32_t a, uint32_t b)
{
    uint32_t p = 0;
    for (int i = 0; i < 32; ++i) {
        if ((a >> (31 - i)) & 1u) p ^= b;
        b = (b & 1u) ? (b >> 1) ^ 0x82F63B78u : b >> 1;
    }
    return p;
}

uint32_t h_xpow(uint64_t n)  // x^n mod P, reflected
{
    uint32_t sq = 1u << 30, r = 1u << 31;
    while (n) {
        if (n & 1) r = h_multmodp(sq, r);
        sq = h_multmodp(sq, sq);
        n >>= 1;
    }
    return r;
}

int ensure_device_constants(int dev)
{
    std::lock_guard<std::mutex> lk(g_mu);
    if (dev < 0 || dev >= kMaxDevices) return RSPT_E_ARG;
    if (g_crc[dev]) return RSPT_OK;
    std::vector<CrcConst> hc(1);
    CrcConst& c = hc[0];
    for (uint32_t i = 0; i < 256; ++i) {
        uint32_t r = i;
        for (int k = 0; k < 8; ++k) r = (r >> 1) ^ (0x82F63B78u & (0u - (r & 1u)));
        c.byte_tab[i] = r;
    }
    for (uint32_t j = 0; j < 1024; ++j) c.lane_mul[j] = h_xpow(32ull * (j + 1));
    for (int t = 0; t < 4; ++t) {
        const uint32_t T = 128u << t;
        const uint32_t z = h_xpow(32ull * T);
        for (int b = 0; b < 4; ++b)
            for (uint32_t v = 0; v < 256; ++v) c.zt[t][b][v] = h_multmodp(z, v << (8 * b));
    }
    {
        const uint32_t z = h_xpow(32ull * 32);
        for (int b = 0; b < 4; ++b)
            for (uint32_t v = 0; v < 256; ++v) c.zt32[b][v] = h_multmodp(z, v << (8 * b));
    }
    CrcConst* d = nullptr;
    if (cudaMalloc(&d, sizeof(CrcConst)) != cudaSuccess) return RSPT_E_CUDA;
    if (cudaMemcpy(d, &c, sizeof(CrcConst), cudaMemcpyHostToDevice) != cudaSuccess) return RSPT_E_CUDA;
    std::vector<int32_t> tab(2 * RSPT_SYNTH_TABLE);
    rspt_synth_build_tables(tab.data(), tab.data() + RSPT_SYNTH_TABLE);
    int32_t* dt = nullptr;
    if (cudaMalloc(&dt, tab.size() * sizeof(int32_t)) != cudaSuccess) return RSPT_E_CUDA;
    if (cudaMemcpy(dt, tab.data(), tab.size() * sizeof(int32_t), cudaMemcpyHostToDevice) != cudaSuccess) return RSPT_E_CUDA;
    uint8_t* ring = nullptr;
    if (cudaMalloc(&ring, 64 * 16) != cudaSuccess) return RSPT_E_CUDA;
    g_result_ring[dev] = ring;
    g_crc[dev] = d;
    g_synth_tab[dev] = dt;
    return RSPT_OK;
}

size_t hzr_max(size_t n) { return 4 + (n ? ((n + kBlock - 1) / kBlock) * 7 + n : 0); }

template <class T>
cudaError_t dalloc(T*& ptr, size_t count)
{
    return cudaMalloc(reinterpret_cast<void**>(&ptr), count * sizeof(T) + 64);
}

template <class K>
cudaError_t allow_smem(K kernel, size_t bytes)
{
    return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev)
    {
        cudaGetDevice(&prev);
        if (prev != dev) cudaSetDevice(dev);
        else prev = -1;
    }
    ~DeviceGuard()
    {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

void destroy_host_pipe(rspt_gpu_packer* p);

uint32_t total_blocks(const rspt_gpu_packer* p, size_t frames) { return (uint32_t)(frames * p->s.nb_alloc * p->s.nblk); }

// tile height (samples) of k_xdelta_planes and the dynamic shared memory it needs
bool xdelta_tile(const Shape& s, uint32_t& ts, size_t& smem)
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

// quads per tile and dynamic shared memory of k_xdelta_planes_fast; false = shape not eligible
bool xdelta_fast_tile(const Shape& s, const uint8_t* d_src, uint32_t& tsq, size_t& smem)
{
    if ((s.ch & 3) || (s.ns & 3) || s.ns < 4 || ((uintptr_t)d_src & 15)) return false;
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


#define RSPT_TMA_SHAPES(X) X(2, 4) X(2, 8) X(2, 12) X(3, 4) X(3, 8) X(3, 12) X(4, 4) X(4, 8) X(4, 12)

// shapes k_xdelta_planes_tma is compiled for (RSPT_TMA_SHAPES), whole tiles of 128 quads, 16-byte aligned input
bool tma_transform_ok(const Shape& s, const uint8_t* d_src)
{
    if ((uintptr_t)d_src & 15) return false;
    if (s.bps < 2 || s.bps > 4 || (s.ch != 4 && s.ch != 8 && s.ch != 12)) return false;
    return s.ns % (4 * kTmaQuads) == 0 && s.ns >= 4 * kTmaQuads;
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// stage timing: events around kernel groups, resolved lazily
// ---------------------------------------------------------------------------------------------
namespace {

cudaEvent_t ev_get(rspt_gpu_packer* p)
{
    if (!p->ev_free->empty()) {
        cudaEvent_t e = p->ev_free->back();
        p->ev_free->pop_back();
        return e;
    }
    cudaEvent_t e = nullptr;
    cudaEventCreate(&e);
    return e;
}

void ev_resolve(rspt_gpu_packer* p)
{
    for (auto& q : *p->ev_pending) {
        float ms = 0;
        if (cudaEventSynchronize(q.b) == cudaSuccess && cudaEventElapsedTime(&ms, q.a, q.b) == cudaSuccess) {
            p->stage_ms[q.stage] += ms;
            p->stage_calls[q.stage] += 1;
        }
        p->ev_free->push_back(q.a);
        p->ev_free->push_back(q.b);
    }
    p->ev_pending->clear();
}

struct StageTimer {
    rspt_gpu_packer* p;
    int stage;
    cudaEvent_t a = nullptr;
    StageTimer(rspt_gpu_packer* p_, int stage_) : p(p_), stage(stage_)
    {
        if (p->timing) {
            a = ev_get(p);
            cudaEventRecord(a, p->stream);
        }
    }
    ~StageTimer()
    {
        if (a) {
            cudaEvent_t b = ev_get(p);
            cudaEventRecord(b, p->stream);
            p->ev_pending->push_back({stage, a, b});
            if (p->ev_pending->size() > 4096) ev_resolve(p);
        }
    }
};

}  // namespace

extern "C" int rspt_gpu_set_stage_timing(rspt_gpu_packer* p, int enable)
{
    if (!p) return RSPT_E_ARG;
    p->timing = enable != 0;
    return RSPT_OK;
}

extern "C" int rspt_gpu_get_stage_times(rspt_gpu_packer* p, double* ms, uint64_t* calls, int reset)
{
    if (!p) return RSPT_E_ARG;
    DeviceGuard dg(p->device);
    ev_resolve(p);
    for (int i = 0; i < RSPT_STAGE_COUNT; ++i) {
        if (ms) ms[i] = p->stage_ms[i];
        if (calls) calls[i] = p->stage_calls[i];
        if (reset) {
            p->stage_ms[i] = 0;
            p->stage_calls[i] = 0;
        }
    }
    return RSPT_OK;
}

// ---------------------------------------------------------------------------------------------
// create / destroy
// ---------------------------------------------------------------------------------------------
extern "C" int rspt_gpu_create(int kind, size_t bps, size_t ch, size_t ns, size_t nb, int device, void* stream,
                               size_t max_batch_frames, rspt_gpu_packer** out)
{
    if (!out) return RSPT_E_ARG;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return RSPT_E_NOGPU;
    if (device < 0 || device >= ndev) return RSPT_E_ARG;
    if (kind < 0 || kind > 3 || bps < 1 || bps > 4 || ch < 1 || ns < 1 || max_batch_frames < 1) return RSPT_E_ARG;
    if (ch > 65535 || (uint64_t)ch * ns > 0x7FFFFFFFull / 4) return RSPT_E_ARG;
    if (kind == RSPT_XDELTA_HZR && (nb < 1 || nb > 4)) return RSPT_E_ARG;
    if (kind == RSPT_HADAMARD && ((ns & (ns - 1)) || ns < 2 || ns > kFwhtMaxN)) return RSPT_E_ARG;  // needs 2^k (fwht.c)
    if (kind == RSPT_DCT && (ns < 2 || ns > kDctMaxN)) return RSPT_E_ARG;
    // A shape that the tile kernels cannot stage in shared memory is refused here, not at the first call:
    // the generic forward tile (xdelta_tile / kPiece sample rows), the inverse kernel's carries + tile.
    {
        Shape t{};
        t.kind = kind; t.bps = (int)bps; t.ch = (int)ch; t.ns = (int)ns;
        uint32_t ts;
        size_t smem;
        if ((kind == RSPT_XDELTA_HZR || kind == RSPT_HZR) && !xdelta_tile(t, ts, smem)) return RSPT_E_ARG;
        const size_t tile_bytes = (size_t)kPiece * ch * bps + 48;
        const size_t pieces = ((ns + kPiece - 1) / kPiece) * ch;
        if (tile_bytes > 200 * 1024 || 2 * pieces * 4 + tile_bytes > 200 * 1024) return RSPT_E_ARG;
    }
    DeviceGuard dg(device);
    int rc = ensure_device_constants(device);
    if (rc != RSPT_OK) return rc;

    rspt_gpu_packer* p = new (std::nothrow) rspt_gpu_packer();
    if (!p) return RSPT_E_ARG;
    memset(p, 0, sizeof(*p));
    Shape& s = p->s;
    s.kind = kind; s.bps = (int)bps; s.ch = (int)ch; s.ns = (int)ns;
    s.N = (uint32_t)(ch * ns);
    s.nblk = (s.N + kBlock - 1) / kBlock;
    // planes: xdelta = ctor argument, escalating up to bps (xdelta.cpp:63-69); hzr 4 (hzr.cpp:39);
    // hadamard 3 (hadamard.cpp:44); dct 2 (dct.cpp:46)
    s.nb_init = kind == RSPT_XDELTA_HZR ? (uint32_t)nb : kind == RSPT_HZR ? 4u : kind == RSPT_HADAMARD ? 3u : 2u;
    p->can_escalate = kind == RSPT_XDELTA_HZR && s.nb_init < (uint32_t)bps;
    s.nb_alloc = p->can_escalate ? (uint32_t)bps : s.nb_init;
    s.hdr_bytes = (kind == RSPT_HADAMARD || kind == RSPT_DCT) ? 3u * (uint32_t)ch : 0u;
    s.plane_stride = (s.N + 15u) & ~15u;
    s.frame_bytes = (uint32_t)(bps * ch * ns);
    s.method = kind == RSPT_DCT ? 1u : (kind == RSPT_HADAMARD ? 2u : 0u);
    p->ev_free = new std::vector<cudaEvent_t>();
    p->ev_pending = new std::vector<rspt_gpu_packer::Pending>();
    p->device = device;
    p->max_batch = max_batch_frames;
    p->d_crc = g_crc[device];
    const uint32_t maxn = s.N < kBlock ? s.N : kBlock;
    p->enc_smem = (size_t)(12 + (maxn + 3) / 4 + 8) * 4;  // staging of the largest block: header + payload at an offset of <= 38 bytes, + slack
    p->dec_smem = ((size_t)(maxn + 30) / 16 + 2) * 16;   // the 16-byte chunks that hold the largest payload (any alignment) + zero slack
    p->stream = (cudaStream_t)stream;  // NULL = the CUDA default stream
    p->own_stream = false;
    const size_t F = max_batch_frames, nblocks = F * s.nb_alloc * s.nblk;
    cudaError_t e = cudaSuccess;
    auto A = [&](cudaError_t r) { if (e == cudaSuccess) e = r; };
    A(dalloc(p->d_planes, F * s.nb_alloc * (size_t)s.plane_stride));
    A(dalloc(p->d_hist, nblocks * kSymStride));
    A(dalloc(p->d_codes, nblocks * kSymStride));
    A(dalloc(p->d_tree, nblocks * kTreeWords));
    A(dalloc(p->d_step_lz, nblocks * kMaxSteps));
    A(dalloc(p->d_lists, nblocks * (size_t)kListCap));
    A(dalloc(p->d_list_n, nblocks));
    A(dalloc(p->d_blk_class, nblocks));
    A(dalloc(p->d_info, nblocks));
    A(dalloc(p->d_frame_nb, F));
    A(dalloc(p->d_need, F));
    A(dalloc(p->d_nb_state, 4));
    A(dalloc(p->d_all_totals, 64));
    A(dalloc(p->d_sizes, F));
    A(dalloc(p->d_blk_off, nblocks));
    A(dalloc(p->d_headers, F * (s.hdr_bytes ? s.hdr_bytes : 1)));
    A(dalloc(p->d_ctr, 1));
    A(dalloc(p->d_status_tmp, F));
    A(dalloc(p->d_dec_nb, F));
    A(cudaMalloc(&p->d_dec, nblocks * sizeof(DecBlk) + 64));
    A(cudaMalloc(&p->d_auto_index, ((F * (1 + s.hdr_bytes + (size_t)s.nb_alloc * (4 + hzr_max(s.N))) >> 6) + nblocks + 2) * sizeof(uint32_t) + 64));
    if (kind == RSPT_HADAMARD || kind == RSPT_DCT) {
        A(dalloc(p->d_words, F * (size_t)s.N));
        A(dalloc(p->d_sums, F * (size_t)s.ch));
    }
    p->dct_direct = kind == RSPT_DCT && dct_choose_direct((uint32_t)ns);
    if (e == cudaSuccess && kind == RSPT_DCT) e = dct_build_tables(p);
    const size_t maxc = rspt_gpu_max_compressed_size(p);
    A(dalloc(p->d_one_src, (size_t)s.frame_bytes));
    A(dalloc(p->d_one_dst, maxc));
    A(dalloc(p->d_one_off, 2));
    p->h_pin_bytes = maxc > s.frame_bytes ? maxc : s.frame_bytes;
    p->h_pin_bytes += 64;
    if (e == cudaSuccess) e = cudaMallocHost(reinterpret_cast<void**>(&p->h_pin), p->h_pin_bytes);
    if (e == cudaSuccess) e = cudaMemsetAsync(p->d_frame_nb, (int)s.nb_init, F, p->stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(p->d_ctr, 0, sizeof(Counters), p->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(p->d_nb_state, &s.nb_init, 4, cudaMemcpyHostToDevice, p->stream);
    if (e == cudaSuccess) e = allow_smem(k_hzr_encode<2>, kEncodeSmem);
    if (e == cudaSuccess) e = allow_smem(k_hzr_encode<3>, kEncodeSmem);
    if (e == cudaSuccess) e = allow_smem(k_hzr_hist<3>, kHistSmemList);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&p->side, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&p->place, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&p->ev_place, cudaEventDisableTiming);
    for (int k = 0; k < rspt_gpu_packer::kPlaceRing && e == cudaSuccess; ++k)
        e = cudaEventCreateWithFlags(&p->ev_placed[k], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&p->ev_fork, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&p->ev_join, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&p->ev_fork2, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&p->ev_join2, cudaEventDisableTiming);
    if (e == cudaSuccess) e = allow_smem(k_hzr_encode_sparse, kSparseSmem);
    {
        // test hook: a smaller staging limit sends listed blocks down the hand-over path to k_hzr_encode
        const char* ev = getenv("RSPT_SPARSE_STAGE_BYTES");
        const long v = ev ? atol(ev) : (long)kSpStageBytes;
        p->sp_stage = (uint32_t)(v < 1 ? 1 : (v > (long)kSpStageBytes ? (long)kSpStageBytes : v));
    }
    if (e == cudaSuccess) e = allow_smem(k_hzr_decode, kDecodeSmem);
    if (e == cudaSuccess) e = allow_smem(k_hzr_verify, kDecodeSmem);
    if (e == cudaSuccess) e = allow_smem(k_hzr_build_index, kDecodeSmem);
    if (e == cudaSuccess) e = allow_smem(k_crc32c, kEncodeSmem);
    if (e == cudaSuccess) e = cudaStreamSynchronize(p->stream);
    if (e != cudaSuccess) {
        fprintf(stderr, "rspt_gpu_create: %s\n", cudaGetErrorString(e));
        rspt_gpu_destroy(p);
        return RSPT_E_CUDA;
    }
    *out = p;
    return RSPT_OK;
}

extern "C" int rspt_gpu_destroy(rspt_gpu_packer* p)
{
    if (!p) return RSPT_E_ARG;
    DeviceGuard dg(p->device);
    cudaStreamSynchronize(p->stream);
    void* ptrs[] = {p->d_planes, p->d_hist, p->d_codes, p->d_tree, p->d_step_lz, p->d_lists, p->d_list_n, p->d_blk_class, p->d_info, p->d_frame_nb,
                    p->d_need, p->d_nb_state, p->d_sizes, p->d_blk_off, p->d_headers, p->d_words, p->d_sums, p->d_ctr,
                    p->d_dec, p->d_dec_nb, p->d_status_tmp, p->d_twiddle, p->d_post, p->d_cos, p->d_one_src, p->d_one_dst,
                    p->d_one_off, p->d_hb_src, p->d_hb_dst, p->d_hb_off, p->d_auto_index, p->d_fir, p->d_words2, p->d_all_totals};
    for (void* q : ptrs)
        if (q) cudaFree(q);
    if (p->h_pin) cudaFreeHost(p->h_pin);
    destroy_host_pipe(p);
    if (p->ev_pending) {
        ev_resolve(p);
        for (cudaEvent_t e : *p->ev_free) cudaEventDestroy(e);
        delete p->ev_pending;
        delete p->ev_free;
    }
    if (p->side) cudaStreamDestroy(p->side);
    if (p->place) cudaStreamDestroy(p->place);
    if (p->ev_place) cudaEventDestroy(p->ev_place);
    for (cudaEvent_t ev : p->ev_placed) if (ev) cudaEventDestroy(ev);
    if (p->ev_fork) cudaEventDestroy(p->ev_fork);
    if (p->ev_join) cudaEventDestroy(p->ev_join);
    if (p->ev_fork2) cudaEventDestroy(p->ev_fork2);
    if (p->ev_join2) cudaEventDestroy(p->ev_join2);
    if (p->own_stream) cudaStreamDestroy(p->stream);
    delete p;
    return RSPT_OK;
}

extern "C" size_t rspt_gpu_frame_bytes(const rspt_gpu_packer* p) { return p ? p->s.frame_bytes : 0; }
extern "C" size_t rspt_gpu_header_bytes(const rspt_gpu_packer* p) { return p ? p->s.hdr_bytes : 0; }

extern "C" size_t rspt_gpu_max_compressed_size(const rspt_gpu_packer* p)
{
    if (!p) return 0;
    return 1 + p->s.hdr_bytes + (size_t)p->s.nb_alloc * (4 + hzr_max(p->s.N));
}

// The decode index has one 32-bit slot per 64 bytes of stream plus one per block (common.cuh); the buffer is
// sized for the worst-case stream, the entries of a batch lie in a prefix of it.
extern "C" size_t rspt_gpu_sidecar_bytes(const rspt_gpu_packer* p, size_t n_frames)
{
    if (!p) return 0;
    return ((n_frames * rspt_gpu_max_compressed_size(p) >> 6) + total_blocks(p, n_frames) + 2) * sizeof(uint32_t);
}

extern "C" size_t rspt_gpu_sidecar_used_bytes(const rspt_gpu_packer* p, size_t n_frames, size_t stream_bytes)
{
    if (!p) return 0;
    return ((stream_bytes >> 6) + total_blocks(p, n_frames) + 2) * sizeof(uint32_t);
}

extern "C" const char* rspt_gpu_last_error(const rspt_gpu_packer* p) { return p ? p->err : "null handle"; }

extern "C" int rspt_gpu_sync(rspt_gpu_packer* p)
{
    if (!p) return RSPT_E_ARG;
    DeviceGuard dg(p->device);
    RSPT_CUDA_CHECK(cudaStreamSynchronize(p->stream));
    return RSPT_OK;
}

extern "C" int rspt_gpu_nb(rspt_gpu_packer* p, unsigned* nb)
{
    if (!p || !nb) return RSPT_E_ARG;
    DeviceGuard dg(p->device);
    uint32_t v = 0;
    RSPT_CUDA_CHECK(cudaMemcpyAsync(&v, p->d_nb_state, 4, cudaMemcpyDeviceToHost, p->stream));
    RSPT_CUDA_CHECK(cudaStreamSynchronize(p->stream));
    *nb = v;
    return RSPT_OK;
}

extern "C" int rspt_gpu_get_counters(rspt_gpu_packer* p, rspt_gpu_counters* out)
{
    if (!p || !out) return RSPT_E_ARG;
    DeviceGuard dg(p->device);
    Counters c;
    RSPT_CUDA_CHECK(cudaMemcpyAsync(&c, p->d_ctr, sizeof(c), cudaMemcpyDeviceToHost, p->stream));
    RSPT_CUDA_CHECK(cudaStreamSynchronize(p->stream));
    out->frames_compressed = c.frames_compressed;
    out->frames_decompressed = c.frames_decompressed;
    out->raw_bytes_in = c.raw_bytes_in;
    out->compressed_bytes_out = c.compressed_bytes_out;
    out->blocks_copy = c.blocks_copy;
    out->blocks_huff = c.blocks_huff;
    out->blocks_fill = c.blocks_fill;
    out->escalations = c.escalations;
    out->crc_failures = c.crc_failures;
    out->kernel_launches = p->launches;
    return RSPT_OK;
}


// ---------------------------------------------------------------------------------------------
// compress
// ---------------------------------------------------------------------------------------------
namespace {

// stage 1: samples -> byte planes (+ header, + need flags)
int launch_forward_transform(rspt_gpu_packer* p, const uint8_t* d_src, size_t F)
{
    const Shape& s = p->s;
    if (s.kind == RSPT_XDELTA_HZR || s.kind == RSPT_HZR) {
        uint32_t* need = p->can_escalate ? p->d_need : nullptr;
        if (need) RSPT_CUDA_CHECK(cudaMemsetAsync(need, 0, F * sizeof(uint32_t), p->stream));
        const bool st = s.kind == RSPT_XDELTA_HZR;
        // TMA-fed tile kernel (xdelta_tma.cuh: k_xdelta_planes_tma) for the shapes it is compiled for; it has no
        // plane-count probe (need): that case keeps k_xdelta_planes_fast
        if (!need && tma_transform_ok(s, d_src)) {
            const uint32_t tiles = (uint32_t)s.ns / (4u * kTmaQuads);
            const size_t tsm = (size_t)(kTmaQuads + 2) * 4u * s.ch * s.bps;
            const dim3 grid((unsigned)(F * tiles));
#define X(B, C)                                                                                                          \
    if (s.bps == B && s.ch == C) {                                                                                       \
        if (st) {                                                                                                        \
            RSPT_CUDA_CHECK(allow_smem(k_xdelta_planes_tma<B, C, true>, tsm));                                           \
            k_xdelta_planes_tma<B, C, true><<<grid, kTmaThreads, tsm, p->stream>>>(d_src, s, tiles, p->d_planes);       \
        } else {                                                                                                         \
            RSPT_CUDA_CHECK(allow_smem(k_xdelta_planes_tma<B, C, false>, tsm));                                          \
            k_xdelta_planes_tma<B, C, false><<<grid, kTmaThreads, tsm, p->stream>>>(d_src, s, tiles, p->d_planes);      \
        }                                                                                                                \
    }
            RSPT_TMA_SHAPES(X)
#undef X
            p->launches += 1;
            RSPT_CUDA_CHECK(cudaGetLastError());
            return RSPT_OK;
        }
        uint32_t tsq;
        size_t fsmem;
        if (xdelta_fast_tile(s, d_src, tsq, fsmem)) {
            const uint32_t nq = (uint32_t)s.ns >> 2, tiles = (nq + tsq - 1) / tsq;
            const dim3 grid((unsigned)(F * tiles));
#define LAUNCH_F(B, ST)                                                                                   \
    do {                                                                                                  \
        RSPT_CUDA_CHECK(allow_smem(k_xdelta_planes_fast<B, ST>, fsmem));                                  \
        k_xdelta_planes_fast<B, ST><<<grid, 128, fsmem, p->stream>>>(d_src, s, tsq, tiles, p->d_planes, need);       \
    } while (0)
            switch (s.bps) {
            case 1: if (st) LAUNCH_F(1, true); else LAUNCH_F(1, false); break;
            case 2: if (st) LAUNCH_F(2, true); else LAUNCH_F(2, false); break;
            case 3: if (st) LAUNCH_F(3, true); else LAUNCH_F(3, false); break;
            default: if (st) LAUNCH_F(4, true); else LAUNCH_F(4, false); break;
            }
#undef LAUNCH_F
            p->launches += 1;
            RSPT_CUDA_CHECK(cudaGetLastError());
            return RSPT_OK;
        }
        uint32_t ts;
        size_t smem;
        if (!xdelta_tile(s, ts, smem)) return fail_arg(p, "too many channels for the tile kernel");
        const uint32_t tiles = ((uint32_t)s.ns + ts - 1) / ts;
        const dim3 grid((unsigned)(F * tiles));
#define LAUNCH_X(B, ST)                                                                              \
    do {                                                                                             \
        RSPT_CUDA_CHECK(allow_smem(k_xdelta_planes<B, ST>, smem));                                   \
        k_xdelta_planes<B, ST><<<grid, 256, smem, p->stream>>>(d_src, s, ts, tiles, p->d_planes, need); \
    } while (0)
        switch (s.bps) {
        case 1: if (st) LAUNCH_X(1, true); else LAUNCH_X(1, false); break;
        case 2: if (st) LAUNCH_X(2, true); else LAUNCH_X(2, false); break;
        case 3: if (st) LAUNCH_X(3, true); else LAUNCH_X(3, false); break;
        default: if (st) LAUNCH_X(4, true); else LAUNCH_X(4, false); break;
        }
#undef LAUNCH_X
        p->launches += 1;
        RSPT_CUDA_CHECK(cudaGetLastError());
        return RSPT_OK;
    }
    return spectral_forward(p, d_src, F);
}

int launch_frame_nb(rspt_gpu_packer* p, size_t F)
{
    if (!p->can_escalate) return RSPT_OK;
    k_frame_nb<<<1, 1024, 0, p->stream>>>(p->d_need, (uint32_t)F, p->d_nb_state, p->d_frame_nb, p->d_ctr);
    p->launches += 1;
    RSPT_CUDA_CHECK(cudaGetLastError());
    return RSPT_OK;
}

}  // namespace

// Dense-encoder CTAs per SM the kernel is compiled for.  Measured per 4096-frame batch: xdelta_hzr 1.075 -> 1.051 ms
// and hadamard 1.121 -> 1.090 ms with 3 (more warps to cover the barriers), hzr 2.344 -> 2.369 and dct
// 0.848 -> 0.890 with 3 (their planes take the spilled slow path more often).
static int encode_ctas_per_sm(const Shape& s)
{
    return (s.kind == RSPT_XDELTA_HZR || s.kind == RSPT_HADAMARD) ? 3 : 2;
}

// A compress that rewrites an offsets array must not overtake a placement still rebasing it.
static int wait_for_placement_of(rspt_gpu_packer* p, const void* d_offsets)
{
    for (int k = 0; k < rspt_gpu_packer::kPlaceRing; ++k)
        if (p->placed_ptr[k] == d_offsets) {
            RSPT_CUDA_CHECK(cudaStreamWaitEvent(p->stream, p->ev_placed[k], 0));
            p->placed_ptr[k] = nullptr;
        }
    return RSPT_OK;
}

extern "C" int rspt_gpu_compress_batch(rspt_gpu_packer* p, const uint8_t* d_src, size_t n_frames, uint8_t* d_dst,
                                       size_t dst_capacity, uint64_t* d_offsets, uint8_t* d_frame_nb, void* d_sidecar)
{
    if (!p || !d_src || !d_dst || !d_offsets) return RSPT_E_ARG;
    if (n_frames == 0) return RSPT_OK;
    if (n_frames > p->max_batch) return fail_arg(p, "n_frames exceeds max_batch_frames"), RSPT_E_CAPACITY;
    if (dst_capacity < n_frames * rspt_gpu_max_compressed_size(p))
        return fail_arg(p, "dst_capacity < n_frames * rspt_gpu_max_compressed_size"), RSPT_E_CAPACITY;
    DeviceGuard dg(p->device);
    const Shape& s = p->s;
    const size_t F = n_frames;
    const uint32_t nblocks = total_blocks(p, F);
    int rc = wait_for_placement_of(p, d_offsets);
    if (rc) return rc;
    uint32_t* sidecar = reinterpret_cast<uint32_t*>(d_sidecar);
    const unsigned tgrid = (nblocks + kTreeWarps - 1) / kTreeWarps;
    {
        StageTimer t(p, RSPT_STAGE_TRANSFORM);
        rc = launch_forward_transform(p, d_src, F);
        if (rc) return rc;
        rc = launch_frame_nb(p, F);
        if (rc) return rc;
    }
    {
        // Two classes of blocks (density probe): the sparse-looking ones go through histogram + tree on
        // the side stream while this stream does the dense-looking ones, whose tree build is long and
        // latency-bound and overlaps with the sparse histogram.  RSPT_STAGE_HIST times the dense
        // histogram, RSPT_STAGE_TREE everything from there to the join.
        RSPT_CUDA_CHECK(cudaEventRecord(p->ev_fork, p->stream));
        RSPT_CUDA_CHECK(cudaStreamWaitEvent(p->side, p->ev_fork, 0));
        k_hzr_hist<3><<<nblocks, kHistThreads, kHistSmemList, p->side>>>(p->d_planes, s, p->d_frame_nb, p->d_hist, p->d_step_lz, p->d_lists, p->d_list_n, p->d_blk_class);
        k_hzr_tree<<<tgrid, 32 * kTreeWarps, 0, p->side>>>(p->d_hist, s, p->d_frame_nb, p->d_blk_class, kClassSparse, nblocks, p->d_codes, p->d_tree, p->d_info, p->d_ctr);
        RSPT_CUDA_CHECK(cudaEventRecord(p->ev_join, p->side));
        {
            StageTimer t(p, RSPT_STAGE_HIST);
            k_hzr_hist<2><<<nblocks, kHistThreads, 0, p->stream>>>(p->d_planes, s, p->d_frame_nb, p->d_hist, p->d_step_lz, p->d_lists, p->d_list_n, p->d_blk_class);
        }
        {
            StageTimer t(p, RSPT_STAGE_TREE);
            k_hzr_tree<<<tgrid, 32 * kTreeWarps, 0, p->stream>>>(p->d_hist, s, p->d_frame_nb, p->d_blk_class, kClassDense, nblocks, p->d_codes, p->d_tree, p->d_info, p->d_ctr);
            RSPT_CUDA_CHECK(cudaStreamWaitEvent(p->stream, p->ev_join, 0));
        }
        p->launches += 4;
    }
    {
        StageTimer t(p, RSPT_STAGE_LAYOUT);
        k_frame_sizes<<<(unsigned)((F + 255) / 256), 256, 0, p->stream>>>(p->d_info, s, p->d_frame_nb, (uint32_t)F, p->d_sizes, p->d_blk_off);
        k_scan_offsets<<<1, 1024, 0, p->stream>>>(p->d_sizes, (uint32_t)F, d_offsets, p->d_ctr, s.frame_bytes);
    }
    {
        // sparse blocks from their lists (side stream) beside everything else from the planes: both kernels
        // decide with the same predicate which of them writes a block
        StageTimer t(p, RSPT_STAGE_ENCODE);
        const SparseOut so{d_dst, d_offsets, p->d_blk_off, p->sp_stage, p->d_headers, sidecar};
        RSPT_CUDA_CHECK(cudaEventRecord(p->ev_fork2, p->stream));
        RSPT_CUDA_CHECK(cudaStreamWaitEvent(p->side, p->ev_fork2, 0));
        k_hzr_encode_sparse<<<nblocks, kSpThreads, kSparseSmem, p->side>>>(s, p->d_frame_nb, p->d_info, p->d_codes, p->d_tree, p->d_lists,
                                                                           p->d_list_n, p->d_crc, so);
        RSPT_CUDA_CHECK(cudaEventRecord(p->ev_join2, p->side));
        if (encode_ctas_per_sm(s) == 3)
            k_hzr_encode<3><<<nblocks, kEncThreads, p->enc_smem, p->stream>>>(p->d_planes, s, p->d_frame_nb, p->d_info, p->d_blk_off,
                                                                               p->d_codes, p->d_tree, p->d_step_lz, p->d_lists, p->d_list_n, p->sp_stage,
                                                                               d_offsets, p->d_headers, p->d_crc, d_dst, sidecar);
        else
            k_hzr_encode<2><<<nblocks, kEncThreads, p->enc_smem, p->stream>>>(p->d_planes, s, p->d_frame_nb, p->d_info, p->d_blk_off,
                                                                               p->d_codes, p->d_tree, p->d_step_lz, p->d_lists, p->d_list_n, p->sp_stage,
                                                                               d_offsets, p->d_headers, p->d_crc, d_dst, sidecar);
        RSPT_CUDA_CHECK(cudaStreamWaitEvent(p->stream, p->ev_join2, 0));
    }
    p->launches += 4;
    RSPT_CUDA_CHECK(cudaGetLastError());
    if (d_frame_nb) RSPT_CUDA_CHECK(cudaMemcpyAsync(d_frame_nb, p->d_frame_nb, F, cudaMemcpyDeviceToDevice, p->stream));
    return RSPT_OK;
}

// ---------------------------------------------------------------------------------------------
// decompress
// ---------------------------------------------------------------------------------------------
namespace {

// frame / block header walk + (for streams without a decode index) the index itself
int launch_parse_and_index(rspt_gpu_packer* p, const uint8_t* d_src, const uint64_t* d_offsets, size_t F,
                           const uint8_t* d_frame_nb, void* d_sidecar_out, int32_t* status)
{
    const Shape& s = p->s;
    const uint32_t nblocks = total_blocks(p, F);
    DecBlk* dec = reinterpret_cast<DecBlk*>(p->d_dec);
    {
        StageTimer t(p, RSPT_STAGE_PARSE);
        k_frame_parse<<<(unsigned)((F + 127) / 128), 128, 0, p->stream>>>(d_src, d_offsets, s, d_frame_nb, p->d_nb_state,
                                                                          (uint32_t)F, dec, p->d_headers, p->d_dec_nb, status, p->d_ctr);
        // code tables of the HUFF blocks from their in-stream trees (unused symbols stay 0)
        RSPT_CUDA_CHECK(cudaMemsetAsync(p->d_codes, 0, (size_t)nblocks * kSymStride * sizeof(uint32_t), p->stream));
        k_hzr_recover_codes<<<(nblocks + kRecoverThreads - 1) / kRecoverThreads, kRecoverThreads, 0, p->stream>>>(d_src, nblocks, dec, p->d_codes, s, status);
        p->launches += 2;
        if (d_sidecar_out) {
            k_hzr_build_index<<<nblocks, kIndexThreads, p->dec_smem, p->stream>>>(d_src, s, dec, d_offsets, p->d_codes,
                                                                                  reinterpret_cast<uint32_t*>(d_sidecar_out), status);
            p->launches += 1;
        }
    }
    RSPT_CUDA_CHECK(cudaGetLastError());
    return RSPT_OK;
}

}  // namespace

extern "C" int rspt_gpu_build_index(rspt_gpu_packer* p, const uint8_t* d_src, const uint64_t* d_offsets, size_t n_frames,
                                    const uint8_t* d_frame_nb, void* d_sidecar, int32_t* d_status)
{
    if (!p || !d_src || !d_offsets || !d_sidecar) return RSPT_E_ARG;
    if (n_frames == 0) return RSPT_OK;
    if (n_frames > p->max_batch) return fail_arg(p, "n_frames exceeds max_batch_frames"), RSPT_E_CAPACITY;
    DeviceGuard dg(p->device);
    return launch_parse_and_index(p, d_src, d_offsets, n_frames, d_frame_nb, d_sidecar, d_status ? d_status : p->d_status_tmp);
}

// payload bits per output byte up to which k_hzr_decode uses its two-literals-per-look-up table (measured)
constexpr uint32_t kDecodePairMaxBits = 4;

extern "C" int rspt_gpu_decompress_batch(rspt_gpu_packer* p, const uint8_t* d_src, const uint64_t* d_offsets,
                                         size_t n_frames, const uint8_t* d_frame_nb, const void* d_sidecar,
                                         uint8_t* d_dst, int32_t* d_status)
{
    if (!p || !d_src || !d_offsets || !d_dst) return RSPT_E_ARG;
    if (n_frames == 0) return RSPT_OK;
    if (n_frames > p->max_batch) return fail_arg(p, "n_frames exceeds max_batch_frames"), RSPT_E_CAPACITY;
    DeviceGuard dg(p->device);
    const Shape& s = p->s;
    const size_t F = n_frames;
    const uint32_t nblocks = total_blocks(p, F);
    int32_t* status = d_status ? d_status : p->d_status_tmp;
    DecBlk* dec = reinterpret_cast<DecBlk*>(p->d_dec);
    // Without an explicit per-frame plane count every frame uses the instance's current count,
    // as the reference's decompress does (signal_packer_xdelta_hzr.cpp:77).
    void* own_index = nullptr;
    if (!d_sidecar) {
        // stream from the CPU reference: build the decode index here first (handle-owned scratch)
        own_index = p->d_auto_index;
        d_sidecar = own_index;
    }
    int rc = launch_parse_and_index(p, d_src, d_offsets, F, d_frame_nb, own_index, status);
    if (rc) return rc;
    const uint32_t* sc = reinterpret_cast<const uint32_t*>(d_sidecar);
    const uint32_t maxn = s.N < kBlock ? s.N : kBlock;
    const uint32_t flags = kDecodePairMaxBits | (s.kind <= RSPT_HZR ? 256u : 0u);
    {
        // the classes with short payloads (few busy threads per CTA, latency-bound) run on the side stream
        // beside the full-size blocks
        StageTimer t(p, RSPT_STAGE_DECODE);
        cudaEventRecord(p->ev_fork, p->stream);
        cudaStreamWaitEvent(p->side, p->ev_fork, 0);
        k_hzr_decode<<<nblocks, decode_class_threads(kSmallPayload), decode_class_smem(kSmallPayload), p->side>>>(
            d_src, s, dec, d_offsets, sc, p->d_codes, p->d_planes, status, flags, 1u);
        if (maxn > kSmallPayload) {
            k_hzr_decode<<<nblocks, decode_class_threads(kMediumPayload), decode_class_smem(kMediumPayload), p->side>>>(
                d_src, s, dec, d_offsets, sc, p->d_codes, p->d_planes, status, flags, 2u);
            p->launches += 1;
        }
        cudaEventRecord(p->ev_join, p->side);
        k_hzr_decode<<<nblocks, kDecodeThreads, p->dec_smem, p->stream>>>(d_src, s, dec, d_offsets, sc, p->d_codes, p->d_planes, status, flags, 0u);
        cudaStreamWaitEvent(p->stream, p->ev_join, 0);
        p->launches += 2;
    }
    RSPT_CUDA_CHECK(cudaGetLastError());
    StageTimer t(p, RSPT_STAGE_INVERSE);
    return launch_inverse_transform(p, d_dst, F);
}

extern "C" int rspt_gpu_verify_batch(rspt_gpu_packer* p, const uint8_t* d_src, const uint64_t* d_offsets, size_t n_frames,
                                     const uint8_t* d_frame_nb, int32_t* d_status)
{
    if (!p || !d_src || !d_offsets || !d_status) return RSPT_E_ARG;
    if (n_frames == 0) return RSPT_OK;
    if (n_frames > p->max_batch) return fail_arg(p, "n_frames exceeds max_batch_frames"), RSPT_E_CAPACITY;
    DeviceGuard dg(p->device);
    const Shape& s = p->s;
    const size_t F = n_frames;
    const uint32_t nblocks = total_blocks(p, F);
    DecBlk* dec = reinterpret_cast<DecBlk*>(p->d_dec);
    k_frame_parse<<<(unsigned)((F + 127) / 128), 128, 0, p->stream>>>(d_src, d_offsets, s, d_frame_nb, p->d_nb_state, (uint32_t)F, dec,
                                                                      p->d_headers, p->d_dec_nb, d_status, p->d_ctr);
    k_hzr_verify<<<nblocks, kVerifyThreads, p->dec_smem, p->stream>>>(d_src, s, dec, p->d_crc, d_status, p->d_ctr);
    p->launches += 2;
    RSPT_CUDA_CHECK(cudaGetLastError());
    return RSPT_OK;
}


// ---------------------------------------------------------------------------------------------
// NCCL through its C API, resolved at run time (no link-time dependency)
// ---------------------------------------------------------------------------------------------
namespace {

struct NcclId { char b[128]; };   // ncclUniqueId, passed by value

struct NcclApi {
    int (*get_unique_id)(void*) = nullptr;
    int (*comm_init_rank)(void**, int, NcclId, int) = nullptr;
    int (*comm_destroy)(void*) = nullptr;
    int (*all_gather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
    bool ok = false;
};

NcclApi* nccl_api()
{
    static NcclApi api = [] {
        NcclApi a;
        void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);   // the copy the process already has (torch's)
        if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (!h) return a;
        a.get_unique_id = reinterpret_cast<decltype(a.get_unique_id)>(dlsym(h, "ncclGetUniqueId"));
        a.comm_init_rank = reinterpret_cast<decltype(a.comm_init_rank)>(dlsym(h, "ncclCommInitRank"));
        a.comm_destroy = reinterpret_cast<decltype(a.comm_destroy)>(dlsym(h, "ncclCommDestroy"));
        a.all_gather = reinterpret_cast<decltype(a.all_gather)>(dlsym(h, "ncclAllGather"));
        a.ok = a.get_unique_id && a.comm_init_rank && a.comm_destroy && a.all_gather;
        return a;
    }();
    return &api;
}
constexpr int kNcclUint64 = 5;   // ncclUint64 (nccl.h: ncclInt8 0, ncclUint8 1, ncclInt32 2, ncclUint32 3, ncclInt64 4, ncclUint64 5)

}  // namespace

extern "C" int rspt_gpu_comm_unique_id(uint8_t id[128])
{
    NcclApi* a = nccl_api();
    if (!id || !a->ok) return RSPT_E_ARG;
    return a->get_unique_id(id) == 0 ? RSPT_OK : RSPT_E_CUDA;
}

extern "C" int rspt_gpu_comm_init(int world, const uint8_t id[128], int rank, int device, void** comm)
{
    NcclApi* a = nccl_api();
    if (!comm || !id || !a->ok || world < 1 || rank < 0 || rank >= world) return RSPT_E_ARG;
    DeviceGuard dg(device);
    NcclId u;
    memcpy(u.b, id, 128);
    return a->comm_init_rank(comm, world, u, rank) == 0 ? RSPT_OK : RSPT_E_CUDA;
}

extern "C" int rspt_gpu_comm_destroy(void* comm)
{
    NcclApi* a = nccl_api();
    if (!comm || !a->ok) return RSPT_E_ARG;
    return a->comm_destroy(comm) == 0 ? RSPT_OK : RSPT_E_CUDA;
}

extern "C" int rspt_gpu_allgather_totals(void* comm, const uint64_t* d_total, uint64_t* d_all_totals, void* stream)
{
    NcclApi* a = nccl_api();
    if (!comm || !d_total || !d_all_totals || !a->ok) return RSPT_E_ARG;
    return a->all_gather(d_total, d_all_totals, 1, kNcclUint64, comm, (cudaStream_t)stream) == 0 ? RSPT_OK : RSPT_E_CUDA;
}

extern "C" int rspt_gpu_place_offsets_async(rspt_gpu_packer* p, void* comm, uint64_t* d_offsets, size_t n_frames, int rank, int world)
{
    if (!p || !d_offsets || rank < 0 || world < 1 || rank >= world || world > 64) return RSPT_E_ARG;
    if (world == 1) return RSPT_OK;
    DeviceGuard dg(p->device);
    cudaStream_t st = p->place;
    RSPT_CUDA_CHECK(cudaEventRecord(p->ev_place, p->stream));
    RSPT_CUDA_CHECK(cudaStreamWaitEvent(p->place, p->ev_place, 0));
    int rc = rspt_gpu_allgather_totals(comm, d_offsets + n_frames, p->d_all_totals, st);
    if (rc) return rc;
    rc = rspt_gpu_rebase_offsets(d_offsets, n_frames + 1, p->d_all_totals, rank, st);
    if (rc) return rc;
    const unsigned slot = p->place_seq++ % rspt_gpu_packer::kPlaceRing;
    if (p->placed_ptr[slot])   // the ring is full: the compute stream takes the oldest placement's completion now
        RSPT_CUDA_CHECK(cudaStreamWaitEvent(p->stream, p->ev_placed[slot], 0));
    RSPT_CUDA_CHECK(cudaEventRecord(p->ev_placed[slot], st));
    p->placed_ptr[slot] = d_offsets;
    return RSPT_OK;
}

extern "C" int rspt_gpu_place_join(rspt_gpu_packer* p)
{
    if (!p) return RSPT_E_ARG;
    DeviceGuard dg(p->device);
    RSPT_CUDA_CHECK(cudaEventRecord(p->ev_place, p->place));
    RSPT_CUDA_CHECK(cudaStreamWaitEvent(p->stream, p->ev_place, 0));
    for (const void*& q : p->placed_ptr) q = nullptr;
    return RSPT_OK;
}

extern "C" int rspt_gpu_set_stream(rspt_gpu_packer* p, void* stream)
{
    if (!p) return RSPT_E_ARG;
    p->stream = (cudaStream_t)stream;
    return RSPT_OK;
}

extern "C" int rspt_gpu_set_dct_exact(rspt_gpu_packer* p, int exact)
{
    if (!p || p->s.kind != RSPT_DCT) return RSPT_E_ARG;
    if (!exact && ((p->s.ns & (p->s.ns - 1)) != 0)) return fail_arg(p, "the FFT path needs a power-of-two length");
    DeviceGuard dg(p->device);
    if (exact && !p->d_cos) {
        // the cosine table is built on first use (the twiddles of the FFT path are rebuilt with it)
        RSPT_CUDA_CHECK(cudaStreamSynchronize(p->stream));
        if (p->d_twiddle) cudaFree(p->d_twiddle);
        if (p->d_post) cudaFree(p->d_post);
        p->d_twiddle = nullptr;
        p->d_post = nullptr;
        p->dct_direct = true;
        RSPT_CUDA_CHECK(dct_build_tables(p));
    }
    p->dct_direct = exact != 0;
    return RSPT_OK;
}

// ---------------------------------------------------------------------------------------------
// streaming ingest ring (io_buffer, lib_ring_buffer/ring_buffers.h:150-201, with pinned packets)
// ---------------------------------------------------------------------------------------------
struct rspt_gpu_ingest {
    rspt_gpu_packer* p;
    size_t packet_bytes, nr_max_packets;
    uint8_t* buffer;                   // pinned, nr_max_packets * packet_bytes
    std::atomic<uint8_t>* rw_states;   // 0 free, 1 being filled, 2 filled, 3 consumed
    size_t it_read, it_write, it_write_last;
};

extern "C" int rspt_gpu_ingest_create(rspt_gpu_packer* p, size_t nr_max_packets, rspt_gpu_ingest** out)
{
    if (!p || !out || nr_max_packets < 2) return RSPT_E_ARG;
    *out = nullptr;
    DeviceGuard dg(p->device);
    rspt_gpu_ingest* g = new (std::nothrow) rspt_gpu_ingest();
    if (!g) return RSPT_E_ARG;
    g->p = p;
    g->packet_bytes = p->s.frame_bytes;
    g->nr_max_packets = nr_max_packets;
    g->it_read = g->it_write = g->it_write_last = 0;
    g->buffer = nullptr;
    g->rw_states = new (std::nothrow) std::atomic<uint8_t>[nr_max_packets];
    if (!g->rw_states || cudaMallocHost(reinterpret_cast<void**>(&g->buffer), nr_max_packets * g->packet_bytes) != cudaSuccess) {
        delete[] g->rw_states;
        delete g;
        return RSPT_E_CUDA;
    }
    for (size_t i = 0; i < nr_max_packets; ++i) g->rw_states[i].store(0, std::memory_order_relaxed);
    *out = g;
    return RSPT_OK;
}

extern "C" int rspt_gpu_ingest_destroy(rspt_gpu_ingest* g)
{
    if (!g) return RSPT_E_ARG;
    DeviceGuard dg(g->p->device);
    cudaStreamSynchronize(g->p->stream);
    if (g->buffer) cudaFreeHost(g->buffer);
    delete[] g->rw_states;
    delete g;
    return RSPT_OK;
}

// io_buffer::get_next_address_to_fill, ring_buffers.h:182-199 (producer side)
extern "C" uint8_t* rspt_gpu_ingest_next_address_to_fill(rspt_gpu_ingest* g)
{
    if (!g) return nullptr;
    const uint8_t st = g->rw_states[g->it_write].load(std::memory_order_acquire);
    if (st != 0 && st != 3) return nullptr;
    if (g->rw_states[g->it_write_last].load(std::memory_order_relaxed) == 1)
        g->rw_states[g->it_write_last].store(2, std::memory_order_release);  // the previous packet is complete
    uint8_t* res = g->buffer + g->it_write * g->packet_bytes;
    g->rw_states[g->it_write].store(1, std::memory_order_relaxed);
    g->it_write_last = g->it_write;
    if (++g->it_write == g->nr_max_packets) g->it_write = 0;
    return res;
}

// consumer side: what a loop over io_buffer::get_next_filled_address (:168-180) + compress would do,
// in batches of contiguous filled packets
extern "C" int rspt_gpu_ingest_drain(rspt_gpu_ingest* g, int flush, uint8_t* h_dst, size_t dst_capacity, uint64_t* h_offsets,
                                     size_t* n_frames)
{
    if (!g || !h_dst || !h_offsets || !n_frames) return RSPT_E_ARG;
    rspt_gpu_packer* p = g->p;
    if (flush && g->rw_states[g->it_write_last].load(std::memory_order_relaxed) == 1)
        g->rw_states[g->it_write_last].store(2, std::memory_order_release);  // only safe once the producer has stopped
    const size_t want = *n_frames, maxc = rspt_gpu_max_compressed_size(p);
    size_t done = 0;
    uint64_t bytes = 0;
    h_offsets[0] = 0;
    while (done < want) {
        // the run of filled packets that starts at it_read and does not wrap
        size_t run = 0;
        while (done + run < want && g->it_read + run < g->nr_max_packets && run < p->max_batch &&
               g->rw_states[g->it_read + run].load(std::memory_order_acquire) == 2)
            ++run;
        if (run == 0) break;
        if (dst_capacity - bytes < run * maxc) {
            if (done == 0) return fail_arg(p, "dst_capacity too small for the filled packets"), RSPT_E_CAPACITY;
            break;
        }
        const int rc = rspt_gpu_compress_batch_host(p, g->buffer + g->it_read * g->packet_bytes, run, h_dst + bytes,
                                                    dst_capacity - bytes, h_offsets + done);
        if (rc != RSPT_OK) return rc;
        // compress_batch_host numbers its offsets from 0: rebase onto what this drain has written so far
        const uint64_t chunk_bytes = h_offsets[done + run];
        for (size_t i = 0; i <= run; ++i) h_offsets[done + i] += bytes;
        bytes += chunk_bytes;
        for (size_t i = 0; i < run; ++i) g->rw_states[g->it_read + i].store(3, std::memory_order_release);
        g->it_read += run;
        if (g->it_read == g->nr_max_packets) g->it_read = 0;
        done += run;
    }
    *n_frames = done;
    return RSPT_OK;
}

// ---------------------------------------------------------------------------------------------
// pre-filter (the step in front of the packers in the reference's pipeline)
// ---------------------------------------------------------------------------------------------
namespace {

int ensure_words(rspt_gpu_packer* p)
{
    const Shape& s = p->s;
    if (!p->d_words) RSPT_CUDA_CHECK(dalloc(p->d_words, p->max_batch * (size_t)s.N));
    if (!p->d_sums) RSPT_CUDA_CHECK(dalloc(p->d_sums, p->max_batch * (size_t)s.ch));
    return RSPT_OK;
}

int launch_words_to_raw(rspt_gpu_packer* p, const int32_t* d_words, uint8_t* d_dst, size_t F)
{
    const Shape& s = p->s;
    const uint32_t tiles = ((uint32_t)s.ns + kPiece - 1) / kPiece;
    const size_t tile_bytes = (size_t)kPiece * s.ch * s.bps + 48;
    if (tile_bytes > 200 * 1024) return fail_arg(p, "too many channels");
    switch (s.bps) {
    case 1: RSPT_CUDA_CHECK(cudaFuncSetAttribute(k_words_to_raw<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tile_bytes)); break;
    case 2: RSPT_CUDA_CHECK(cudaFuncSetAttribute(k_words_to_raw<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tile_bytes)); break;
    case 3: RSPT_CUDA_CHECK(cudaFuncSetAttribute(k_words_to_raw<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tile_bytes)); break;
    default: RSPT_CUDA_CHECK(cudaFuncSetAttribute(k_words_to_raw<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tile_bytes)); break;
    }
    SPECTRAL_BPS_SWITCH(k_words_to_raw, <<<(unsigned)(F * tiles), 256, tile_bytes, p->stream>>>(d_words, s, tiles, d_dst));
    p->launches += 1;
    RSPT_CUDA_CHECK(cudaGetLastError());
    return RSPT_OK;
}

int launch_raw_to_words(rspt_gpu_packer* p, const uint8_t* d_src, size_t F)
{
    const Shape& s = p->s;
    const uint32_t tiles = ((uint32_t)s.ns + kPiece - 1) / kPiece;
    const size_t tile_smem = (size_t)kPiece * s.ch * s.bps + 48;
    if (tile_smem > 200 * 1024) return fail_arg(p, "too many channels");
    switch (s.bps) {
    case 1: RSPT_CUDA_CHECK(cudaFuncSetAttribute(k_raw_to_words<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tile_smem)); break;
    case 2: RSPT_CUDA_CHECK(cudaFuncSetAttribute(k_raw_to_words<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tile_smem)); break;
    case 3: RSPT_CUDA_CHECK(cudaFuncSetAttribute(k_raw_to_words<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tile_smem)); break;
    default: RSPT_CUDA_CHECK(cudaFuncSetAttribute(k_raw_to_words<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tile_smem)); break;
    }
    SPECTRAL_BPS_SWITCH(k_raw_to_words, <<<(unsigned)(F * tiles), 256, tile_smem, p->stream>>>(d_src, s, tiles, p->d_words, p->d_sums));
    p->launches += 1;
    RSPT_CUDA_CHECK(cudaGetLastError());
    return RSPT_OK;
}

}  // namespace

extern "C" int rspt_gpu_prefilter_iir(rspt_gpu_packer* p, uint8_t* d_frames, size_t n_frames, const double* n, const double* d,
                                      int nr_coefficients, int init_nr_samples)
{
    if (!p || !d_frames || !n || !d || init_nr_samples < 0) return RSPT_E_ARG;
    if (nr_coefficients < 2 || nr_coefficients > 5) return fail_arg(p, "iir: 2..5 coefficients (iir_filter.cpp:84-100)");
    if (n_frames == 0) return RSPT_OK;
    if (n_frames > p->max_batch) return fail_arg(p, "n_frames exceeds max_batch_frames"), RSPT_E_CAPACITY;
    DeviceGuard dg(p->device);
    const Shape& s = p->s;
    const size_t F = n_frames;
    int rc = ensure_words(p);
    if (rc) return rc;
    rc = launch_raw_to_words(p, d_frames, F);
    if (rc) return rc;
    IirCoef c;
    memset(&c, 0, sizeof c);
    c.nc = nr_coefficients;
    c.init_calls = 4 * init_nr_samples;
    for (int i = 0; i < nr_coefficients; ++i) {
        c.n[i] = n[i];
        c.d[i] = d[i];
    }
    const unsigned grid = (unsigned)((F + 31) / 32);
    switch (nr_coefficients) {
    case 2: k_iir_frames<2><<<grid, 32, 0, p->stream>>>(p->d_words, s, (uint32_t)F, c); break;
    case 3: k_iir_frames<3><<<grid, 32, 0, p->stream>>>(p->d_words, s, (uint32_t)F, c); break;
    case 4: k_iir_frames<4><<<grid, 32, 0, p->stream>>>(p->d_words, s, (uint32_t)F, c); break;
    default: k_iir_frames<5><<<grid, 32, 0, p->stream>>>(p->d_words, s, (uint32_t)F, c); break;
    }
    p->launches += 1;
    RSPT_CUDA_CHECK(cudaGetLastError());
    return launch_words_to_raw(p, p->d_words, d_frames, F);
}

extern "C" int rspt_gpu_prefilter_fir(rspt_gpu_packer* p, uint8_t* d_frames, size_t n_frames, const double* kernel, int kernel_size)
{
    if (!p || !d_frames || !kernel || kernel_size < 1 || kernel_size > 65536) return RSPT_E_ARG;
    if (n_frames == 0) return RSPT_OK;
    if (n_frames > p->max_batch) return fail_arg(p, "n_frames exceeds max_batch_frames"), RSPT_E_CAPACITY;
    DeviceGuard dg(p->device);
    const Shape& s = p->s;
    const size_t F = n_frames;
    int rc = ensure_words(p);
    if (rc) return rc;
    if (p->fir_cap < (size_t)kernel_size) {
        if (p->d_fir) cudaFree(p->d_fir);
        p->d_fir = nullptr;
        RSPT_CUDA_CHECK(dalloc(p->d_fir, (size_t)kernel_size));
        p->fir_cap = (size_t)kernel_size;
    }
    RSPT_CUDA_CHECK(cudaMemcpyAsync(p->d_fir, kernel, sizeof(double) * (size_t)kernel_size, cudaMemcpyHostToDevice, p->stream));
    if (!p->d_words2) RSPT_CUDA_CHECK(dalloc(p->d_words2, p->max_batch * (size_t)s.N));
    rc = launch_raw_to_words(p, d_frames, F);
    if (rc) return rc;
    const size_t sm = (size_t)(2 * kernel_size + kFirTile) * sizeof(double);
    if (sm > 200 * 1024) return fail_arg(p, "fir kernel too long for the shared-memory tile");
    RSPT_CUDA_CHECK(allow_smem(k_fir_words, sm));
    const uint32_t tiles = ((uint32_t)s.ns + kFirTile - 1) / kFirTile;
    k_fir_words<<<(unsigned)(F * s.ch * tiles), kFirTile, sm, p->stream>>>(p->d_words, s, tiles, p->d_fir, kernel_size, p->d_words2);
    p->launches += 1;
    RSPT_CUDA_CHECK(cudaGetLastError());
    return launch_words_to_raw(p, p->d_words2, d_frames, F);
}

// ---------------------------------------------------------------------------------------------
// host-buffer entry points
// ---------------------------------------------------------------------------------------------
extern "C" int rspt_gpu_compress_host(rspt_gpu_packer* p, const uint8_t* h_src, uint8_t* h_dst, size_t dst_max_len,
                                      size_t* dst_len)
{
    if (!p || !h_src || !h_dst || !dst_len) return RSPT_E_ARG;
    DeviceGuard dg(p->device);
    const size_t fb = p->s.frame_bytes, maxc = rspt_gpu_max_compressed_size(p);
    memcpy(p->h_pin, h_src, fb);
    RSPT_CUDA_CHECK(cudaMemcpyAsync(p->d_one_src, p->h_pin, fb, cudaMemcpyHostToDevice, p->stream));
    int rc = rspt_gpu_compress_batch(p, p->d_one_src, 1, p->d_one_dst, maxc, p->d_one_off, nullptr, nullptr);
    if (rc) return rc;
    uint64_t off[2];
    RSPT_CUDA_CHECK(cudaMemcpyAsync(off, p->d_one_off, sizeof(off), cudaMemcpyDeviceToHost, p->stream));
    RSPT_CUDA_CHECK(cudaStreamSynchronize(p->stream));
    const size_t len = (size_t)off[1];
    if (len > dst_max_len) return fail_arg(p, "dst_max_len too small"), RSPT_E_CAPACITY;
    RSPT_CUDA_CHECK(cudaMemcpyAsync(p->h_pin, p->d_one_dst, len, cudaMemcpyDeviceToHost, p->stream));
    RSPT_CUDA_CHECK(cudaStreamSynchronize(p->stream));
    memcpy(h_dst, p->h_pin, len);
    *dst_len = len;
    return RSPT_OK;
}

namespace {
// Length of one frame found by walking its chunk length fields on the host
// (signal_packer_base.cpp:101-121: frames are self-delimiting given the plane count).
size_t host_frame_len(const rspt_gpu_packer* p, const uint8_t* h, unsigned nb)
{
    size_t pos = 1 + p->s.hdr_bytes;
    for (unsigned k = 0; k < nb; ++k) {
        const uint32_t len = (uint32_t)h[pos] | ((uint32_t)h[pos + 1] << 8) | ((uint32_t)h[pos + 2] << 16) |
                             ((uint32_t)h[pos + 3] << 24);
        pos += 4 + (size_t)len;
        if (pos > rspt_gpu_max_compressed_size(p)) return 0;
    }
    return pos;
}
}  // namespace

extern "C" int rspt_gpu_decompress_host(rspt_gpu_packer* p, const uint8_t* h_src, size_t* src_len, uint8_t* h_dst)
{
    if (!p || !h_src || !src_len || !h_dst) return RSPT_E_ARG;
    DeviceGuard dg(p->device);
    unsigned nb = 0;
    int rc = rspt_gpu_nb(p, &nb);
    if (rc) return rc;
    const size_t len = host_frame_len(p, h_src, nb);
    if (!len) return fail_arg(p, "malformed frame"), RSPT_E_STREAM;
    memcpy(p->h_pin, h_src, len);
    uint64_t off[2] = {0, (uint64_t)len};
    RSPT_CUDA_CHECK(cudaMemcpyAsync(p->d_one_dst, p->h_pin, len, cudaMemcpyHostToDevice, p->stream));
    RSPT_CUDA_CHECK(cudaMemcpyAsync(p->d_one_off, off, sizeof(off), cudaMemcpyHostToDevice, p->stream));
    rc = rspt_gpu_decompress_batch(p, p->d_one_dst, p->d_one_off, 1, nullptr, nullptr, p->d_one_src, nullptr);
    if (rc) return rc;
    int32_t st = 0;
    RSPT_CUDA_CHECK(cudaMemcpyAsync(&st, p->d_status_tmp, 4, cudaMemcpyDeviceToHost, p->stream));
    RSPT_CUDA_CHECK(cudaStreamSynchronize(p->stream));
    RSPT_CUDA_CHECK(cudaMemcpyAsync(p->h_pin, p->d_one_src, p->s.frame_bytes, cudaMemcpyDeviceToHost, p->stream));
    RSPT_CUDA_CHECK(cudaStreamSynchronize(p->stream));
    memcpy(h_dst, p->h_pin, p->s.frame_bytes);
    *src_len = len;
    return st ? RSPT_E_STREAM : RSPT_OK;
}

namespace {
// Host-buffer compress runs as a three-stage pipeline over chunks of frames: H2D of chunk i+1,
// the kernels of chunk i and D2H of chunk i-1 overlap on three streams with two device buffers.
// The payload D2H of a chunk needs its byte total on the host, so the host waits for the (tiny)
// offsets copy of the previous chunk while the next chunk is already queued.
int ensure_host_pipe(rspt_gpu_packer* p)
{
    HostPipe& hp = p->pipe;
    if (hp.chunk) return RSPT_OK;
    size_t c = (size_t)(32u << 20) / p->s.frame_bytes;  // ~32 MB of raw input per chunk
    if (const char* e = getenv("RSPT_HOST_CHUNK_FRAMES")) c = (size_t)atol(e);
    if (c < 1) c = 1;
    if (c > p->max_batch) c = p->max_batch;
    RSPT_CUDA_CHECK(cudaStreamCreateWithFlags(&hp.s_in, cudaStreamNonBlocking));
    RSPT_CUDA_CHECK(cudaStreamCreateWithFlags(&hp.s_out, cudaStreamNonBlocking));
    for (int b = 0; b < 2; ++b) {
        RSPT_CUDA_CHECK(cudaEventCreateWithFlags(&hp.ev_in[b], cudaEventDisableTiming));
        RSPT_CUDA_CHECK(cudaEventCreateWithFlags(&hp.ev_comp[b], cudaEventDisableTiming));
        RSPT_CUDA_CHECK(cudaEventCreateWithFlags(&hp.ev_off[b], cudaEventDisableTiming));
        RSPT_CUDA_CHECK(cudaEventCreateWithFlags(&hp.ev_out[b], cudaEventDisableTiming));
        RSPT_CUDA_CHECK(dalloc(hp.d_src[b], c * (size_t)p->s.frame_bytes));
        RSPT_CUDA_CHECK(dalloc(hp.d_dst[b], c * rspt_gpu_max_compressed_size(p)));
        RSPT_CUDA_CHECK(dalloc(hp.d_off[b], c + 1));
        RSPT_CUDA_CHECK(cudaMallocHost(reinterpret_cast<void**>(&hp.h_off[b]), (c + 1) * sizeof(uint64_t)));
    }
    hp.chunk = c;
    return RSPT_OK;
}

void destroy_host_pipe(rspt_gpu_packer* p)
{
    HostPipe& hp = p->pipe;
    if (!hp.s_in && !hp.s_out) return;
    if (hp.s_in) cudaStreamSynchronize(hp.s_in);
    if (hp.s_out) cudaStreamSynchronize(hp.s_out);
    for (int b = 0; b < 2; ++b) {
        if (hp.ev_in[b]) cudaEventDestroy(hp.ev_in[b]);
        if (hp.ev_comp[b]) cudaEventDestroy(hp.ev_comp[b]);
        if (hp.ev_off[b]) cudaEventDestroy(hp.ev_off[b]);
        if (hp.ev_out[b]) cudaEventDestroy(hp.ev_out[b]);
        if (hp.d_src[b]) cudaFree(hp.d_src[b]);
        if (hp.d_dst[b]) cudaFree(hp.d_dst[b]);
        if (hp.d_off[b]) cudaFree(hp.d_off[b]);
        if (hp.h_off[b]) cudaFreeHost(hp.h_off[b]);
    }
    if (hp.s_in) cudaStreamDestroy(hp.s_in);
    if (hp.s_out) cudaStreamDestroy(hp.s_out);
    memset(&hp, 0, sizeof(hp));
}
}  // namespace

extern "C" int rspt_gpu_compress_batch_host(rspt_gpu_packer* p, const uint8_t* h_src, size_t n_frames, uint8_t* h_dst,
                                            size_t dst_capacity, uint64_t* h_offsets)
{
    if (!p || !h_src || !h_dst || !h_offsets) return RSPT_E_ARG;
    DeviceGuard dg(p->device);
    int rc = ensure_host_pipe(p);
    if (rc) return rc;
    HostPipe& hp = p->pipe;
    const size_t fb = p->s.frame_bytes, maxc = rspt_gpu_max_compressed_size(p), C = hp.chunk;
    const size_t nchunks = (n_frames + C - 1) / C;
    uint64_t running = 0;  // bytes of the chunks whose offsets have reached the host
    h_offsets[0] = 0;
    int status = RSPT_OK;
    // stage 3 of chunk j: wait for its offsets, rebase them, start the payload copy
    auto drain = [&](size_t j) -> int {
        const int b = (int)(j & 1);
        const size_t f0 = j * C, nf = (n_frames - f0 < C) ? n_frames - f0 : C;
        RSPT_CUDA_CHECK(cudaEventSynchronize(hp.ev_off[b]));
        for (size_t i = 1; i <= nf; ++i) h_offsets[f0 + i] = running + hp.h_off[b][i];
        const uint64_t total = hp.h_off[b][nf];
        if (running + total > dst_capacity) return fail_arg(p, "dst_capacity too small"), RSPT_E_CAPACITY;
        RSPT_CUDA_CHECK(cudaMemcpyAsync(h_dst + running, hp.d_dst[b], (size_t)total, cudaMemcpyDeviceToHost, hp.s_out));
        RSPT_CUDA_CHECK(cudaEventRecord(hp.ev_out[b], hp.s_out));
        running += total;
        return RSPT_OK;
    };
    for (size_t j = 0; j < nchunks && status == RSPT_OK; ++j) {
        const int b = (int)(j & 1);
        const size_t f0 = j * C, nf = (n_frames - f0 < C) ? n_frames - f0 : C;
        // stage 1: H2D once the kernels of chunk j-2 have released the input buffer
        RSPT_CUDA_CHECK(cudaStreamWaitEvent(hp.s_in, hp.ev_comp[b], 0));
        RSPT_CUDA_CHECK(cudaMemcpyAsync(hp.d_src[b], h_src + f0 * fb, nf * fb, cudaMemcpyHostToDevice, hp.s_in));
        RSPT_CUDA_CHECK(cudaEventRecord(hp.ev_in[b], hp.s_in));
        // stage 2: kernels, once the input is there and the payload of chunk j-2 has left the output buffer
        RSPT_CUDA_CHECK(cudaStreamWaitEvent(p->stream, hp.ev_in[b], 0));
        RSPT_CUDA_CHECK(cudaStreamWaitEvent(p->stream, hp.ev_out[b], 0));
        status = rspt_gpu_compress_batch(p, hp.d_src[b], nf, hp.d_dst[b], nf * maxc, hp.d_off[b], nullptr, nullptr);
        if (status != RSPT_OK) break;
        RSPT_CUDA_CHECK(cudaEventRecord(hp.ev_comp[b], p->stream));
        // stage 3 of the previous chunk, then queue this chunk's offsets copy behind it
        if (j > 0) status = drain(j - 1);
        RSPT_CUDA_CHECK(cudaStreamWaitEvent(hp.s_out, hp.ev_comp[b], 0));
        RSPT_CUDA_CHECK(cudaMemcpyAsync(hp.h_off[b], hp.d_off[b], (nf + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, hp.s_out));
        RSPT_CUDA_CHECK(cudaEventRecord(hp.ev_off[b], hp.s_out));
    }
    if (status == RSPT_OK && nchunks > 0) status = drain(nchunks - 1);
    RSPT_CUDA_CHECK(cudaStreamSynchronize(hp.s_out));
    RSPT_CUDA_CHECK(cudaStreamSynchronize(p->stream));
    return status;
}

// The mirror image: H2D of the compressed bytes of chunk i+1 (with its offsets, rebased to the chunk), the
// kernels of chunk i and D2H of the samples of chunk i-1 overlap on the same three streams and buffers.
// The stream arrives as the reference would store it -- no decode index -- so the index is rebuilt per chunk
// on the device (k_hzr_build_index); the call is bound by the D2H of the raw samples all the same.
extern "C" int rspt_gpu_decompress_batch_host(rspt_gpu_packer* p, const uint8_t* h_src, const uint64_t* h_offsets,
                                              size_t n_frames, uint8_t* h_dst)
{
    if (!p || !h_src || !h_offsets || !h_dst) return RSPT_E_ARG;
    if (n_frames == 0) return RSPT_OK;
    DeviceGuard dg(p->device);
    int rc = ensure_host_pipe(p);
    if (rc) return rc;
    HostPipe& hp = p->pipe;
    const size_t fb = p->s.frame_bytes, maxc = rspt_gpu_max_compressed_size(p), C = hp.chunk;
    const size_t nchunks = (n_frames + C - 1) / C;
    for (size_t f = 0; f < n_frames; ++f)
        if (h_offsets[f + 1] < h_offsets[f] || h_offsets[f + 1] - h_offsets[f] > maxc) return fail_arg(p, "offsets exceed the frame bound"), RSPT_E_STREAM;
    for (size_t j = 0; j < nchunks; ++j) {
        const int b = (int)(j & 1);
        const size_t f0 = j * C, nf = (n_frames - f0 < C) ? n_frames - f0 : C;
        const uint64_t base = h_offsets[f0], bytes = h_offsets[f0 + nf] - base;
        // stage 1: H2D once the kernels of chunk j-2 have released the compressed buffer; the pinned offsets
        // staging is free once ITS copy of chunk j-2 has gone out
        if (j >= 2) RSPT_CUDA_CHECK(cudaEventSynchronize(hp.ev_in[b]));
        for (size_t i = 0; i <= nf; ++i) hp.h_off[b][i] = h_offsets[f0 + i] - base;
        RSPT_CUDA_CHECK(cudaStreamWaitEvent(hp.s_in, hp.ev_comp[b], 0));
        RSPT_CUDA_CHECK(cudaMemcpyAsync(hp.d_dst[b], h_src + base, (size_t)bytes, cudaMemcpyHostToDevice, hp.s_in));
        RSPT_CUDA_CHECK(cudaMemcpyAsync(hp.d_off[b], hp.h_off[b], (nf + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, hp.s_in));
        RSPT_CUDA_CHECK(cudaEventRecord(hp.ev_in[b], hp.s_in));
        // stage 2: kernels, once the input is there and the samples of chunk j-2 have left the output buffer
        RSPT_CUDA_CHECK(cudaStreamWaitEvent(p->stream, hp.ev_in[b], 0));
        RSPT_CUDA_CHECK(cudaStreamWaitEvent(p->stream, hp.ev_out[b], 0));
        rc = rspt_gpu_decompress_batch(p, hp.d_dst[b], hp.d_off[b], nf, nullptr, nullptr, hp.d_src[b], nullptr);
        if (rc) return rc;
        RSPT_CUDA_CHECK(cudaEventRecord(hp.ev_comp[b], p->stream));
        // stage 3: D2H of the samples
        RSPT_CUDA_CHECK(cudaStreamWaitEvent(hp.s_out, hp.ev_comp[b], 0));
        RSPT_CUDA_CHECK(cudaMemcpyAsync(h_dst + f0 * fb, hp.d_src[b], nf * fb, cudaMemcpyDeviceToHost, hp.s_out));
        RSPT_CUDA_CHECK(cudaEventRecord(hp.ev_out[b], hp.s_out));
    }
    RSPT_CUDA_CHECK(cudaStreamSynchronize(hp.s_out));
    RSPT_CUDA_CHECK(cudaStreamSynchronize(p->stream));
    return RSPT_OK;
}

// ---------------------------------------------------------------------------------------------
// stage-level entry points for the parity tests
// ---------------------------------------------------------------------------------------------
extern "C" int rspt_gpu_debug_planes(rspt_gpu_packer* p, const uint8_t* d_src, size_t n_frames, uint8_t* d_planes,
                                     uint8_t* d_header)
{
    if (!p || !d_src || !d_planes || n_frames > p->max_batch) return RSPT_E_ARG;
    DeviceGuard dg(p->device);
    int rc = launch_forward_transform(p, d_src, n_frames);
    if (rc) return rc;
    const Shape& s = p->s;
    RSPT_CUDA_CHECK(cudaMemcpy2DAsync(d_planes, s.N, p->d_planes, s.plane_stride, s.N, n_frames * s.nb_alloc,
                                      cudaMemcpyDeviceToDevice, p->stream));
    if (d_header && s.hdr_bytes)
        RSPT_CUDA_CHECK(cudaMemcpyAsync(d_header, p->d_headers, n_frames * s.hdr_bytes, cudaMemcpyDeviceToDevice, p->stream));
    return RSPT_OK;
}

extern "C" int rspt_gpu_debug_hzr_tables(rspt_gpu_packer* p, const uint8_t* d_block, size_t n, uint32_t* d_hist,
                                         uint32_t* d_codes, uint32_t* d_info)
{
    if (!p || !d_block || n < 1 || n > kBlock || ((uintptr_t)d_block & 15)) return RSPT_E_ARG;
    DeviceGuard dg(p->device);
    Shape s = p->s;
    s.N = (uint32_t)n; s.nblk = 1; s.nb_alloc = 1; s.plane_stride = (uint32_t)((n + 15) & ~(size_t)15);
    k_hzr_hist<3><<<1, kHistThreads, kHistSmemList, p->stream>>>(d_block, s, p->d_frame_nb, p->d_hist, p->d_step_lz, p->d_lists, p->d_list_n, p->d_blk_class);
    k_hzr_hist<2><<<1, kHistThreads, 0, p->stream>>>(d_block, s, p->d_frame_nb, p->d_hist, p->d_step_lz, p->d_lists, p->d_list_n, p->d_blk_class);
    k_hzr_tree<<<1, 32 * kTreeWarps, 0, p->stream>>>(p->d_hist, s, p->d_frame_nb, p->d_blk_class, kClassSparse, 1, p->d_codes, p->d_tree, p->d_info, p->d_ctr);
    k_hzr_tree<<<1, 32 * kTreeWarps, 0, p->stream>>>(p->d_hist, s, p->d_frame_nb, p->d_blk_class, kClassDense, 1, p->d_codes, p->d_tree, p->d_info, p->d_ctr);
    p->launches += 4;
    RSPT_CUDA_CHECK(cudaGetLastError());
    if (d_hist) RSPT_CUDA_CHECK(cudaMemcpyAsync(d_hist, p->d_hist, kNumSymbols * 4, cudaMemcpyDeviceToDevice, p->stream));
    if (d_codes) RSPT_CUDA_CHECK(cudaMemcpyAsync(d_codes, p->d_codes, kNumSymbols * 4, cudaMemcpyDeviceToDevice, p->stream));
    if (d_info) {
        RSPT_CUDA_CHECK(cudaStreamSynchronize(p->stream));
        BlkInfo bi;
        RSPT_CUDA_CHECK(cudaMemcpy(&bi, p->d_info, sizeof(bi), cudaMemcpyDeviceToHost));
        uint32_t v[4] = {bi.mode, bi.payload_len, bi.tree_nbits, bi.n_used};
        RSPT_CUDA_CHECK(cudaMemcpy(d_info, v, sizeof(v), cudaMemcpyHostToDevice));
    }
    return RSPT_OK;
}

extern "C" int rspt_gpu_crc32c(const uint8_t* d_data, size_t n, uint32_t* h_crc, void* stream)
{
    if (!d_data || !h_crc || n > kBlock) return RSPT_E_ARG;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return RSPT_E_NOGPU;
    int rc = ensure_device_constants(dev);
    if (rc) return rc;
    uint32_t* d_out = static_cast<uint32_t*>(result_slot(dev));
    allow_smem(k_crc32c, kEncodeSmem);
    k_crc32c<<<1, 1024, kEncodeSmem, (cudaStream_t)stream>>>(d_data, (uint32_t)n, g_crc[dev], 3, d_out);
    cudaError_t e = cudaMemcpyAsync(h_crc, d_out, 4, cudaMemcpyDeviceToHost, (cudaStream_t)stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize((cudaStream_t)stream);
    return e == cudaSuccess ? RSPT_OK : RSPT_E_CUDA;
}

// ---------------------------------------------------------------------------------------------
// synthetic workload, PRDN terms, offset rebasing
// ---------------------------------------------------------------------------------------------
namespace {

template <int BPS>
__global__ void __launch_bounds__(256) k_synth(uint8_t* __restrict__ dst, uint64_t first, uint32_t n_frames, int ch, int ns,
                                               rspt_synth_params prm, const int32_t* __restrict__ tab)
{
    // one CTA per (frame, 256-sample tile); threads run along samples, loop over channels
    const uint32_t tiles = ((uint32_t)ns + 255u) / 256u;
    const uint32_t f = blockIdx.x / tiles, s = (blockIdx.x % tiles) * 256u + threadIdx.x;
    if (f >= n_frames || s >= (uint32_t)ns) return;
    const int32_t* beat = tab;
    const int32_t* sine = tab + RSPT_SYNTH_TABLE;
    uint8_t* out = dst + ((size_t)f * ns + s) * ch * BPS;
    for (int c = 0; c < ch; ++c) {
        const rspt_synth_chan k = rspt_synth_channel(&prm, first + f, (uint32_t)c);
        const uint32_t v = (uint32_t)rspt_synth_sample(&prm, &k, beat, sine, first + f, (uint32_t)c, s, BPS);
#pragma unroll
        for (int b = 0; b < BPS; ++b) out[c * BPS + b] = (uint8_t)(v >> (8 * b));
    }
}

template <int BPS>
__global__ void __launch_bounds__(256) k_prdn(const uint8_t* __restrict__ a, const uint8_t* __restrict__ b, uint32_t n_frames,
                                              int ch, int ns, double* __restrict__ out)
{
    // one CTA per (frame, channel): mean = average_32 (utils.cpp:30-40), then the two sums of
    // lib_rspt_test/rspt_test.cpp:98-111
    __shared__ long long s_sum[8];
    __shared__ double s_d[2][8];
    const uint32_t f = blockIdx.x / ch, c = blockIdx.x % ch;
    const uint8_t* pa = a + (size_t)f * ns * ch * BPS + (size_t)c * BPS;
    const uint8_t* pb = b + (size_t)f * ns * ch * BPS + (size_t)c * BPS;
    const size_t step = (size_t)ch * BPS;
    long long sum = 0;
    for (int i = threadIdx.x; i < ns; i += blockDim.x) sum += load_sample<BPS>(pa + i * step);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xFFFFFFFFu, sum, o);
    if (lane_id() == 0) s_sum[warp_id()] = sum;
    __syncthreads();
    long long tot = 0;
    for (int w = 0; w < 8; ++w) tot += s_sum[w];
    const int32_t mean = (int32_t)(long long)((unsigned long long)tot / (unsigned long long)ns);
    double e2 = 0, d2 = 0;
    for (int i = threadIdx.x; i < ns; i += blockDim.x) {
        const double x = load_sample<BPS>(pa + i * step), y = load_sample<BPS>(pb + i * step);
        e2 += (x - y) * (x - y);
        d2 += (x - mean) * (x - mean);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        e2 += __shfl_xor_sync(0xFFFFFFFFu, e2, o);
        d2 += __shfl_xor_sync(0xFFFFFFFFu, d2, o);
    }
    if (lane_id() == 0) {
        s_d[0][warp_id()] = e2;
        s_d[1][warp_id()] = d2;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double x = 0, y = 0;
        for (int w = 0; w < 8; ++w) {
            x += s_d[0][w];
            y += s_d[1][w];
        }
        atomicAdd(out, x);
        atomicAdd(out + 1, y);
    }
}

__global__ void k_rebase(uint64_t* off, size_t n, const uint64_t* totals, int rank)
{
    unsigned long long base = 0;
    for (int r = 0; r < rank; ++r) base += totals[r];
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) off[i] += base;
}

}  // namespace

extern "C" int rspt_gpu_synth_ecg(uint8_t* d_dst, uint64_t first_frame, size_t n_frames, int bps, int ch, int ns,
                                  uint64_t seed, int32_t amplitude, int32_t sigma, void* stream)
{
    if (!d_dst || bps < 1 || bps > 4 || ch < 1 || ns < 1) return RSPT_E_ARG;
    if (n_frames == 0) return RSPT_OK;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return RSPT_E_NOGPU;
    int rc = ensure_device_constants(dev);
    if (rc) return rc;
    rspt_synth_params prm = {seed, amplitude, sigma};
    const uint32_t tiles = ((uint32_t)ns + 255u) / 256u;
    const dim3 grid((unsigned)(n_frames * tiles));
    cudaStream_t st = (cudaStream_t)stream;
    switch (bps) {
    case 1: k_synth<1><<<grid, 256, 0, st>>>(d_dst, first_frame, (uint32_t)n_frames, ch, ns, prm, g_synth_tab[dev]); break;
    case 2: k_synth<2><<<grid, 256, 0, st>>>(d_dst, first_frame, (uint32_t)n_frames, ch, ns, prm, g_synth_tab[dev]); break;
    case 3: k_synth<3><<<grid, 256, 0, st>>>(d_dst, first_frame, (uint32_t)n_frames, ch, ns, prm, g_synth_tab[dev]); break;
    default: k_synth<4><<<grid, 256, 0, st>>>(d_dst, first_frame, (uint32_t)n_frames, ch, ns, prm, g_synth_tab[dev]); break;
    }
    return cudaGetLastError() == cudaSuccess ? RSPT_OK : RSPT_E_CUDA;
}

extern "C" int rspt_gpu_prdn_terms(const uint8_t* d_orig, const uint8_t* d_dec, size_t n_frames, int bps, int ch, int ns,
                                   double* h_out, void* stream)
{
    if (!d_orig || !d_dec || !h_out || bps < 1 || bps > 4) return RSPT_E_ARG;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return RSPT_E_NOGPU;
    int rc = ensure_device_constants(dev);
    if (rc) return rc;
    double* d_out = static_cast<double*>(result_slot(dev));
    cudaStream_t st = (cudaStream_t)stream;
    cudaMemsetAsync(d_out, 0, 16, st);
    const dim3 grid((unsigned)(n_frames * ch));
    switch (bps) {
    case 1: k_prdn<1><<<grid, 256, 0, st>>>(d_orig, d_dec, (uint32_t)n_frames, ch, ns, d_out); break;
    case 2: k_prdn<2><<<grid, 256, 0, st>>>(d_orig, d_dec, (uint32_t)n_frames, ch, ns, d_out); break;
    case 3: k_prdn<3><<<grid, 256, 0, st>>>(d_orig, d_dec, (uint32_t)n_frames, ch, ns, d_out); break;
    default: k_prdn<4><<<grid, 256, 0, st>>>(d_orig, d_dec, (uint32_t)n_frames, ch, ns, d_out); break;
    }
    cudaError_t e = cudaMemcpyAsync(h_out, d_out, 16, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    return e == cudaSuccess ? RSPT_OK : RSPT_E_CUDA;
}

extern "C" int rspt_gpu_rebase_offsets(uint64_t* d_offsets, size_t n, const uint64_t* d_all_totals, int rank, void* stream)
{
    if (!d_offsets || !d_all_totals || rank < 0) return RSPT_E_ARG;
    if (n == 0 || rank == 0) return RSPT_OK;
    k_rebase<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(d_offsets, n, d_all_totals, rank);
    return cudaGetLastError() == cudaSuccess ? RSPT_OK : RSPT_E_CUDA;
}
