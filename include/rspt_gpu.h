/* rspt_gpu.h -- C ABI of the B200-native signal-packer library (librspt_gpu.so).
 *
 * This is the drop-in boundary for rspt's packer hot path.  The reference has no FFI of its own:
 * its only plugin interface is the C++ abstract class i_signal_packer
 * (/root/reference/lib_rspt/signal_packer.h:29-73).  The entry points below are what a binding
 * for that path needs: one handle per packer instance (= one `new_*` factory call), batched
 * compress / decompress over many independent fixed-shape frames, and the size bound.  The C++
 * class in include/signal_packer.h is implemented on top of exactly these calls
 * (rspt_b200/csrc/signal_packer_gpu.cpp); INTEGRATION.md shows the binding stubs.
 *
 * Conventions: plain pointers and sizes only; every function returns 0 on success or a negative
 * RSPT_E_* code and never throws; `d_` pointers are CUDA device pointers on the handle's device,
 * `h_` pointers are host pointers.  Batch calls are asynchronous on the handle's stream unless
 * stated otherwise.  A handle is not thread-safe; distinct handles are independent
 * (reference: instances are not re-entrant either, signal_packer_base.h:20-21).
 * There is no CPU fallback anywhere in this library.
 */
#ifndef RSPT_GPU_H_
#define RSPT_GPU_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RSPT_GPU_ABI_VERSION 1

/* packer kinds <-> reference factories */
enum {
    RSPT_XDELTA_HZR = 0, /* i_signal_packer::new_xdelta_hzr, signal_packer.h:59 */
    RSPT_HZR = 1,        /* i_signal_packer::new_hzr,        signal_packer.h:62 */
    RSPT_HADAMARD = 2,   /* i_signal_packer::new_hadamard,   signal_packer.h:68 */
    RSPT_DCT = 3         /* i_signal_packer::new_dct,        signal_packer.h:65 */
};

enum {
    RSPT_OK = 0,
    RSPT_E_ARG = -1,      /* bad argument / unsupported shape */
    RSPT_E_CUDA = -2,     /* CUDA runtime error (see rspt_gpu_last_error) */
    RSPT_E_CAPACITY = -3, /* destination or batch capacity too small */
    RSPT_E_STREAM = -4,   /* malformed compressed stream */
    RSPT_E_NOGPU = -5,    /* no usable CUDA device: the library refuses to run */
    RSPT_E_CRC = -6       /* a block's CRC-32C does not match its payload (verify only) */
};

typedef struct rspt_gpu_packer rspt_gpu_packer;

/* Replaces the constructor behind new_xdelta_hzr / new_hzr / new_hadamard / new_dct
 * (signal_packer_xdelta_hzr.cpp:42-50, signal_packer_hzr.cpp, signal_packer_hadamard.cpp:47-55,
 * signal_packer_dct.cpp:49-58).  `nb` = nr_bytes_to_encode, used by RSPT_XDELTA_HZR only.
 * `stream` is a cudaStream_t (NULL = the CUDA default stream); all work of the handle is ordered on it.  `max_batch_frames` sizes the
 * device scratch (planes, histograms, code tables); batches larger than that are rejected. */
int rspt_gpu_create(int kind, size_t bytes_per_sample, size_t nr_channels, size_t nr_samples,
                    size_t nb, int device, void* stream, size_t max_batch_frames,
                    rspt_gpu_packer** out);

/* Replaces delete_xdelta_hzr / delete_hzr / delete_hadamard / delete_dct (signal_packer.h:60-69). */
int rspt_gpu_destroy(rspt_gpu_packer* p);

size_t rspt_gpu_frame_bytes(const rspt_gpu_packer* p); /* bps * ch * ns */
size_t rspt_gpu_header_bytes(const rspt_gpu_packer* p); /* 3*ch for hadamard/dct, else 0 */

/* Worst-case bytes of ONE compressed frame: 1 + header + planes * (4 + hzr_max_compressed_size(ch*ns))
 * (signal_packer_base.cpp:83-95, hzr_encode.c:489-497), with `planes` the largest count the
 * instance can reach (xdelta_hzr may escalate up to bytes_per_sample). */
size_t rspt_gpu_max_compressed_size(const rspt_gpu_packer* p);

/* Current plane count: the reference's nr_bytes_to_compress_ (signal_packer_xdelta_hzr.cpp:39,66).
 * Synchronises the handle's stream. */
int rspt_gpu_nb(rspt_gpu_packer* p, unsigned* nb);

/* Replaces i_signal_packer::compress (signal_packer.h:44) for `n_frames` frames at once.
 *   d_src      [n_frames][frame_bytes]  interleaved little-endian samples ([ns][ch][bps])
 *   d_dst      the frames' streams, concatenated back to back, each byte-identical to what the
 *              reference writes for that frame (xdelta_hzr, hzr, hadamard; dct: on its exact path,
 *              see rspt_gpu_set_dct_exact -- its default FFT path is held to a tolerance instead)
 *   d_offsets  [n_frames + 1] byte offset of every frame in d_dst; d_offsets[n_frames] = total
 *   d_frame_nb [n_frames] planes used per frame (the reference does not store this in the
 *              stream; decompress needs it); may be NULL
 *   d_sidecar  optional out-of-band decode index (rspt_gpu_sidecar_bytes(p, n_frames) bytes);
 *              NULL = not produced.  The stream itself never depends on it.
 * Frames are processed as if by ONE reference instance in order: the xdelta_hzr plane count
 * carries from frame to frame and from batch to batch (signal_packer_xdelta_hzr.cpp:63-69). */
int rspt_gpu_compress_batch(rspt_gpu_packer* p, const uint8_t* d_src, size_t n_frames,
                            uint8_t* d_dst, size_t dst_capacity, uint64_t* d_offsets,
                            uint8_t* d_frame_nb, void* d_sidecar);

/* Replaces i_signal_packer::decompress (signal_packer.h:57) for `n_frames` frames.
 *   d_src      concatenated frames; d_offsets [n_frames + 1] as produced by compress (frames are
 *              self-delimiting but carry no index, signal_packer_base.cpp:121)
 *   d_frame_nb per-frame plane count or NULL = the handle's current count for every frame
 *   d_sidecar  optional decode index produced by compress_batch (or rspt_gpu_build_index) for these
 *              same frames, or NULL (streams from the CPU reference): the index is then rebuilt on
 *              the device first, into scratch owned by the handle
 *   d_dst      [n_frames][frame_bytes]
 *   d_status   [n_frames] 0 = ok, else RSPT_E_STREAM-style code; may be NULL */
int rspt_gpu_decompress_batch(rspt_gpu_packer* p, const uint8_t* d_src, const uint64_t* d_offsets,
                              size_t n_frames, const uint8_t* d_frame_nb, const void* d_sidecar,
                              uint8_t* d_dst, int32_t* d_status);

/* The same two calls with the samples as int32 words [n_frames][ch][ns] (flat channel-major: the reference's
 * own int32 matrix, convert_native_to_i32) instead of interleaved native bytes.  Frame format, handle state,
 * counters (raw bytes count bps * ch * ns per frame) and stage timers are shared with the native calls: the
 * xdelta_hzr plane count carries across batches whichever entry point compressed them.
 *   compress    only the low 8 * bps bits of a word are the sample, higher bits are ignored.  Stream,
 *               offsets, frame_nb and sidecar equal what rspt_gpu_compress_batch writes for the native frame
 *               holding the low bps bytes of every word, for all four packers (and both dct paths).
 *   decompress  every word is the sample rspt_gpu_decompress_batch writes, sign-extended from 8 * bps bits
 *               (for every stream, including ones from the CPU reference).
 * d_src / d_dst (the word side) must be 4-byte aligned, else RSPT_E_ARG; 16-byte alignment is faster. */
int rspt_gpu_compress_batch_i32(rspt_gpu_packer* p, const int32_t* d_src, size_t n_frames, uint8_t* d_dst,
                                size_t dst_capacity, uint64_t* d_offsets, uint8_t* d_frame_nb, void* d_sidecar);
int rspt_gpu_decompress_batch_i32(rspt_gpu_packer* p, const uint8_t* d_src, const uint64_t* d_offsets, size_t n_frames,
                                  const uint8_t* d_frame_nb, const void* d_sidecar, int32_t* d_dst, int32_t* d_status);

/* Compress n_frames frames and append them to a stored batch (a "store") of n_stored frames / stored_bytes stream
 * bytes, so that a store can grow far beyond max_batch_frames.  Writes frames n_stored .. n_stored + n_frames - 1
 * of the store and nothing else of it:
 *   d_store          the stream from byte stored_bytes on (store_capacity bytes in all)
 *   d_store_offsets  entries n_stored .. n_stored + n_frames; entry n_stored is (re)written as stored_bytes
 *   d_store_frame_nb entries n_stored .. n_stored + n_frames - 1 (may be NULL)
 *   d_store_sidecar  the decode-index entries of the new blocks at their places in the store's index (may be NULL;
 *                    sidecar_capacity bytes in all)
 * stored_bytes must equal d_store_offsets[n_stored] as the previous append left it (0 for an empty store); it is
 * passed from the host so that capacities are checked without a read-back and the call stays asynchronous on the
 * handle's stream.  Appending B1 .. Bk on one handle writes, byte for byte, the stream [0, total), offsets,
 * frame_nb and used sidecar prefix that one rspt_gpu_compress_batch over all their frames writes on a fresh handle
 * of the same arguments: the xdelta_hzr plane count carries across appends as across batches.  Counters add
 * n_frames and this call's bytes; stage timers as for compress_batch.  Refused before anything is launched:
 *   n_frames > max_batch_frames                                                    RSPT_E_CAPACITY
 *   (n_stored + n_frames) * planes * blocks per plane >= 2^32 (block ordinals)     RSPT_E_ARG
 *   stored_bytes + n_frames * rspt_gpu_max_compressed_size > store_capacity        RSPT_E_CAPACITY
 *   a sidecar whose index words could reach 2^32 (the limit of the decode calls)   RSPT_E_ARG
 *   a sidecar with sidecar_capacity < rspt_gpu_sidecar_used_bytes(p, n_stored + n_frames,
 *                         stored_bytes + n_frames * rspt_gpu_max_compressed_size)  RSPT_E_CAPACITY
 * rspt_gpu_compress_batch is this call with n_stored = stored_bytes = 0.  _i32: d_src is int32 [n][ch][ns] as for
 * rspt_gpu_compress_batch_i32 (4-byte aligned, else RSPT_E_ARG); both may be mixed on one store. */
int rspt_gpu_compress_append(rspt_gpu_packer* p, const uint8_t* d_src, size_t n_frames,
                             uint8_t* d_store, size_t store_capacity, uint64_t* d_store_offsets,
                             size_t n_stored, size_t stored_bytes, uint8_t* d_store_frame_nb,
                             void* d_store_sidecar, size_t sidecar_capacity);
int rspt_gpu_compress_append_i32(rspt_gpu_packer* p, const int32_t* d_src, size_t n_frames,
                                 uint8_t* d_store, size_t store_capacity, uint64_t* d_store_offsets,
                                 size_t n_stored, size_t stored_bytes, uint8_t* d_store_frame_nb,
                                 void* d_store_sidecar, size_t sidecar_capacity);

/* Decode any list of frames of a stored batch (seek in a recording, a random minibatch of a dataset kept
 * compressed in HBM).  Output slot j receives stored frame d_frame_ids[j]: its bytes (words) equal row
 * d_frame_ids[j] of what rspt_gpu_decompress_batch (_i32) writes for the whole stored batch.  Ids may come in
 * any order and repeat.
 *   d_src, d_offsets [n_stored + 1], d_frame_nb [n_stored], d_sidecar
 *              the stored batch exactly as compress_batch produced it: d_offsets is the batch's full array, not
 *              a slice; d_frame_nb is indexed by stored id (NULL = the handle's current plane count for every
 *              frame); d_sidecar needs only its used prefix (rspt_gpu_sidecar_used_bytes(p, n_stored, ...)).
 *              d_sidecar NULL: an index is built for the selected frames only, in scratch owned by the handle
 *              (the cost follows n_frames, not n_stored).
 *   d_frame_ids [n_frames] int64 stored ids, on the device.  An id < 0 or >= n_stored gives d_status[j] =
 *              RSPT_E_ARG: nothing is read for it and the slot is written like a frame that fails to parse.
 *   d_dst      [n_frames][frame_bytes] (_i32: [n_frames][ch][ns] words, aligned as for decompress_batch_i32)
 *   d_status   [n_frames] per output slot, as for decompress_batch; may be NULL
 * n_frames <= max_batch_frames, else RSPT_E_CAPACITY; n_stored is not limited by the handle, but a stored batch
 * of more than 2^32 - 1 blocks (n_stored * planes * blocks per plane) is refused with RSPT_E_ARG, and a block
 * whose index entries would lie at or beyond word 2^32 of the index fails its frame with RSPT_E_STREAM.  A
 * malformed frame or a wrong index entry costs only the slots that name that frame.  Asynchronous on the
 * handle's stream; counters (frames_decompressed += n_frames) and the PARSE / DECODE / INVERSE stage timers
 * as for decompress_batch.  The decode index of a stored batch depends on the largest plane count of the
 * handle that wrote it: it is valid for any handle of the same kind, shape and `nb` argument. */
int rspt_gpu_decompress_frames(rspt_gpu_packer* p, const uint8_t* d_src, const uint64_t* d_offsets, size_t n_stored,
                               const uint8_t* d_frame_nb, const void* d_sidecar, const int64_t* d_frame_ids,
                               size_t n_frames, uint8_t* d_dst, int32_t* d_status);
int rspt_gpu_decompress_frames_i32(rspt_gpu_packer* p, const uint8_t* d_src, const uint64_t* d_offsets, size_t n_stored,
                                   const uint8_t* d_frame_nb, const void* d_sidecar, const int64_t* d_frame_ids,
                                   size_t n_frames, int32_t* d_dst, int32_t* d_status);

/* Output element types of the _float calls. */
enum {
    RSPT_OUT_F32 = 0,  /* float32 */
    RSPT_OUT_BF16 = 1  /* bfloat16 */
};

/* rspt_gpu_decompress_batch_i32 and rspt_gpu_decompress_frames_i32 with the samples in physical units, as float32
 * or bfloat16 [n_frames][ch][ns] (a training loop's input), dequantized per channel inside the kernels that
 * produce the samples.  With v the int32 word the _i32 call writes for an element of channel c:
 *   f32   y = float32((int64) v - (int64) zero_point[c]) * scale[c]   int64 -> float32 rounded to nearest even,
 *                                                                      then one float32 multiply rounded to nearest
 *   bf16  y above, rounded to nearest even to bfloat16 (not the exact product rounded once)
 * which is bit for bit what numpy ((v.astype(int64) - zp).astype(float32) * scale) or torch ((v.long() - zp).float()
 * * scale, then .to(torch.bfloat16)) computes from the int32 output.  IEEE throughout: subnormal results are kept,
 * overflow gives +-inf.  Results are specified for finite scales.
 *   out_type        RSPT_OUT_F32 or RSPT_OUT_BF16
 *   d_zero_point    int32 [ch] on the device, or NULL = 0 for every channel
 *   d_scale         float32 [ch] on the device, or NULL = 1.0 for every channel
 *   d_dst           [n_frames][ch][ns] elements of 4 (f32) or 2 (bf16) bytes, aligned to its element size;
 *                   16-byte alignment is faster
 * Everything else (sidecar or none, ids in any order with repeats, RSPT_E_ARG in the status slot of an id outside
 * [0, n_stored), n_stored not limited by the handle, counters, the PARSE / DECODE / INVERSE stage timers) is as for
 * the _i32 calls, and so is the call: asynchronous on the handle's stream.  The kernels read d_zero_point and d_scale
 * while the call runs, so the caller keeps them alive and unchanged until the stream has passed it.  Refused before
 * anything is launched: an unknown out_type, a NULL d_dst or one not aligned to its element size (RSPT_E_ARG),
 * n_frames > max_batch_frames (RSPT_E_CAPACITY). */
int rspt_gpu_decompress_batch_float(rspt_gpu_packer* p, const uint8_t* d_src, const uint64_t* d_offsets, size_t n_frames,
                                    const uint8_t* d_frame_nb, const void* d_sidecar, int out_type,
                                    const int32_t* d_zero_point, const float* d_scale, void* d_dst, int32_t* d_status);
int rspt_gpu_decompress_frames_float(rspt_gpu_packer* p, const uint8_t* d_src, const uint64_t* d_offsets, size_t n_stored,
                                     const uint8_t* d_frame_nb, const void* d_sidecar, const int64_t* d_frame_ids,
                                     size_t n_frames, int out_type, const int32_t* d_zero_point, const float* d_scale,
                                     void* d_dst, int32_t* d_status);

/* Integrity check without decoding: replaces hzr_verify (lib_hzr/hzr_decode.c:569-624) applied to
 * every hzr stream of `n_frames` frames -- frame / chunk / block headers are walked as in
 * decompress, and the CRC-32C of every block payload is compared with the block header.
 *   d_status   [n_frames] 0 = ok, RSPT_E_STREAM = malformed framing, RSPT_E_CRC = checksum mismatch
 * (The reference's decompress never checks the CRC, hzr_decode.c:343; neither does
 * rspt_gpu_decompress_batch.  This is the separate check a receiver runs on streams from either
 * implementation.) */
int rspt_gpu_verify_batch(rspt_gpu_packer* p, const uint8_t* d_src, const uint64_t* d_offsets,
                          size_t n_frames, const uint8_t* d_frame_nb, int32_t* d_status);

/* Decode index ("sidecar"), out of band.  The payload bits of every HUFF block are cut into at most 512 equal
 * intervals of at least 512 bits; the index holds one 32-bit entry per interval: where the first token that
 * ends at or behind the interval's first bit starts (12 bits, relative to the interval) and the output byte it
 * starts at (20 bits).  A block's entries sit at word (payload offset in the batch's stream >> 6) + block number,
 * so the index is valid only together with the d_src / d_offsets layout it was produced for.
 * rspt_gpu_sidecar_bytes is the buffer size to allocate (worst-case stream); the entries of a batch whose
 * stream has `stream_bytes` bytes lie in the first rspt_gpu_sidecar_used_bytes of it (one word per 64 stream
 * bytes + one per block: 5.4 KB for a 294 912-byte frame of 12 ch x 3 B x 8192, 6 % of its stream) -- that
 * prefix is what has to be stored next to the stream.  Code tables are NOT part of it: the decoder recovers
 * them from the tree bits in the stream (hzr_decode.c:263-333).  Entries are range-checked on use; a wrong
 * index yields RSPT_E_STREAM or wrong bytes in that frame, never an out-of-bounds access. */
size_t rspt_gpu_sidecar_bytes(const rspt_gpu_packer* p, size_t n_frames);
size_t rspt_gpu_sidecar_used_bytes(const rspt_gpu_packer* p, size_t n_frames, size_t stream_bytes);

/* Decode index for frames that came without one (written by the CPU reference, or stored without
 * the sidecar): header walk, then every HUFF block is cut into bit sub-sequences that are decoded
 * in parallel from guessed starts until the token boundaries stop moving (a prefix code
 * re-synchronises by itself).  The result equals the index compress_batch emits and can be kept
 * next to the stream: build once, decode many times.  d_sidecar: rspt_gpu_sidecar_bytes bytes. */
int rspt_gpu_build_index(rspt_gpu_packer* p, const uint8_t* d_src, const uint64_t* d_offsets,
                         size_t n_frames, const uint8_t* d_frame_nb, void* d_sidecar, int32_t* d_status);

/* rspt_gpu_build_index for the listed frames d_frame_ids[0 .. n_frames) of a stored batch of n_stored frames
 * (d_offsets [n_stored + 1], d_frame_nb [n_stored] or NULL, as for rspt_gpu_decompress_frames): their entries are
 * written into the stored batch's own index d_sidecar, at the words a whole-batch build_index would write, so a
 * store of any length is indexed in pieces of at most max_batch_frames frames.  n_frames > max_batch_frames gives
 * RSPT_E_CAPACITY; n_stored is not limited by the handle (but by 32-bit block ordinals, RSPT_E_ARG).  Per slot,
 * d_status[j] (may be NULL): RSPT_E_ARG for an id outside [0, n_stored), RSPT_E_STREAM for a malformed frame or
 * one whose entries would lie at or beyond byte sidecar_capacity of d_sidecar; such a slot writes nothing.
 * Asynchronous on the handle's stream. */
int rspt_gpu_build_index_frames(rspt_gpu_packer* p, const uint8_t* d_src, const uint64_t* d_offsets, size_t n_stored,
                                const uint8_t* d_frame_nb, const int64_t* d_frame_ids, size_t n_frames,
                                void* d_sidecar, size_t sidecar_capacity, int32_t* d_status);

/* Single-frame convenience with HOST buffers -- the exact shape of the reference calls
 * (signal_packer.h:44,57): stages host<->device, runs the batch path with n_frames = 1 and
 * synchronises.  decompress reports the consumed length through *src_len like the reference. */
int rspt_gpu_compress_host(rspt_gpu_packer* p, const uint8_t* h_src, uint8_t* h_dst,
                           size_t dst_max_len, size_t* dst_len);
int rspt_gpu_decompress_host(rspt_gpu_packer* p, const uint8_t* h_src, size_t* src_len, uint8_t* h_dst);

/* Host-buffer batch (what bench.py times as the end-to-end leg): H2D of the frames, the batch
 * path, D2H of offsets and payload.  h_offsets [n_frames + 1]. */
int rspt_gpu_compress_batch_host(rspt_gpu_packer* p, const uint8_t* h_src, size_t n_frames,
                                 uint8_t* h_dst, size_t dst_capacity, uint64_t* h_offsets);
int rspt_gpu_decompress_batch_host(rspt_gpu_packer* p, const uint8_t* h_src, const uint64_t* h_offsets,
                                   size_t n_frames, uint8_t* h_dst);

/* Pre-filter step in front of the packers, in place on `n_frames` device-resident frames of the
 * handle's shape: what the reference's pipeline does per frame with i_filter before packing
 * (lib_rspt_test/rspt_test.cpp:116-136; lib_rspt/filter.h:23-89) -- native -> int32 matrix, ONE
 * filter object walked over the channels (init_history_values(first sample, init_nr_samples), then
 * filter_opt per sample, result truncated to int32), back to native.  Bit-identical to the reference.
 *   iir: i_filter::new_iir(n, d, nr_coefficients), lib_filter/iir_filter.cpp:46-116; 2..5 coefficients
 *   fir: i_filter::new_fir(kernel, kernel_size), lib_filter/fir_filter.cpp:26-68
 * n / d / kernel are HOST arrays (a handful of doubles). */
int rspt_gpu_prefilter_iir(rspt_gpu_packer* p, uint8_t* d_frames, size_t n_frames, const double* n,
                           const double* d, int nr_coefficients, int init_nr_samples);
int rspt_gpu_prefilter_fir(rspt_gpu_packer* p, uint8_t* d_frames, size_t n_frames, const double* kernel,
                           int kernel_size);

/* Streaming ingest: a packet ring in PINNED host memory in front of a packer, modelled on the
 * reference's io_buffer (lib_ring_buffer/ring_buffers.h:150-201): one packet = one frame, the same
 * single-producer / single-consumer protocol and slot states (0 free, 1 being filled, 2 filled,
 * 3 consumed).  The producer (an acquisition thread) asks for the next address to fill exactly as with
 * io_buffer::get_next_address_to_fill -- NULL means the ring is full; a packet counts as filled once the
 * producer asks for the next one (:186-187), or when `flush` is set.  The consumer does not take the
 * filled packets one by one (get_next_filled_address) but drains them in batches: every run of filled
 * packets goes through the pipelined host-buffer path (H2D of chunk i+1, kernels of chunk i, D2H of chunk
 * i-1) and the compressed frames are appended to h_dst.
 *   h_offsets   [max frames of this drain + 1] offsets of the frames inside h_dst, starting at 0
 *   *n_frames   in: capacity of h_offsets - 1 (frames to take at most); out: frames compressed
 * The handle `p` must not be used for anything else while the ring exists. */
typedef struct rspt_gpu_ingest rspt_gpu_ingest;
int rspt_gpu_ingest_create(rspt_gpu_packer* p, size_t nr_max_packets, rspt_gpu_ingest** out);
int rspt_gpu_ingest_destroy(rspt_gpu_ingest* g);
uint8_t* rspt_gpu_ingest_next_address_to_fill(rspt_gpu_ingest* g);
int rspt_gpu_ingest_drain(rspt_gpu_ingest* g, int flush, uint8_t* h_dst, size_t dst_capacity,
                          uint64_t* h_offsets, size_t* n_frames);

int rspt_gpu_sync(rspt_gpu_packer* p);
const char* rspt_gpu_last_error(const rspt_gpu_packer* p);

/* Counters since creation (SURVEY.md section 5: never silent). Synchronises. */
typedef struct {
    uint64_t frames_compressed, frames_decompressed;
    uint64_t raw_bytes_in, compressed_bytes_out;
    uint64_t blocks_copy, blocks_huff, blocks_fill;
    uint64_t escalations;    /* "Compression needs one more byte to encode." events */
    uint64_t crc_failures;   /* blocks whose CRC-32C did not match (rspt_gpu_verify_batch) */
    uint64_t kernel_launches;
} rspt_gpu_counters;
int rspt_gpu_get_counters(rspt_gpu_packer* p, rspt_gpu_counters* out);

/* Per-stage device timing (CUDA events recorded on the handle's stream around each kernel group).
 * Off by default.  get: accumulated milliseconds and launch-group counts since the last reset;
 * synchronises the stream. */
enum {
    RSPT_STAGE_TRANSFORM = 0, /* samples -> byte planes (xdelta / fwht / dct) */
    RSPT_STAGE_HIST = 1,      /* per-block token histogram */
    RSPT_STAGE_TREE = 2,      /* Huffman tree + code tables + block plan */
    RSPT_STAGE_LAYOUT = 3,    /* frame sizes + offset scan */
    RSPT_STAGE_ENCODE = 4,    /* bit packing + CRC-32C + framing */
    RSPT_STAGE_PARSE = 5,     /* decode: frame / block header walk */
    RSPT_STAGE_DECODE = 6,    /* decode: hzr blocks -> planes */
    RSPT_STAGE_INVERSE = 7,   /* decode: planes -> samples */
    RSPT_STAGE_COUNT = 8
};
int rspt_gpu_set_stage_timing(rspt_gpu_packer* p, int enable);
int rspt_gpu_get_stage_times(rspt_gpu_packer* p, double* ms /*[RSPT_STAGE_COUNT]*/,
                             uint64_t* calls /*[RSPT_STAGE_COUNT]*/, int reset);

/* Stage-level entry points used by the parity tests (same device code as the batch path). */
int rspt_gpu_debug_planes(rspt_gpu_packer* p, const uint8_t* d_src, size_t n_frames,
                          uint8_t* d_planes /*[n][planes][ch*ns]*/, uint8_t* d_header /*[n][hdr]*/);
int rspt_gpu_debug_hzr_tables(rspt_gpu_packer* p, const uint8_t* d_block, size_t n,
                              uint32_t* d_hist /*[261]*/, uint32_t* d_codes /*[261]: code | len<<27*/,
                              uint32_t* d_info /*[4]: mode, payload_len, tree_nbits, n_used*/);
int rspt_gpu_crc32c(const uint8_t* d_data, size_t n, uint32_t* h_crc, void* stream);

/* Synthetic ECG-like workload (include/rspt_synth.h), frames [first_frame, first_frame + n). */
int rspt_gpu_synth_ecg(uint8_t* d_dst, uint64_t first_frame, size_t n_frames, int bps, int ch, int ns,
                       uint64_t seed, int32_t amplitude, int32_t sigma, void* stream);

/* Quality metric on device: PRDN as printed by the reference's test harness
 * (lib_rspt_test/rspt_test.cpp:98-111), accumulated over n_frames.  h_out = {sum_sq_err, sum_sq_dev}. */
int rspt_gpu_prdn_terms(const uint8_t* d_orig, const uint8_t* d_dec, size_t n_frames, int bps, int ch,
                        int ns, double* h_out, void* stream);

/* ---- multi-GPU placement of the concatenated stream (SURVEY.md section 8e) ---------------------------------
 * Frames shard over ranks; the path's only collective is ONE all-gather of a uint64 per rank (each rank's
 * compressed byte total).  NCCL is reached through its C API, resolved at run time from libnccl.so.2 (the copy
 * already loaded in the process, e.g. torch's, else the system one): no link-time dependency.
 *
 * rspt_gpu_comm_unique_id / _init / _destroy are ncclGetUniqueId / ncclCommInitRank / ncclCommDestroy for a
 * caller that has no NCCL communicator of its own (`id`: 128 bytes, produced on rank 0 and handed to the other
 * ranks by whatever means the host program has).  `comm` is an ncclComm_t; one created elsewhere works too. */
int rspt_gpu_comm_unique_id(uint8_t id[128]);
int rspt_gpu_comm_init(int world, const uint8_t id[128], int rank, int device, void** comm);
int rspt_gpu_comm_destroy(void* comm);

/* ncclAllGather(sendcount = 1, ncclUint64) of d_total into d_all_totals [world], on `stream`. */
int rspt_gpu_allgather_totals(void* comm, const uint64_t* d_total, uint64_t* d_all_totals, void* stream);

/* Rebase this rank's frame offsets by the exclusive prefix of the totals.  d_all_totals [world]. */
int rspt_gpu_rebase_offsets(uint64_t* d_offsets, size_t n_frames_plus_1, const uint64_t* d_all_totals,
                            int rank, void* stream);

/* Both steps for the batch rspt_gpu_compress_batch has just produced into d_offsets, OFF the handle's stream:
 * they run on a side stream of the handle ordered behind the compress, so the next batch's kernels start at
 * once.  A later rspt_gpu_compress_batch into the SAME d_offsets array waits for that array's placement first
 * (the handle remembers the last four placements); anything else that reads the rebased offsets needs
 * rspt_gpu_place_join, which makes the handle's stream wait for every placement issued so far. */
int rspt_gpu_place_offsets_async(rspt_gpu_packer* p, void* comm, uint64_t* d_offsets, size_t n_frames, int rank, int world);
int rspt_gpu_place_join(rspt_gpu_packer* p);

/* All later work of the handle is ordered on `stream` (a cudaStream_t) instead of the one given at create;
 * the caller orders the two streams against each other if work is still in flight. */
int rspt_gpu_set_stream(rspt_gpu_packer* p, void* stream);

/* dct only: 1 = the O(n^2) float-product / double-accumulate path over the reference's cosine table, whose
 * stream is byte-identical to the reference's (signal_packer_dct.cpp:76-100); 0 = the FP64 FFT path (default
 * for power-of-two lengths), held to the stated tolerance.  The RSPT_DCT_DIRECT environment variable sets
 * the default at create time. */
int rspt_gpu_set_dct_exact(rspt_gpu_packer* p, int exact);

#ifdef __cplusplus
}
#endif
#endif
