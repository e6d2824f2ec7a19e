"""ctypes binding of include/rspt_gpu.h.  No CPU fallback: importing the symbols fails loudly when
the CUDA library has not been built, and every call fails when there is no GPU."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "librspt_gpu.so")

KINDS = {"xdelta_hzr": 0, "hzr": 1, "hadamard": 2, "dct": 3}
OUT_TYPES = {"float32": 0, "bfloat16": 1}  # RSPT_OUT_F32 / RSPT_OUT_BF16
STAGES = ["transform", "hist", "tree", "layout", "encode", "parse", "decode", "inverse"]
ERRORS = {0: "ok", -1: "bad argument / unsupported shape", -2: "CUDA error", -3: "capacity too small",
          -4: "malformed stream", -5: "no CUDA device", -6: "CRC-32C mismatch"}

# every symbol include/rspt_gpu.h declares
EXPORTS = [
    "rspt_gpu_create", "rspt_gpu_destroy", "rspt_gpu_frame_bytes", "rspt_gpu_header_bytes",
    "rspt_gpu_max_compressed_size", "rspt_gpu_nb", "rspt_gpu_compress_batch", "rspt_gpu_decompress_batch",
    "rspt_gpu_compress_batch_i32", "rspt_gpu_decompress_batch_i32",
    "rspt_gpu_compress_append", "rspt_gpu_compress_append_i32", "rspt_gpu_build_index_frames",
    "rspt_gpu_decompress_frames", "rspt_gpu_decompress_frames_i32",
    "rspt_gpu_decompress_batch_float", "rspt_gpu_decompress_frames_float",
    "rspt_gpu_sidecar_bytes", "rspt_gpu_sidecar_used_bytes", "rspt_gpu_compress_host", "rspt_gpu_decompress_host",
    "rspt_gpu_compress_batch_host", "rspt_gpu_decompress_batch_host", "rspt_gpu_sync", "rspt_gpu_last_error",
    "rspt_gpu_get_counters", "rspt_gpu_debug_planes", "rspt_gpu_debug_hzr_tables", "rspt_gpu_crc32c",
    "rspt_gpu_synth_ecg", "rspt_gpu_prdn_terms", "rspt_gpu_rebase_offsets",
    "rspt_gpu_set_stage_timing", "rspt_gpu_get_stage_times", "rspt_gpu_verify_batch", "rspt_gpu_build_index",
    "rspt_gpu_prefilter_iir", "rspt_gpu_prefilter_fir",
    "rspt_gpu_ingest_create", "rspt_gpu_ingest_destroy", "rspt_gpu_ingest_next_address_to_fill", "rspt_gpu_ingest_drain",
    "rspt_gpu_comm_unique_id", "rspt_gpu_comm_init", "rspt_gpu_comm_destroy", "rspt_gpu_allgather_totals",
    "rspt_gpu_place_offsets_async", "rspt_gpu_place_join", "rspt_gpu_set_stream", "rspt_gpu_set_dct_exact",
]


class Counters(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in (
        "frames_compressed", "frames_decompressed", "raw_bytes_in", "compressed_bytes_out",
        "blocks_copy", "blocks_huff", "blocks_fill", "escalations", "crc_failures", "kernel_launches")]


class RsptError(RuntimeError):
    pass


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RsptError(f"{LIB_PATH} is missing: run `python -m rspt_b200.build` (nvcc, sm_100a). "
                        "There is no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    sz, vp, u64 = C.c_size_t, C.c_void_p, C.c_uint64
    L.rspt_gpu_create.restype = C.c_int
    L.rspt_gpu_create.argtypes = [C.c_int, sz, sz, sz, sz, C.c_int, vp, sz, C.POINTER(vp)]
    L.rspt_gpu_destroy.restype = C.c_int
    L.rspt_gpu_destroy.argtypes = [vp]
    for name in ("rspt_gpu_frame_bytes", "rspt_gpu_header_bytes", "rspt_gpu_max_compressed_size"):
        getattr(L, name).restype = sz
        getattr(L, name).argtypes = [vp]
    L.rspt_gpu_sidecar_bytes.restype = sz
    L.rspt_gpu_sidecar_bytes.argtypes = [vp, sz]
    L.rspt_gpu_sidecar_used_bytes.restype = sz
    L.rspt_gpu_sidecar_used_bytes.argtypes = [vp, sz, sz]
    L.rspt_gpu_nb.restype = C.c_int
    L.rspt_gpu_nb.argtypes = [vp, C.POINTER(C.c_uint)]
    L.rspt_gpu_compress_batch.restype = C.c_int
    L.rspt_gpu_compress_batch.argtypes = [vp, vp, sz, vp, sz, vp, vp, vp]
    L.rspt_gpu_decompress_batch.restype = C.c_int
    L.rspt_gpu_decompress_batch.argtypes = [vp, vp, vp, sz, vp, vp, vp, vp]
    L.rspt_gpu_compress_batch_i32.restype = C.c_int
    L.rspt_gpu_compress_batch_i32.argtypes = [vp, vp, sz, vp, sz, vp, vp, vp]
    L.rspt_gpu_decompress_batch_i32.restype = C.c_int
    L.rspt_gpu_decompress_batch_i32.argtypes = [vp, vp, vp, sz, vp, vp, vp, vp]
    for name in ("rspt_gpu_compress_append", "rspt_gpu_compress_append_i32"):
        getattr(L, name).restype = C.c_int
        getattr(L, name).argtypes = [vp, vp, sz, vp, sz, vp, sz, sz, vp, vp, sz]
    L.rspt_gpu_build_index_frames.restype = C.c_int
    L.rspt_gpu_build_index_frames.argtypes = [vp, vp, vp, sz, vp, vp, sz, vp, sz, vp]
    for name in ("rspt_gpu_decompress_frames", "rspt_gpu_decompress_frames_i32"):
        getattr(L, name).restype = C.c_int
        getattr(L, name).argtypes = [vp, vp, vp, sz, vp, vp, vp, sz, vp, vp]
    L.rspt_gpu_decompress_batch_float.restype = C.c_int
    L.rspt_gpu_decompress_batch_float.argtypes = [vp, vp, vp, sz, vp, vp, C.c_int, vp, vp, vp, vp]
    L.rspt_gpu_decompress_frames_float.restype = C.c_int
    L.rspt_gpu_decompress_frames_float.argtypes = [vp, vp, vp, sz, vp, vp, vp, sz, C.c_int, vp, vp, vp, vp]
    dp = C.POINTER(C.c_double)
    L.rspt_gpu_prefilter_iir.restype = C.c_int
    L.rspt_gpu_prefilter_iir.argtypes = [vp, vp, sz, dp, dp, C.c_int, C.c_int]
    L.rspt_gpu_prefilter_fir.restype = C.c_int
    L.rspt_gpu_prefilter_fir.argtypes = [vp, vp, sz, dp, C.c_int]
    L.rspt_gpu_ingest_create.restype = C.c_int
    L.rspt_gpu_ingest_create.argtypes = [vp, sz, C.POINTER(vp)]
    L.rspt_gpu_ingest_destroy.restype = C.c_int
    L.rspt_gpu_ingest_destroy.argtypes = [vp]
    L.rspt_gpu_ingest_next_address_to_fill.restype = vp
    L.rspt_gpu_ingest_next_address_to_fill.argtypes = [vp]
    L.rspt_gpu_ingest_drain.restype = C.c_int
    L.rspt_gpu_ingest_drain.argtypes = [vp, C.c_int, vp, sz, vp, C.POINTER(sz)]
    L.rspt_gpu_build_index.restype = C.c_int
    L.rspt_gpu_build_index.argtypes = [vp, vp, vp, sz, vp, vp, vp]
    L.rspt_gpu_verify_batch.restype = C.c_int
    L.rspt_gpu_verify_batch.argtypes = [vp, vp, vp, sz, vp, vp]
    L.rspt_gpu_compress_host.restype = C.c_int
    L.rspt_gpu_compress_host.argtypes = [vp, vp, vp, sz, C.POINTER(sz)]
    L.rspt_gpu_decompress_host.restype = C.c_int
    L.rspt_gpu_decompress_host.argtypes = [vp, vp, C.POINTER(sz), vp]
    L.rspt_gpu_compress_batch_host.restype = C.c_int
    L.rspt_gpu_compress_batch_host.argtypes = [vp, vp, sz, vp, sz, vp]
    L.rspt_gpu_decompress_batch_host.restype = C.c_int
    L.rspt_gpu_decompress_batch_host.argtypes = [vp, vp, vp, sz, vp]
    L.rspt_gpu_sync.restype = C.c_int
    L.rspt_gpu_sync.argtypes = [vp]
    L.rspt_gpu_last_error.restype = C.c_char_p
    L.rspt_gpu_last_error.argtypes = [vp]
    L.rspt_gpu_get_counters.restype = C.c_int
    L.rspt_gpu_get_counters.argtypes = [vp, C.POINTER(Counters)]
    L.rspt_gpu_debug_planes.restype = C.c_int
    L.rspt_gpu_debug_planes.argtypes = [vp, vp, sz, vp, vp]
    L.rspt_gpu_debug_hzr_tables.restype = C.c_int
    L.rspt_gpu_debug_hzr_tables.argtypes = [vp, vp, sz, vp, vp, vp]
    L.rspt_gpu_crc32c.restype = C.c_int
    L.rspt_gpu_crc32c.argtypes = [vp, sz, C.POINTER(C.c_uint32), vp]
    L.rspt_gpu_synth_ecg.restype = C.c_int
    L.rspt_gpu_synth_ecg.argtypes = [vp, u64, sz, C.c_int, C.c_int, C.c_int, u64, C.c_int32, C.c_int32, vp]
    L.rspt_gpu_prdn_terms.restype = C.c_int
    L.rspt_gpu_prdn_terms.argtypes = [vp, vp, sz, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double), vp]
    L.rspt_gpu_rebase_offsets.restype = C.c_int
    L.rspt_gpu_rebase_offsets.argtypes = [vp, sz, vp, C.c_int, vp]
    L.rspt_gpu_set_stage_timing.restype = C.c_int
    L.rspt_gpu_set_stage_timing.argtypes = [vp, C.c_int]
    L.rspt_gpu_get_stage_times.restype = C.c_int
    L.rspt_gpu_get_stage_times.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(u64), C.c_int]
    L.rspt_gpu_comm_unique_id.restype = C.c_int
    L.rspt_gpu_comm_unique_id.argtypes = [vp]
    L.rspt_gpu_comm_init.restype = C.c_int
    L.rspt_gpu_comm_init.argtypes = [C.c_int, vp, C.c_int, C.c_int, C.POINTER(vp)]
    L.rspt_gpu_comm_destroy.restype = C.c_int
    L.rspt_gpu_comm_destroy.argtypes = [vp]
    L.rspt_gpu_allgather_totals.restype = C.c_int
    L.rspt_gpu_allgather_totals.argtypes = [vp, vp, vp, vp]
    L.rspt_gpu_place_offsets_async.restype = C.c_int
    L.rspt_gpu_place_offsets_async.argtypes = [vp, vp, vp, sz, C.c_int, C.c_int]
    L.rspt_gpu_place_join.restype = C.c_int
    L.rspt_gpu_place_join.argtypes = [vp]
    L.rspt_gpu_set_stream.restype = C.c_int
    L.rspt_gpu_set_stream.argtypes = [vp, vp]
    L.rspt_gpu_set_dct_exact.restype = C.c_int
    L.rspt_gpu_set_dct_exact.argtypes = [vp, C.c_int]
    _lib = L
    return L


def check(rc: int, handle=None, what: str = "") -> None:
    if rc == 0:
        return
    msg = ERRORS.get(rc, f"error {rc}")
    if handle:
        detail = lib().rspt_gpu_last_error(handle)
        if detail:
            msg += ": " + detail.decode(errors="replace")
    raise RsptError(f"{what or 'rspt_gpu'} failed ({rc}): {msg}")
