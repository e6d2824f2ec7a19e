"""Host-side mirror of the reference's packer interface (lib_rspt/signal_packer.h:29-73) over the
C ABI in include/rspt_gpu.h.

`SignalPacker.new_xdelta_hzr / new_hzr / new_hadamard / new_dct` take the reference factories'
arguments; `compress(src) -> bytes` and `decompress(src) -> (bytes, consumed)` have the reference
methods' meaning for ONE frame in host memory (signal_packer.h:44,57).  `compress_batch` /
`decompress_batch` are the B200 path proper: many independent frames resident in HBM per call.
torch is used only to own device memory and to name the CUDA stream.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field

import numpy as np
import torch

from . import _lib
from ._lib import KINDS, Counters, RsptError, check


@dataclass
class CompressedBatch:
    """The concatenated frames of one batch plus the out-of-band facts a decoder needs
    (the reference stream carries neither a frame index nor the plane count)."""
    stream: torch.Tensor      # uint8, capacity-sized; valid bytes = offsets[-1]
    offsets: torch.Tensor     # uint64-as-int64 [n + 1], device
    frame_nb: torch.Tensor    # uint8 [n], device
    sidecar: torch.Tensor | None
    n_frames: int

    def total_bytes(self) -> int:
        return int(self.offsets[-1].item())

    def frame(self, i: int) -> bytes:
        off = self.offsets[i:i + 2].cpu().tolist()
        return bytes(self.stream[off[0]:off[1]].cpu().numpy())


# bytes behind the last frame that the decoder's 16-byte staging reads may touch (decompress_stream pads the same way)
STREAM_PAD = 16


@dataclass
class CompressedStore(CompressedBatch):
    """A stored batch that grows past max_batch_frames by appends (SignalPacker.new_store / append_batch /
    append_tensor), e.g. a dataset kept compressed in HBM.  Frames [0, n_frames) and stream bytes [0, stored_bytes)
    are used; the buffers have room behind them.  Offsets are store-relative and the decode index is addressed
    from the store's start, so the used prefix of every buffer is the whole store: growth copies it and trim()
    cuts the buffers down to it.  Accepted wherever a CompressedBatch is (decompress_frames(_tensor), frame(),
    slices for verify_batch)."""
    stored_bytes: int = 0
    packer: "SignalPacker | None" = field(default=None, repr=False)

    def total_bytes(self) -> int:
        return self.stored_bytes

    def sidecar_used_bytes(self) -> int:
        return self.packer.sidecar_used_bytes(self.n_frames, self.stored_bytes)

    def trim(self) -> "CompressedStore":
        """Shrink every buffer to what the store uses: the stream to stored_bytes + STREAM_PAD zero bytes, offsets
        and frame_nb to n_frames + 1 and n_frames entries, the sidecar to sidecar_used_bytes().  Ordered on torch's
        current stream."""
        n, used = self.n_frames, self.stored_bytes
        stream = torch.zeros(used + STREAM_PAD, dtype=torch.uint8, device=self.stream.device)
        stream[:used].copy_(self.stream[:used])
        self.stream = stream
        self.offsets = self.offsets[:n + 1].clone()
        self.frame_nb = self.frame_nb[:n].clone()
        if self.sidecar is not None:
            self.sidecar = self.sidecar[:self.sidecar_used_bytes()].clone()
        return self

    def index_all(self, p: "SignalPacker", status: torch.Tensor | None = None) -> "CompressedStore":
        """Build the decode index of every stored frame (e.g. for a store appended without one) with
        p.index_frames, p.max_batch frames per call.  status: optional int32 [n_frames], as for index_frames."""
        for a in range(0, self.n_frames, p.max_batch):
            b = min(self.n_frames, a + p.max_batch)
            ids = torch.arange(a, b, dtype=torch.int64, device=self.stream.device)
            p.index_frames(self, ids, status[a:b] if status is not None else None)
        return self


class SignalPacker:
    """One reference packer instance (= one `i_signal_packer::new_*` call) on one GPU."""

    def __init__(self, kind: str, bytes_per_sample: int, nr_channels: int, nr_samples: int,
                 nr_bytes_to_encode: int = 3, device: int | None = None, max_batch_frames: int = 1):
        if kind not in KINDS:
            raise ValueError(f"unknown packer kind {kind!r}")
        if not torch.cuda.is_available():
            raise RsptError("no CUDA device: rspt_b200 has no CPU fallback")
        self.L = _lib.lib()
        self.kind, self.bps, self.ch, self.ns = kind, bytes_per_sample, nr_channels, nr_samples
        self.device = torch.cuda.current_device() if device is None else device
        self.max_batch = max_batch_frames
        self.stream_ptr = torch.cuda.current_stream(self.device).cuda_stream
        h = C.c_void_p()
        rc = self.L.rspt_gpu_create(KINDS[kind], bytes_per_sample, nr_channels, nr_samples, nr_bytes_to_encode,
                                    self.device, self.stream_ptr, max_batch_frames, C.byref(h))
        check(rc, None, "rspt_gpu_create")
        self.h = h
        self.frame_bytes = self.L.rspt_gpu_frame_bytes(h)
        self.header_bytes = self.L.rspt_gpu_header_bytes(h)
        self.max_compressed_size = self.L.rspt_gpu_max_compressed_size(h)

    # -- reference factories (signal_packer.h:59-69) ------------------------------------------
    @classmethod
    def new_xdelta_hzr(cls, bytes_per_channel, nr_of_channels, nr_of_samples_in_each_channel, nr_bytes_to_encode, **kw):
        return cls("xdelta_hzr", bytes_per_channel, nr_of_channels, nr_of_samples_in_each_channel, nr_bytes_to_encode, **kw)

    @classmethod
    def new_hzr(cls, bytes_per_channel, nr_of_channels, nr_of_samples_in_each_channel, **kw):
        return cls("hzr", bytes_per_channel, nr_of_channels, nr_of_samples_in_each_channel, 4, **kw)

    @classmethod
    def new_hadamard(cls, bytes_per_channel, nr_of_channels, nr_of_samples_in_each_channel, **kw):
        return cls("hadamard", bytes_per_channel, nr_of_channels, nr_of_samples_in_each_channel, 3, **kw)

    @classmethod
    def new_dct(cls, bytes_per_channel, nr_of_channels, nr_of_samples_in_each_channel, **kw):
        return cls("dct", bytes_per_channel, nr_of_channels, nr_of_samples_in_each_channel, 2, **kw)

    def close(self):
        if getattr(self, "h", None):
            self.L.rspt_gpu_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- state ------------------------------------------------------------------------------
    @property
    def nb(self) -> int:
        v = C.c_uint(0)
        check(self.L.rspt_gpu_nb(self.h, C.byref(v)), self.h, "rspt_gpu_nb")
        return v.value

    def counters(self) -> dict:
        c = Counters()
        check(self.L.rspt_gpu_get_counters(self.h, C.byref(c)), self.h, "rspt_gpu_get_counters")
        return {n: getattr(c, n) for n, _ in Counters._fields_}

    def sync(self):
        check(self.L.rspt_gpu_sync(self.h), self.h, "rspt_gpu_sync")

    def set_stage_timing(self, enable: bool = True):
        check(self.L.rspt_gpu_set_stage_timing(self.h, int(enable)), self.h, "set_stage_timing")

    def stage_times(self, reset: bool = True) -> dict:
        """{stage: (milliseconds, calls)} accumulated since the last reset (device time, CUDA events)."""
        ms = (C.c_double * len(_lib.STAGES))()
        calls = (C.c_uint64 * len(_lib.STAGES))()
        check(self.L.rspt_gpu_get_stage_times(self.h, ms, calls, int(reset)), self.h, "get_stage_times")
        return {n: (ms[i], calls[i]) for i, n in enumerate(_lib.STAGES)}

    # -- single frame, host buffers: the reference call shapes -----------------------------------
    def compress(self, src) -> bytes:
        s = np.ascontiguousarray(np.frombuffer(src, np.uint8) if not isinstance(src, np.ndarray) else src.view(np.uint8).reshape(-1))
        if s.size != self.frame_bytes:
            raise ValueError(f"expected {self.frame_bytes} bytes, got {s.size}")
        dst = np.empty(self.max_compressed_size, np.uint8)
        n = C.c_size_t(0)
        check(self.L.rspt_gpu_compress_host(self.h, s.ctypes.data, dst.ctypes.data, dst.size, C.byref(n)), self.h, "compress")
        return dst[: n.value].tobytes()

    def decompress(self, src):
        c = np.frombuffer(src, np.uint8) if not isinstance(src, np.ndarray) else src.view(np.uint8).reshape(-1)
        c = np.ascontiguousarray(np.concatenate([c, np.zeros(8, np.uint8)]))
        out = np.empty(self.frame_bytes, np.uint8)
        n = C.c_size_t(0)
        check(self.L.rspt_gpu_decompress_host(self.h, c.ctypes.data, C.byref(n), out.ctypes.data), self.h, "decompress")
        return out.tobytes(), n.value

    # -- batches, device buffers ------------------------------------------------------------
    def _dev(self):
        return torch.device("cuda", self.device)

    def _bind_stream(self):
        """Order the handle's work on torch's CURRENT stream (the handle was created on the stream that was
        current then).  The switch itself is ordered: the new stream waits for what the old one still holds."""
        cur = torch.cuda.current_stream(self.device)
        if cur.cuda_stream != self.stream_ptr:
            ev = torch.cuda.Event()
            ev.record(torch.cuda.ExternalStream(self.stream_ptr, device=self._dev()) if self.stream_ptr else torch.cuda.default_stream(self.device))
            cur.wait_event(ev)
            check(self.L.rspt_gpu_set_stream(self.h, cur.cuda_stream), self.h, "rspt_gpu_set_stream")
            self.stream_ptr = cur.cuda_stream

    def sidecar_used_bytes(self, n_frames: int, stream_bytes: int) -> int:
        """Bytes of the decode index that belong to a batch whose stream has `stream_bytes` bytes (a prefix of
        the sidecar buffer): what has to be kept next to the stream."""
        return int(self.L.rspt_gpu_sidecar_used_bytes(self.h, n_frames, stream_bytes))

    # -- multi-GPU placement (the path's only collective), through the C ABI -------------------------
    def place_offsets_async(self, comm, batch: "CompressedBatch", rank: int, world: int) -> None:
        """All-gather of the ranks' byte totals + rebase of this batch's offsets into the global stream, on the
        handle's side stream (ordered behind the compress that produced `batch`)."""
        check(self.L.rspt_gpu_place_offsets_async(self.h, comm, batch.offsets.data_ptr(), batch.n_frames, rank, world), self.h,
              "rspt_gpu_place_offsets_async")

    def place_join(self) -> None:
        check(self.L.rspt_gpu_place_join(self.h), self.h, "rspt_gpu_place_join")

    def set_dct_exact(self, exact: bool) -> None:
        check(self.L.rspt_gpu_set_dct_exact(self.h, int(exact)), self.h, "rspt_gpu_set_dct_exact")

    def alloc_output(self, n_frames: int, sidecar: bool = True) -> CompressedBatch:
        dev = self._dev()
        stream = torch.empty(n_frames * self.max_compressed_size, dtype=torch.uint8, device=dev)
        offsets = torch.empty(n_frames + 1, dtype=torch.int64, device=dev)
        frame_nb = torch.empty(n_frames, dtype=torch.uint8, device=dev)
        sc = torch.empty(self.L.rspt_gpu_sidecar_bytes(self.h, n_frames), dtype=torch.uint8, device=dev) if sidecar else None
        return CompressedBatch(stream, offsets, frame_nb, sc, n_frames)

    def compress_batch(self, frames: torch.Tensor, out: CompressedBatch | None = None, sidecar: bool = True) -> CompressedBatch:
        """frames: uint8 CUDA tensor of n * frame_bytes bytes.  Asynchronous on torch's current stream (the
        handle is re-bound to it when it changed since the last call)."""
        return self._compress(self.L.rspt_gpu_compress_batch, frames, self._check_frames(frames), out, sidecar)

    def _check_frames(self, frames) -> int:
        if not (frames.is_cuda and frames.dtype == torch.uint8 and frames.is_contiguous()):
            raise ValueError("frames must be a contiguous uint8 CUDA tensor")
        n = frames.numel() // self.frame_bytes
        if n * self.frame_bytes != frames.numel():
            raise ValueError("frames is not a whole number of frames")
        return n

    def compress_tensor(self, x: torch.Tensor, out: CompressedBatch | None = None, sidecar: bool = True) -> CompressedBatch:
        """x: contiguous int32 CUDA tensor [n, ch, ns] on the handle's device, the samples in the low 8 * bps bits of
        each word (higher bits are ignored).  The batch equals what compress_batch writes for the same samples in
        the native layout; both calls share the handle's state.  Asynchronous on torch's current stream."""
        self._check_words(x)
        return self._compress(self.L.rspt_gpu_compress_batch_i32, x, x.shape[0], out, sidecar)

    def _check_words(self, x, n: int | None = None) -> None:
        shape = (x.shape[0] if n is None else n, self.ch, self.ns) if isinstance(x, torch.Tensor) and x.dim() == 3 else None
        if not (isinstance(x, torch.Tensor) and x.dtype == torch.int32 and x.is_cuda and x.device.index == self.device
                and tuple(x.shape) == shape and x.is_contiguous()):
            want = f"[{'n' if n is None else n}, {self.ch}, {self.ns}]"
            raise ValueError(f"expected a contiguous torch.int32 tensor {want} on cuda:{self.device}")

    def _compress(self, fn, src: torch.Tensor, n: int, out: CompressedBatch | None, sidecar: bool) -> CompressedBatch:
        if out is None:
            out = self.alloc_output(n, sidecar)
        if out.offsets.numel() < n + 1 or out.frame_nb.numel() < n or out.stream.numel() < n * self.max_compressed_size:
            raise ValueError("the output batch is too small for these frames")
        if out.sidecar is not None and out.sidecar.numel() < self.L.rspt_gpu_sidecar_bytes(self.h, n):
            raise ValueError("the output batch's sidecar is too small for these frames")
        self._bind_stream()
        sc = out.sidecar.data_ptr() if out.sidecar is not None else None
        rc = fn(self.h, src.data_ptr(), n, out.stream.data_ptr(), out.stream.numel(), out.offsets.data_ptr(),
                out.frame_nb.data_ptr(), sc)
        check(rc, self.h, fn.__name__)
        out.n_frames = n
        return out

    # -- stores: batches appended past max_batch_frames ---------------------------------------------
    def new_store(self, frames_capacity: int, bytes_capacity: int | None = None, sidecar: bool = True) -> CompressedStore:
        """An empty store with room for frames_capacity frames and bytes_capacity stream bytes (None: the worst case
        of frames_capacity frames, max_compressed_size each -- raw-sized; pass an estimate for a large store).  The
        store grows when an append does not fit, so the capacities are only a starting point."""
        dev = self._dev()
        if bytes_capacity is None:
            bytes_capacity = frames_capacity * self.max_compressed_size
        stream = torch.empty(bytes_capacity + STREAM_PAD, dtype=torch.uint8, device=dev)
        offsets = torch.zeros(frames_capacity + 1, dtype=torch.int64, device=dev)
        frame_nb = torch.zeros(frames_capacity, dtype=torch.uint8, device=dev)
        sc = torch.zeros(self.sidecar_used_bytes(frames_capacity, bytes_capacity), dtype=torch.uint8, device=dev) if sidecar else None
        return CompressedStore(stream, offsets, frame_nb, sc, 0, 0, self)

    def append_batch(self, store: CompressedStore, frames: torch.Tensor) -> CompressedStore:
        """Compress frames (as for compress_batch, at most max_batch_frames of them) and append them to the store
        (rspt_gpu_compress_append): the store then equals what one compress_batch over all its frames writes.  Runs
        on torch's current stream, then reads the new stream total back (one 8-byte copy and a synchronisation), so
        that the next append can be checked and placed from the host."""
        return self._append(self.L.rspt_gpu_compress_append, store, frames, self._check_frames(frames))

    def append_tensor(self, store: CompressedStore, x: torch.Tensor) -> CompressedStore:
        """append_batch for an int32 tensor [n, ch, ns], as compress_tensor takes it.  Native and int32 appends may be
        mixed on one store."""
        self._check_words(x)
        return self._append(self.L.rspt_gpu_compress_append_i32, store, x, x.shape[0])

    def _append(self, fn, store: CompressedStore, src: torch.Tensor, n: int) -> CompressedStore:
        if n > self.max_batch:
            raise ValueError(f"{n} frames in one append: max_batch_frames is {self.max_batch}")
        if n == 0:
            return store
        self._bind_stream()
        self._reserve(store, store.n_frames + n, store.stored_bytes + n * self.max_compressed_size)
        sc = store.sidecar
        rc = fn(self.h, src.data_ptr(), n, store.stream.data_ptr(), store.stream.numel() - STREAM_PAD, store.offsets.data_ptr(),
                store.n_frames, store.stored_bytes, store.frame_nb.data_ptr(), sc.data_ptr() if sc is not None else None,
                sc.numel() if sc is not None else 0)
        check(rc, self.h, fn.__name__)
        store.n_frames += n
        store.stored_bytes = int(store.offsets[store.n_frames].item())
        return store

    def _reserve(self, store: CompressedStore, frames: int, stream_bytes: int) -> None:
        """Grow the store's buffers (at least doubling a buffer that is too small) so that `frames` frames and
        `stream_bytes` stream bytes fit; the used prefix of each is copied over."""
        def grown(t, used, need, zero):
            if t.numel() >= need:
                return t
            new = (torch.zeros if zero else torch.empty)(max(need, 2 * t.numel()), dtype=t.dtype, device=t.device)
            new[:used].copy_(t[:used])
            return new
        n = store.n_frames
        store.offsets = grown(store.offsets, n + 1, frames + 1, True)
        store.frame_nb = grown(store.frame_nb, n, frames, True)
        store.stream = grown(store.stream, store.stored_bytes, stream_bytes + STREAM_PAD, False)
        if store.sidecar is not None:
            need = self.sidecar_used_bytes(frames, stream_bytes)
            if store.sidecar.numel() < need:
                used = self.sidecar_used_bytes(n, store.stored_bytes)
                room = self.sidecar_used_bytes(store.offsets.numel() - 1, store.stream.numel() - STREAM_PAD)
                new = torch.zeros(max(need, room), dtype=torch.uint8, device=store.sidecar.device)
                new[:used].copy_(store.sidecar[:used])
                store.sidecar = new

    def index_frames(self, batch: CompressedBatch, frame_ids, status: torch.Tensor | None = None) -> CompressedBatch:
        """Write the decode-index entries of stored frames frame_ids[0], frame_ids[1], ... (at most max_batch_frames
        ids, as for decompress_frames) into the batch's own index (rspt_gpu_build_index_frames): indexing a batch
        in pieces gives the words one build_index over the whole batch gives.  A batch without a sidecar first gets
        a zeroed one of sidecar_used_bytes(n_frames, total).  status: optional int32 per id, -1 for an id outside
        the batch, -4 for a malformed frame.  Asynchronous on torch's current stream."""
        ids = self._frame_ids(frame_ids)
        if batch.sidecar is None:
            total = int(batch.offsets[batch.n_frames].item())
            batch.sidecar = torch.zeros(self.sidecar_used_bytes(batch.n_frames, total), dtype=torch.uint8, device=self._dev())
        nbp = batch.frame_nb.data_ptr() if batch.frame_nb is not None else None
        self._bind_stream()
        rc = self.L.rspt_gpu_build_index_frames(self.h, batch.stream.data_ptr(), batch.offsets.data_ptr(), batch.n_frames, nbp,
                                                ids.data_ptr(), ids.numel(), batch.sidecar.data_ptr(), batch.sidecar.numel(),
                                                status.data_ptr() if status is not None else None)
        check(rc, self.h, "rspt_gpu_build_index_frames")
        return batch

    def decompress_batch(self, batch: CompressedBatch, out: torch.Tensor | None = None, status: torch.Tensor | None = None,
                         use_sidecar: bool = True) -> torch.Tensor:
        n = batch.n_frames
        if out is None:
            out = torch.empty(n * self.frame_bytes, dtype=torch.uint8, device=self._dev())
        return self._decompress(self.L.rspt_gpu_decompress_batch, batch, out, status, use_sidecar)

    def decompress_tensor(self, batch: CompressedBatch, out: torch.Tensor | None = None, status: torch.Tensor | None = None,
                          use_sidecar: bool = True, *, dtype: torch.dtype = torch.int32, zero_point=None,
                          scale=None) -> torch.Tensor:
        """The batch's samples as an int32 tensor [n, ch, ns]: every word is the sample decompress_batch writes,
        sign-extended from 8 * bps bits.  `out`, when given, must be a contiguous int32 tensor of that shape on the
        handle's device.

        dtype torch.float32 or torch.bfloat16: the samples in physical units, dequantized per channel c inside the
        decode kernels (rspt_gpu_decompress_batch_float).  With x the int32 output, the result is bit for bit
        (x.long() - zero_point).float() * scale, and for bfloat16 that value's .to(torch.bfloat16).  zero_point: an
        int32 CUDA tensor [ch] on the handle's device or a sequence of ints (None = 0); scale: a float32 CUDA tensor
        [ch] or a sequence of floats (None = 1.0).  `out` must then have that dtype.  The call is asynchronous and
        its kernels read zero_point and scale: keep tensors passed for them unchanged until the stream passes it."""
        n = batch.n_frames
        dq = self._dequant(dtype, zero_point, scale)
        out = self._samples_out(out, n, dtype)
        if dq is None:
            return self._decompress(self.L.rspt_gpu_decompress_batch_i32, batch, out, status, use_sidecar)
        return self._decompress(self.L.rspt_gpu_decompress_batch_float, batch, out, status, use_sidecar, dq=dq)

    def _samples_out(self, out: torch.Tensor | None, n: int, dtype: torch.dtype) -> torch.Tensor:
        if out is None:
            out = torch.empty((n, self.ch, self.ns), dtype=dtype, device=self._dev())
        if dtype == torch.int32:
            self._check_words(out, n)
        elif not (isinstance(out, torch.Tensor) and out.dtype == dtype and out.is_cuda and out.device.index == self.device
                  and tuple(out.shape) == (n, self.ch, self.ns) and out.is_contiguous()):
            raise ValueError(f"expected a contiguous {dtype} tensor [{n}, {self.ch}, {self.ns}] on cuda:{self.device}")
        return out

    def _dequant(self, dtype: torch.dtype, zero_point, scale):
        """(out_type, zero point, scale) of the _float calls, the last two as device tensors or None; None for int32
        output.  Sequences become tensors allocated on the current stream, which the call runs on: once the caller
        drops them, the caching allocator hands their memory only to work ordered behind the call."""
        if dtype == torch.int32:
            if zero_point is not None or scale is not None:
                raise ValueError("zero_point and scale apply to float32 / bfloat16 output only")
            return None
        out_type = {torch.float32: _lib.OUT_TYPES["float32"], torch.bfloat16: _lib.OUT_TYPES["bfloat16"]}.get(dtype)
        if out_type is None:
            raise ValueError(f"dtype must be torch.int32, torch.float32 or torch.bfloat16, not {dtype}")

        def per_channel(v, want: torch.dtype, name: str):
            if v is None:
                return None
            if not isinstance(v, torch.Tensor):
                v = torch.tensor(list(v), dtype=want, device=self._dev())
            if not (v.dtype == want and v.is_cuda and v.device.index == self.device and tuple(v.shape) == (self.ch,)
                    and v.is_contiguous()):
                raise ValueError(f"{name} must be a contiguous {want} tensor [{self.ch}] on cuda:{self.device}, "
                                 f"or a sequence of {self.ch} numbers")
            return v

        zp = per_channel(zero_point, torch.int32, "zero_point")
        sc = per_channel(scale, torch.float32, "scale")
        return out_type, zp, sc

    def _decompress(self, fn, batch: CompressedBatch, out: torch.Tensor, status: torch.Tensor | None,
                    use_sidecar: bool, ids: torch.Tensor | None = None, dq: tuple = ()) -> torch.Tensor:
        """The whole batch, or (ids given: the gather calls) its frames ids[0], ids[1], ...; dq: the _float calls'
        (out_type, zero point, scale), the tensors held here until the call is enqueued"""
        sc = batch.sidecar.data_ptr() if (use_sidecar and batch.sidecar is not None) else None
        nbp = batch.frame_nb.data_ptr() if batch.frame_nb is not None else None
        sel = () if ids is None else (ids.data_ptr(), ids.numel())
        fargs = tuple(a.data_ptr() if isinstance(a, torch.Tensor) else a for a in dq)
        self._bind_stream()
        rc = fn(self.h, batch.stream.data_ptr(), batch.offsets.data_ptr(), batch.n_frames, nbp, sc, *sel, *fargs,
                out.data_ptr(), status.data_ptr() if status is not None else None)
        check(rc, self.h, fn.__name__)
        return out

    def decompress_frames(self, batch: CompressedBatch, frame_ids, out: torch.Tensor | None = None,
                          status: torch.Tensor | None = None, use_sidecar: bool = True) -> torch.Tensor:
        """Stored frames frame_ids[0], frame_ids[1], ... of `batch` (any order, repeats allowed) as native uint8
        [n * frame_bytes]: row j equals row frame_ids[j] of decompress_batch(batch).  frame_ids: an int64 CUDA
        tensor on the handle's device, or a sequence / range of ints (copied to one).  An id outside
        [0, batch.n_frames) gives status -1 in its slot.  The handle's max_batch_frames bounds len(frame_ids),
        not batch.n_frames.  Asynchronous on torch's current stream."""
        ids = self._frame_ids(frame_ids)
        if out is None:
            out = torch.empty(ids.numel() * self.frame_bytes, dtype=torch.uint8, device=self._dev())
        if not (out.is_cuda and out.dtype == torch.uint8 and out.is_contiguous() and out.numel() >= ids.numel() * self.frame_bytes):
            raise ValueError(f"out must be a contiguous uint8 CUDA tensor of at least {ids.numel() * self.frame_bytes} bytes")
        return self._decompress(self.L.rspt_gpu_decompress_frames, batch, out, status, use_sidecar, ids)

    def decompress_frames_tensor(self, batch: CompressedBatch, frame_ids, out: torch.Tensor | None = None,
                                 status: torch.Tensor | None = None, use_sidecar: bool = True, *,
                                 dtype: torch.dtype = torch.int32, zero_point=None, scale=None) -> torch.Tensor:
        """decompress_frames with the samples as an int32 tensor [n, ch, ns], as decompress_tensor writes them; dtype,
        zero_point and scale as for decompress_tensor (rspt_gpu_decompress_frames_float): a minibatch of stored
        frames in physical units."""
        ids = self._frame_ids(frame_ids)
        n = ids.numel()
        dq = self._dequant(dtype, zero_point, scale)
        out = self._samples_out(out, n, dtype)
        if dq is None:
            return self._decompress(self.L.rspt_gpu_decompress_frames_i32, batch, out, status, use_sidecar, ids)
        return self._decompress(self.L.rspt_gpu_decompress_frames_float, batch, out, status, use_sidecar, ids, dq)

    def _frame_ids(self, frame_ids) -> torch.Tensor:
        if isinstance(frame_ids, (list, tuple, range)):
            return torch.tensor(list(frame_ids), dtype=torch.int64, device=self._dev())
        if not (isinstance(frame_ids, torch.Tensor) and frame_ids.dtype == torch.int64 and frame_ids.is_cuda
                and frame_ids.device.index == self.device and frame_ids.dim() == 1 and frame_ids.is_contiguous()):
            raise ValueError(f"frame_ids must be a contiguous 1-D torch.int64 tensor on cuda:{self.device}, or a sequence of ints")
        return frame_ids

    def prefilter_iir(self, frames: torch.Tensor, n, d, init_nr_samples: int) -> torch.Tensor:
        """In place on device frames: the IIR pre-filter step of rspt_test.cpp:116-136 (i_filter::new_iir)."""
        na, da = np.ascontiguousarray(n, np.float64), np.ascontiguousarray(d, np.float64)
        dp = C.POINTER(C.c_double)
        self._bind_stream()
        rc = self.L.rspt_gpu_prefilter_iir(self.h, frames.data_ptr(), frames.numel() // self.frame_bytes,
                                           na.ctypes.data_as(dp), da.ctypes.data_as(dp), len(na), init_nr_samples)
        check(rc, self.h, "rspt_gpu_prefilter_iir")
        return frames

    def prefilter_fir(self, frames: torch.Tensor, kernel) -> torch.Tensor:
        """In place on device frames: the same step with i_filter::new_fir(kernel)."""
        ka = np.ascontiguousarray(kernel, np.float64)
        self._bind_stream()
        rc = self.L.rspt_gpu_prefilter_fir(self.h, frames.data_ptr(), frames.numel() // self.frame_bytes,
                                           ka.ctypes.data_as(C.POINTER(C.c_double)), len(ka))
        check(rc, self.h, "rspt_gpu_prefilter_fir")
        return frames

    def build_index(self, batch: CompressedBatch, status: torch.Tensor | None = None) -> CompressedBatch:
        """Give a batch that came without a decode index (CPU-written frames) one, on the device."""
        n = batch.n_frames
        sc = torch.empty(self.L.rspt_gpu_sidecar_bytes(self.h, n), dtype=torch.uint8, device=self._dev())
        nbp = batch.frame_nb.data_ptr() if batch.frame_nb is not None else None
        self._bind_stream()
        rc = self.L.rspt_gpu_build_index(self.h, batch.stream.data_ptr(), batch.offsets.data_ptr(), n, nbp, sc.data_ptr(),
                                         status.data_ptr() if status is not None else None)
        check(rc, self.h, "rspt_gpu_build_index")
        return CompressedBatch(batch.stream, batch.offsets, batch.frame_nb, sc, n)

    def verify_batch(self, batch: CompressedBatch, status: torch.Tensor | None = None) -> torch.Tensor:
        """hzr_verify (hzr_decode.c:569-624) over every block of every frame: int32 status per frame,
        0 = ok, -4 = malformed framing, -6 = CRC-32C mismatch.  Asynchronous on the current stream."""
        n = batch.n_frames
        if status is None:
            status = torch.zeros(n, dtype=torch.int32, device=self._dev())
        nbp = batch.frame_nb.data_ptr() if batch.frame_nb is not None else None
        self._bind_stream()
        rc = self.L.rspt_gpu_verify_batch(self.h, batch.stream.data_ptr(), batch.offsets.data_ptr(), n, nbp, status.data_ptr())
        check(rc, self.h, "rspt_gpu_verify_batch")
        return status

    def decompress_stream(self, stream: bytes, offsets, frame_nb=None) -> tuple[np.ndarray, np.ndarray]:
        """Decode frames produced elsewhere (e.g. by the CPU reference): no decode index."""
        dev = self._dev()
        off = torch.tensor(list(offsets), dtype=torch.int64, device=dev)
        n = off.numel() - 1
        buf = torch.from_numpy(np.frombuffer(stream, np.uint8).copy()).to(dev)
        pad = torch.zeros(16, dtype=torch.uint8, device=dev)
        buf = torch.cat([buf, pad])
        nb = torch.tensor(list(frame_nb), dtype=torch.uint8, device=dev) if frame_nb is not None else None
        status = torch.zeros(n, dtype=torch.int32, device=dev)
        b = CompressedBatch(buf, off, nb, None, n)
        out = self.decompress_batch(b, status=status, use_sidecar=False)
        torch.cuda.synchronize(dev)
        return out.cpu().numpy().reshape(n, self.frame_bytes), status.cpu().numpy()

    # -- batches, host buffers (end-to-end leg) ------------------------------------------------
    def compress_batch_host(self, frames: np.ndarray, dst: np.ndarray, offsets: np.ndarray) -> int:
        n = frames.size // self.frame_bytes
        rc = self.L.rspt_gpu_compress_batch_host(self.h, frames.ctypes.data, n, dst.ctypes.data, dst.size, offsets.ctypes.data)
        check(rc, self.h, "rspt_gpu_compress_batch_host")
        return int(offsets[n])

    def decompress_batch_host(self, src: np.ndarray, offsets: np.ndarray, out: np.ndarray) -> None:
        n = offsets.size - 1
        rc = self.L.rspt_gpu_decompress_batch_host(self.h, src.ctypes.data, offsets.ctypes.data, n, out.ctypes.data)
        check(rc, self.h, "rspt_gpu_decompress_batch_host")

    # -- stage-level (parity tests) -----------------------------------------------------------
    def debug_planes(self, frames: torch.Tensor):
        n = frames.numel() // self.frame_bytes
        unsigned = C.c_uint(0)
        nb_alloc = (self.max_compressed_size - 1 - self.header_bytes) // (4 + 4 + 7 * ((self.ch * self.ns + 65535) // 65536) + self.ch * self.ns)
        planes = torch.empty(n * nb_alloc * self.ch * self.ns, dtype=torch.uint8, device=self._dev())
        hdr = torch.zeros(max(1, n * self.header_bytes), dtype=torch.uint8, device=self._dev())
        check(self.L.rspt_gpu_debug_planes(self.h, frames.data_ptr(), n, planes.data_ptr(), hdr.data_ptr()), self.h, "debug_planes")
        torch.cuda.synchronize(self._dev())
        return planes.cpu().numpy().reshape(n, nb_alloc, self.ch * self.ns), hdr.cpu().numpy()[: n * self.header_bytes].reshape(n, -1)

    def debug_hzr_tables(self, block: np.ndarray):
        dev = self._dev()
        b = torch.from_numpy(np.ascontiguousarray(block, np.uint8)).to(dev)
        pad = torch.zeros(64, dtype=torch.uint8, device=dev)
        b = torch.cat([b, pad])
        hist = torch.zeros(264, dtype=torch.int32, device=dev)
        codes = torch.zeros(264, dtype=torch.int32, device=dev)
        info = torch.zeros(4, dtype=torch.int32, device=dev)
        check(self.L.rspt_gpu_debug_hzr_tables(self.h, b.data_ptr(), block.size, hist.data_ptr(), codes.data_ptr(), info.data_ptr()),
              self.h, "debug_hzr_tables")
        torch.cuda.synchronize(dev)
        return (hist.cpu().numpy().view(np.uint32)[:261], codes.cpu().numpy().view(np.uint32)[:261],
                info.cpu().numpy().view(np.uint32))


class IngestRing:
    """Pinned-host packet ring in front of a packer (the reference's io_buffer, ring_buffers.h:150-201):
    the producer writes frames into `next_packet()`, the consumer calls `drain()`."""

    def __init__(self, packer: SignalPacker, nr_max_packets: int):
        self.p = packer
        self.L = packer.L
        self.h = C.c_void_p()
        check(self.L.rspt_gpu_ingest_create(packer.h, nr_max_packets, C.byref(self.h)), packer.h, "rspt_gpu_ingest_create")

    def close(self):
        if self.h:
            self.L.rspt_gpu_ingest_destroy(self.h)
            self.h = C.c_void_p()

    def next_packet(self):
        """numpy view of the next packet to fill (frame_bytes bytes), or None when the ring is full."""
        addr = self.L.rspt_gpu_ingest_next_address_to_fill(self.h)
        if not addr:
            return None
        return np.ctypeslib.as_array(C.cast(addr, C.POINTER(C.c_uint8)), shape=(self.p.frame_bytes,))

    def drain(self, dst: np.ndarray, offsets: np.ndarray, max_frames: int | None = None, flush: bool = False) -> int:
        """Compress the filled packets into dst; offsets[0..n] are filled in.  Returns n."""
        n = C.c_size_t(offsets.size - 1 if max_frames is None else min(max_frames, offsets.size - 1))
        rc = self.L.rspt_gpu_ingest_drain(self.h, int(flush), dst.ctypes.data, dst.size, offsets.ctypes.data, C.byref(n))
        check(rc, self.p.h, "rspt_gpu_ingest_drain")
        return int(n.value)


def crc32c(data: np.ndarray) -> int:
    t = torch.from_numpy(np.array(data, dtype=np.uint8, copy=True)).cuda() if data.size else torch.zeros(1, dtype=torch.uint8, device="cuda")
    out = C.c_uint32(0)
    check(_lib.lib().rspt_gpu_crc32c(t.data_ptr(), data.size, C.byref(out), torch.cuda.current_stream().cuda_stream), None, "crc32c")
    return out.value


def synth_ecg(first_frame: int, n_frames: int, bps: int, ch: int, ns: int, seed: int = 42, amplitude: int = 20000,
              sigma: int = 3, out: torch.Tensor | None = None, device=None) -> torch.Tensor:
    """Synthetic ECG-like frames generated on the device (include/rspt_synth.h)."""
    dev = torch.device("cuda", torch.cuda.current_device() if device is None else device)
    if out is None:
        out = torch.empty(n_frames * bps * ch * ns, dtype=torch.uint8, device=dev)
    check(_lib.lib().rspt_gpu_synth_ecg(out.data_ptr(), first_frame, n_frames, bps, ch, ns, seed, amplitude, sigma,
                                        torch.cuda.current_stream(dev).cuda_stream), None, "synth_ecg")
    return out


def prdn_terms(orig: torch.Tensor, dec: torch.Tensor, n_frames: int, bps: int, ch: int, ns: int) -> tuple[float, float]:
    """Numerator and denominator sums of PRDN (rspt_test.cpp:98-111) over the given frames, so that a
    caller can accumulate them over batches."""
    out = (C.c_double * 2)()
    check(_lib.lib().rspt_gpu_prdn_terms(orig.data_ptr(), dec.data_ptr(), n_frames, bps, ch, ns, out,
                                         torch.cuda.current_stream().cuda_stream), None, "prdn")
    return float(out[0]), float(out[1])


def prdn(orig: torch.Tensor, dec: torch.Tensor, n_frames: int, bps: int, ch: int, ns: int) -> float:
    num, den = prdn_terms(orig, dec, n_frames, bps, ch, ns)
    return float(np.sqrt(num / den) * 100.0) if den > 0 else 0.0
