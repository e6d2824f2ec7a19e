"""Every sample-stage kernel variant held to the CPU oracle, one table row per path.

Which kernel turns samples into byte planes (and back) depends on the packer, bps, the channel count, the length,
the plane-count probe and the alignment of the caller's pointer (sample_stages.cuh, rspt_gpu_prefilter_*).  The
same output bytes can come from very different code: a TMA kernel compiled per (bps, ch), a quad-tiled kernel, a
generic one.  Each row of ROWS names one call (entry point, packer, shape, pointer offset) and the sample-stage
kernels it must launch, in launch order.  For every row:

* test_row_matches_oracle runs the call on frames that reach the edges of the sample range (full-range noise,
  per-sample / per-channel min-max alternation, constant min and max, min-max steps on the 128 / 256 / 512-sample
  tile and piece boundaries, ECG, all zero) from a buffer with guard bands on both sides, and compares with the
  oracle bit for bit (dct's fast path: with the aligned native call);
* test_rows_launch_their_kernels traces the whole table under torch.profiler in a child process and checks that
  each call launched exactly its listed kernels;
* test_table_covers_every_sample_stage_kernel reads the kernels the library compiles (cuobjdump) and checks that
  the table reaches every one, so a new kernel or a changed eligibility predicate fails until the table says so.

Needs a B200, except the coverage check, which needs only the built library and cuobjdump."""
import json
import os
import re
import shutil
import subprocess
import sys
from collections import namedtuple

import numpy as np
import pytest

torch = pytest.importorskip("torch")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "rspt_b200", "librspt_gpu.so")
GUARD = 64          # sentinel bytes on both sides of every buffer
FILL_U8 = 0xA5
FILL_I32 = 0x5A5A5A5A
N_FRAMES = 7
NB = {"hzr": 4, "hadamard": 3, "dct": 2}   # the reference factories' nr_bytes_to_encode (xdelta_hzr: per row)

# ---- the case table -------------------------------------------------------------------------------------------

Row = namedtuple("Row", "entry kind bps ch ns nb exact off kernels")
# entry: compress / decompress / decompress_frames take native uint8 buffers, `off` in bytes;
#        compress_i32 / decompress_i32 take int32 [n, ch, ns] tensors, `off` in words;
#        iir2..iir5 / fir run the pre-filter in place on native frames, `off` in bytes.

ROWS = []


def tf(v):
    return "true" if v else "false"


def TMA(b, c, st): return f"k_xdelta_planes_tma<{b},{c},{tf(st)}>"
def FAST(b, st): return f"k_xdelta_planes_fast<{b},{tf(st)}>"
def GEN(b, st): return f"k_xdelta_planes<{b},{tf(st)}>"
def I32(b, st): return f"k_xdelta_planes_i32<{b},{tf(st)}>"
def INVF(b, sc, words=False): return f"k_planes_to_samples_fast<{b},{tf(sc)},{tf(words)}>"
def INVG(b, sc, raw): return f"k_planes_to_samples<{b},{tf(sc)},{tf(raw)}>"
def RAWF(lg, b): return f"k_fwht_raw_fwd<{lg},{b}>"
def RAWI(lg, b): return f"k_fwht_raw_inv<{lg},{b}>"
def FFWD(lg): return f"k_fwht_fast_fwd<{lg}>"
def FINV(lg): return f"k_fwht_fast_inv<{lg}>"
def R2W(b): return f"k_raw_to_words<{b}>"
def R2W4(b): return f"k_raw_to_words_g4<{b}>"
def W2R(b): return f"k_words_to_raw<{b}>"
def W2R4(b): return f"k_words_to_raw_g4<{b}>"
def I2W(b): return f"k_i32_to_words<{b}>"
def SEXT(b): return f"k_words_sext<{b}>"
def IIR(nc): return f"k_iir_frames<{nc}>"


FWD, INV, STENCIL, FIR = "k_fwht_fwd", "k_fwht_inv", "k_words_stencil_planes", "k_fir_words"
TMA_SHAPES = [(b, c) for b in (2, 3, 4) for c in (4, 8, 12)]   # RSPT_TMA_SHAPES (xdelta_tma.cuh)
MISALIGNED = (1, 2, 3, 4, 8)


def add(entry, kind, bps, ch, ns, off, kernels, nb=None, exact=False):
    ROWS.append(Row(entry, kind, bps, ch, ns, nb if nb is not None else NB.get(kind, bps), exact, off, tuple(kernels)))


def st(kind):
    return kind == "xdelta_hzr"


# -- stage 1 of compress from native samples: xdelta_hzr / hzr
for b, c in TMA_SHAPES:   # every compiled (bps, ch), both stencil flags: one 512-sample tile, 2 and 4 tiles
    for kind in ("xdelta_hzr", "hzr"):
        add("compress", kind, b, c, {4: 2048, 8: 512, 12: 1024}[c], 0, [TMA(b, c, st(kind))])
add("compress", "xdelta_hzr", 3, 12, 8192, 0, [TMA(3, 12, True)])           # 98 304 samples per frame
# the plane-count probe (nb < bps) keeps the quad-tiled kernel on TMA shapes
add("compress", "xdelta_hzr", 3, 12, 1024, 0, [FAST(3, True)], nb=1)
add("compress", "xdelta_hzr", 2, 4, 512, 0, [FAST(2, True)], nb=1)
add("compress", "xdelta_hzr", 4, 8, 512, 0, [FAST(4, True)], nb=2)
for kind, b, c, ns in (("xdelta_hzr", 1, 4, 512), ("hzr", 1, 8, 1000), ("xdelta_hzr", 2, 16, 1000), ("hzr", 2, 16, 512),
                       ("xdelta_hzr", 3, 4, 1000), ("hzr", 3, 4, 1000), ("xdelta_hzr", 4, 4, 4),
                       ("hzr", 4, 32, 1024), ("xdelta_hzr", 4, 56, 256)):
    # 4 samples: the shortest quad frame; 32 and 56 x 4 B: 64- and 32-quad tiles
    add("compress", kind, b, c, ns, 0, [FAST(b, st(kind))])
for kind, b, c, ns in (("xdelta_hzr", 1, 3, 700), ("hzr", 1, 2, 40000), ("xdelta_hzr", 2, 3, 30000), ("hzr", 2, 5, 1000),
                       ("xdelta_hzr", 2, 4, 6), ("xdelta_hzr", 3, 2, 1), ("hzr", 3, 7, 33), ("xdelta_hzr", 4, 3, 2),
                       ("hzr", 4, 1, 257)):
    add("compress", kind, b, c, ns, 0, [GEN(b, st(kind))])
for off in MISALIGNED:   # a pointer off 16-byte alignment takes the generic kernel on any shape
    add("compress", "xdelta_hzr", 3, 12, 1024, off, [GEN(3, True)])
    add("compress", "hzr", 2, 16, 512, off, [GEN(2, False)])
    add("compress", "hzr", 1, 3, 700, off, [GEN(1, False)])
# -- hadamard / dct: the fused raw kernels, or native -> words + the word-matrix transform
for b in (1, 2, 3, 4):
    add("compress", "hadamard", b, 4, 4096, 0, [RAWF(12, b)])
    add("compress", "hadamard", b, 4, 8192, 0, [RAWF(13, b)])
add("compress", "hadamard", 3, 12, 4096, 0, [RAWF(12, 3)])
for off in MISALIGNED:
    add("compress", "hadamard", 3, 4, 4096, off, [R2W(3), FFWD(12)])
    add("compress", "dct", 2, 4, 1024, off, [R2W(2), STENCIL], exact=True)
add("compress", "hadamard", 2, 3, 8192, 0, [R2W(2), FFWD(13)])
add("compress", "hadamard", 1, 4, 1024, 0, [R2W4(1), FWD])
add("compress", "hadamard", 4, 3, 64, 0, [R2W(4), FWD])
add("compress", "hadamard", 2, 2, 8, 0, [R2W(2), FWD])
add("compress", "dct", 2, 4, 1024, 0, [R2W4(2), STENCIL], exact=True)
add("compress", "dct", 3, 8, 1024, 0, [R2W4(3), STENCIL], exact=True)
add("compress", "dct", 4, 4, 1024, 0, [R2W4(4), STENCIL], exact=True)
add("compress", "dct", 1, 3, 77, 0, [R2W(1), STENCIL], exact=True)
for off in (1, 4):   # the fast dct path: same bytes as the aligned call
    add("compress", "dct", 3, 4, 1024, off, [R2W(3), STENCIL])

# -- stage 1 of compress from int32 words (any 4-byte offset: one kernel per bps and packer)
for kind, b, c, ns in (("xdelta_hzr", 1, 4, 512), ("hzr", 1, 3, 700), ("xdelta_hzr", 2, 5, 1000), ("hzr", 2, 4, 1000),
                       ("xdelta_hzr", 2, 3, 30000), ("xdelta_hzr", 3, 2, 1), ("hzr", 3, 7, 33), ("xdelta_hzr", 4, 3, 2),
                       ("hzr", 4, 8, 512)):
    add("compress_i32", kind, b, c, ns, 0, [I32(b, st(kind))])
for off in (0, 1, 2, 3):
    add("compress_i32", "xdelta_hzr", 3, 12, 1024, off, [I32(3, True)])
    add("compress_i32", "hadamard", 2, 4, 4096, off, [I2W(2), FFWD(12)])
add("compress_i32", "xdelta_hzr", 4, 4, 512, 0, [I32(4, True)], nb=2)
add("compress_i32", "hadamard", 1, 4, 4096, 0, [I2W(1), FFWD(12)])
add("compress_i32", "hadamard", 3, 3, 8192, 0, [I2W(3), FFWD(13)])
add("compress_i32", "hadamard", 4, 4, 1024, 0, [I2W(4), FWD])
add("compress_i32", "dct", 4, 4, 1024, 0, [I2W(4), STENCIL], exact=True)
for off in (0, 1):
    add("compress_i32", "dct", 3, 4, 1024, off, [I2W(3), STENCIL])

# -- last stage of decompress to native samples
# k_planes_to_samples_fast: 4-channel groups, 128-sample pieces; 16, 28 and 56 x 4 B drop the sample tiles per
# output group (tpg) from 8 to 4, 2 and 1.  An even number of pieces per channel and an even tpg take the two-tile
# loop, an odd one (128, 384, 640, 1152 samples; tpg 1) the one-tile loop.
for kind, b, c, ns in (("xdelta_hzr", 1, 4, 512), ("hzr", 1, 8, 1024), ("xdelta_hzr", 1, 4, 128), ("xdelta_hzr", 2, 4, 512),
                       ("hzr", 2, 16, 512), ("hzr", 2, 8, 384), ("xdelta_hzr", 3, 12, 1024), ("xdelta_hzr", 3, 12, 640),
                       ("hzr", 3, 4, 1024), ("xdelta_hzr", 4, 16, 1024), ("hzr", 4, 16, 1152), ("hzr", 4, 28, 256),
                       ("xdelta_hzr", 4, 56, 256)):
    add("decompress", kind, b, c, ns, 0, [INVF(b, st(kind))])
GENERIC_SHAPES = (("xdelta_hzr", 1, 3, 700), ("hzr", 1, 2, 40000), ("xdelta_hzr", 2, 3, 30000), ("hzr", 2, 4, 1000),
                  ("xdelta_hzr", 3, 2, 1), ("hzr", 3, 7, 33), ("xdelta_hzr", 4, 3, 2), ("hzr", 4, 1, 257))
for kind, b, c, ns in GENERIC_SHAPES:
    add("decompress", kind, b, c, ns, 0, [INVG(b, st(kind), True)])
for off in MISALIGNED:
    add("decompress", "xdelta_hzr", 3, 12, 1024, off, [INVG(3, True, True)])
    add("decompress", "hzr", 2, 16, 512, off, [INVG(2, False, True)])
    add("decompress", "hadamard", 3, 4, 4096, off, [FINV(12), W2R(3)])
    add("decompress", "dct", 2, 4, 1024, off, [INVF(4, True, True), W2R(2)], exact=True)
for b in (1, 2, 3, 4):
    add("decompress", "hadamard", b, 4, 4096, 0, [RAWI(12, b)])
    add("decompress", "hadamard", b, 4, 8192, 0, [RAWI(13, b)])
add("decompress", "hadamard", 3, 12, 4096, 0, [RAWI(12, 3)])
add("decompress", "hadamard", 2, 3, 8192, 0, [FINV(13), W2R(2)])
add("decompress", "hadamard", 1, 4, 1024, 0, [INV, W2R4(1)])
add("decompress", "hadamard", 4, 3, 64, 0, [INV, W2R(4)])
add("decompress", "dct", 2, 4, 1024, 0, [INVF(4, True, True), W2R4(2)], exact=True)
add("decompress", "dct", 3, 8, 1024, 0, [INVF(4, True, True), W2R4(3)], exact=True)
add("decompress", "dct", 4, 4, 1024, 0, [INVF(4, True, True), W2R4(4)], exact=True)
add("decompress", "dct", 1, 3, 77, 0, [INVG(4, True, False), W2R(1)], exact=True)
for off in (1, 3):
    add("decompress", "dct", 3, 4, 1024, off, [INVF(4, True, True), W2R(3)])
for off in (0,) + MISALIGNED:
    add("decompress_frames", "xdelta_hzr", 3, 12, 1024, off, [INVF(3, True) if off == 0 else INVG(3, True, True)])
for off in (0, 1):
    add("decompress_frames", "hadamard", 3, 4, 4096, off, [RAWI(12, 3)] if off == 0 else [FINV(12), W2R(3)])

# -- last stage of decompress to int32 words: the fast kernel needs 128-sample pieces in groups of 4 and 16-byte
# alignment (3 ch x 128 samples: 3 pieces, generic)
for kind, b, c, ns in (("xdelta_hzr", 1, 4, 512), ("hzr", 1, 8, 1024), ("xdelta_hzr", 2, 4, 512), ("hzr", 2, 16, 512),
                       ("hzr", 3, 4, 1024), ("xdelta_hzr", 3, 12, 640), ("xdelta_hzr", 4, 16, 1024), ("hzr", 4, 28, 256)):
    add("decompress_i32", kind, b, c, ns, 0, [INVF(b, st(kind), True)])
for kind, b, c, ns in GENERIC_SHAPES + (("xdelta_hzr", 2, 3, 128),):
    add("decompress_i32", kind, b, c, ns, 0, [INVG(b, st(kind), False)])
for off in (0, 1, 2, 3):
    add("decompress_i32", "xdelta_hzr", 3, 12, 1024, off, [INVF(3, True, True) if off == 0 else INVG(3, True, False)])
    add("decompress_i32", "hadamard", 2, 4, 4096, off, [FINV(12), SEXT(2)])
add("decompress_i32", "hadamard", 4, 4, 4096, 0, [FINV(12)])    # 4-byte samples: written by the transform itself
add("decompress_i32", "hadamard", 4, 3, 64, 0, [INV])
add("decompress_i32", "hadamard", 1, 4, 1024, 0, [INV, SEXT(1)])
add("decompress_i32", "hadamard", 3, 3, 8192, 0, [FINV(13), SEXT(3)])
add("decompress_i32", "dct", 4, 4, 1024, 0, [INVF(4, True, True), SEXT(4)], exact=True)
add("decompress_i32", "dct", 1, 3, 77, 0, [INVG(4, True, False), SEXT(1)], exact=True)
add("decompress_i32", "dct", 3, 4, 1024, 1, [INVF(4, True, True), SEXT(3)])

# -- the pre-filters, in place
for off in (0, 1, 4):
    g4 = off == 0
    add("iir5", "xdelta_hzr", 3, 12, 1024, off, [R2W4(3) if g4 else R2W(3), IIR(5), W2R4(3) if g4 else W2R(3)])
    add("iir4", "xdelta_hzr", 4, 4, 2048, off, [R2W4(4) if g4 else R2W(4), IIR(4), W2R4(4) if g4 else W2R(4)])
    add("fir", "xdelta_hzr", 2, 8, 1024, off, [R2W4(2) if g4 else R2W(2), FIR, W2R4(2) if g4 else W2R(2)])
add("iir2", "xdelta_hzr", 1, 4, 1024, 0, [R2W4(1), IIR(2), W2R4(1)])
add("iir3", "xdelta_hzr", 2, 3, 300, 0, [R2W(2), IIR(3), W2R(2)])
add("fir", "xdelta_hzr", 4, 1, 257, 0, [R2W(4), FIR, W2R(4)])

# Sample-stage kernels the library compiles that no call can reach, with the reason (none today).
UNREACHABLE: dict[str, str] = {}

# (n, d, init_nr_samples) of the IIR rows: Butterworth low-passes of order 1..3 and the reference's band-pass
N5 = [1.00000000000, -3.14332095199, 3.70064088865, -1.97083923944, 0.41351972908]
D5 = [0.06722876941, 0.00000000000, -0.13445753881, 0.00000000000, 0.06722876941]
IIR_FILTERS = {
    2: ([1.0, -0.5095254], [0.2452373, 0.2452373], 0),
    3: ([1.0, -1.1429805, 0.4128016], [0.06745527, 0.13491055, 0.06745527], 50),
    4: ([1.0, -1.76004188, 1.18289326, -0.27805992], [0.01809893, 0.0542968, 0.0542968, 0.01809893], 20),
    5: (N5, D5, 2000),
}
FIR_KERNEL = np.array([0.05, -0.1, 0.15, 0.2, 0.3, 0.2, 0.15, -0.1, 0.05])
FRAME_IDS = [6, 0, 3, 3, 1, 5, 2]   # decompress_frames: any order, a repeat


def row_id(r):
    return (f"{r.entry}-{r.kind}{'-exact' if r.exact else ''}-b{r.bps}c{r.ch}n{r.ns}"
            f"{f'-nb{r.nb}' if r.kind == 'xdelta_hzr' else ''}-o{r.off}")


# ---- frames that reach the edges ------------------------------------------------------------------------------

def native(x, bps):
    """int64 samples [ns, ch] -> the frame's interleaved little-endian bytes."""
    ns, ch = x.shape
    return np.ascontiguousarray(x.astype("<i8").view(np.uint8).reshape(ns, ch, 8)[:, :, :bps]).reshape(-1)


def make_frames(oracle, bps, ch, ns):
    """uint8 [N_FRAMES, frame_bytes]: all zero (FILL blocks), ECG, min -> max steps on the 128 / 256 / 512-sample
    boundaries (channel c steps every 2^(7 + c % 3) samples), min / max alternating per sample and per channel,
    constant min, constant max, full-range noise with both extremes scattered in.  The quiet frames come first, so
    that a plane-count probe escalates inside the batch."""
    lo, hi = -(1 << (8 * bps - 1)), (1 << (8 * bps - 1)) - 1
    rng = np.random.default_rng(7 * ns + 31 * ch + bps)
    s, c = np.arange(ns)[:, None], np.arange(ch)[None, :]
    noise = rng.integers(lo, hi + 1, (ns, ch), dtype=np.int64)
    flat = noise.reshape(-1)
    pos = rng.integers(0, flat.size, 2 + flat.size // 32)
    flat[pos[0::2]], flat[pos[1::2]] = lo, hi
    flat[0], flat[-1] = lo, hi
    ecg = oracle.synth_ecg(ns + ch, 1, bps, ch, ns, amplitude=min(20000, 1 << (8 * bps - 2)))[0]
    frames = [np.zeros((ns, ch), np.int64), None, np.where((s >> (7 + c % 3)) & 1, hi, lo),
              np.where((s + c) & 1, hi, lo), np.full((ns, ch), lo), np.full((ns, ch), hi), noise]
    return np.stack([ecg if x is None else native(x, bps) for x in frames])


def sext(w, bps):
    """The low 8*bps bits of int32 words, sign-extended."""
    sh = 32 - 8 * bps
    return ((np.asarray(w, np.int32).astype(np.uint32) << np.uint32(sh)).view(np.int32) >> sh).astype(np.int32)


def native_to_words(raw, bps, ch, ns, rng=None):
    """uint8 [n, ns*ch*bps] interleaved samples -> int32 [n, ch, ns]; with `rng`, random bits above 8*bps."""
    x = np.asarray(raw, np.uint8).reshape(-1, ns, ch, bps).astype(np.uint32)
    v = np.zeros(x.shape[:3], np.uint32)
    for b in range(bps):
        v |= x[..., b] << np.uint32(8 * b)
    w = sext(v.view(np.int32), bps).view(np.uint32)
    if rng is not None and bps < 4:
        hi = np.uint32((0xFFFFFFFF << (8 * bps)) & 0xFFFFFFFF)
        w = (w & ~hi) | (rng.integers(0, 1 << 32, w.shape, dtype=np.uint64).astype(np.uint32) & hi)
    return np.ascontiguousarray(w.view(np.int32).transpose(0, 2, 1))


# ---- what the oracle writes, once per shape -------------------------------------------------------------------

Expect = namedtuple("Expect", "raws streams frame_nb nb dec")
_EXPECT = {}


def expected(oracle, r):
    """The frames of a row's shape and, except for dct's fast path, the oracle's streams, per-frame plane counts,
    final plane count and decode."""
    key = (r.kind, r.bps, r.ch, r.ns, r.nb, r.exact)
    if key not in _EXPECT:
        raws = make_frames(oracle, r.bps, r.ch, r.ns)
        if r.kind == "dct" and not r.exact:
            _EXPECT[key] = Expect(raws, None, None, None, None)
        else:
            o = oracle.OraclePacker(r.kind, r.bps, r.ch, r.ns, r.nb)
            streams, fnb, dec = [], [], []
            for f in raws:
                streams.append(o.compress(f))
                fnb.append(o.nb)
                dec.append(np.frombuffer(o.decompress(streams[-1])[0], np.uint8))
            _EXPECT[key] = Expect(raws, streams, fnb, o.nb, np.stack(dec))
    return _EXPECT[key]


# ---- buffers with guard bands ---------------------------------------------------------------------------------

class Guarded:
    """`data` (uint8 or int32, 1-D) at element offset `off` behind GUARD bytes of sentinels, GUARD bytes of
    sentinels behind it, on the device."""

    def __init__(self, data, off):
        data = np.asarray(data).reshape(-1)
        fill = FILL_U8 if data.dtype == np.uint8 else FILL_I32
        g = GUARD // data.itemsize
        self.lo, self.hi = g + off, g + off + data.size
        self.host = np.full(self.hi + g, fill, data.dtype)
        self.host[self.lo:self.hi] = data
        self.buf = torch.from_numpy(self.host.copy()).cuda()
        self.view = self.buf[self.lo:self.hi]
        assert self.view.data_ptr() % 16 == (off * data.itemsize) % 16

    def get(self):
        """(the whole buffer on the host, the data part)."""
        torch.cuda.synchronize()
        a = self.buf.cpu().numpy()
        return a, a[self.lo:self.hi]

    def assert_guards(self, what):
        a, _ = self.get()
        assert np.array_equal(a[:self.lo], self.host[:self.lo]), f"{what}: written before the buffer"
        assert np.array_equal(a[self.hi:], self.host[self.hi:]), f"{what}: written past the buffer"


def make_packer(R, r):
    p = R.SignalPacker(r.kind, r.bps, r.ch, r.ns, r.nb, max_batch_frames=N_FRAMES)
    if r.exact:
        p.set_dct_exact(True)
    return p


def batch_on_host(b):
    torch.cuda.synchronize()
    offs = b.offsets.cpu().numpy()
    return offs, b.stream.cpu().numpy()[:int(offs[b.n_frames])], b.frame_nb.cpu().numpy()


def frames_of(b):
    offs, stream, _ = batch_on_host(b)
    return [stream[offs[i]:offs[i + 1]].tobytes() for i in range(b.n_frames)]


def to_dev(a):
    return torch.from_numpy(np.ascontiguousarray(a).reshape(-1).copy()).cuda()


# ---- the calls of a row ---------------------------------------------------------------------------------------

def row_call(R, r, raws, rng):
    """(packer, guarded buffer, thunk, batch): everything a row's call needs is set up, the thunk makes the call;
    for the decompress entries, `batch` is the aligned native compress of `raws` that the call decodes."""
    p = make_packer(R, r)
    n = len(raws)
    if r.entry == "compress":
        g = Guarded(raws, r.off)
        return p, g, lambda: p.compress_batch(g.view), None
    if r.entry == "compress_i32":
        g = Guarded(native_to_words(raws, r.bps, r.ch, r.ns, rng), r.off)
        return p, g, lambda: p.compress_tensor(g.view.view(n, r.ch, r.ns)), None
    if r.entry.startswith("iir") or r.entry == "fir":
        g = Guarded(raws, r.off)
        if r.entry == "fir":
            return p, g, lambda: p.prefilter_fir(g.view, FIR_KERNEL), None
        nn, dd, init = IIR_FILTERS[int(r.entry[3:])]
        return p, g, lambda: p.prefilter_iir(g.view, nn, dd, init), None
    batch = p.compress_batch(to_dev(raws))
    if r.entry == "decompress":
        g = Guarded(np.zeros(raws.size, np.uint8), r.off)
        return p, g, lambda: p.decompress_batch(batch, out=g.view), batch
    if r.entry == "decompress_frames":
        g = Guarded(np.zeros(len(FRAME_IDS) * p.frame_bytes, np.uint8), r.off)
        ids = torch.tensor(FRAME_IDS, dtype=torch.int64, device="cuda")
        return p, g, lambda: p.decompress_frames(batch, ids, out=g.view), batch
    assert r.entry == "decompress_i32", r.entry
    g = Guarded(np.zeros(n * r.ch * r.ns, np.int32), r.off)
    return p, g, lambda: p.decompress_tensor(batch, out=g.view.view(n, r.ch, r.ns)), batch


@pytest.fixture(scope="module")
def R():
    import rspt_b200  # noqa: F401
    from rspt_b200 import packer
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return packer


@pytest.mark.gpu
@pytest.mark.timeout(600)
@pytest.mark.parametrize("r", ROWS, ids=row_id)
def test_row_matches_oracle(R, oracle, r):
    e = expected(oracle, r)
    raws, n, fb = e.raws, len(e.raws), r.bps * r.ch * r.ns
    p, g, call, batch = row_call(R, r, raws, np.random.default_rng(r.ns + r.off))
    before = g.get()[0]
    out = call()
    what = row_id(r)

    if r.entry.startswith("iir") or r.entry == "fir":
        g.assert_guards(what)
        got = g.get()[1].reshape(n, fb)
        from conftest import has_ref
        impl = "reference" if has_ref() else "port"
        for i in range(n):
            if r.entry == "fir":
                want = oracle.prefilter_fir(raws[i], r.bps, r.ch, r.ns, FIR_KERNEL, impl)
            else:
                nn, dd, init = IIR_FILTERS[int(r.entry[3:])]
                want = oracle.prefilter_iir(raws[i], r.bps, r.ch, r.ns, nn, dd, init, impl)
            assert np.array_equal(got[i], want), (what, "frame", i)
        return

    fast_dct = r.kind == "dct" and not r.exact
    ref = None
    if fast_dct:   # the aligned native call of a second handle is the yardstick
        ref = make_packer(R, r)
        ref_batch = ref.compress_batch(to_dev(raws))

    if r.entry in ("compress", "compress_i32"):
        assert np.array_equal(g.get()[0], before), f"{what}: the input buffer or its guards changed"
        got = frames_of(out)
        if fast_dct:
            assert got == frames_of(ref_batch), what
            return
        for i in range(n):
            assert got[i] == e.streams[i], (what, "frame", i)
        assert batch_on_host(out)[2].tolist() == e.frame_nb, what
        assert p.nb == e.nb, what
        return

    g.assert_guards(what)
    got = g.get()[1]
    if fast_dct:
        want = ref.decompress_batch(ref_batch).cpu().numpy().reshape(n, fb)
    else:
        want = e.dec
        assert frames_of(batch) == e.streams, f"{what}: the decoded batch is not the oracle's stream"
    if r.entry == "decompress":
        assert np.array_equal(got.reshape(n, fb), want), what
    elif r.entry == "decompress_frames":
        assert np.array_equal(got.reshape(len(FRAME_IDS), fb), want[FRAME_IDS]), what
    else:
        assert np.array_equal(got.reshape(n, r.ch, r.ns), native_to_words(want, r.bps, r.ch, r.ns)), what


# ---- kernel identity ------------------------------------------------------------------------------------------

FAMILY = re.compile(r"^k_(xdelta_planes|planes_to_samples|raw_to_words|words_to_raw|fwht_|i32_to_words|words_sext|"
                    r"words_stencil_planes|iir_frames|fir_words)")


def kernel_name(demangled):
    """'void rspt::k_xdelta_planes_tma<(int)2, (int)4, (bool)1>(...)' or '... k_xdelta_planes_tma<2, 4, true>(...)'
    -> 'k_xdelta_planes_tma<2,4,true>'; None for a name without a k_ kernel."""
    s = demangled.replace("(bool)0", "false").replace("(bool)1", "true")
    s = re.sub(r"\((?:unsigned )?int\)", "", s)
    m = re.search(r"\bk_\w+(?:<[^>]*>)?", s)
    return m.group(0).replace(" ", "") if m else None


def trace_rows(out_path):
    """Child process: every row's call under torch.profiler, one window per call between two marker kernels;
    writes {row id: [sample-stage kernels in launch order]}."""
    sys.path.insert(0, ROOT)
    from rspt_b200 import packer as R
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.set_device(0)
    marker = torch.zeros(1, dtype=torch.int64, device="cuda")
    rng = np.random.default_rng(11)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        marker.bitwise_not_()   # the first two kernels of the trace name the window markers
        marker.neg_()
        torch.cuda.synchronize()
        for r in ROWS:
            raws = rng.integers(0, 256, (N_FRAMES, r.bps * r.ch * r.ns), dtype=np.uint8)
            p, _, call, _ = row_call(R, r, raws, rng)
            torch.cuda.synchronize()
            marker.bitwise_not_()
            call()
            torch.cuda.synchronize()
            marker.neg_()
            p.close()
        torch.cuda.synchronize()
    path = out_path + ".trace.json"
    prof.export_chrome_trace(path)
    with open(path) as f:
        events = json.load(f)["traceEvents"]
    os.remove(path)
    kernels = [e["name"] for e in sorted((e for e in events if e.get("cat") == "kernel"), key=lambda e: e["ts"])]
    opening, closing = kernels[:2]
    windows, cur = [], None
    for name in kernels[2:]:
        if name == opening:
            cur = []
        elif name == closing:
            windows.append(cur)
            cur = None
        elif cur is not None:
            k = kernel_name(name)
            if k and FAMILY.match(k):
                cur.append(k)
    assert len(windows) == len(ROWS), f"{len(windows)} call windows in the trace for {len(ROWS)} rows"
    with open(out_path, "w") as f:
        json.dump({row_id(r): w for r, w in zip(ROWS, windows)}, f)


@pytest.mark.gpu
@pytest.mark.timeout(600)
def test_rows_launch_their_kernels(tmp_path):
    out = str(tmp_path / "kernels.json")
    p = subprocess.run([sys.executable, os.path.abspath(__file__), out], capture_output=True, text=True, timeout=500)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-4000:]
    with open(out) as f:
        got = json.load(f)
    bad = [f"{row_id(r)}: launched {got[row_id(r)]}, the table says {list(r.kernels)}"
           for r in ROWS if got[row_id(r)] != list(r.kernels)]
    assert not bad, "\n".join(bad)


# ---- coverage of the compiled kernels -------------------------------------------------------------------------

def _cuda_tool(name):
    for d in (os.environ.get("CUDA_HOME"), os.environ.get("CUDA_PATH"), "/usr/local/cuda"):
        if d and os.path.exists(os.path.join(d, "bin", name)):
            return os.path.join(d, "bin", name)
    return shutil.which(name)


def compiled_sample_kernels():
    """The sample-stage kernel instantiations in the library's sm_100a code, normalised like the table's names."""
    dump, filt = _cuda_tool("cuobjdump"), _cuda_tool("cu++filt")
    if not (dump and filt):
        pytest.skip("cuobjdump / cu++filt not found (CUDA toolkit bin): cannot list the library's kernels")
    syms = subprocess.run([dump, "-symbols", LIB], capture_output=True, text=True, check=True).stdout
    mangled = [line.split()[-1] for line in syms.splitlines() if "STO_ENTRY" in line]
    names = subprocess.run([filt], input="\n".join(mangled), capture_output=True, text=True, check=True).stdout
    return {k for k in map(kernel_name, names.splitlines()) if k and FAMILY.match(k)}


def test_table_covers_every_sample_stage_kernel():
    assert os.path.exists(LIB), "build the library first (python -m rspt_b200.build)"
    compiled = compiled_sample_kernels()
    table = {k for r in ROWS for k in r.kernels}
    assert table <= compiled, f"table names kernels the library does not compile: {sorted(table - compiled)}"
    assert not set(UNREACHABLE) - compiled, sorted(set(UNREACHABLE) - compiled)
    missing = compiled - table - set(UNREACHABLE)
    assert not missing, f"compiled sample-stage kernels no row reaches: {sorted(missing)}"
    print(f"{len(table)} of {len(compiled) - len(UNREACHABLE)} sample-stage instantiations covered")


if __name__ == "__main__":
    trace_rows(sys.argv[1])
