"""Parity of the CUDA path (through the C ABI) against the CPU oracle, the committed golden vectors
and -- where oracle/_ref/libref.so travelled with the repo -- the unmodified reference.
Bit-exact for everything integer; stated tolerances for the dct packer.  Needs a B200."""
import hashlib
import os

import numpy as np
import pytest

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600)]

torch = pytest.importorskip("torch")


def sha(b):
    return hashlib.sha256(bytes(b)).hexdigest()


@pytest.fixture(scope="module")
def R():
    import rspt_b200
    from rspt_b200 import packer
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return packer


def to_dev(a):
    return torch.from_numpy(np.array(a, dtype=np.uint8, copy=True).reshape(-1)).cuda()


def make_raw(rng, bps, ch, ns, amp=None, kind="walk"):
    amp = amp or (1 << min(8 * bps - 2, 14))
    if kind == "walk":
        x = np.cumsum(rng.integers(-amp // 16 - 1, amp // 16 + 2, (ns, ch)), axis=0)
    else:
        x = rng.integers(-amp, amp, (ns, ch))
    x = np.clip(x, -(1 << (8 * bps - 1)), (1 << (8 * bps - 1)) - 1).astype(np.int32)
    return x.astype("<i4").view(np.uint8).reshape(ns, ch, 4)[:, :, :bps].copy().reshape(-1)


# ---------------------------------------------------------------------------------------------
def test_synth_generator_matches_cpu(R, oracle):
    for (first, n, bps, ch, ns) in [(0, 3, 3, 12, 8192), (7, 2, 4, 12, 4096), (1000000, 3, 2, 5, 1000), (3, 2, 1, 1, 77)]:
        amp = 20000 if bps >= 3 else (100 if bps == 1 else 5000)
        g = R.synth_ecg(first, n, bps, ch, ns, amplitude=amp).cpu().numpy()
        c = oracle.synth_ecg(first, n, bps, ch, ns, amplitude=amp).reshape(-1)
        assert np.array_equal(g, c), (first, n, bps, ch, ns)


def test_crc32c_kernel(R, oracle):
    rng = np.random.default_rng(5)
    for n in (1, 2, 3, 7, 8, 9, 11, 12, 63, 64, 65, 1000, 4097, 65535, 65536):
        buf = rng.integers(0, 256, n, dtype=np.uint8)
        assert R.crc32c(buf) == oracle.crc32c(buf), n
    assert R.crc32c(np.frombuffer(b"123456789", np.uint8)) == 0xE3069283


def _hzr_buffers(rng):
    out = []
    for n in (1, 2, 3, 7, 22, 23, 278, 279, 1000, 16662, 16663, 33324, 40000, 65535, 65536):
        out.append(np.zeros(n, np.uint8))
        out.append(rng.integers(0, 256, n, dtype=np.uint8))
        out.append(rng.integers(0, 4, n, dtype=np.uint8))
        sp = np.zeros(n, np.uint8)
        k = max(1, n // 50)
        sp[rng.integers(0, n, k)] = rng.integers(1, 256, k, dtype=np.uint8)
        out.append(sp)
        out.append(np.clip(np.rint(rng.laplace(0, 6, n)), -120, 120).astype(np.int8).view(np.uint8))
        out.append(np.full(n, 255, np.uint8))
        z = np.zeros(n, np.uint8)
        z[-1] = 9
        out.append(z)
        z = np.zeros(n, np.uint8)
        z[0] = 9
        out.append(z)
    for p in (0.5, 0.9, 0.99):
        out.append((rng.random(65536) < p).astype(np.uint8) * 3 + 1)
    out.append(rng.integers(0, 200, 65536, dtype=np.uint8))
    out.append(np.tile(np.arange(256, dtype=np.uint8), 256))          # every count equal: tie-breaking
    out.append(np.repeat(np.arange(1, 24, dtype=np.uint8), [2 ** min(i, 11) for i in range(23)])[:65536])
    return out


def test_hzr_histogram_tree_and_plan(R, oracle):
    """Per-block stages: token histogram, non-canonical Huffman codes, mode + payload size."""
    p = R.SignalPacker.new_hzr(1, 1, 65536, max_batch_frames=1)
    rng = np.random.default_rng(7)
    for buf in _hzr_buffers(rng):
        hist, codes, info = p.debug_hzr_tables(buf)
        want_hist = oracle.hzr_histogram(buf)
        assert np.array_equal(hist, want_hist), buf.size
        mode, plen = oracle.hzr_block_plan(buf)
        assert (int(info[0]), int(info[1])) == (mode, plen), (buf.size, info, mode, plen)
        if mode == 1:
            n_used, code, ln, tree, tree_nbits = oracle.hzr_build_codes(want_hist)
            used = want_hist > 0
            assert np.array_equal(codes[used] & 0x07FFFFFF, code[used])
            assert np.array_equal(codes[used] >> 27, ln[used])
            assert int(info[2]) == tree_nbits and int(info[3]) == n_used


PLANE_CASES = [
    ("xdelta_hzr", 3, 12, 8192, 3), ("xdelta_hzr", 4, 12, 4096, 3), ("xdelta_hzr", 2, 5, 1000, 2),
    ("xdelta_hzr", 1, 3, 700, 1), ("xdelta_hzr", 4, 1, 8192, 4), ("xdelta_hzr", 3, 2, 1, 3),
    ("xdelta_hzr", 4, 3, 2, 3), ("xdelta_hzr", 3, 7, 33, 3),
    # shapes of the quad-tiled fast transform (ch % 4 == 0, ns % 4 == 0): partial tiles, planes > bps
    ("xdelta_hzr", 2, 4, 1000, 2), ("xdelta_hzr", 1, 8, 700, 1), ("xdelta_hzr", 3, 4, 4, 3),
    ("xdelta_hzr", 3, 8, 516, 4), ("xdelta_hzr", 4, 16, 2052, 2), ("hzr", 2, 8, 2052, 0), ("hzr", 1, 4, 8, 0),
    ("hzr", 3, 12, 8192, 0), ("hzr", 1, 2, 999, 0), ("hzr", 4, 3, 5000, 0),
    ("hadamard", 4, 12, 4096, 0), ("hadamard", 3, 3, 16384, 0), ("hadamard", 2, 2, 8, 0), ("hadamard", 1, 1, 32768, 0),
    ("hadamard", 3, 5, 4096, 0), ("hadamard", 2, 1, 4096, 0),   # radix-16 register path (ns = 4096), odd channel counts
]


@pytest.mark.parametrize("kind,bps,ch,ns,nb", PLANE_CASES)
def test_transform_planes_bit_exact(R, oracle, kind, bps, ch, ns, nb):
    """Stage 1 (de-interleave, delta/offset/xor or FWHT+quantise, plane split) against the oracle's words."""
    rng = np.random.default_rng(ns * 7 + ch)
    nfr = 3
    raws = [make_raw(rng, bps, ch, ns, kind="walk" if i else "noise") for i in range(nfr)]
    p = R.SignalPacker(kind, bps, ch, ns, nb or 3, max_batch_frames=nfr)
    planes, hdr = p.debug_planes(to_dev(np.concatenate(raws)))
    o = oracle.OraclePacker(kind, bps, ch, ns, nb or 3)
    for i, raw in enumerate(raws):
        words, header = o.transform(raw)
        for k in range(planes.shape[1]):
            want = ((words.view(np.uint32) >> (8 * k)) & 0xFF).astype(np.uint8)
            assert np.array_equal(planes[i, k], want), (kind, i, k)
        if o.header_bytes:
            assert np.array_equal(hdr[i], header)


STREAM_CASES = [
    ("xdelta_hzr", 3, 12, 8192, 3, 4), ("xdelta_hzr", 4, 12, 4096, 3, 3), ("xdelta_hzr", 4, 1, 8192, 3, 2),
    ("xdelta_hzr", 2, 5, 1000, 2, 5), ("xdelta_hzr", 1, 3, 700, 1, 3), ("xdelta_hzr", 3, 3, 20000, 3, 2),
    ("xdelta_hzr", 4, 12, 16384, 3, 2), ("xdelta_hzr", 3, 2, 1, 3, 4), ("xdelta_hzr", 3, 7, 33, 3, 4),
    ("xdelta_hzr", 4, 2, 70001, 4, 2),
    ("hzr", 3, 12, 8192, 0, 3), ("hzr", 4, 12, 4096, 0, 2), ("hzr", 1, 2, 999, 0, 3), ("hzr", 2, 1, 140000, 0, 2),
    ("hadamard", 4, 12, 4096, 0, 3), ("hadamard", 3, 3, 16384, 0, 2), ("hadamard", 2, 2, 8, 0, 3), ("hadamard", 2, 3, 4096, 0, 2),
    ("hadamard", 3, 12, 8192, 0, 3), ("hadamard", 4, 1, 8192, 0, 2),
    # fused raw <-> planes kernels (ch % 4 == 0, ns 4096 / 8192), every sample width
    ("hadamard", 2, 4, 4096, 0, 2), ("hadamard", 1, 8, 8192, 0, 2), ("hadamard", 4, 4, 8192, 0, 2), ("hadamard", 3, 4, 4096, 0, 3),
    ("hadamard", 1, 4, 4096, 0, 2), ("hadamard", 2, 8, 8192, 0, 2),
]


@pytest.mark.parametrize("kind,bps,ch,ns,nb,nfr", STREAM_CASES)
def test_stream_bit_exact_and_round_trip(R, oracle, kind, bps, ch, ns, nb, nfr):
    """Whole path: the concatenated frames equal the oracle's bytes; decode (indexed and serial)
    restores the oracle's decode, which for the lossless packers is the input."""
    rng = np.random.default_rng(ns + 13 * ch + bps)
    fb = bps * ch * ns
    if bps >= 2 and ns >= 64:
        raws = oracle.synth_ecg(11, nfr, bps, ch, ns, amplitude=20000 if bps >= 3 else 3000)
    else:
        raws = np.stack([make_raw(rng, bps, ch, ns) for _ in range(nfr)])
    raws[nfr - 1] = 0 if nfr > 2 else raws[nfr - 1]  # an all-zero frame: FILL blocks
    p = R.SignalPacker(kind, bps, ch, ns, nb or 3, max_batch_frames=nfr)
    batch = p.compress_batch(to_dev(raws))
    torch.cuda.synchronize()
    offs = batch.offsets.cpu().numpy()
    stream = batch.stream.cpu().numpy()
    o = oracle.OraclePacker(kind, bps, ch, ns, nb or 3)
    want_dec = []
    for i in range(nfr):
        want = o.compress(raws[i])
        got = stream[offs[i]:offs[i + 1]].tobytes()
        assert len(got) == len(want), (kind, i, len(got), len(want))
        assert got == want, (kind, i)
        want_dec.append(np.frombuffer(o.decompress(want)[0], np.uint8))
    assert np.array_equal(batch.frame_nb.cpu().numpy(), np.full(nfr, o.nb, np.uint8))
    want_dec = np.stack(want_dec)
    if kind in ("xdelta_hzr", "hzr"):
        assert np.array_equal(want_dec, raws.reshape(nfr, fb))
    for use_sc in (True, False):
        status = torch.full((nfr,), 7, dtype=torch.int32, device="cuda")
        dec = p.decompress_batch(batch, status=status, use_sidecar=use_sc)
        torch.cuda.synchronize()
        assert not status.cpu().numpy().any()
        assert np.array_equal(dec.cpu().numpy().reshape(nfr, fb), want_dec), (kind, use_sc)
    c = p.counters()
    assert c["frames_compressed"] == nfr and c["frames_decompressed"] == 2 * nfr
    assert c["compressed_bytes_out"] == offs[nfr]
    assert c["blocks_copy"] + c["blocks_huff"] + c["blocks_fill"] == nfr * o.nb * ((ch * ns + 65535) // 65536)


def test_golden_vectors(R, golden, golden_inputs):
    """The committed vectors produced by the unmodified reference (tests/golden/make_golden.py)."""
    for case in golden["cases"]:
        kind, bps, ch, ns = case["kind"], case["bps"], case["ch"], case["ns"]
        fb = bps * ch * ns
        data = golden_inputs[case["input"]]
        nfr = len(case["frames"])
        if kind == "dct":
            os.environ["RSPT_DCT_DIRECT"] = "1"  # the bit-exact path; the fast path has its own test
        try:
            p = R.SignalPacker(kind, bps, ch, ns, case["nb"] or 3, max_batch_frames=nfr)
        finally:
            os.environ.pop("RSPT_DCT_DIRECT", None)
        batch = p.compress_batch(to_dev(data[: nfr * fb]))
        torch.cuda.synchronize()
        offs = batch.offsets.cpu().numpy()
        stream = batch.stream.cpu().numpy()
        dec = p.decompress_batch(batch).cpu().numpy().reshape(nfr, fb)
        for i, want in enumerate(case["frames"]):
            got = stream[offs[i]:offs[i + 1]]
            assert len(got) == want["len"], (case["name"], i, len(got), want["len"])
            assert sha(got) == want["sha256"], (case["name"], i)
            assert sha(dec[i]) == want["dec_sha256"], (case["name"], i)
        assert p.nb == case["final_nb"], case["name"]


def test_xdelta_plane_escalation(R, oracle):
    """nb < bps: the plane count is a sticky running max over frames, across batches
    (signal_packer_xdelta_hzr.cpp:63-69).  Frames are built so that 1, then 2, 3 and 4 planes
    are needed: a flat-order ramp with increments in [0, 200] keeps every post-xor word in int8."""
    rng = np.random.default_rng(3)
    bps, ch, ns = 4, 3, 500

    def ramp(maxinc, jump_at=None, jump=0):
        inc = rng.integers(0, maxinc + 1, ch * ns).astype(np.int64)
        if jump_at is not None:
            inc[jump_at] += jump
        x = np.cumsum(inc).reshape(ch, ns).T.astype(np.int32)      # flat (channel-major) order is monotone
        return np.ascontiguousarray(x).astype("<i4").view(np.uint8).reshape(-1)

    raws = np.stack([ramp(200), ramp(200), ramp(200, 700, 20000), ramp(200), ramp(200, 5, 3000000), ramp(100),
                     ramp(200, 1499, 1 << 29), ramp(50)])
    p = R.SignalPacker.new_xdelta_hzr(bps, ch, ns, 1, max_batch_frames=8)
    o = oracle.OraclePacker("xdelta_hzr", bps, ch, ns, 1)
    want_nb = []
    want = []
    for r in raws:
        want.append(o.compress(r))
        want_nb.append(o.nb)
    assert want_nb == [1, 1, 2, 2, 3, 3, 4, 4], want_nb
    got_nb = []
    for lo, hi in ((0, 3), (3, 8)):  # two batches: the state must carry over
        batch = p.compress_batch(to_dev(raws[lo:hi]))
        torch.cuda.synchronize()
        offs = batch.offsets.cpu().numpy()
        stream = batch.stream.cpu().numpy()
        for i in range(hi - lo):
            assert stream[offs[i]:offs[i + 1]].tobytes() == want[lo + i], (lo, i)
        got_nb += batch.frame_nb.cpu().numpy().tolist()
        dec = p.decompress_batch(batch).cpu().numpy().reshape(hi - lo, -1)
        assert np.array_equal(dec, raws[lo:hi].reshape(hi - lo, -1))
    assert got_nb == want_nb
    assert p.nb == o.nb == 4 and p.counters()["escalations"] == o.escalations == 3


def test_host_api_single_frame_readme_example(R, oracle):
    """The README / test_5 call sequence (rspt_test.cpp:225-256) through the host entry points."""
    import math
    import zlib
    sine = np.array([int(math.sin(i / 100.0) * 1000.0) for i in range(8192)], np.int32).view(np.uint8)
    c = R.SignalPacker.new_xdelta_hzr(4, 1, 8192, 3)
    comp = c.compress(sine)
    assert len(comp) == 2028 and "%08x" % zlib.crc32(comp) == "672647f0"   # BASELINE.md section 3
    dec, used = c.decompress(comp)
    assert used == 2028 and dec == sine.tobytes()


def test_decodes_streams_from_cpu_reference(R, oracle):
    """Interop: frames written by the CPU side (no decode index) are decoded on the GPU."""
    from conftest import has_ref
    impl = "reference" if has_ref() else "port"
    for kind, bps, ch, ns in (("xdelta_hzr", 3, 12, 8192), ("hzr", 3, 3, 5000), ("hadamard", 4, 4, 4096)):
        raws = oracle.synth_ecg(0, 3, bps, ch, ns)
        cpu = oracle.make_packer(kind, bps, ch, ns, 3, impl)
        frames = [cpu.compress(r) for r in raws]
        offs = np.concatenate([[0], np.cumsum([len(f) for f in frames])])
        p = R.SignalPacker(kind, bps, ch, ns, 3, max_batch_frames=3)
        dec, status = p.decompress_stream(b"".join(frames), offs)
        assert not status.any()
        for i, f in enumerate(frames):
            assert dec[i].tobytes() == cpu.decompress(f)[0]


def test_listed_block_handed_to_general_encoder(R, oracle, monkeypatch):
    """A sparse block whose payload exceeds k_hzr_encode_sparse's staging is handed to k_hzr_encode,
    which needs the per-step leading-zero counts rebuilt from the list.  That size is out of reach of
    real data (5120 entries x ~15 bits), so the limit is lowered for this test."""
    monkeypatch.setenv("RSPT_SPARSE_STAGE_BYTES", "300")
    bps, ch, ns, n = 3, 12, 8192, 6
    raws = oracle.synth_ecg(40, n, bps, ch, ns)
    raws[5] = 0
    p = R.SignalPacker.new_xdelta_hzr(bps, ch, ns, 3, max_batch_frames=n)
    batch = p.compress_batch(to_dev(raws))
    torch.cuda.synchronize()
    offs = batch.offsets.cpu().numpy()
    stream = batch.stream.cpu().numpy()
    o = oracle.OraclePacker("xdelta_hzr", bps, ch, ns, 3)
    for i in range(n):
        assert stream[offs[i]:offs[i + 1]].tobytes() == o.compress(raws[i]), i
    for use_sc in (True, False):
        dec = p.decompress_batch(batch, use_sidecar=use_sc)
        assert np.array_equal(dec.cpu().numpy().reshape(n, -1), raws)
    # ragged single-channel planes: short last block, long zero runs across the step boundaries
    rng = np.random.default_rng(8)
    x = np.zeros((3, 70001), np.uint8)
    for r in x:
        idx = rng.choice(70001, 900, replace=False)
        r[idx] = rng.integers(1, 256, 900)
    # bursts: few chunks are touched (the density probe says "sparse") but the list overflows its 5120
    # entries, so the block falls back to the dense scan half-way through
    x[2] = 0
    for c0 in rng.choice(4000, 450, replace=False):
        x[2, c0 * 16:(c0 + 1) * 16] = rng.integers(1, 256, 16)
    ph = R.SignalPacker.new_hzr(1, 1, 70001, max_batch_frames=3)
    bh = ph.compress_batch(to_dev(x))
    torch.cuda.synchronize()
    oh = oracle.OraclePacker("hzr", 1, 1, 70001, 3)
    so, st = bh.offsets.cpu().numpy(), bh.stream.cpu().numpy()
    for i in range(3):
        assert st[so[i]:so[i + 1]].tobytes() == oh.compress(x[i]), i
    assert np.array_equal(ph.decompress_batch(bh).cpu().numpy().reshape(3, -1), x)


def test_ingest_ring_streams_frames_in_order(R, oracle):
    """The pinned packet ring (io_buffer protocol, ring_buffers.h:150-201): a packet becomes visible to
    the consumer when the producer asks for the next one, a full ring refuses, wrap-around keeps the frame
    order, and every drained frame is byte-identical to the oracle's."""
    bps, ch, ns, total, slots = 3, 4, 2048, 23, 6
    raws = oracle.synth_ecg(77, total, bps, ch, ns)
    p = R.SignalPacker.new_xdelta_hzr(bps, ch, ns, 3, max_batch_frames=4)  # smaller than the ring: several batches per drain
    ring = R.IngestRing(p, slots)
    o = oracle.OraclePacker("xdelta_hzr", bps, ch, ns, 3)
    dst = np.zeros(slots * p.max_compressed_size, np.uint8)
    offs = np.zeros(slots + 1, np.uint64)
    got = []
    produced = 0

    def take(flush=False):
        n = ring.drain(dst, offs, flush=flush)
        for i in range(n):
            got.append(dst[int(offs[i]):int(offs[i + 1])].tobytes())
        return n

    # nothing filled yet; the first packet alone stays "being filled"
    assert take() == 0
    pk = ring.next_packet()
    pk[:] = raws[produced]; produced += 1
    assert take() == 0
    while produced < total:
        pk = ring.next_packet()
        if pk is None:                 # ring full: the consumer has to run
            assert take() >= 1
            continue
        pk[:] = raws[produced]; produced += 1
        if produced % 5 == 0:
            take()
    take(flush=True)                   # the last packet is only released by flush
    assert take(flush=True) == 0
    assert len(got) == total
    for i in range(total):
        assert got[i] == o.compress(raws[i]), i
    # the same with the producer on its own thread (single producer / single consumer, like io_buffer)
    import threading
    import time
    got.clear()

    def producer():
        sent = 0
        while sent < total:
            pk2 = ring.next_packet()
            if pk2 is None:
                time.sleep(0.0005)
                continue
            pk2[:] = raws[sent]
            sent += 1

    th = threading.Thread(target=producer)
    th.start()
    deadline = time.time() + 60
    while th.is_alive() and time.time() < deadline:
        if take() == 0:
            time.sleep(0.0005)
    th.join(timeout=5)
    assert not th.is_alive()
    while take(flush=True):
        pass
    assert len(got) == total
    for i in range(total):
        assert got[i] == o.compress(raws[i]), i
    ring.close()
    p.close()


def test_prefilter_bit_exact(R, oracle):
    """rspt_gpu_prefilter_iir / _fir (the step in front of the packers, rspt_test.cpp:116-136) give the
    bytes the CPU side gives, for the reference's own band-pass and for shorter filters."""
    from conftest import has_ref
    impl = "reference" if has_ref() else "port"
    n5 = [1.00000000000, -3.14332095199, 3.70064088865, -1.97083923944, 0.41351972908]
    d5 = [0.06722876941, 0.00000000000, -0.13445753881, 0.00000000000, 0.06722876941]
    rng = np.random.default_rng(9)
    for bps, ch, ns, nfr in ((3, 12, 8192, 5), (4, 3, 1000, 3), (2, 5, 300, 4), (1, 1, 1, 2), (2, 3, 33, 35), (4, 1, 257, 3)):
        raws = oracle.synth_ecg(21, nfr, bps, ch, ns, amplitude=20000 if bps >= 3 else (3000 if bps == 2 else 40))
        p = R.SignalPacker.new_xdelta_hzr(bps, ch, ns, bps, max_batch_frames=nfr)
        # 2nd / 1st order Butterworth low-passes, and the band-pass cut to 3 taps (unstable: the output
        # leaves the int32 range and must turn into 0x80000000 like the reference's x86 conversion)
        filters = ((n5, d5, 2000), ([1.0, -1.1429805, 0.4128016], [0.06745527, 0.13491055, 0.06745527], 50),
                   ([1.0, -0.5095254], [0.2452373, 0.2452373], 0), (n5[:3], d5[:3], 10))
        for nn, dd, init in filters:
            nc = len(nn)
            got = p.prefilter_iir(to_dev(raws), nn, dd, init)
            torch.cuda.synchronize()
            got = got.cpu().numpy().reshape(nfr, -1)
            for i in range(nfr):
                want = oracle.prefilter_iir(raws[i], bps, ch, ns, nn, dd, init, impl)
                assert np.array_equal(got[i], want), ("iir", bps, ch, ns, nc, i)
        for K in (1, 9, 64, 300):
            k = rng.normal(size=K)
            k /= np.abs(k).sum()
            got = p.prefilter_fir(to_dev(raws), k)
            torch.cuda.synchronize()
            got = got.cpu().numpy().reshape(nfr, -1)
            for i in range(nfr):
                assert np.array_equal(got[i], oracle.prefilter_fir(raws[i], bps, ch, ns, k, impl)), ("fir", bps, ch, ns, K, i)
        # filtered frames then go through the packer like any other input
        f = p.prefilter_iir(to_dev(raws), n5, d5, 2000)
        b = p.compress_batch(f)
        assert torch.equal(p.decompress_batch(b), f)
        p.close()


def test_index_rebuilt_on_device_for_cpu_streams(R, oracle):
    """Frames written by the CPU reference carry no decode index: rspt_gpu_build_index rebuilds it by
    self-synchronising parallel decode, and decoding with it equals the CPU decode.  Crafted planes
    stress the token kinds: zero runs far beyond the 16 662 chunk cap, isolated zeros, a lone
    symbol, incompressible bytes (COPY blocks), a ragged tail block."""
    from conftest import has_ref
    impl = "reference" if has_ref() else "port"
    bps, ch, ns, n = 1, 1, 150000, 6   # hzr packer, 1 B/sample: the plane IS the input; 3 blocks, last one ragged
    rng = np.random.default_rng(5)
    raws = np.zeros((n, ns), np.uint8)
    raws[0, [7, 70000, 149999]] = [1, 2, 3]                       # three literals in 150 000 zeros
    raws[1] = rng.integers(0, 256, ns)                            # incompressible
    raws[2] = np.where(rng.random(ns) < 0.03, 0, rng.integers(1, 9, ns))   # dense, isolated zeros
    raws[3] = np.repeat(rng.integers(0, 3, ns // 50), 50)         # runs of 50 of {0,1,2}
    raws[4] = 0
    raws[4, 40000:40010] = 255                                    # FILL blocks next to a sparse one
    raws[5] = (rng.random(ns) < 0.5) * 7                          # two symbols, short runs
    cpu = oracle.make_packer("hzr", bps, ch, ns, 3, impl)
    frames = [cpu.compress(r) for r in raws]
    offs = np.concatenate([[0], np.cumsum([len(f) for f in frames])])
    p = R.SignalPacker.new_hzr(bps, ch, ns, max_batch_frames=n)
    buf = torch.from_numpy(np.frombuffer(b"".join(frames) + bytes(16), np.uint8).copy()).cuda()
    b0 = R.CompressedBatch(buf, torch.tensor(offs, dtype=torch.int64, device="cuda"), None, None, n)
    st = torch.zeros(n, dtype=torch.int32, device="cuda")
    b1 = p.build_index(b0, status=st)
    dec = p.decompress_batch(b1, status=st)
    torch.cuda.synchronize()
    assert not st.cpu().numpy().any()
    assert np.array_equal(dec.cpu().numpy().reshape(n, ns), raws)
    # and through the implicit path (no index given)
    dec2, st2 = p.decompress_stream(b"".join(frames), offs)
    assert not st2.any() and np.array_equal(dec2, raws)
    # the GPU's own stream of the same frames is byte-identical to the CPU's, index or not
    gb = p.compress_batch(to_dev(raws))
    torch.cuda.synchronize()
    assert bytes(gb.stream[: int(gb.offsets[n].item())].cpu().numpy()) == b"".join(frames)


def test_verify_batch_matches_hzr_verify(R, oracle):
    """rspt_gpu_verify_batch = hzr_verify (hzr_decode.c:569-624) on every plane of every frame: clean
    streams from the GPU and from the CPU reference pass; a flipped payload byte fails the CRC of
    that frame only (and the CPU hzr_verify agrees on the damaged plane); broken framing is -4."""
    from conftest import has_ref
    impl = "reference" if has_ref() else "port"
    bps, ch, ns, n = 3, 12, 8192, 6
    raws = oracle.synth_ecg(3, n, bps, ch, ns)
    raws[4] = 0  # FILL blocks
    p = R.SignalPacker.new_xdelta_hzr(bps, ch, ns, 3, max_batch_frames=n)
    batch = p.compress_batch(to_dev(raws))
    st = p.verify_batch(batch)
    torch.cuda.synchronize()
    assert not st.cpu().numpy().any()
    assert p.counters()["crc_failures"] == 0
    # CPU-produced streams
    cpu = oracle.make_packer("xdelta_hzr", bps, ch, ns, 3, impl)
    frames = [bytearray(cpu.compress(r)) for r in raws]
    offs = np.concatenate([[0], np.cumsum([len(f) for f in frames])])

    def run(frs):
        buf = torch.from_numpy(np.frombuffer(b"".join(bytes(f) for f in frs) + bytes(16), np.uint8).copy()).cuda()
        b = R.CompressedBatch(buf, torch.tensor(offs, dtype=torch.int64, device="cuda"), None, None, n)
        s_ = p.verify_batch(b)
        torch.cuda.synchronize()
        return s_.cpu().numpy()

    assert not run(frames).any()
    # flip one byte inside the last block's payload of frame 2, and one in the first HUFF payload of frame 0
    frames[2][len(frames[2]) - 3] ^= 0x40
    frames[0][1 + 8 + 7 + 50] ^= 0x01
    # frame 5: truncate the chunk length field -> malformed framing
    frames[5][1] ^= 0xFF
    st = run(frames)
    assert list(st) == [-6, 0, -6, 0, 0, -4], st
    assert p.counters()["crc_failures"] == 2
    # the CPU's hzr_verify flags the same damaged plane streams
    f0 = bytes(frames[0])
    clen = int.from_bytes(f0[1:5], "little")
    assert oracle.hzr_verify(f0[5:5 + clen], impl) is False
    good = bytes(frames[1])
    clen = int.from_bytes(good[1:5], "little")
    assert oracle.hzr_verify(good[5:5 + clen], impl) is True


def test_corrupt_stream_is_reported_not_silent(R, oracle):
    raws = oracle.synth_ecg(0, 2, 3, 4, 2048)
    cpu = oracle.OraclePacker("xdelta_hzr", 3, 4, 2048, 3)
    frames = [bytearray(cpu.compress(r)) for r in raws]
    frames[1][0] = 9            # bad method byte
    offs = np.concatenate([[0], np.cumsum([len(f) for f in frames])])
    p = R.SignalPacker.new_xdelta_hzr(3, 4, 2048, 3, max_batch_frames=2)
    dec, status = p.decompress_stream(b"".join(bytes(f) for f in frames), offs)
    assert status[0] == 0 and status[1] != 0
    assert dec[0].tobytes() == raws[0].tobytes()


def test_oversized_block_size_field_is_rejected(R, oracle):
    """A block whose 16-bit size field exceeds the block it decodes to (inside a consistently lengthened
    chunk) must come back as a stream error from decompress, index build and verify -- the kernels stage
    payload_len bytes in shared memory sized for the largest LEGITIMATE payload (hzr_encode.c:377-382)."""
    bps, ch, ns = 3, 4, 1000                      # N = 4000: staging is ~4 KB, the forged payload 64 KB
    raws = oracle.synth_ecg(9, 3, bps, ch, ns)
    cpu = oracle.OraclePacker("xdelta_hzr", bps, ch, ns, 3)
    frames = [bytearray(cpu.compress(r)) for r in raws]
    for mode in (0, 1, 2):                        # forged COPY, HUFF and FILL headers
        f = bytearray(frames[1])
        clen = int.from_bytes(f[1:5], "little")
        q = 1 + 4 + 4                             # first block header of plane 0
        plen = int.from_bytes(f[q:q + 2], "little") + 1
        grow = 65536 - plen
        body = f[q + 7:q + 7 + plen] + bytes(grow)
        f2 = f[:1] + (clen + grow).to_bytes(4, "little") + f[5:q] + (0xFFFF).to_bytes(2, "little") + f[q + 2:q + 6] + bytes([mode]) + body + f[q + 7 + plen:]
        fr = [frames[0], f2, frames[2]]
        offs = np.concatenate([[0], np.cumsum([len(x) for x in fr])])
        p = R.SignalPacker.new_xdelta_hzr(bps, ch, ns, 3, max_batch_frames=3)
        blob = b"".join(bytes(x) for x in fr)
        dec, status = p.decompress_stream(blob, offs)
        assert status[0] == 0 and status[1] == -4 and status[2] == 0, (mode, status)
        assert dec[0].tobytes() == raws[0].tobytes() and dec[2].tobytes() == raws[2].tobytes()
        buf = torch.from_numpy(np.frombuffer(blob + bytes(16), np.uint8).copy()).cuda()
        b = R.CompressedBatch(buf, torch.tensor(offs, dtype=torch.int64, device="cuda"), None, None, 3)
        st = p.verify_batch(b)
        torch.cuda.synchronize()
        assert list(st.cpu().numpy()) == [0, -4, 0], (mode, st)
        p.close()


@pytest.mark.parametrize("bps,ch,ns", [(4, 4, 4096), (4, 8, 8192), (3, 4, 8192), (2, 4, 4096)])
def test_hadamard_extreme_sample_values(R, oracle, bps, ch, ns):
    """The fused hadamard kernel rebuilds the 64-bit channel sum (average_32, utils.cpp:30-40) from the
    transform's DC coefficient and the sum of the samples' upper halves: full-range random samples and
    constant frames at the extremes must give the reference's means and stream."""
    rng = np.random.default_rng(5 * ns + bps)
    lo, hi = -(1 << (8 * bps - 1)), (1 << (8 * bps - 1)) - 1
    vals = [rng.integers(lo, hi + 1, size=(ns, ch), dtype=np.int64),
            np.full((ns, ch), lo, np.int64), np.full((ns, ch), hi, np.int64), np.full((ns, ch), -1, np.int64),
            np.where(rng.random((ns, ch)) < 0.5, lo, hi).astype(np.int64),
            rng.integers(lo, lo // 2, size=(ns, ch), dtype=np.int64)]
    raws = np.stack([v.astype("<i4").view(np.uint8).reshape(ns, ch, 4)[:, :, :bps].reshape(-1) for v in vals])
    nfr, fb = len(vals), bps * ch * ns
    p = R.SignalPacker.new_hadamard(bps, ch, ns, max_batch_frames=nfr)
    batch = p.compress_batch(to_dev(raws))
    dec = p.decompress_batch(batch).cpu().numpy().reshape(nfr, fb)
    torch.cuda.synchronize()
    offs = batch.offsets.cpu().numpy()
    stream = batch.stream.cpu().numpy()
    o = oracle.OraclePacker("hadamard", bps, ch, ns)
    for i in range(nfr):
        want = o.compress(raws[i])
        assert stream[offs[i]:offs[i + 1]].tobytes() == want, i
        assert dec[i].tobytes() == o.decompress(want)[0], i


DCT_CASES = [(4, 12, 4096, 4), (3, 3, 4096, 2), (4, 2, 512, 6), (2, 3, 64, 4), (3, 4, 1024, 3), (2, 8, 2048, 2)]
DCT_EQUAL_FRACTION = 0.9999   # stated fraction of quantised coefficients that equal the reference's (DESIGN.md section 6)


def unstencil16(words16):
    """Coefficients mod 2^16 from the post-stencil plane words (signal_packer_dct.cpp:117-119 undone):
    d = prefix-xor(y), x = prefix-sum(d + 128).  Both scans only carry upwards, so they are closed
    under mod 2^16 -- exactly the two byte planes the dct packer keeps."""
    d = np.bitwise_xor.accumulate(words16.astype(np.uint32) & 0xFFFF)
    return (np.cumsum((d + 128) & 0xFFFF, dtype=np.uint64) & 0xFFFF).astype(np.uint32)


def dct_coefficient_diff(oracle_words, planes):
    """Signed difference (GPU - reference) of the quantised coefficients, mod 2^16, from the reference's
    post-stencil words and the GPU's two byte planes of one frame."""
    want = unstencil16(oracle_words.view(np.uint32) & 0xFFFF)
    got = unstencil16(planes[0].astype(np.uint32) | (planes[1].astype(np.uint32) << 8))
    return ((got.astype(np.int64) - want.astype(np.int64) + 0x8000) & 0xFFFF) - 0x8000


@pytest.mark.parametrize("bps,ch,ns,nfr", DCT_CASES)
def test_dct_fast_path_tolerance(R, oracle, bps, ch, ns, nfr):
    """dct, FFT-based FP64 path (signal_packer_dct.cpp:76-100 is an O(n^2) float-product sum): the
    QUANTISED COEFFICIENTS (stencil undone) never differ from the reference's by more than 1 LSB and
    are equal on >= 99.99 % of values; reconstruction PRDN within 0.01 percentage points."""
    raws = oracle.synth_ecg(3, nfr, bps, ch, ns, amplitude=20000 if bps >= 3 else 3000)
    fb = bps * ch * ns
    p = R.SignalPacker.new_dct(bps, ch, ns, max_batch_frames=nfr)
    batch = p.compress_batch(to_dev(raws))
    dec = p.decompress_batch(batch).cpu().numpy().reshape(nfr, fb)
    torch.cuda.synchronize()
    planes, gh = p.debug_planes(to_dev(raws))
    o = oracle.OraclePacker("dct", bps, ch, ns)
    n_all = n_bad = 0
    for i in range(nfr):
        want = o.compress(raws[i])
        wd, _ = o.decompress(want)
        ww, wh = o.transform(raws[i])
        diff = dct_coefficient_diff(ww, planes[i])
        assert np.abs(diff).max() <= 1, (i, int(np.abs(diff).max()))   # the +-1 LSB clause
        n_all += diff.size
        n_bad += int((diff != 0).sum())
        assert np.array_equal(gh[i], wh)                               # the means are integer: exact
        prd_ref = oracle.prdn(raws[i], wd, bps, ch, ns)
        prd_gpu = oracle.prdn(raws[i], dec[i], bps, ch, ns)
        assert abs(prd_ref - prd_gpu) < 0.01, (prd_ref, prd_gpu)
    # the stated fraction; a case smaller than 10 000 coefficients may hold one such coefficient
    assert n_bad <= max(1, int(n_all * (1.0 - DCT_EQUAL_FRACTION))), (n_bad, n_all)


DCT_DIRECT_CASES = [(4, 3, 512), (3, 2, 300), (4, 2, 4096), (1, 3, 2), (1, 2, 3), (1, 4, 5), (1, 3, 77), (3, 2, 77),
                    (1, 2, 1000), (4, 3, 1000), (1, 2, 4095), (3, 2, 4095), (1, 1, 8192), (4, 12, 4096)]


def test_dct_direct_path_bit_exact(R, oracle):
    """dct, O(n^2) path with the reference's float-product / double-accumulate arithmetic: two synthetic ECG
    and two full-range noise frames per shape, lengths 2 to 8192 (powers of two through set_dct_exact).
    Full-range 3- and 4-byte noise decodes to inverse sums outside int32, which the reference converts to
    0x80000000."""
    for bps, ch, ns in DCT_DIRECT_CASES:
        lo, hi = -(1 << (8 * bps - 1)), 1 << (8 * bps - 1)
        noise = [np.random.default_rng(seed).integers(lo, hi, (ns, ch)).astype("<i4").view(np.uint8).reshape(ns, ch, 4)[:, :, :bps]
                 for seed in (1, 2)]
        raws = np.concatenate([oracle.synth_ecg(1, 2, bps, ch, ns, amplitude=100 if bps == 1 else 20000),
                               np.stack([x.reshape(-1) for x in noise])])
        nfr = len(raws)
        p = R.SignalPacker.new_dct(bps, ch, ns, max_batch_frames=nfr)
        p.set_dct_exact(True)
        batch = p.compress_batch(to_dev(raws))
        dec = p.decompress_batch(batch).cpu().numpy().reshape(nfr, -1)
        offs = batch.offsets.cpu().numpy()
        stream = batch.stream.cpu().numpy()
        p.close()
        o = oracle.OraclePacker("dct", bps, ch, ns)
        for i in range(nfr):
            want = o.compress(raws[i])
            assert stream[offs[i]:offs[i + 1]].tobytes() == want, (bps, ch, ns, i)
            wd = np.frombuffer(o.decompress(want)[0], np.uint8)
            n_diff = int((dec[i] != wd).reshape(-1, bps).any(axis=1).sum())
            assert n_diff == 0, (bps, ch, ns, i, f"{n_diff} decoded samples differ")


def test_prdn_kernel(R, oracle):
    raws = oracle.synth_ecg(0, 2, 4, 12, 4096)
    p = R.SignalPacker.new_hadamard(4, 12, 4096, max_batch_frames=2)
    d = to_dev(raws)
    dec = p.decompress_batch(p.compress_batch(d))
    torch.cuda.synchronize()
    got = R.prdn(d, dec, 2, 4, 12, 4096)
    # oracle: same formula over both frames
    o = oracle.OraclePacker("hadamard", 4, 12, 4096)
    both = np.concatenate([np.frombuffer(o.decompress(o.compress(r))[0], np.uint8) for r in raws])
    a = raws.reshape(-1).view("<i4").reshape(2, 4096, 12).astype(np.float64)
    b = both.view("<i4").reshape(2, 4096, 12).astype(np.float64)
    mean = np.floor(a.sum(axis=1, keepdims=True) / 4096)
    want = np.sqrt(((a - b) ** 2).sum() / ((a - mean) ** 2).sum()) * 100
    assert abs(got - want) < 1e-9 * max(1.0, want)


def test_large_batch_round_trip_property(R):
    """BASELINE config 2 shape at a batch big enough to fill the GPU: size-independent checks --
    encode -> decode is the identity, offsets are a strictly increasing scan, CR is sane."""
    bps, ch, ns, nfr = 3, 12, 8192, 2048
    p = R.SignalPacker.new_xdelta_hzr(bps, ch, ns, 3, max_batch_frames=nfr)
    raw = R.synth_ecg(0, nfr, bps, ch, ns)
    batch = p.compress_batch(raw)
    dec = p.decompress_batch(batch)
    torch.cuda.synchronize()
    assert torch.equal(raw, dec)
    offs = batch.offsets.cpu().numpy()
    assert offs[0] == 0 and np.all(np.diff(offs) > 0)
    cr = raw.numel() / offs[-1]
    assert 2.5 < cr < 5.0, cr


@pytest.mark.parametrize("chunk", [1, 3, 64])
def test_host_batch_pipeline_matches_device_batch(R, oracle, chunk, monkeypatch):
    """rspt_gpu_compress_batch_host (chunked H2D / kernels / D2H pipeline) returns the same bytes and
    offsets as the device-resident batch call, for ragged chunk counts; and the host decompress
    call restores the input."""
    monkeypatch.setenv("RSPT_HOST_CHUNK_FRAMES", str(chunk))
    bps, ch, ns, nfr = 3, 12, 2048, 10
    raws = oracle.synth_ecg(5, nfr, bps, ch, ns)
    p = R.SignalPacker.new_xdelta_hzr(bps, ch, ns, 3, max_batch_frames=nfr)
    batch = p.compress_batch(to_dev(raws))
    torch.cuda.synchronize()
    offs = batch.offsets.cpu().numpy().astype(np.uint64)
    stream = batch.stream.cpu().numpy()[: int(offs[nfr])]
    src = torch.from_numpy(raws.reshape(-1).copy()).pin_memory()
    dst = torch.empty(nfr * p.max_compressed_size, dtype=torch.uint8).pin_memory()
    hoff = np.zeros(nfr + 1, np.uint64)
    total = p.compress_batch_host(src.numpy(), dst.numpy(), hoff)
    assert total == int(offs[nfr])
    assert np.array_equal(hoff, offs)
    assert np.array_equal(dst.numpy()[:total], stream)
    out = np.empty(nfr * bps * ch * ns, np.uint8)
    p.decompress_batch_host(dst.numpy()[: total + 16], hoff, out)
    assert np.array_equal(out, raws.reshape(-1))


# ---------------------------------------------------------------------------------------------
# round 2: decode index v2, fused front end, one-pass inverse kernels, C-ABI collective
# ---------------------------------------------------------------------------------------------
def test_decode_index_is_small_and_equivalent_to_a_rebuilt_one(R, oracle):
    """The decode index of a batch: a prefix of the sidecar buffer, about 6 % of the compressed size (one 32-bit
    slot per 64 stream bytes), well under 6 KB per 12 ch x 3 B x 8192 frame; decoding with it, with one rebuilt
    on the device, or with none gives the same samples."""
    bps, ch, ns, n = 3, 12, 8192, 16
    raws = oracle.synth_ecg(100, n, bps, ch, ns)
    p = R.SignalPacker.new_xdelta_hzr(bps, ch, ns, 3, max_batch_frames=n)
    b = p.compress_batch(to_dev(raws))
    torch.cuda.synchronize()
    total = int(b.offsets[n].item())
    used = p.sidecar_used_bytes(n, total)
    assert used / n < 6 * 1024, used / n
    assert used <= b.sidecar.numel()
    d1 = p.decompress_batch(b).cpu().numpy()
    b2 = p.build_index(R.CompressedBatch(b.stream, b.offsets, b.frame_nb, None, n))
    d2 = p.decompress_batch(b2).cpu().numpy()
    d3 = p.decompress_batch(b, use_sidecar=False).cpu().numpy()
    assert np.array_equal(d1, raws.reshape(-1)) and np.array_equal(d2, d1) and np.array_equal(d3, d1)
    # only the used prefix matters: garbage behind it changes nothing
    b.sidecar[used:] = 0xA5
    assert np.array_equal(p.decompress_batch(b).cpu().numpy(), d1)


def test_wrong_decode_index_cannot_leave_its_frame(R, oracle):
    """Entries are range-checked on use: an index that does not belong to the stream (all ones, zeros, noise)
    gives RSPT_E_STREAM or wrong bytes in the frames it covers -- never a fault, never a write outside them.
    The frames behind an intact part of the index stay correct."""
    bps, ch, ns, n = 3, 12, 8192, 6
    raws = oracle.synth_ecg(7, n, bps, ch, ns)
    p = R.SignalPacker.new_xdelta_hzr(bps, ch, ns, 3, max_batch_frames=n)
    b = p.compress_batch(to_dev(raws))
    torch.cuda.synchronize()
    good = b.sidecar.clone()
    offs = b.offsets.cpu().numpy()
    cut = (int(offs[3]) >> 6) * 4 + 3 * 6 * 4          # slots of the frames 0..2 (4 bytes per 64 stream bytes + 1 per block)
    rng = np.random.default_rng(1)
    for fill in ("ones", "zeros", "noise"):
        sc = good.clone()
        if fill == "ones":
            sc[:cut] = 0xFF
        elif fill == "zeros":
            sc[:cut] = 0
        else:
            sc[:cut] = torch.from_numpy(rng.integers(0, 256, cut, dtype=np.uint8)).cuda()
        bb = R.CompressedBatch(b.stream, b.offsets, b.frame_nb, sc, n)
        st = torch.zeros(n, dtype=torch.int32, device="cuda")
        guard = torch.full((n * bps * ch * ns + 4096,), 0x5A, dtype=torch.uint8, device="cuda")
        out = guard[: n * bps * ch * ns]
        p.decompress_batch(bb, out=out, status=st)
        torch.cuda.synchronize()
        assert bool((guard[n * bps * ch * ns:] == 0x5A).all())
        dec = out.cpu().numpy().reshape(n, -1)
        assert np.array_equal(dec[4:], raws[4:].reshape(2, -1)), fill      # frames well behind the damage
    assert np.array_equal(p.decompress_batch(R.CompressedBatch(b.stream, b.offsets, b.frame_nb, good, n)).cpu().numpy(), raws.reshape(-1))


FRONT_CASES = [("xdelta_hzr", 3, 12, 8192, 3), ("xdelta_hzr", 4, 12, 4096, 4), ("hzr", 3, 12, 8192, 0), ("xdelta_hzr", 2, 8, 1024, 2),
               ("xdelta_hzr", 3, 4, 512, 3), ("hzr", 4, 8, 2048, 0), ("xdelta_hzr", 4, 4, 16384, 4)]


@pytest.mark.parametrize("kind,bps,ch,ns,nb", FRONT_CASES)
def test_fused_front_end_streams_are_bit_exact(R, oracle, kind, bps, ch, ns, nb):
    """The compress front end (transform, token histograms, sparse lists) on the shapes of the TMA-fed transform:
    byte-identical streams and an exact round trip for frames that change character half-way (a quiet first
    tile, then dense upper planes: where the density probe sees only zeros, the list overflows and the block
    falls back to the dense scan), all-zero frames and noise."""
    nfr = 6
    rng = np.random.default_rng(ns + ch)
    raws = oracle.synth_ecg(31, nfr, bps, ch, ns, amplitude=20000 if bps >= 3 else 3000)
    fb = bps * ch * ns
    raws[2] = 0
    raws[3] = make_raw(rng, bps, ch, ns, kind="noise")
    quiet_then_wild = raws[4].copy().reshape(ns, ch * bps)
    quiet_then_wild[:600] = 0
    quiet_then_wild[600:] = make_raw(rng, bps, ch, ns, kind="noise").reshape(ns, ch * bps)[600:]
    raws[4] = quiet_then_wild.reshape(-1)
    p = R.SignalPacker(kind, bps, ch, ns, nb or 3, max_batch_frames=nfr)
    batch = p.compress_batch(to_dev(raws))
    torch.cuda.synchronize()
    offs = batch.offsets.cpu().numpy()
    stream = batch.stream.cpu().numpy()
    o = oracle.OraclePacker(kind, bps, ch, ns, nb or 3)
    for i in range(nfr):
        assert stream[offs[i]:offs[i + 1]].tobytes() == o.compress(raws[i]), (kind, i)
    assert np.array_equal(p.decompress_batch(batch).cpu().numpy().reshape(nfr, fb), raws.reshape(nfr, fb))


def test_fused_front_end_hands_oversized_lists_back(R, oracle, monkeypatch):
    """With the list encoder's staging limit lowered, the listed blocks it cannot take are packed by k_hzr_encode
    from the plane, with the per-step leading-zero counts derived from the list: the streams stay byte-identical."""
    monkeypatch.setenv("RSPT_SPARSE_STAGE_BYTES", "300")
    bps, ch, ns, n = 3, 12, 8192, 5
    raws = oracle.synth_ecg(40, n, bps, ch, ns)
    p = R.SignalPacker.new_xdelta_hzr(bps, ch, ns, 3, max_batch_frames=n)
    batch = p.compress_batch(to_dev(raws))
    torch.cuda.synchronize()
    offs = batch.offsets.cpu().numpy()
    stream = batch.stream.cpu().numpy()
    o = oracle.OraclePacker("xdelta_hzr", bps, ch, ns, 3)
    for i in range(n):
        assert stream[offs[i]:offs[i + 1]].tobytes() == o.compress(raws[i]), i


def test_host_decompress_pipeline_small_chunks(R, oracle, monkeypatch):
    """rspt_gpu_decompress_batch_host: chunked H2D / kernels / D2H pipeline over ragged chunk counts."""
    monkeypatch.setenv("RSPT_HOST_CHUNK_FRAMES", "3")
    bps, ch, ns, nfr = 3, 4, 2048, 11
    raws = oracle.synth_ecg(9, nfr, bps, ch, ns)
    cpu = oracle.OraclePacker("xdelta_hzr", bps, ch, ns, 3)
    frames = [cpu.compress(r) for r in raws]
    offs = np.concatenate([[0], np.cumsum([len(f) for f in frames])]).astype(np.uint64)
    blob = np.frombuffer(b"".join(frames) + bytes(64), np.uint8).copy()
    p = R.SignalPacker.new_xdelta_hzr(bps, ch, ns, 3, max_batch_frames=nfr)
    out = np.empty(nfr * bps * ch * ns, np.uint8)
    p.decompress_batch_host(blob, offs, out)
    assert np.array_equal(out, raws.reshape(-1))


@pytest.mark.skipif(torch.cuda.is_available() and torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_c_abi_allgather_places_two_shards():
    """rspt_gpu_comm_* + rspt_gpu_place_offsets_async: two processes, one GPU each, no torch.distributed -- the
    NCCL unique id travels through a file.  Every rank's offsets end up rebased by the totals of the ranks before it."""
    import subprocess
    import sys
    import tempfile
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = (
        "import ctypes as C, os, sys, time, numpy as np, torch\n"
        "sys.path.insert(0, %r)\n"
        "from rspt_b200 import packer as R, _lib\n"
        "rank, path = int(sys.argv[1]), sys.argv[2]\n"
        "torch.cuda.set_device(rank)\n"
        "L = _lib.lib()\n"
        "buf = (C.c_uint8 * 128)()\n"
        "if rank == 0:\n"
        "    _lib.check(L.rspt_gpu_comm_unique_id(buf), None, 'uid')\n"
        "    open(path + '.tmp', 'wb').write(bytes(buf)); os.rename(path + '.tmp', path)\n"
        "else:\n"
        "    while not os.path.exists(path): time.sleep(0.05)\n"
        "    buf = (C.c_uint8 * 128)(*open(path, 'rb').read())\n"
        "comm = C.c_void_p()\n"
        "_lib.check(L.rspt_gpu_comm_init(2, buf, rank, rank, C.byref(comm)), None, 'init')\n"
        "n = 4 + rank\n"
        "p = R.SignalPacker.new_xdelta_hzr(3, 4, 2048, 3, max_batch_frames=n)\n"
        "x = R.synth_ecg(100 * rank, n, 3, 4, 2048)\n"
        "b = p.compress_batch(x)\n"
        "local = b.offsets.clone()\n"
        "p.place_offsets_async(comm, b, rank, 2); p.place_join(); torch.cuda.synchronize()\n"
        "print('RESULT', rank, int(local[n].item()), int(b.offsets[0].item()), int(b.offsets[n].item()))\n"
        "L.rspt_gpu_comm_destroy(comm)\n") % root
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "uid")
        procs = [subprocess.Popen([sys.executable, "-c", code, str(r), path], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
                 for r in range(2)]
        outs = [pr.communicate(timeout=300) for pr in procs]
    res = {}
    for (so, se), pr in zip(outs, procs):
        assert pr.returncode == 0, se[-2000:]
        for ln in so.splitlines():
            if ln.startswith("RESULT"):
                _, r, tot, first, last = ln.split()
                res[int(r)] = (int(tot), int(first), int(last))
    assert res[0][1] == 0 and res[0][2] == res[0][0]
    assert res[1][1] == res[0][0] and res[1][2] == res[0][0] + res[1][0]


def test_create_refuses_shapes_the_tile_kernels_cannot_stage(R):
    """A shape that would only fail at the first compress call (too many channels for the shared-memory tiles) is
    refused by rspt_gpu_create instead (the reference has no such limit, so the refusal has to be visible early)."""
    from rspt_b200._lib import RsptError
    for kind, bps, ch, ns in (("xdelta_hzr", 4, 4000, 64), ("hzr", 4, 4000, 64), ("dct", 4, 4000, 64)):
        with pytest.raises(RsptError):
            R.SignalPacker(kind, bps, ch, ns, 3, max_batch_frames=1)
    p = R.SignalPacker("xdelta_hzr", 2, 300, 64, 2, max_batch_frames=1)   # many channels, still feasible
    x = np.random.default_rng(5).integers(-2000, 2000, size=(64, 300)).astype("<i2")
    y, used = p.decompress(p.compress(x.tobytes()))
    assert y == x.tobytes()
    p.close()
