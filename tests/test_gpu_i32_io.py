"""compress_tensor / decompress_tensor (rspt_gpu_compress_batch_i32 / rspt_gpu_decompress_batch_i32): int32
[n, ch, ns] samples in and out.  The batch must equal what the native entry writes for the same samples, and
for xdelta_hzr, hzr and hadamard what the CPU oracle writes.  Needs a B200."""
import numpy as np
import pytest

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900)]

torch = pytest.importorskip("torch")

E_ARG, E_CAPACITY = -1, -3


@pytest.fixture(scope="module")
def R():
    import rspt_b200  # noqa: F401
    from rspt_b200 import packer
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return packer


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


def words_to_native(w, bps):
    """int32 [n, ch, ns] -> uint8 [n, ns*ch*bps]: the low bps bytes of every word."""
    w = np.ascontiguousarray(np.asarray(w, np.int32).transpose(0, 2, 1))
    n = w.shape[0]
    return w.astype("<i4").view(np.uint8).reshape(*w.shape, 4)[..., :bps].reshape(n, -1).copy()


def make_frames(oracle, rng, bps, ch, ns, nfr):
    """ECG-like (or a random walk for tiny shapes), full-range noise, then ECG again: native uint8 [nfr, fb]."""
    frames = []
    for i in range(nfr):
        if i % 3 == 1:
            lo, hi = -(1 << (8 * bps - 1)), 1 << (8 * bps - 1)
            x = rng.integers(lo, hi, (ns, ch)).astype(np.int32)
            frames.append(x.astype("<i4").view(np.uint8).reshape(ns, ch, 4)[:, :, :bps].reshape(-1))
        elif bps >= 2 and ns >= 64:
            frames.append(oracle.synth_ecg(5 + i, 1, bps, ch, ns, amplitude=20000 if bps >= 3 else 3000)[0])
        else:
            amp = 1 << min(8 * bps - 2, 14)
            x = np.cumsum(rng.integers(-amp // 16 - 1, amp // 16 + 2, (ns, ch)), axis=0)
            x = np.clip(x, -(1 << (8 * bps - 1)), (1 << (8 * bps - 1)) - 1).astype(np.int32)
            frames.append(x.astype("<i4").view(np.uint8).reshape(ns, ch, 4)[:, :, :bps].reshape(-1))
    return np.stack(frames)


def dev_u8(a):
    return torch.from_numpy(np.array(a, dtype=np.uint8, copy=True).reshape(-1)).cuda()


def dev_i32(a):
    return torch.from_numpy(np.array(a, dtype=np.int32, copy=True)).cuda()


def zeroed_output(p, n):
    """An output batch whose decode index starts as zeros: the encoder writes only the entries the stream
    needs, so comparing two indexes byte for byte needs the same background."""
    out = p.alloc_output(n, sidecar=True)
    out.sidecar.zero_()
    return out


def host_batch(p, b):
    torch.cuda.synchronize()
    n = b.n_frames
    offs = b.offsets.cpu().numpy()
    total = int(offs[n])
    sc = None
    if b.sidecar is not None:
        sc = b.sidecar.cpu().numpy()[: p.sidecar_used_bytes(n, total)]
    return offs, b.stream.cpu().numpy()[:total], b.frame_nb.cpu().numpy(), sc


# (kind, bps, ch, ns, nb, frames, dct_exact)
CASES = [
    # TMA- and quad-tiled shapes of the native transform, N % 4 != 0, N % 16 != 0, ns = 1 / 2, > 65536 words
    ("xdelta_hzr", 3, 12, 8192, 3, 3, False), ("xdelta_hzr", 4, 12, 4096, 3, 3, False),
    ("xdelta_hzr", 2, 5, 1000, 2, 3, False), ("xdelta_hzr", 1, 3, 700, 1, 3, False),
    ("xdelta_hzr", 3, 7, 33, 3, 4, False), ("xdelta_hzr", 3, 2, 1, 3, 4, False), ("xdelta_hzr", 4, 3, 2, 3, 3, False),
    ("xdelta_hzr", 4, 2, 70001, 4, 2, False), ("xdelta_hzr", 2, 4, 1000, 2, 3, False), ("xdelta_hzr", 4, 1, 8192, 3, 3, False),
    ("xdelta_hzr", 3, 4, 6, 2, 3, False),
    ("hzr", 3, 12, 8192, 0, 3, False), ("hzr", 1, 2, 999, 0, 3, False), ("hzr", 2, 1, 140000, 0, 2, False),
    ("hzr", 4, 3, 5000, 0, 3, False), ("hzr", 2, 7, 33, 0, 3, False), ("hzr", 1, 4, 1024, 0, 3, False),
    ("hadamard", 4, 12, 4096, 0, 3, False), ("hadamard", 3, 12, 8192, 0, 3, False), ("hadamard", 3, 3, 16384, 0, 2, False),
    ("hadamard", 2, 2, 8, 0, 3, False), ("hadamard", 2, 3, 4096, 0, 3, False), ("hadamard", 1, 4, 4096, 0, 3, False),
    ("hadamard", 4, 1, 8192, 0, 2, False), ("hadamard", 2, 7, 64, 0, 3, False), ("hadamard", 1, 12, 1024, 0, 3, False),
    ("dct", 3, 12, 4096, 0, 3, False), ("dct", 2, 3, 256, 0, 3, False), ("dct", 4, 1, 8192, 0, 2, False),
    ("dct", 1, 4, 64, 0, 3, False), ("dct", 3, 2, 8, 0, 3, False), ("dct", 2, 7, 1024, 0, 3, False),
    ("dct", 3, 3, 1000, 0, 3, True), ("dct", 2, 4, 256, 0, 3, True), ("dct", 4, 2, 77, 0, 3, True),
]


@pytest.mark.parametrize("kind,bps,ch,ns,nb,nfr,exact", CASES)
def test_i32_streams_and_decode(R, oracle, kind, bps, ch, ns, nb, nfr, exact):
    rng = np.random.default_rng(ns * 31 + ch * 7 + bps)
    raws = make_frames(oracle, rng, bps, ch, ns, nfr)
    words = native_to_words(raws, bps, ch, ns, rng)
    assert np.array_equal(words_to_native(words, bps), raws)
    pi = R.SignalPacker(kind, bps, ch, ns, nb or 3, max_batch_frames=nfr)
    pn = R.SignalPacker(kind, bps, ch, ns, nb or 3, max_batch_frames=nfr)
    if exact:
        pi.set_dct_exact(True)
        pn.set_dct_exact(True)
    x = dev_i32(words)
    bi = pi.compress_tensor(x, out=zeroed_output(pi, nfr))
    bn = pn.compress_batch(dev_u8(raws), out=zeroed_output(pn, nfr))
    gi, gn = host_batch(pi, bi), host_batch(pn, bn)
    offs, stream, fnb, sc = gi
    assert np.array_equal(offs, gn[0]) and np.array_equal(stream, gn[1]), kind
    assert np.array_equal(fnb, gn[2]) and np.array_equal(sc, gn[3])
    assert torch.equal(x, dev_i32(words)), "the input tensor was modified"
    ci, cn = pi.counters(), pn.counters()
    for k in ("frames_compressed", "raw_bytes_in", "compressed_bytes_out", "escalations"):
        assert ci[k] == cn[k], k
    assert pi.nb == pn.nb
    lossless = kind in ("xdelta_hzr", "hzr")
    if kind != "dct":
        o = oracle.OraclePacker(kind, bps, ch, ns, nb or 3)
        ofr, want_nb, want_o = [], [], []
        for i in range(nfr):
            ofr.append(o.compress(raws[i]))
            assert stream[offs[i]:offs[i + 1]].tobytes() == ofr[-1], (kind, i)
            want_nb.append(o.nb)
            want_o.append(np.frombuffer(o.decompress(ofr[-1])[0], np.uint8))
        assert fnb.tolist() == want_nb
        # streams written by the CPU oracle (no decode index)
        buf = torch.from_numpy(np.frombuffer(b"".join(ofr) + bytes(16), np.uint8).copy()).cuda()
        ooff = torch.tensor(np.concatenate([[0], np.cumsum([len(f) for f in ofr])]), dtype=torch.int64, device="cuda")
        ob = R.CompressedBatch(buf, ooff, torch.tensor(want_nb, dtype=torch.uint8, device="cuda"), None, nfr)
        status = torch.full((nfr,), 7, dtype=torch.int32, device="cuda")
        got = pi.decompress_tensor(ob, status=status, use_sidecar=False)
        torch.cuda.synchronize()
        assert not status.cpu().numpy().any()
        assert np.array_equal(got.cpu().numpy(), native_to_words(np.stack(want_o), bps, ch, ns))
    for use_sc in (True, False):
        status = torch.full((nfr,), 7, dtype=torch.int32, device="cuda")
        dec_w = pi.decompress_tensor(bi, status=status, use_sidecar=use_sc)
        dec_n = pn.decompress_batch(bn, use_sidecar=use_sc)
        torch.cuda.synchronize()
        assert not status.cpu().numpy().any()
        assert dec_w.shape == (nfr, ch, ns) and dec_w.dtype == torch.int32
        got = dec_w.cpu().numpy()
        assert np.array_equal(got, native_to_words(dec_n.cpu().numpy(), bps, ch, ns)), (kind, use_sc)
        if lossless:
            assert np.array_equal(got, sext(words, bps))


def test_i32_unaligned_views(R, oracle):
    """Tensors that start 4 bytes into their storage take the scalar / unaligned paths and give the same bytes."""
    for kind, bps, ch, ns in (("xdelta_hzr", 3, 12, 8192), ("hzr", 2, 4, 1024), ("hadamard", 4, 4, 4096),
                              ("hadamard", 2, 12, 4096), ("dct", 3, 4, 1024)):
        nfr = 3
        rng = np.random.default_rng(ch * ns + bps)
        raws = make_frames(oracle, rng, bps, ch, ns, nfr)
        words = native_to_words(raws, bps, ch, ns, rng)
        buf = torch.zeros(words.size + 1, dtype=torch.int32, device="cuda")
        xu = buf[1:].view(nfr, ch, ns)
        xu.copy_(dev_i32(words))
        assert xu.data_ptr() % 16 == 4
        pa = R.SignalPacker(kind, bps, ch, ns, 3, max_batch_frames=nfr)
        pb = R.SignalPacker(kind, bps, ch, ns, 3, max_batch_frames=nfr)
        ba = pa.compress_tensor(dev_i32(words), out=zeroed_output(pa, nfr))
        bu = pb.compress_tensor(xu, out=zeroed_output(pb, nfr))
        ga, gu = host_batch(pa, ba), host_batch(pb, bu)
        for a, u in zip(ga, gu):
            assert np.array_equal(a, u), kind
        obuf = torch.full((words.size + 1,), 12345, dtype=torch.int32, device="cuda")
        outu = obuf[1:].view(nfr, ch, ns)
        pa.decompress_tensor(ba, out=outu)
        want = pa.decompress_tensor(ba)
        torch.cuda.synchronize()
        assert torch.equal(outu, want), kind
        assert int(obuf[0].item()) == 12345
        if kind in ("xdelta_hzr", "hzr"):
            assert np.array_equal(want.cpu().numpy(), sext(words, bps))


def test_i32_escalation_alternating_entry_points(R, oracle):
    """nb < bps: the sticky plane count carries across batches whichever entry point compressed them (the
    flat-order ramps of test_xdelta_plane_escalation: 1, then 2, 3 and 4 planes)."""
    rng = np.random.default_rng(3)
    bps, ch, ns = 4, 3, 500

    def ramp(maxinc, jump_at=None, jump=0):
        inc = rng.integers(0, maxinc + 1, ch * ns).astype(np.int64)
        if jump_at is not None:
            inc[jump_at] += jump
        x = np.cumsum(inc).reshape(ch, ns).T.astype(np.int32)
        return np.ascontiguousarray(x).astype("<i4").view(np.uint8).reshape(-1)

    raws = np.stack([ramp(200), ramp(200), ramp(200, 700, 20000), ramp(200), ramp(200, 5, 3000000), ramp(100),
                     ramp(200, 1499, 1 << 29), ramp(50)])
    o = oracle.OraclePacker("xdelta_hzr", bps, ch, ns, 1)
    want, want_nb = [], []
    for r in raws:
        want.append(o.compress(r))
        want_nb.append(o.nb)
    assert want_nb == [1, 1, 2, 2, 3, 3, 4, 4], want_nb
    p = R.SignalPacker.new_xdelta_hzr(bps, ch, ns, 1, max_batch_frames=8)
    got_nb = []
    for j, (lo, hi) in enumerate(((0, 2), (2, 3), (3, 5), (5, 7), (7, 8))):
        words = native_to_words(raws[lo:hi], bps, ch, ns)
        b = p.compress_tensor(dev_i32(words)) if j % 2 == 0 else p.compress_batch(dev_u8(raws[lo:hi]))
        offs, stream, fnb, _ = host_batch(p, b)
        for i in range(hi - lo):
            assert stream[offs[i]:offs[i + 1]].tobytes() == want[lo + i], (lo, i)
        got_nb += fnb.tolist()
        dec = p.decompress_tensor(b)
        torch.cuda.synchronize()
        assert np.array_equal(dec.cpu().numpy(), words)
    assert got_nb == want_nb
    assert p.nb == o.nb == 4 and p.counters()["escalations"] == o.escalations == 3


def test_i32_round_trip_at_scale(R):
    """4096 frames of 3 B x 12 x 8192 generated on the device: same batch as the native entry, exact round trip."""
    bps, ch, ns, n = 3, 12, 8192, 4096
    raw = R.synth_ecg(0, n, bps, ch, ns)
    b = raw.view(n, ns, ch, bps)
    x = (b[..., 0].to(torch.int32) | (b[..., 1].to(torch.int32) << 8) | (b[..., 2].view(torch.int8).to(torch.int32) << 16))
    x = x.permute(0, 2, 1).contiguous()
    del b
    p = R.SignalPacker.new_xdelta_hzr(bps, ch, ns, 3, max_batch_frames=n)
    bi = p.compress_tensor(x, sidecar=True)
    pn = R.SignalPacker.new_xdelta_hzr(bps, ch, ns, 3, max_batch_frames=n)
    bn = pn.compress_batch(raw, sidecar=False)
    torch.cuda.synchronize()
    total = int(bi.offsets[-1].item())
    assert torch.equal(bi.offsets, bn.offsets)
    assert torch.equal(bi.stream[:total], bn.stream[:total])
    del bn, raw
    dec = p.decompress_tensor(bi)
    torch.cuda.synchronize()
    assert torch.equal(dec, x)
    c = p.counters()
    assert c["frames_compressed"] == n and c["raw_bytes_in"] == n * bps * ch * ns


def test_i32_refusals(R):
    bps, ch, ns, n = 3, 4, 256, 2
    p = R.SignalPacker.new_xdelta_hzr(bps, ch, ns, 3, max_batch_frames=n)
    x = torch.zeros((n, ch, ns), dtype=torch.int32, device="cuda")
    for bad in (x.to(torch.int64), x.to(torch.int16), x.view(n, ns, ch), x.view(n * ch, ns), x.reshape(n, ch, ns, 1),
                x.cpu(), x.transpose(1, 2).contiguous().transpose(1, 2), torch.zeros((n, ch, ns + 1), dtype=torch.int32, device="cuda"),
                x.view(torch.uint8).view(n, ch, ns * 4)[:, :, : ns].contiguous(), x.numpy(force=True)):
        with pytest.raises(ValueError):
            p.compress_tensor(bad)
    b = p.compress_tensor(x)
    for bad in (torch.empty((n, ch, ns), dtype=torch.float32, device="cuda"), torch.empty((n + 1, ch, ns), dtype=torch.int32, device="cuda"),
                torch.empty((n, ch, ns), dtype=torch.int32), torch.empty((n, ns, ch), dtype=torch.int32, device="cuda").transpose(1, 2)):
        with pytest.raises(ValueError):
            p.decompress_tensor(b, out=bad)
    if torch.cuda.device_count() > 1:
        with pytest.raises(ValueError):
            p.compress_tensor(x.to("cuda:1"))

    L, h = p.L, p.h
    out = p.alloc_output(n + 1)
    cap = out.stream.numel()
    args = (out.stream.data_ptr(), cap, out.offsets.data_ptr(), out.frame_nb.data_ptr(), None)
    assert L.rspt_gpu_compress_batch_i32(None, x.data_ptr(), n, *args) == E_ARG
    assert L.rspt_gpu_compress_batch_i32(h, None, n, *args) == E_ARG
    assert L.rspt_gpu_compress_batch_i32(h, x.data_ptr() + 2, n, *args) == E_ARG
    assert L.rspt_gpu_compress_batch_i32(h, x.data_ptr(), n, None, cap, out.offsets.data_ptr(), None, None) == E_ARG
    assert L.rspt_gpu_compress_batch_i32(h, x.data_ptr(), n, out.stream.data_ptr(), cap, None, None, None) == E_ARG
    big = torch.zeros((n + 1, ch, ns), dtype=torch.int32, device="cuda")
    assert L.rspt_gpu_compress_batch_i32(h, big.data_ptr(), n + 1, *args) == E_CAPACITY
    assert L.rspt_gpu_compress_batch_i32(h, x.data_ptr(), n, out.stream.data_ptr(), n * p.max_compressed_size - 1,
                                         out.offsets.data_ptr(), None, None) == E_CAPACITY
    assert L.rspt_gpu_compress_batch_i32(h, x.data_ptr(), 0, *args) == 0
    dst = torch.zeros((n, ch, ns), dtype=torch.int32, device="cuda")
    dargs = (b.stream.data_ptr(), b.offsets.data_ptr())
    assert L.rspt_gpu_decompress_batch_i32(h, *dargs, n, None, None, None, None) == E_ARG
    assert L.rspt_gpu_decompress_batch_i32(h, *dargs, n, None, None, dst.data_ptr() + 2, None) == E_ARG
    assert L.rspt_gpu_decompress_batch_i32(h, None, b.offsets.data_ptr(), n, None, None, dst.data_ptr(), None) == E_ARG
    assert L.rspt_gpu_decompress_batch_i32(h, b.stream.data_ptr(), None, n, None, None, dst.data_ptr(), None) == E_ARG
    assert L.rspt_gpu_decompress_batch_i32(None, *dargs, n, None, None, dst.data_ptr(), None) == E_ARG
    assert L.rspt_gpu_decompress_batch_i32(h, *dargs, n + 1, None, None, big.data_ptr(), None) == E_CAPACITY
    # a 4-byte offset is accepted: 16-byte alignment is only a fast-path condition
    xs = torch.zeros(n * ch * ns + 1, dtype=torch.int32, device="cuda")
    assert L.rspt_gpu_compress_batch_i32(h, xs.data_ptr() + 4, n, *args) == 0
    assert L.rspt_gpu_decompress_batch_i32(h, out.stream.data_ptr(), out.offsets.data_ptr(), n, out.frame_nb.data_ptr(), None,
                                           xs.data_ptr() + 4, None) == 0
    torch.cuda.synchronize()
    assert not xs[1:].any()
