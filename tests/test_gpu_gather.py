"""decompress_frames / decompress_frames_tensor (rspt_gpu_decompress_frames / _i32): any list of frames of a stored
batch, decoded by a handle whose max_batch_frames is smaller than the stored batch.  Every slot must equal the
matching row of the whole batch's decode, with the stored decode index and without one.  Needs a B200."""
import numpy as np
import pytest

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900)]

torch = pytest.importorskip("torch")

E_ARG, E_CAPACITY, E_STREAM = -1, -3, -4
N_STORED, MAX_BATCH = 40, 8


@pytest.fixture(scope="module")
def R():
    import rspt_b200  # noqa: F401
    from rspt_b200 import packer
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return packer


def make_frames(oracle, rng, bps, ch, ns, nfr, escalate=False):
    """uint8 [nfr, frame_bytes]: all-zero frames (FILL blocks), noise (COPY blocks) and ECG-like frames.  With
    `escalate` the noise gets one bit wider every other frame, so that an xdelta_hzr handle with nb < bps
    escalates in the middle of the batch."""
    lo, hi = -(1 << (8 * bps - 1)), 1 << (8 * bps - 1)
    frames = []
    for i in range(nfr):
        if i % 5 == 0:
            x = np.zeros((ns, ch), np.int32)
        elif i % 5 == 2:
            r = 1 << (min(8 * bps, 6 + i // 2) - 1) if escalate else hi
            x = rng.integers(-r, r, (ns, ch)).astype(np.int32)
        elif bps >= 2 and ns >= 64:
            frames.append(oracle.synth_ecg(5 + i, 1, bps, ch, ns, amplitude=20000 if bps >= 3 else 3000)[0])
            continue
        else:
            amp = 1 << min(8 * bps - 2, 14)
            x = np.cumsum(rng.integers(-amp // 16 - 1, amp // 16 + 2, (ns, ch)), axis=0)
            x = np.clip(x, lo, hi - 1).astype(np.int32)
        frames.append(x.astype("<i4").view(np.uint8).reshape(ns, ch, 4)[:, :, :bps].reshape(-1))
    return np.stack(frames)


def dev_u8(a):
    return torch.from_numpy(np.array(a, dtype=np.uint8, copy=True).reshape(-1)).cuda()


def id_lists(n, offsets, rng):
    """The id lists every case decodes, each at most MAX_BATCH long."""
    chunks = lambda ids: [ids[i:i + MAX_BATCH] for i in range(0, len(ids), MAX_BATCH)]
    lists = chunks(list(range(n))) + chunks(list(range(n - 1, -1, -1)))
    lists += chunks(rng.integers(0, n, 3 * MAX_BATCH).tolist())
    lists += [[0], [n - 1]]
    lo = next(i for i in range(1, n) if offsets[i] % 64)
    lists.append(list(range(lo, min(n, lo + MAX_BATCH))))
    return lists


def planes_alloc(kind, bps, nb):
    return (bps if nb < bps else nb) if kind == "xdelta_hzr" else {"hzr": 4, "hadamard": 3, "dct": 2}[kind]


class Stored:
    """A stored batch of N_STORED frames and its whole decode (native and int32), from a handle that holds all."""

    def __init__(self, R, oracle, kind, bps, ch, ns, nb, exact=False, escalate=False):
        self.kind, self.bps, self.ch, self.ns, self.nb, self.exact = kind, bps, ch, ns, nb, exact
        rng = np.random.default_rng(ns * 31 + ch * 7 + bps)
        self.raw = make_frames(oracle, rng, bps, ch, ns, N_STORED, escalate)
        self.pc = self.handle(R, N_STORED)
        self.batch = self.pc.compress_batch(dev_u8(self.raw))
        self.full = self.pc.decompress_batch(self.batch).view(N_STORED, -1)
        self.full_w = self.pc.decompress_tensor(self.batch)
        torch.cuda.synchronize()
        self.offsets = self.batch.offsets.cpu().numpy()
        self.counters = self.pc.counters()

    def handle(self, R, max_batch):
        p = R.SignalPacker(self.kind, self.bps, self.ch, self.ns, self.nb, max_batch_frames=max_batch)
        if self.exact:
            p.set_dct_exact(True)
        return p


# (kind, bps, ch, ns, nb, dct_exact, escalate, expect COPY blocks, expect FILL blocks)
CASES = [
    ("xdelta_hzr", 3, 12, 8192, 3, False, False, True, True),   # two blocks per plane
    ("xdelta_hzr", 4, 3, 5000, 1, False, True, True, False),    # frame_nb 1, 2, 3, 4 across the batch
    ("hzr", 2, 1, 140000, 4, False, False, True, True),
    ("hadamard", 4, 12, 4096, 3, False, False, True, True),
    ("hadamard", 3, 3, 16384, 3, False, False, True, True),
    ("dct", 3, 12, 4096, 2, False, False, False, False),        # fast path
    ("dct", 4, 2, 77, 2, True, False, False, False),            # exact path
]


@pytest.mark.parametrize("kind,bps,ch,ns,nb,exact,escalate,copy,fill", CASES)
def test_gather_equals_full_decode(R, oracle, kind, bps, ch, ns, nb, exact, escalate, copy, fill):
    st = Stored(R, oracle, kind, bps, ch, ns, nb, exact, escalate)
    if copy:
        assert st.counters["blocks_copy"] > 0
    if fill:
        assert st.counters["blocks_fill"] > 0
    if escalate:
        assert len(set(st.batch.frame_nb.cpu().tolist())) > 1
    pd = st.handle(R, MAX_BATCH)
    rng = np.random.default_rng(7)
    for ids in id_lists(N_STORED, st.offsets, rng):
        want = st.full[torch.tensor(ids, device="cuda")]
        want_w = st.full_w[torch.tensor(ids, device="cuda")]
        for use_sc in (True, False):
            status = torch.full((len(ids),), 7, dtype=torch.int32, device="cuda")
            got = pd.decompress_frames(st.batch, torch.tensor(ids, dtype=torch.int64, device="cuda"), status=status, use_sidecar=use_sc)
            status_w = torch.full((len(ids),), 7, dtype=torch.int32, device="cuda")
            got_w = pd.decompress_frames_tensor(st.batch, ids, status=status_w, use_sidecar=use_sc)
            torch.cuda.synchronize()
            assert not status.any() and not status_w.any(), (ids, use_sc, status.tolist(), status_w.tolist())
            assert got.shape == (len(ids) * pd.frame_bytes,) and got.dtype == torch.uint8
            assert got_w.shape == (len(ids), ch, ns) and got_w.dtype == torch.int32
            assert torch.equal(got.view(len(ids), -1), want), (ids, use_sc)
            assert torch.equal(got_w, want_w), (ids, use_sc)


@pytest.mark.parametrize("kind,bps,ch,ns,nb", [("xdelta_hzr", 3, 12, 8192, 3), ("hadamard", 4, 12, 4096, 3)])
def test_gather_cpu_written_streams(R, oracle, kind, bps, ch, ns, nb):
    """Frames written by the CPU packer carry no decode index: a gather indexes the selected frames on the device."""
    rng = np.random.default_rng(11)
    raw = make_frames(oracle, rng, bps, ch, ns, 24)
    o = oracle.OraclePacker(kind, bps, ch, ns, nb)
    frames, fnb, want = [], [], []
    for r in raw:
        frames.append(o.compress(r))
        fnb.append(o.nb)
        want.append(np.frombuffer(o.decompress(frames[-1])[0], np.uint8))
    want = np.stack(want)
    buf = torch.from_numpy(np.frombuffer(b"".join(frames) + bytes(16), np.uint8).copy()).cuda()
    off = torch.tensor(np.concatenate([[0], np.cumsum([len(f) for f in frames])]), dtype=torch.int64, device="cuda")
    b = R.CompressedBatch(buf, off, torch.tensor(fnb, dtype=torch.uint8, device="cuda"), None, len(frames))
    p = R.SignalPacker(kind, bps, ch, ns, nb, max_batch_frames=MAX_BATCH)
    for ids in ([23, 0, 5, 5, 17, 2, 11, 9], [3], list(range(13, 21))):
        status = torch.full((len(ids),), 7, dtype=torch.int32, device="cuda")
        got = p.decompress_frames(b, ids, status=status)
        torch.cuda.synchronize()
        assert not status.any()
        assert np.array_equal(got.cpu().numpy().reshape(len(ids), -1), want[ids]), ids


def test_gather_bad_ids(R, oracle):
    st = Stored(R, oracle, "xdelta_hzr", 3, 12, 8192, 3)
    pd = st.handle(R, MAX_BATCH)
    ids = [3, -1, 39, N_STORED, 0, 2 ** 40, 7, 3]
    bad = [1, 3, 5]
    for use_sc in (True, False):
        status = torch.full((len(ids),), 7, dtype=torch.int32, device="cuda")
        got = pd.decompress_frames(st.batch, ids, status=status, use_sidecar=use_sc).view(len(ids), -1)
        status_w = torch.full((len(ids),), 7, dtype=torch.int32, device="cuda")
        got_w = pd.decompress_frames_tensor(st.batch, ids, status=status_w, use_sidecar=use_sc)
        torch.cuda.synchronize()
        for j, g in enumerate(ids):
            if j in bad:
                assert int(status[j]) == E_ARG and int(status_w[j]) == E_ARG, (j, use_sc)
            else:
                assert int(status[j]) == 0 and int(status_w[j]) == 0, (j, use_sc)
                assert torch.equal(got[j], st.full[g]) and torch.equal(got_w[j], st.full_w[g]), (j, use_sc)


def test_gather_corrupted_frame(R, oracle):
    """A stored frame whose framing is broken costs only the slots that name it."""
    st = Stored(R, oracle, "xdelta_hzr", 3, 12, 8192, 3)
    pd = st.handle(R, MAX_BATCH)
    k = 13
    stream = st.batch.stream.clone()
    stream[int(st.offsets[k]) + 1:int(st.offsets[k]) + 5] = 0xFF   # first chunk length: far beyond the frame
    b = R.CompressedBatch(stream, st.batch.offsets, st.batch.frame_nb, st.batch.sidecar, N_STORED)
    ids = [12, 13, 14, 13, 0, 39, 13, 1]
    for use_sc in (True, False):
        status = torch.full((len(ids),), 7, dtype=torch.int32, device="cuda")
        got = pd.decompress_frames(b, ids, status=status, use_sidecar=use_sc).view(len(ids), -1)
        torch.cuda.synchronize()
        for j, g in enumerate(ids):
            if g == k:
                assert int(status[j]) == E_STREAM, (j, use_sc)
            else:
                assert int(status[j]) == 0 and torch.equal(got[j], st.full[g]), (j, use_sc)


def test_gather_garbage_index_entries(R, oracle):
    """Random words over one frame's part of the stored decode index affect only the slots that name that frame."""
    kind, bps, ch, ns, nb = "xdelta_hzr", 3, 12, 8192, 3
    st = Stored(R, oracle, kind, bps, ch, ns, nb)
    pd = st.handle(R, MAX_BATCH)
    k = 21
    per_frame = planes_alloc(kind, bps, nb) * ((ch * ns + 65535) // 65536)
    # frame k's entries lie in words [(offsets[k] >> 6) + k * blocks per frame, (offsets[k + 1] >> 6) + (k + 1) * blocks per frame)
    w0 = (int(st.offsets[k]) >> 6) + k * per_frame
    w1 = (int(st.offsets[k + 1]) >> 6) + (k + 1) * per_frame
    sc = st.batch.sidecar.clone()
    words = sc.view(torch.int32)
    words[w0:w1] = torch.from_numpy(np.random.default_rng(5).integers(-2 ** 31, 2 ** 31, w1 - w0, dtype=np.int64).astype(np.int32)).cuda()
    b = R.CompressedBatch(st.batch.stream, st.batch.offsets, st.batch.frame_nb, sc, N_STORED)
    ids = [20, 21, 22, 21, 0, 39, 21, 5]
    status = torch.full((len(ids),), 7, dtype=torch.int32, device="cuda")
    got = pd.decompress_frames(b, ids, status=status).view(len(ids), -1)
    torch.cuda.synchronize()
    hit = 0
    for j, g in enumerate(ids):
        if g == k:
            hit += int(status[j]) == E_STREAM or not torch.equal(got[j], st.full[g])
        else:
            assert int(status[j]) == 0 and torch.equal(got[j], st.full[g]), j
    assert hit == 3, "the garbage entries were not used"


def test_gather_refusals_and_counters(R, oracle):
    st = Stored(R, oracle, "hadamard", 4, 12, 4096, 3)
    pd = st.handle(R, MAX_BATCH)
    ids = torch.arange(MAX_BATCH, dtype=torch.int64, device="cuda")
    for bad in (ids.to(torch.int32), ids.cpu(), ids.numpy(force=True), ids.view(2, -1), ids[::2], 3, "0,1", None):
        with pytest.raises(ValueError):
            pd.decompress_frames(st.batch, bad)
        with pytest.raises(ValueError):
            pd.decompress_frames_tensor(st.batch, bad)
    if torch.cuda.device_count() > 1:
        with pytest.raises(ValueError):
            pd.decompress_frames(st.batch, ids.to("cuda:1"))
    with pytest.raises(ValueError):
        pd.decompress_frames_tensor(st.batch, ids, out=torch.empty((MAX_BATCH, 12, 4095), dtype=torch.int32, device="cuda"))

    c0 = pd.counters()["frames_decompressed"]
    pd.decompress_frames(st.batch, [5, 5, 9])
    pd.decompress_frames_tensor(st.batch, ids, use_sidecar=False)
    assert pd.counters()["frames_decompressed"] == c0 + 3 + MAX_BATCH

    L, h, b = pd.L, pd.h, st.batch
    dst = torch.zeros((MAX_BATCH + 1) * pd.frame_bytes, dtype=torch.uint8, device="cuda")
    dst_w = torch.zeros((MAX_BATCH + 1) * 12 * 4096 + 1, dtype=torch.int32, device="cuda")
    many = torch.zeros(MAX_BATCH + 1, dtype=torch.int64, device="cuda")
    src, off, fnb, sc = b.stream.data_ptr(), b.offsets.data_ptr(), b.frame_nb.data_ptr(), b.sidecar.data_ptr()
    for fn, d in ((L.rspt_gpu_decompress_frames, dst.data_ptr()), (L.rspt_gpu_decompress_frames_i32, dst_w.data_ptr())):
        assert fn(h, src, off, N_STORED, fnb, sc, many.data_ptr(), MAX_BATCH + 1, d, None) == E_CAPACITY
        assert fn(None, src, off, N_STORED, fnb, sc, ids.data_ptr(), MAX_BATCH, d, None) == E_ARG
        assert fn(h, None, off, N_STORED, fnb, sc, ids.data_ptr(), MAX_BATCH, d, None) == E_ARG
        assert fn(h, src, None, N_STORED, fnb, sc, ids.data_ptr(), MAX_BATCH, d, None) == E_ARG
        assert fn(h, src, off, N_STORED, fnb, sc, None, MAX_BATCH, d, None) == E_ARG
        assert fn(h, src, off, N_STORED, fnb, sc, ids.data_ptr(), MAX_BATCH, None, None) == E_ARG
        # more stored blocks than 32-bit ordinals can number
        assert fn(h, src, off, 1 << 32, fnb, sc, ids.data_ptr(), MAX_BATCH, d, None) == E_ARG
        assert fn(h, src, off, N_STORED, fnb, sc, ids.data_ptr(), 0, d, None) == 0
    assert L.rspt_gpu_decompress_frames_i32(h, src, off, N_STORED, fnb, sc, ids.data_ptr(), MAX_BATCH, dst_w.data_ptr() + 2, None) == E_ARG
    # a 4-byte offset is accepted, as for decompress_batch_i32
    assert L.rspt_gpu_decompress_frames_i32(h, src, off, N_STORED, fnb, sc, ids.data_ptr(), MAX_BATCH, dst_w.data_ptr() + 4, None) == 0
    torch.cuda.synchronize()
    assert torch.equal(dst_w[1:1 + MAX_BATCH * 12 * 4096].view(MAX_BATCH, 12, 4096), st.full_w[:MAX_BATCH])
    assert pd.counters()["frames_decompressed"] == c0 + 3 + 2 * MAX_BATCH


def test_gather_at_scale(R):
    """4096 random ids (with repeats) from a 4096-frame batch of 3 B x 12 x 8192 equal the whole batch's decode."""
    bps, ch, ns, n = 3, 12, 8192, 4096
    raw = R.synth_ecg(0, n, bps, ch, ns)
    p = R.SignalPacker.new_xdelta_hzr(bps, ch, ns, 3, max_batch_frames=n)
    b = p.compress_batch(raw)
    ids = torch.from_numpy(np.random.default_rng(3).integers(0, n, n)).cuda()
    status = torch.full((n,), 7, dtype=torch.int32, device="cuda")
    got = p.decompress_frames(b, ids, status=status)
    torch.cuda.synchronize()
    assert not status.any()
    assert torch.equal(got.view(n, -1), raw.view(n, -1)[ids])
    del got
    got = p.decompress_frames(b, ids, status=status, use_sidecar=False)
    torch.cuda.synchronize()
    assert not status.any()
    assert torch.equal(got.view(n, -1), raw.view(n, -1)[ids])
