"""Stores: stored batches grown by appends past max_batch_frames (SignalPacker.new_store / append_batch / append_tensor,
rspt_gpu_compress_append(_i32)), and decode indexes built over any list of stored frames (index_frames / index_all,
rspt_gpu_build_index_frames).  A store appended batch by batch must equal, byte for byte, one compress_batch over all
its frames on a fresh handle of the same arguments.  Needs a B200."""
import numpy as np
import pytest

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(1800)]

torch = pytest.importorskip("torch")

E_ARG, E_CAPACITY, E_STREAM = -1, -3, -4
N, MAX_BATCH = 40, 8
APPENDS = [1, 7, 3, 8, 5, 8, 2, 6]   # uneven: most appends start at a byte base that is not a multiple of 64
assert sum(APPENDS) == N and max(APPENDS) <= MAX_BATCH

# (kind, bps, ch, ns, nb, dct_exact, escalate): the shapes of the gather tests
CASES = [
    ("xdelta_hzr", 3, 12, 8192, 3, False, False),
    ("xdelta_hzr", 4, 3, 5000, 1, False, True),
    ("hzr", 2, 1, 140000, 4, False, False),
    ("hadamard", 4, 12, 4096, 3, False, False),
    ("hadamard", 3, 3, 16384, 3, False, False),
    ("dct", 3, 12, 4096, 2, False, False),   # fast path
    ("dct", 4, 2, 77, 2, True, False),       # exact path
]


@pytest.fixture(scope="module")
def R():
    import rspt_b200  # noqa: F401
    from rspt_b200 import packer
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return packer


def make_frames(oracle, rng, bps, ch, ns, nfr, escalate=False):
    """uint8 [nfr, frame_bytes]: all-zero frames (FILL blocks), noise (COPY blocks) and ECG-like frames.  With
    `escalate` the noise gets wider frame by frame, so that an xdelta_hzr handle with nb < bps escalates late."""
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


def to_words(frames_u8, bps, ch, ns):
    """Native frames [n, ns, ch, bps] as the int32 tensor [n, ch, ns] compress_tensor takes (the low bps bytes)."""
    b = frames_u8.view(-1, ns, ch, bps).to(torch.int32)
    w = sum(b[..., i] << (8 * i) for i in range(bps))
    return w.transpose(1, 2).contiguous()


def handle(R, kind, bps, ch, ns, nb, exact, max_batch):
    p = R.SignalPacker(kind, bps, ch, ns, nb, max_batch_frames=max_batch)
    if exact:
        p.set_dct_exact(True)
    return p


def one_shot(R, kind, bps, ch, ns, nb, exact, frames):
    """One compress_batch over all frames on a fresh handle that holds them all, sidecar zero-filled beforehand."""
    n = frames.numel() // (bps * ch * ns)
    p = handle(R, kind, bps, ch, ns, nb, exact, n)
    out = p.alloc_output(n)
    out.sidecar.zero_()
    p.compress_batch(frames, out=out)
    torch.cuda.synchronize()
    return p, out


def append_all(p, store, frames, sizes, bps, ch, ns, layouts="mixed"):
    """Append the frames in pieces of `sizes`, alternating native and int32 input; the handle's nb after each."""
    fb = bps * ch * ns
    nbs, a = [], 0
    for j, k in enumerate(sizes):
        piece = frames[a * fb:(a + k) * fb]
        if layouts == "mixed" and j % 2:
            p.append_tensor(store, to_words(piece, bps, ch, ns))
        else:
            p.append_batch(store, piece)
        a += k
        nbs.append(p.nb)
    return nbs


def assert_same_store(p, store, one):
    n = one.n_frames
    total = int(one.offsets[n].item())
    assert store.n_frames == n and store.stored_bytes == total
    assert torch.equal(store.offsets[:n + 1], one.offsets[:n + 1])
    assert torch.equal(store.frame_nb[:n], one.frame_nb[:n])
    assert torch.equal(store.stream[:total], one.stream[:total])
    used = p.sidecar_used_bytes(n, total)
    assert store.sidecar.numel() >= used
    assert torch.equal(store.sidecar[:used], one.sidecar[:used])


def assert_gathers(pd, store, want, want_w, rng, n):
    """Every stored frame (in pieces of MAX_BATCH) and a random list, with the stored index and without one."""
    lists = [list(range(a, min(n, a + MAX_BATCH))) for a in range(0, n, MAX_BATCH)]
    lists.append(rng.integers(0, n, MAX_BATCH).tolist())
    for ids in lists:
        t = torch.tensor(ids, dtype=torch.int64, device="cuda")
        for use_sc in (True, False):
            status = torch.full((len(ids),), 7, dtype=torch.int32, device="cuda")
            got = pd.decompress_frames(store, t, status=status, use_sidecar=use_sc)
            status_w = torch.full((len(ids),), 7, dtype=torch.int32, device="cuda")
            got_w = pd.decompress_frames_tensor(store, t, status=status_w, use_sidecar=use_sc)
            torch.cuda.synchronize()
            assert not status.any() and not status_w.any(), (ids, use_sc)
            assert torch.equal(got.view(len(ids), -1), want[t]), (ids, use_sc)
            assert torch.equal(got_w, want_w[t]), (ids, use_sc)


@pytest.mark.parametrize("kind,bps,ch,ns,nb,exact,escalate", CASES)
def test_append_equals_one_shot(R, oracle, kind, bps, ch, ns, nb, exact, escalate):
    rng = np.random.default_rng(ns * 31 + ch * 7 + bps)
    frames = torch.from_numpy(make_frames(oracle, rng, bps, ch, ns, N, escalate).reshape(-1)).cuda()
    p1, one = one_shot(R, kind, bps, ch, ns, nb, exact, frames)
    want = p1.decompress_batch(one).view(N, -1)
    want_w = p1.decompress_tensor(one)

    p = handle(R, kind, bps, ch, ns, nb, exact, MAX_BATCH)
    store = p.new_store(N)
    append_all(p, store, frames, APPENDS, bps, ch, ns)
    torch.cuda.synchronize()
    assert any(int(o) % 64 for o in store.offsets[1:N].tolist())
    assert_same_store(p, store, one)
    assert p.nb == p1.nb
    c, c1 = p.counters(), p1.counters()
    for k in ("frames_compressed", "raw_bytes_in", "compressed_bytes_out", "blocks_copy", "blocks_huff", "blocks_fill", "escalations"):
        assert c[k] == c1[k], k
    assert store.frame(N - 1) == one.frame(N - 1)

    pd = handle(R, kind, bps, ch, ns, nb, exact, MAX_BATCH)
    assert_gathers(pd, store, want, want_w, np.random.default_rng(3), N)


def test_escalation_across_appends(R, oracle):
    """xdelta_hzr 4 B with nb = 1: the plane count rises in later appends and carries from append to append."""
    kind, bps, ch, ns, nb = "xdelta_hzr", 4, 3, 5000, 1
    frames = torch.from_numpy(make_frames(oracle, np.random.default_rng(1), bps, ch, ns, N, True).reshape(-1)).cuda()
    p1, one = one_shot(R, kind, bps, ch, ns, nb, False, frames)
    p = handle(R, kind, bps, ch, ns, nb, False, MAX_BATCH)
    store = p.new_store(N)
    nbs = append_all(p, store, frames, APPENDS, bps, ch, ns)
    assert nbs[0] == 1 and nbs[-1] == p1.nb > 2
    assert sum(b > a for a, b in zip(nbs, nbs[1:])) >= 2, nbs   # escalated in at least two later appends
    assert nbs == sorted(nbs)
    assert len(set(store.frame_nb[:N].tolist())) > 2
    assert_same_store(p, store, one)
    assert p.counters()["escalations"] == p1.counters()["escalations"] == p1.nb - 1


def test_growth_and_trim(R, oracle):
    kind, bps, ch, ns, nb = "xdelta_hzr", 3, 12, 8192, 3
    frames = torch.from_numpy(make_frames(oracle, np.random.default_rng(2), bps, ch, ns, N).reshape(-1)).cuda()
    p1, one = one_shot(R, kind, bps, ch, ns, nb, False, frames)
    want = p1.decompress_batch(one).view(N, -1)
    want_w = p1.decompress_tensor(one)
    p = handle(R, kind, bps, ch, ns, nb, False, MAX_BATCH)
    store = p.new_store(2, bytes_capacity=1000)
    caps = [(store.offsets.numel(), store.stream.numel(), store.sidecar.numel())]
    a = 0
    for k in APPENDS[:5]:
        p.append_batch(store, frames[a * p.frame_bytes:(a + k) * p.frame_bytes])
        a += k
        caps.append((store.offsets.numel(), store.stream.numel(), store.sidecar.numel()))
    assert all(x < y for x, y in zip(caps[0], caps[-1])), caps
    # growth reallocates; trimming then cuts every buffer to the used prefix
    pd = handle(R, kind, bps, ch, ns, nb, False, MAX_BATCH)
    assert_gathers(pd, store, want[:a], want_w[:a], np.random.default_rng(4), a)
    store.trim()
    torch.cuda.synchronize()
    assert store.stream.numel() == store.stored_bytes + 16
    assert store.offsets.numel() == a + 1 and store.frame_nb.numel() == a
    assert store.sidecar.numel() == p.sidecar_used_bytes(a, store.stored_bytes)
    assert_gathers(pd, store, want[:a], want_w[:a], np.random.default_rng(5), a)
    # a trimmed store takes further appends (it grows again) and still equals the one-shot batch
    for k in APPENDS[5:]:
        p.append_batch(store, frames[a * p.frame_bytes:(a + k) * p.frame_bytes])
        a += k
    torch.cuda.synchronize()
    assert_same_store(p, store, one)
    assert_gathers(pd, store, want, want_w, np.random.default_rng(6), N)


@pytest.mark.parametrize("kind,bps,ch,ns,nb", [("xdelta_hzr", 3, 12, 8192, 3), ("hadamard", 4, 12, 4096, 3)])
def test_cpu_written_store_indexed_in_pieces(R, oracle, kind, bps, ch, ns, nb):
    """Frames from the CPU packer, loaded as one store and indexed MAX_BATCH frames at a time, get the words one
    build_index over all of them gives."""
    n = 24
    raw = make_frames(oracle, np.random.default_rng(11), bps, ch, ns, n)
    o = oracle.OraclePacker(kind, bps, ch, ns, nb)
    frames, fnb, want = [], [], []
    for r in raw:
        frames.append(o.compress(r))
        fnb.append(o.nb)
        want.append(np.frombuffer(o.decompress(frames[-1])[0], np.uint8))
    want = np.stack(want)
    total = sum(len(f) for f in frames)
    buf = torch.from_numpy(np.frombuffer(b"".join(frames) + bytes(16), np.uint8).copy()).cuda()
    offs = np.concatenate([[0], np.cumsum([len(f) for f in frames])])
    off = torch.tensor(offs, dtype=torch.int64, device="cuda")
    nbt = torch.tensor(fnb, dtype=torch.uint8, device="cuda")
    p = R.SignalPacker(kind, bps, ch, ns, nb, max_batch_frames=MAX_BATCH)
    used = p.sidecar_used_bytes(n, total)

    # reference: one build_index over all frames on a handle that holds them all
    pa = R.SignalPacker(kind, bps, ch, ns, nb, max_batch_frames=n)
    ref = torch.zeros(used, dtype=torch.uint8, device="cuda")
    assert pa.L.rspt_gpu_build_index(pa.h, buf.data_ptr(), off.data_ptr(), n, nbt.data_ptr(), ref.data_ptr(), None) == 0

    store = R.CompressedStore(buf, off, nbt, None, n, total, p)
    status = torch.full((n,), 7, dtype=torch.int32, device="cuda")
    store.index_all(p, status)
    torch.cuda.synchronize()
    assert not status.any()
    assert store.sidecar.numel() == used
    assert torch.equal(store.sidecar, ref)
    for ids in ([23, 0, 5, 5, 17, 2, 11, 9], [3], list(range(13, 21))):
        st = torch.full((len(ids),), 7, dtype=torch.int32, device="cuda")
        got = p.decompress_frames(store, ids, status=st)
        torch.cuda.synchronize()
        assert not st.any()
        assert np.array_equal(got.cpu().numpy().reshape(len(ids), -1), want[ids]), ids

    # bad ids fail their own slots and write nothing
    sc = torch.zeros(used, dtype=torch.uint8, device="cuda")
    b = R.CompressedBatch(buf, off, nbt, sc, n)
    st = torch.full((4,), 7, dtype=torch.int32, device="cuda")
    p.index_frames(b, [-1, n, 2 ** 40, -2 ** 40], st)
    torch.cuda.synchronize()
    assert st.tolist() == [E_ARG] * 4
    assert not sc.any()

    # a frame whose entries would reach sidecar_capacity fails with RSPT_E_STREAM and nothing is written there
    planes = (bps if nb < bps else nb) if kind == "xdelta_hzr" else 3
    bpf = planes * ((ch * ns + 65535) // 65536)   # blocks per stored frame
    k = 6                                         # an ECG frame: HUFF blocks
    cap = 4 * ((int(offs[k]) >> 6) + k * bpf)     # frame k's entries start at or beyond this byte
    guard = torch.full((used + 4096,), 0xAB, dtype=torch.uint8, device="cuda")
    ids = torch.tensor([0, k, 1], dtype=torch.int64, device="cuda")
    st = torch.full((3,), 7, dtype=torch.int32, device="cuda")
    assert p.L.rspt_gpu_build_index_frames(p.h, buf.data_ptr(), off.data_ptr(), n, nbt.data_ptr(), ids.data_ptr(), 3,
                                           guard.data_ptr(), cap, st.data_ptr()) == 0
    torch.cuda.synchronize()
    assert st.tolist() == [0, E_STREAM, 0]
    assert bool((guard[cap:] == 0xAB).all())
    # the frames below the capacity got their reference words
    w1 = (int(offs[2]) >> 6) + 2 * bpf
    written = guard[:4 * w1].view(torch.int32) != int(np.int32(np.uint32(0xABABABAB)))
    assert torch.equal(guard[:4 * w1].view(torch.int32)[written], ref[:4 * w1].view(torch.int32)[written])
    assert bool(written.any())


def test_append_refusals(R, oracle):
    """Every refusal of the append and ranged-index calls, through ctypes; a refused call leaves the store as it was."""
    kind, bps, ch, ns, nb = "xdelta_hzr", 3, 12, 8192, 3
    frames = torch.from_numpy(make_frames(oracle, np.random.default_rng(3), bps, ch, ns, MAX_BATCH + 1).reshape(-1)).cuda()
    p = R.SignalPacker(kind, bps, ch, ns, nb, max_batch_frames=MAX_BATCH)
    fb, maxc = p.frame_bytes, p.max_compressed_size
    store = p.new_store(2 * MAX_BATCH + 1)
    p.append_batch(store, frames[:3 * fb])
    torch.cuda.synchronize()
    snap = [t.clone() for t in (store.stream, store.offsets, store.frame_nb, store.sidecar)]
    L, h = p.L, p.h
    n0, b0 = store.n_frames, store.stored_bytes
    src, s, off, fnb, sc = (frames.data_ptr(), store.stream.data_ptr(), store.offsets.data_ptr(), store.frame_nb.data_ptr(),
                            store.sidecar.data_ptr())
    cap, sc_cap = store.stream.numel() - 16, store.sidecar.numel()
    words = to_words(frames, bps, ch, ns)
    for fn, sp in ((L.rspt_gpu_compress_append, src), (L.rspt_gpu_compress_append_i32, words.data_ptr())):
        n = 4
        need_sc = p.sidecar_used_bytes(n0 + n, b0 + n * maxc)
        assert fn(h, sp, MAX_BATCH + 1, s, cap, off, n0, b0, fnb, sc, sc_cap) == E_CAPACITY
        assert fn(h, sp, n, s, b0 + n * maxc - 1, off, n0, b0, fnb, sc, sc_cap) == E_CAPACITY
        assert fn(h, sp, n, s, b0 - 1, off, n0, b0, fnb, sc, sc_cap) == E_CAPACITY
        assert fn(h, sp, n, s, cap, off, n0, b0, fnb, sc, need_sc - 1) == E_CAPACITY
        assert fn(h, sp, n, s, cap, off, 1 << 32, b0, fnb, sc, sc_cap) == E_ARG                  # block ordinals
        big = 1 << 38                                                                             # index words reach 2^32
        assert fn(h, sp, n, s, big + n * maxc, off, n0, big, fnb, sc, 1 << 40) == E_ARG
        assert fn(None, sp, n, s, cap, off, n0, b0, fnb, sc, sc_cap) == E_ARG
        assert fn(h, None, n, s, cap, off, n0, b0, fnb, sc, sc_cap) == E_ARG
        assert fn(h, sp, n, None, cap, off, n0, b0, fnb, sc, sc_cap) == E_ARG
        assert fn(h, sp, n, s, cap, None, n0, b0, fnb, sc, sc_cap) == E_ARG
        assert fn(h, sp, 0, s, cap, off, n0, b0, fnb, sc, sc_cap) == 0
    assert L.rspt_gpu_compress_append_i32(h, words.data_ptr() + 2, 4, s, cap, off, n0, b0, fnb, sc, sc_cap) == E_ARG
    ids = torch.arange(MAX_BATCH + 1, dtype=torch.int64, device="cuda")
    bi = L.rspt_gpu_build_index_frames
    assert bi(h, s, off, n0, fnb, ids.data_ptr(), MAX_BATCH + 1, sc, sc_cap, None) == E_CAPACITY
    assert bi(h, s, off, 1 << 32, fnb, ids.data_ptr(), 2, sc, sc_cap, None) == E_ARG
    for args in ((None, s, off), (h, None, off), (h, s, None)):
        assert bi(*args, n0, fnb, ids.data_ptr(), 2, sc, sc_cap, None) == E_ARG
    assert bi(h, s, off, n0, fnb, None, 2, sc, sc_cap, None) == E_ARG
    assert bi(h, s, off, n0, fnb, ids.data_ptr(), 2, None, sc_cap, None) == E_ARG
    assert bi(h, s, off, n0, fnb, ids.data_ptr(), 0, sc, sc_cap, None) == 0
    torch.cuda.synchronize()
    for a, b in zip(snap, (store.stream, store.offsets, store.frame_nb, store.sidecar)):
        assert torch.equal(a, b)
    # the Python layer checks its inputs before anything is written
    with pytest.raises(ValueError):
        p.append_batch(store, frames[:MAX_BATCH * fb + fb])
    for bad in (frames[:fb + 1], frames[:2 * fb].view(torch.int8), words[:2].to(torch.int64)):
        with pytest.raises(ValueError):
            p.append_batch(store, bad)
    with pytest.raises(ValueError):
        p.append_tensor(store, words[:2, :, :-1])
    torch.cuda.synchronize()
    assert store.n_frames == n0 and store.stored_bytes == b0
    for a, b in zip(snap, (store.stream, store.offsets, store.frame_nb, store.sidecar)):
        assert torch.equal(a, b)
    # the same store then takes an append that fits exactly
    p.append_batch(store, frames[3 * fb:7 * fb])
    assert store.n_frames == n0 + 4


def test_store_at_scale(R):
    """32 appends of 2048 shape-A synth_ecg frames (65 536 frames, 19 GB raw); 4096 random ids gathered from it equal
    the regenerated frames, with the stored index and without one."""
    bps, ch, ns, per, k = 3, 12, 8192, 2048, 32
    p = R.SignalPacker.new_xdelta_hzr(bps, ch, ns, 3, max_batch_frames=per)
    store = p.new_store(per)
    for j in range(k):
        p.append_batch(store, R.synth_ecg(j * per, per, bps, ch, ns))
    n = per * k
    assert store.n_frames == n
    ids = torch.from_numpy(np.random.default_rng(9).integers(0, n, 4096)).cuda()
    fb = p.frame_bytes
    want = torch.empty(4096 * fb, dtype=torch.uint8, device="cuda")
    for j, g in enumerate(ids.tolist()):
        R.synth_ecg(g, 1, bps, ch, ns, out=want[j * fb:(j + 1) * fb])
    pg = R.SignalPacker.new_xdelta_hzr(bps, ch, ns, 3, max_batch_frames=4096)
    status = torch.full((4096,), 7, dtype=torch.int32, device="cuda")
    for use_sc in (True, False):
        got = pg.decompress_frames(store, ids, status=status, use_sidecar=use_sc)
        torch.cuda.synchronize()
        assert not status.any(), use_sc
        assert torch.equal(got, want), use_sc
        del got
