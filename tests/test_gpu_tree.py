"""The dense and sparse tree builds (k_hzr_tree) against the oracle's MakeTree on chosen histograms:
code words, code lengths, tree_nbits and n_used through the per-block debug entry, and the serialised
tree through a one-block hzr frame compared byte for byte with the oracle's stream and decoded back.  Needs a B200."""
import numpy as np
import pytest

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600)]

torch = pytest.importorskip("torch")

# zero-run symbols and a run length that tokenises to each (hzr_internal.h:113-121)
RUN_LEN = {0: 1, 256: 2, 257: 3, 258: 7, 259: 23, 260: 279}
MAX_BLOCK = 65536


@pytest.fixture(scope="module")
def R():
    import rspt_b200  # noqa: F401
    from rspt_b200 import packer
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return packer


@pytest.fixture(scope="module")
def O():
    from oracle import oracle
    return oracle


def symbols(L):
    """L used symbols: literals first, the zero-run symbols once all 255 literals are used."""
    lit = list(range(1, 256))
    return lit[:L] if L <= 255 else lit + sorted(RUN_LEN)[: L - 255]


def block_from_hist(hist, rng):
    """A byte block whose token histogram is `hist`: literals in random order, every zero-run token
    in its own gap between two literals."""
    lits = np.repeat(np.arange(1, 256), hist[1:256]).astype(np.uint8)
    rng.shuffle(lits)
    runs = [s for s in RUN_LEN for _ in range(int(hist[s]))]
    rng.shuffle(runs)
    assert len(runs) <= lits.size + 1, "not enough literals to separate the zero runs"
    gaps = np.sort(rng.choice(lits.size + 1, len(runs), replace=False))
    parts, prev = [], 0
    for g, s in zip(gaps, runs):
        parts += [lits[prev:g], np.zeros(RUN_LEN[s], np.uint8)]
        prev = g
    parts.append(lits[prev:])
    return np.concatenate(parts)


def hist_of(L, kind, rng):
    syms = symbols(L)
    h = np.zeros(261, np.int64)
    if kind == "equal":
        c = np.full(L, 3)
    elif kind == "ones_twos":           # long runs of equal-weight internal nodes
        c = np.where(np.arange(L) % 3 == 0, 2, 1)
    elif kind == "fibonacci":           # the deepest trees a block allows
        f = [1, 1]
        while len(f) < L:
            f.append(f[-1] + f[-2])
        m = L
        while sum(f[:m]) + (L - m) > 40000:
            m -= 1
        c = np.array([1] * (L - m) + f[:m])
    elif kind == "near_full":           # one count close to 65 536
        c = np.ones(L, np.int64)
        c[L // 2] = 0
        room = MAX_BLOCK - sum(RUN_LEN.get(s, 1) for s in syms)
        c[L // 2] = room + 1
    else:                               # random counts
        c = rng.integers(1, 200, L)
    h[syms] = c
    if kind != "near_full":
        for s in RUN_LEN:               # zero runs: at most 4 tokens each, inside the block
            h[s] = min(h[s], 4)
    assert sum(h[s] * RUN_LEN.get(s, 1) for s in range(261)) <= MAX_BLOCK
    return h


LENGTHS = [2, 3, 31, 32, 33, 63, 64, 65, 127, 128, 129, 255, 256, 257, 258, 259, 260, 261]
KINDS = ["equal", "ones_twos", "fibonacci", "near_full", "random"]


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("L", LENGTHS)
def test_tree_matches_oracle(R, O, L, kind):
    rng = np.random.default_rng(L * 31 + KINDS.index(kind))
    hist = hist_of(L, kind, rng)
    block = block_from_hist(hist, rng)
    assert block.size < MAX_BLOCK or kind == "near_full"
    want_hist = O.hzr_histogram(block)
    assert np.array_equal(want_hist, hist), "test block does not have the chosen histogram"

    p = R.SignalPacker.new_hzr(1, 1, MAX_BLOCK, max_batch_frames=1)
    got_hist, codes, info = p.debug_hzr_tables(block)
    assert np.array_equal(got_hist, want_hist)
    n_used, code, ln, tree, tree_nbits = O.hzr_build_codes(want_hist)
    used = want_hist > 0
    assert int(info[3]) == n_used == L
    assert int(info[2]) == tree_nbits
    assert np.array_equal(codes[used] & 0x07FFFFFF, code[used])
    assert np.array_equal(codes[used] >> 27, ln[used])
    assert not np.any(codes[~used])

    # the serialised tree: the block as the low byte plane of a one-channel hzr frame
    q = R.SignalPacker.new_hzr(1, 1, block.size, max_batch_frames=1)
    batch = q.compress_batch(torch.from_numpy(block.copy()).cuda())
    torch.cuda.synchronize()
    offs = batch.offsets.cpu().numpy()
    got = batch.stream.cpu().numpy()[offs[0]:offs[1]].tobytes()
    assert got == O.OraclePacker("hzr", 1, 1, block.size, 0).compress(block)

    # and back: with the encoder's decode index and with one rebuilt from the stream
    bare = R.CompressedBatch(batch.stream, batch.offsets, batch.frame_nb, None, 1)
    for what, b in (("encoder index", batch), ("rebuilt index", q.build_index(bare))):
        status = torch.full((1,), 7, dtype=torch.int32, device="cuda")
        dec = q.decompress_batch(b, status=status)
        torch.cuda.synchronize()
        assert status.item() == 0, what
        assert np.array_equal(dec.cpu().numpy(), block), what
