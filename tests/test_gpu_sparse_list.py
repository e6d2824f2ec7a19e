"""The sparse class (k_hzr_hist<3> builds a block's list of non-zero bytes, k_hzr_encode_sparse packs the block
from it) against the oracle: whole streams over the plane shapes of the parity suite, and single blocks at the
edges of the list builder (list capacity, the n/4 density limit, chunk and step boundaries, ragged block ends).
Needs a B200."""
import numpy as np
import pytest

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900)]

torch = pytest.importorskip("torch")

LIST_CAP = 5120

# the xdelta_hzr / hzr / hadamard shapes of test_gpu_parity.PLANE_CASES, plus a single-channel hzr plane of
# 70001 bytes (ragged 4465-byte last block); 3 x 12 x 8192 is the benchmark's shape (65536 + 32768-byte blocks)
STREAM_CASES = [
    ("xdelta_hzr", 3, 12, 8192, 3), ("xdelta_hzr", 4, 12, 4096, 3), ("xdelta_hzr", 2, 5, 1000, 2),
    ("xdelta_hzr", 1, 3, 700, 1), ("xdelta_hzr", 4, 1, 8192, 4), ("xdelta_hzr", 3, 2, 1, 3),
    ("xdelta_hzr", 4, 3, 2, 3), ("xdelta_hzr", 3, 7, 33, 3),
    ("xdelta_hzr", 2, 4, 1000, 2), ("xdelta_hzr", 1, 8, 700, 1), ("xdelta_hzr", 3, 4, 4, 3),
    ("xdelta_hzr", 3, 8, 516, 4), ("xdelta_hzr", 4, 16, 2052, 2), ("hzr", 2, 8, 2052, 4), ("hzr", 1, 4, 8, 4),
    ("hzr", 3, 12, 8192, 4), ("hzr", 1, 2, 999, 4), ("hzr", 4, 3, 5000, 4), ("hzr", 1, 1, 70001, 4),
    ("hadamard", 4, 12, 4096, 3), ("hadamard", 3, 3, 16384, 3), ("hadamard", 2, 2, 8, 3), ("hadamard", 1, 1, 32768, 3),
    ("hadamard", 3, 5, 4096, 3), ("hadamard", 2, 1, 4096, 3),
]


@pytest.fixture(scope="module")
def R():
    import rspt_b200
    from rspt_b200 import packer
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return packer


def _adversarial_blocks(rng):
    """Single blocks at the edges of the list builder; each is (name, bytes)."""
    def nz(k):
        return rng.integers(1, 256, k, dtype=np.uint8)
    out = []
    for m in (LIST_CAP, LIST_CAP + 1):
        # one burst inside the first warp's range: the density probe still says "sparse"
        b = np.zeros(65536, np.uint8)
        b[1000:1000 + m] = nz(m)
        out.append(("cap%d" % m, b))
    for m in (2000, 2001):
        # n = 8000: the n/4 limit binds before the list capacity; the bytes sit in the steps the probe skips
        b = np.zeros(8000, np.uint8)
        pos = np.concatenate([np.arange(512 * s, 512 * (s + 1)) for s in (1, 3, 5, 7)])[:m]
        b[pos] = nz(m)
        out.append(("quarter%d" % m, b))
    b = np.zeros(65536, np.uint8)
    b[1600:1616] = nz(16)
    out.append(("one_chunk", b))
    b = np.zeros(65536, np.uint8)
    c = np.arange(32)
    b[5 * 512 + 16 * c + (c % 16)] = nz(32)
    out.append(("every_chunk_of_a_step", b))
    for n in (1000, 65535, 4465):
        b = np.zeros(n, np.uint8)
        t = n & ~15
        b[t:] = nz(n - t)
        out.append(("last_partial_chunk_%d" % n, b))
    for n in (65536, 1000, 513):
        for at in (0, n - 1):
            b = np.zeros(n, np.uint8)
            b[at] = 7
            out.append(("lone_%d_at_%d" % (n, at), b))
    # scattered bytes with long runs (> 16662) between some of them, and odd step boundaries
    b = np.zeros(65536, np.uint8)
    b[[0, 17, 511, 512, 513, 20000, 40000, 65535]] = nz(8)
    out.append(("long_runs", b))
    return out


def _inputs(oracle):
    """The frames of every STREAM_CASES shape and the single blocks, drawn in one fixed order from one seed."""
    rng = np.random.default_rng(1234)
    frames = []
    for c, (kind, bps, ch, ns, nb) in enumerate(STREAM_CASES):
        nfr = 3
        raws = np.array(oracle.synth_ecg(50 + c, nfr, bps, ch, ns), np.uint8).reshape(nfr, -1)
        if kind == "hzr" and ch == 1 and ns == 70001:
            raws[:] = 0
            for r in raws:
                idx = rng.choice(70001, 900, replace=False)
                r[idx] = rng.integers(1, 256, 900)
        raws[nfr - 1][:] = 0   # a frame of FILL blocks
        frames.append(raws)
    return frames, _adversarial_blocks(rng)


@pytest.mark.parametrize("part", ["streams", "tables"])
def test_sparse_list_streams_and_tables_match_oracle(R, oracle, part):
    """streams: whole batches of every STREAM_CASES shape; tables: histogram and plan of the single blocks."""
    frames, blocks = _inputs(oracle)
    if part == "streams":
        for (kind, bps, ch, ns, nb), raws in zip(STREAM_CASES, frames):
            nfr = raws.shape[0]
            cpu = oracle.OraclePacker(kind, bps, ch, ns, nb)
            p = R.SignalPacker(kind, bps, ch, ns, nb, max_batch_frames=nfr)
            b = p.compress_batch(torch.from_numpy(raws.reshape(-1).copy()).cuda())
            torch.cuda.synchronize()
            offs = b.offsets.cpu().numpy()
            st = b.stream[: int(offs[nfr])].cpu().numpy()
            for i, r in enumerate(raws):
                assert st[offs[i]:offs[i + 1]].tobytes() == cpu.compress(r), ((kind, bps, ch, ns, nb), i)
            p.close()
    else:
        p = R.SignalPacker.new_hzr(1, 1, 65536, max_batch_frames=1)
        for name, b in blocks:
            hist, codes, info = p.debug_hzr_tables(b)
            assert np.array_equal(hist, oracle.hzr_histogram(b)), name
            mode, plen = oracle.hzr_block_plan(b)
            assert (int(info[0]), int(info[1])) == (mode, plen), name

