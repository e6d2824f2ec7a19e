"""The two builds of the sparse class (RSPT_SPARSE_LIST=1: k_hzr_hist<3> + one-pass k_hzr_encode_sparse, the
default; RSPT_SPARSE_LIST=0: the earlier k_hzr_hist<1> + two-pass encoder) against the oracle: whole streams over
the plane shapes of the parity suite, and single blocks at the edges of the list builder (list capacity, the n/4
density limit, chunk and step boundaries, ragged block ends).  The switch is read when a handle is created; each
value runs in a child process, which gets its inputs and returns its results through files.  Needs a B200."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900)]

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
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

CHILD = r"""
import sys, numpy as np, torch
sys.path.insert(0, sys.argv[1])
from rspt_b200 import packer as R
z = np.load(sys.argv[2])
out = {}
for c, (kind, (bps, ch, ns, nb)) in enumerate(zip(z["kinds"].tolist(), z["dims"].tolist())):
    x = z["raw%d" % c]
    n = x.shape[0]
    p = R.SignalPacker(kind, bps, ch, ns, nb, max_batch_frames=n)
    b = p.compress_batch(torch.from_numpy(x.reshape(-1).copy()).cuda())
    torch.cuda.synchronize()
    offs = b.offsets.cpu().numpy()
    out["stream%d" % c] = b.stream[: int(offs[n])].cpu().numpy()
    out["offs%d" % c] = offs[: n + 1].astype(np.int64)
    p.close()
p = R.SignalPacker.new_hzr(1, 1, 65536, max_batch_frames=1)
for j in range(int(z["nblocks"])):
    hist, codes, info = p.debug_hzr_tables(z["blk%d" % j])
    out["hist%d" % j], out["info%d" % j] = hist, info
np.savez(sys.argv[3], **out)
"""


def _run_child(tmp_path, inputs, env_extra):
    src, dst = str(tmp_path / "in.npz"), str(tmp_path / ("out_%s.npz" % "_".join(env_extra.values())))
    np.savez(src, **inputs)
    env = dict(os.environ, **env_extra)
    r = subprocess.run([sys.executable, "-c", CHILD, ROOT, src, dst], env=env, capture_output=True, text=True, timeout=800)
    assert r.returncode == 0, r.stderr[-3000:]
    return np.load(dst)


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


@pytest.mark.parametrize("switch", ["1", "0"])
def test_sparse_list_streams_and_tables_match_oracle(switch, oracle, tmp_path):
    rng = np.random.default_rng(1234)
    inputs = {"kinds": np.array([c[0] for c in STREAM_CASES]), "dims": np.array([c[1:] for c in STREAM_CASES])}
    want = []
    for c, (kind, bps, ch, ns, nb) in enumerate(STREAM_CASES):
        nfr = 3
        raws = np.array(oracle.synth_ecg(50 + c, nfr, bps, ch, ns), np.uint8).reshape(nfr, -1)
        if kind == "hzr" and ch == 1 and ns == 70001:
            raws[:] = 0
            for r in raws:
                idx = rng.choice(70001, 900, replace=False)
                r[idx] = rng.integers(1, 256, 900)
        raws[nfr - 1][:] = 0   # a frame of FILL blocks
        inputs["raw%d" % c] = raws
        cpu = oracle.OraclePacker(kind, bps, ch, ns, nb)
        want.append([cpu.compress(r) for r in raws])
    blocks = _adversarial_blocks(rng)
    inputs["nblocks"] = np.array(len(blocks))
    for j, (_, b) in enumerate(blocks):
        inputs["blk%d" % j] = b
    got = _run_child(tmp_path, inputs, {"RSPT_SPARSE_LIST": switch})
    for c, case in enumerate(STREAM_CASES):
        st, offs = got["stream%d" % c], got["offs%d" % c]
        for i, w in enumerate(want[c]):
            assert st[offs[i]:offs[i + 1]].tobytes() == w, (case, i)
    for j, (name, b) in enumerate(blocks):
        assert np.array_equal(got["hist%d" % j], oracle.hzr_histogram(b)), name
        mode, plen = oracle.hzr_block_plan(b)
        assert (int(got["info%d" % j][0]), int(got["info%d" % j][1])) == (mode, plen), name


@pytest.mark.parametrize("switch", ["1", "0"])
def test_sparse_list_hand_over_to_general_encoder(switch, oracle, tmp_path):
    """RSPT_SPARSE_STAGE_BYTES=300: listed blocks whose payload exceeds the list encoder's staging go to
    k_hzr_encode, which rebuilds the per-step leading-zero counts from the list."""
    bps, ch, ns, nfr = 3, 12, 8192, 4
    raws = np.array(oracle.synth_ecg(40, nfr, bps, ch, ns), np.uint8).reshape(nfr, -1)
    raws[nfr - 1][:] = 0
    inputs = {"kinds": np.array(["xdelta_hzr"]), "dims": np.array([[bps, ch, ns, 3]]), "raw0": raws, "nblocks": np.array(0)}
    got = _run_child(tmp_path, inputs, {"RSPT_SPARSE_LIST": switch, "RSPT_SPARSE_STAGE_BYTES": "300"})
    cpu = oracle.OraclePacker("xdelta_hzr", bps, ch, ns, 3)
    st, offs = got["stream0"], got["offs0"]
    for i in range(nfr):
        assert st[offs[i]:offs[i + 1]].tobytes() == cpu.compress(raws[i]), i
