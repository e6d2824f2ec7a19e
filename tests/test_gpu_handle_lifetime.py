"""Lifetime of a packer handle.  A create whose first device allocation is refused returns RSPT_E_CUDA, hands out no
handle and leaves the device usable.  A handle whose lazy buffers were grown and reused, whose dct paths were
switched back and forth and whose host pipeline was set up is destroyed, together with an ingest ring and its own
packer, while work is still queued, over many cycles in one process.  Needs a B200."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600)]

torch = pytest.importorskip("torch")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BPS, CH, NS, N = 2, 4, 1024, 6
FIR_LENGTHS = (300, 9, 64)  # grow, reuse the larger buffer, reuse it again
CYCLES = 20


def walk_frames(rng, n, bps, ch, ns):
    """uint8 [n, bps * ch * ns]: bounded random walks, interleaved by channel."""
    lim = (1 << (8 * bps - 1)) - 1
    x = np.clip(np.cumsum(rng.integers(-40, 41, (n, ns * ch)), axis=1), -lim, lim).astype(np.int32)
    return np.ascontiguousarray(x.view(np.uint8).reshape(n, ns * ch, 4)[:, :, :bps]).reshape(n, -1)


def stream_frames(batch):
    offs, stream = batch.offsets.cpu().numpy(), batch.stream.cpu().numpy()
    return [stream[offs[i]:offs[i + 1]].tobytes() for i in range(batch.n_frames)]


def test_create_refused_on_its_first_allocation(oracle):
    from rspt_b200 import _lib
    from rspt_b200 import packer as R
    L = _lib.lib()
    dev = torch.cuda.current_device()
    # 2^30 frames of 12 ch x 3 B x 8192 samples: the byte planes alone would take 384 TiB
    h = C.c_void_p(1)
    rc = L.rspt_gpu_create(_lib.KINDS["hzr"], 3, 12, 8192, 4, dev, torch.cuda.current_stream().cuda_stream, 1 << 30, C.byref(h))
    assert rc == -2 and h.value is None, (rc, h.value)

    frames = walk_frames(np.random.default_rng(5), 4, 3, 12, 8192)
    p = R.SignalPacker("hzr", 3, 12, 8192, max_batch_frames=4)
    x = torch.from_numpy(frames.reshape(-1).copy()).cuda()
    batch = p.compress_batch(x)
    dec = p.decompress_batch(batch)
    torch.cuda.synchronize()
    o = oracle.OraclePacker("hzr", 3, 12, 8192, 4)
    assert stream_frames(batch) == [o.compress(f) for f in frames]
    assert np.array_equal(dec.cpu().numpy().reshape(4, -1), frames)
    p.close()


def child():
    sys.path.insert(0, ROOT)
    from oracle import oracle as O
    from rspt_b200 import packer as R
    torch.cuda.set_device(0)
    rng = np.random.default_rng(11)
    frames = walk_frames(rng, N, BPS, CH, NS)
    kernels = {k: rng.standard_normal(k) / k for k in FIR_LENGTHS}
    o = O.OraclePacker("dct", BPS, CH, NS, 2)
    exact = [o.compress(f) for f in frames]
    exact_dec = np.stack([np.frombuffer(o.decompress(c)[0], np.uint8) for c in exact])
    fir9 = np.stack([O.prefilter_fir(f, BPS, CH, NS, kernels[9]) for f in frames])
    x = torch.from_numpy(frames.reshape(-1).copy()).cuda()
    first_fir, first_fast = {}, None
    for cycle in range(CYCLES):
        p = R.SignalPacker("dct", BPS, CH, NS, max_batch_frames=N)
        for k in FIR_LENGTHS:
            y = p.prefilter_fir(x.clone(), kernels[k]).cpu().numpy().reshape(N, -1)
            first_fir.setdefault(k, y)
            assert np.array_equal(y, first_fir[k]), (cycle, k)
        assert np.array_equal(first_fir[9], fir9)
        for exact_path in (True, False, True):
            p.set_dct_exact(exact_path)
            got = stream_frames(p.compress_batch(x))
            if exact_path:
                assert got == exact, cycle
            else:
                first_fast = first_fast or got
                assert got == first_fast, cycle
        dst = np.empty(N * p.max_compressed_size, np.uint8)
        offs = np.zeros(N + 1, np.uint64)
        p.compress_batch_host(frames, dst, offs)
        assert [dst[offs[i]:offs[i + 1]].tobytes() for i in range(N)] == exact, cycle

        q = R.SignalPacker("hzr", BPS, CH, NS, max_batch_frames=N)
        ring = R.IngestRing(q, 4)
        for i in range(3):
            ring.next_packet()[:] = frames[i]
        q_dst, q_offs = np.empty(3 * q.max_compressed_size, np.uint8), np.zeros(4, np.uint64)
        assert ring.drain(q_dst, q_offs, flush=True) == 3
        ring.next_packet()[:] = frames[3]
        ring.close()
        q.close()

        batch = p.compress_batch(x)
        dec = p.decompress_batch(batch)
        p.close()
        assert stream_frames(batch) == exact, cycle
        assert np.array_equal(dec.cpu().numpy().reshape(N, -1), exact_dec), cycle
    print("ok", CYCLES)


def test_destroy_with_work_in_flight(oracle):
    r = subprocess.run([sys.executable, os.path.abspath(__file__)], capture_output=True, text=True, timeout=500)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert r.stdout.split() == ["ok", str(CYCLES)], r.stdout


if __name__ == "__main__":
    child()
