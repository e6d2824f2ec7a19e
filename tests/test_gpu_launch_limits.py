"""Dynamic shared-memory limits in a fresh process.  A kernel's default limit is 48 KB minus its static shared memory,
and the hzr kernels declare up to 12 544 bytes of that, so a launch that asks for a little less than 48 KB of dynamic
shared memory can still need a raised limit.  At 1 B x 5 ch x 8000 samples (40 000 bytes per plane) k_hzr_encode
asks for 40 080 bytes (its default limit is 40 064), k_hzr_decode's full-size class and k_hzr_build_index for
40 048 (38 784 and 36 608).  The limits belong to the process, so the shape is run in a child process in which no
other shape has raised them.  Needs a B200."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600)]

torch = pytest.importorskip("torch")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BPS, CH, NS, N = 1, 5, 8000, 8


def make_frames(rng):
    """uint8 [N, frame_bytes]: a slow walk, narrow noise (HUFF payloads above 16 KB: the full-size decode class),
    full-range noise (COPY blocks) and all-zero frames (FILL blocks)."""
    frames = []
    for i in range(N):
        if i % 4 == 0:
            x = np.clip(np.cumsum(rng.integers(-2, 3, NS * CH)), -128, 127)
        elif i % 4 == 1:
            x = rng.integers(-12, 13, NS * CH)
        elif i % 4 == 2:
            x = rng.integers(-128, 128, NS * CH)
        else:
            x = np.zeros(NS * CH, np.int64)
        frames.append(x.astype(np.int8).view(np.uint8))
    return np.stack(frames)


def child():
    sys.path.insert(0, ROOT)
    from oracle import oracle as O
    from rspt_b200 import packer as R
    torch.cuda.set_device(0)
    frames = make_frames(np.random.default_rng(48))
    x = torch.from_numpy(frames.reshape(-1).copy()).cuda()
    for kind, nb in (("hzr", 4), ("xdelta_hzr", 1)):
        p = R.SignalPacker(kind, BPS, CH, NS, nb, max_batch_frames=N)
        batch = p.compress_batch(x)
        status = torch.full((N,), 7, dtype=torch.int32, device="cuda")
        dec = p.decompress_batch(batch, status=status)
        no_index = R.CompressedBatch(batch.stream, batch.offsets, batch.frame_nb, None, N)
        rebuilt = p.build_index(no_index)
        dec_rebuilt = p.decompress_batch(rebuilt)
        dec_own = p.decompress_batch(no_index, use_sidecar=False)
        verified = p.verify_batch(batch)
        torch.cuda.synchronize()
        offs, stream = batch.offsets.cpu().numpy(), batch.stream.cpu().numpy()
        o = O.OraclePacker(kind, BPS, CH, NS, nb)
        for i in range(N):
            assert stream[offs[i]:offs[i + 1]].tobytes() == o.compress(frames[i]), (kind, i)
        assert not status.any().item(), (kind, status.cpu().numpy())
        assert not verified.any().item(), (kind, verified.cpu().numpy())
        for name, d in (("stored index", dec), ("rebuilt index", dec_rebuilt), ("own index", dec_own)):
            assert np.array_equal(d.cpu().numpy().reshape(N, -1), frames), (kind, name)
        p.close()
        print("ok", kind)


def test_shapes_just_under_48_kb_of_dynamic_shared_memory(oracle):
    r = subprocess.run([sys.executable, os.path.abspath(__file__)], capture_output=True, text=True, timeout=500)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert r.stdout.split() == ["ok", "hzr", "ok", "xdelta_hzr"], r.stdout


if __name__ == "__main__":
    child()
