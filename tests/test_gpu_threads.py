"""Handles driven from several host threads at once.  The dynamic shared-memory limit of a kernel belongs to the
process, not to a handle, so a handle whose shape needs less of it must never lower it under another handle's
launch.  Needs a B200."""
import threading

import numpy as np
import pytest

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600)]

torch = pytest.importorskip("torch")


def test_two_threads_one_kernel_different_shared_memory(oracle):
    from rspt_b200 import packer as R
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    # 3-byte samples and ns = 1000 (no multiple of 512, so no TMA transform): both shapes take
    # k_xdelta_planes_fast<3, true>, which needs about 19 KB of dynamic shared memory at 12 channels and about
    # 50 KB, above the 48 KB default, at 32
    bps, ns, n, batches = 3, 1000, 6, 3
    frames = {ch: [oracle.synth_ecg(1000 * ch + b * n, n, bps, ch, ns) for b in range(batches)] for ch in (12, 32)}
    got, errors = {}, []
    start = threading.Barrier(2)

    def run(ch):
        try:
            stream = torch.cuda.Stream()
            with torch.cuda.stream(stream):
                p = R.SignalPacker.new_xdelta_hzr(bps, ch, ns, bps, max_batch_frames=n)
                inputs = [torch.from_numpy(np.ascontiguousarray(f).reshape(-1)).cuda() for f in frames[ch]]
                stream.synchronize()
                start.wait(timeout=120)
                out = []
                for raw in inputs:
                    batch = p.compress_batch(raw)
                    dec = p.decompress_batch(batch)
                    out.append((batch, dec))
                stream.synchronize()
                got[ch] = [(b.offsets.cpu().numpy(), b.stream.cpu().numpy(), d.cpu().numpy()) for b, d in out]
                p.close()
        except Exception as e:  # reported by the main thread
            start.abort()
            errors.append((ch, repr(e)))

    threads = [threading.Thread(target=run, args=(ch,)) for ch in frames]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    for ch, batches_out in got.items():
        o = oracle.OraclePacker("xdelta_hzr", bps, ch, ns, bps)
        for raw, (offs, stream, dec) in zip(frames[ch], batches_out):
            host = np.asarray(raw, np.uint8).reshape(n, -1)
            assert np.array_equal(dec.reshape(n, -1), host), ch
            for i in range(n):
                assert stream[offs[i]:offs[i + 1]].tobytes() == o.compress(host[i]), (ch, i)
