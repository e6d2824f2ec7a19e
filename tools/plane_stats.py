"""What the byte planes of a packer look like, per hzr block (CPU only: the oracle's transform, counts only).

    python tools/plane_stats.py [--kind xdelta_hzr] [--bps 3] [--ch 12] [--ns 8192] [--nb 3] [--frames 48]

Per (plane, block length): the density class the histogram kernel's probe gives the block (the first 16-byte chunk
of every warp's range of steps; "dense" when more than a quarter of the probed chunks hold >= 2 non-zero bytes),
and, averaged over the blocks of that kind, the non-zero bytes, the 512-byte warp steps, the steps that hold any
non-zero byte, the non-zero 16-byte chunks per such step, and what scattering them into the sparse list costs:
iterations of the half-warp scatter (two non-zero chunks per iteration) against a loop in which every lane walks
its own chunk's non-zero bytes (the most in any lane of the step).  The planes follow the flat channel-major
split of the packer (plane k = byte k of every transformed word)."""
import argparse
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import oracle as O  # noqa: E402

BLOCK, STEP, CHUNK, WARPS = 65536, 512, 16, 8


def block_stats(b):
    n = b.size
    nsteps = (n + STEP - 1) // STEP
    pad = np.zeros(nsteps * STEP, np.uint8)
    pad[:n] = b
    nzc = (pad.reshape(nsteps, STEP // CHUNK, CHUNK) != 0).sum(axis=2)  # non-zero bytes per chunk
    spw = (nsteps + WARPS - 1) // WARPS
    probe = [min(nsteps, w * spw) for w in range(WARPS)]
    probe = [s for s in probe if s < nsteps]
    valid = sum(int(((np.arange(STEP // CHUNK) * CHUNK + s * STEP) < n).sum()) for s in probe)
    dense_chunks = sum(int((nzc[s] >= 2).sum()) for s in probe)
    dense = dense_chunks * 4 > valid
    active = nzc.any(axis=1)
    chunks = (nzc > 0).sum(axis=1)[active]
    return {
        "class": "dense" if dense else "sparse",
        "nonzero": int(nzc.sum()),
        "steps": nsteps,
        "active_steps": int(active.sum()),
        "chunks_per_active_step": float(chunks.mean()) if chunks.size else 0.0,
        "half_warp_iters": int(((chunks + 1) // 2).sum()),
        "per_lane_iters": int(nzc.max(axis=1)[active].sum()),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--kind", default="xdelta_hzr")
    ap.add_argument("--bps", type=int, default=3)
    ap.add_argument("--ch", type=int, default=12)
    ap.add_argument("--ns", type=int, default=8192)
    ap.add_argument("--nb", type=int, default=3, help="planes (xdelta_hzr: its argument; hzr 4, hadamard 3, dct 2)")
    ap.add_argument("--frames", type=int, default=48)
    ap.add_argument("--first", type=int, default=0, help="first frame index of the synthetic recording")
    a = ap.parse_args()
    O.build()
    pk = O.OraclePacker(a.kind, a.bps, a.ch, a.ns, a.nb)
    raws = O.synth_ecg(a.first, a.frames, a.bps, a.ch, a.ns)
    rows = {}
    for r in raws:
        words = pk.transform(r)[0]
        planes = words.astype("<i4").view(np.uint8).reshape(-1, 4)[:, :a.nb].T
        for k, pl in enumerate(planes):
            for off in range(0, pl.size, BLOCK):
                s = block_stats(pl[off:off + BLOCK])
                rows.setdefault((k, min(BLOCK, pl.size - off), s["class"]), []).append(s)
    hdr = ("plane", "block bytes", "class", "blocks", "non-zero bytes", "steps", "steps with a non-zero byte",
           "non-zero chunks per such step", "half-warp scatter iterations", "per-lane-loop iterations")
    print("| " + " | ".join(hdr) + " |")
    print("|" + "---|" * len(hdr))
    for (k, n, cls), ss in sorted(rows.items()):
        m = lambda f: np.mean([s[f] for s in ss])  # noqa: E731
        print("| %d | %d | %s | %d | %.0f | %d | %.0f | %.1f | %.0f | %.0f |" % (
            k, n, cls, len(ss), m("nonzero"), ss[0]["steps"], m("active_steps"), m("chunks_per_active_step"),
            m("half_warp_iters"), m("per_lane_iters")))


if __name__ == "__main__":
    main()
