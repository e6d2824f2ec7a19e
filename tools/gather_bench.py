"""What decoding a list of frames out of a stored batch costs (decompress_frames), device resident.

    python tools/gather_bench.py [--stored 4096] [--sizes 64,256,1024,4096] [--window 1.0] [--out profiles/r06_gather.json]

Per packer (xdelta_hzr on bench.py's shape A = BASELINE configs[1], hadamard on shape B) one stored batch of
`stored` frames (xdelta_hzr: 1.2 GB raw, far larger than the 126 MB L2) with its decode index.  For every B in
`sizes`, on a handle with max_batch_frames = B, three arms:
  gather_index     decompress_frames of B random ids (drawn with replacement) with the stored index
  gather_noindex   the same without an index: one is built for the B selected frames first
  batch            decompress_batch of B contiguous frames with their own index: the stored frames compressed as
                   stored / B batches of B frames (the reference point)
Each arm rotates over max(4, stored / B) id lists or batches, so that it reads about as much distinct stream as
the stored batch holds instead of one L2-resident working set.  Timed with CUDA events after a warm-up, in
windows of at least `window` seconds, the arms alternating; three windows per arm.  Rate = B * frame_bytes / time.
Also timed: rspt_gpu_build_index over the whole stored batch (what a caller without the gather call would pay to
re-index it).  Before timing, every arm's output is compared with the stored batch's whole decode.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = {"A": dict(bps=3, ch=12, ns=8192), "B": dict(bps=4, ch=12, ns=4096)}
PACKERS = (("xdelta_hzr", "A"), ("hadamard", "B"))


def gpu_info(dev: int) -> dict:
    q = subprocess.run(["nvidia-smi", "-i", str(dev), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip()
    name, power, clk = [s.strip() for s in q.split(",")]
    return {"name": name, "power_limit": power, "clocks_max_sm": clk}


def timed(torch, fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def window(torch, fn, seconds):
    """Milliseconds per call over a window of at least `seconds` (the call count from a short calibration)."""
    ms = timed(torch, fn, 3)
    n = max(3, int(np.ceil(seconds * 1e3 / ms)))
    return timed(torch, fn, n), n


def measure(R, torch, kind, sh, stored, sizes, seconds):
    dev = torch.device("cuda", torch.cuda.current_device())
    bps, ch, ns = sh["bps"], sh["ch"], sh["ns"]
    fb = bps * ch * ns
    raw = R.synth_ecg(0, stored, **sh)
    ps = R.SignalPacker(kind, bps, ch, ns, 3, max_batch_frames=stored)
    sb = ps.compress_batch(raw)
    full = ps.decompress_batch(sb).view(stored, fb)
    torch.cuda.synchronize()
    total = int(sb.offsets[-1].item())
    res = {"kind": kind, "shape": sh, "stored_frames": stored, "frame_bytes": fb, "stored_raw_bytes": stored * fb,
           "stored_stream_bytes": total, "sizes": []}
    # re-indexing the whole stored batch
    ps.build_index(sb)
    res["build_index_whole_ms"] = min(window(torch, lambda i: ps.build_index(sb), seconds)[0] for _ in range(3))
    rng = np.random.default_rng(1)
    for B in sizes:
        p = R.SignalPacker(kind, bps, ch, ns, 3, max_batch_frames=B)
        nrot = max(4, stored // B)
        ids = [torch.from_numpy(rng.integers(0, stored, B)).to(dev) for _ in range(nrot)]
        nwin = max(1, stored // B)
        wins = [p.compress_batch(raw[w * B * fb:(w + 1) * B * fb]) for w in range(nwin)]
        out = torch.empty(B * fb, dtype=torch.uint8, device=dev)
        status = torch.zeros(B, dtype=torch.int32, device=dev)
        arms = {
            "gather_index": lambda i: p.decompress_frames(sb, ids[i % nrot], out=out, status=status),
            "gather_noindex": lambda i: p.decompress_frames(sb, ids[i % nrot], out=out, status=status, use_sidecar=False),
            "batch": lambda i: p.decompress_batch(wins[i % nwin], out=out, status=status),
        }
        checks = {}
        for a, fn in arms.items():
            fn(0)
            torch.cuda.synchronize()
            want = full[ids[0]] if a != "batch" else full[:B]
            checks[a] = bool(torch.equal(out.view(B, fb), want)) and not bool(status.any())
        assert all(checks.values()), (kind, B, checks)
        for fn in arms.values():   # warm-up of every arm
            timed(torch, fn, 3)
        ms = {a: [] for a in arms}
        calls = {a: [] for a in arms}
        for _ in range(3):
            for a, fn in arms.items():
                t, n = window(torch, fn, seconds)
                ms[a].append(t)
                calls[a].append(n)
        row = {"B": B, "rotation": {"id_lists": nrot, "batches": nwin}, "checks": checks}
        for a in arms:
            med = float(np.median(ms[a]))
            row[a] = {"ms_median": med, "ms_all": ms[a], "calls_per_window": calls[a], "raw_GBps": B * fb / (med * 1e-3) / 1e9}
        row["gather_index_vs_batch"] = row["batch"]["ms_median"] / row["gather_index"]["ms_median"]
        row["gather_noindex_vs_whole_reindex"] = row["gather_noindex"]["ms_median"] / res["build_index_whole_ms"]
        res["sizes"].append(row)
        print(json.dumps({"kind": kind, "B": B, **{a: round(row[a]["raw_GBps"], 1) for a in arms},
                          "gather_index_vs_batch": round(row["gather_index_vs_batch"], 3),
                          "gather_noindex_vs_whole_reindex": round(row["gather_noindex_vs_whole_reindex"], 3)}), flush=True)
        p.close()
        del wins, out, ids
        torch.cuda.empty_cache()
    ps.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--stored", type=int, default=4096)
    ap.add_argument("--sizes", default="64,256,1024,4096")
    ap.add_argument("--window", type=float, default=1.0, help="seconds per timed window")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_gather.json"))
    args = ap.parse_args()
    import torch
    from rspt_b200 import packer as R
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.cuda.current_device()
    info = gpu_info(dev)
    print(json.dumps({"gpu": info}), flush=True)
    sizes = [int(s) for s in args.sizes.split(",")]
    results = {"gpu": info, "window_s": args.window, "packers": []}
    for kind, shape in PACKERS:
        results["packers"].append(measure(R, torch, kind, SHAPES[shape], args.stored, sizes, args.window))
        torch.cuda.empty_cache()
    results["gpu_after"] = gpu_info(dev)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
