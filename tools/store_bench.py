"""What building and serving a store costs (SignalPacker.new_store / append_batch / index_all, decompress_frames),
device resident, on bench.py's shape A (3 B x 12 ch x 8192 samples = 294 912 bytes per frame, xdelta_hzr nb 3).

    python tools/store_bench.py [--frames 1048576] [--batch 4096] [--window 1.0] [--out profiles/r07_store.json]

1. append vs compress: append_batch of one `batch`-frame batch into a store (reset after every call, so it stays
   small) against compress_batch of the same frames, in alternating windows of at least `window` seconds; CUDA
   events, three windows each.  append_batch includes its 8-byte read-back of the new total and the synchronisation.
2. build: a store of `frames` synth_ecg frames (fewer if they would not fit in 75 % of free device memory), appended
   `batch` frames at a time, the store pre-sized from the first batch's compressed size (2 % over, plus the worst
   case of one append, so that it never grows).  Host clock around the
   whole build (it ends in a synchronisation), synth_ecg generation included and timed separately.  Stream and
   index bytes, CR = raw / stream and CR with the index counted = raw / (stream + index).
3. gather: decompress_frames of B random ids (drawn with replacement, rotated over 64 lists) from the store, with
   the stored index and without one, for B in `sizes`; CUDA events, windows as in 1.  Every arm's first output is
   compared with the regenerated frames.  profiles/r06_gather.json's rates from a 4096-frame batch are set beside.
4. index_all: the store's index is dropped and rebuilt with index_all (max_batch_frames = `batch` per call); host
   clock around it, ending in a synchronisation.  Its words are counted against the ones the appends wrote, and
   a gather of `batch` random frames with it must equal the regenerated frames.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from gather_bench import gpu_info, timed, window  # noqa: E402

SHAPE = dict(bps=3, ch=12, ns=8192)


def r06_rates(path: str) -> dict:
    """{B: {arm: raw GB/s}} of xdelta_hzr in profiles/r06_gather.json, when it is there."""
    if not os.path.exists(path):
        return {}
    with open(path) as f:
        r = json.load(f)
    for pk in r["packers"]:
        if pk["kind"] == "xdelta_hzr":
            return {row["B"]: {a: row[a]["raw_GBps"] for a in ("gather_index", "gather_noindex", "batch")} for row in pk["sizes"]}
    return {}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1 << 20)
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--sizes", default="256,4096")
    ap.add_argument("--window", type=float, default=1.0, help="seconds per timed window")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_store.json"))
    args = ap.parse_args()
    import torch
    from rspt_b200 import packer as R
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda", torch.cuda.current_device())
    info = gpu_info(dev.index)
    print(json.dumps({"gpu": info}), flush=True)
    res = {"gpu": info, "shape": SHAPE, "kind": "xdelta_hzr", "batch": args.batch, "window_s": args.window}
    B0 = args.batch
    p = R.SignalPacker.new_xdelta_hzr(3, 12, 8192, 3, max_batch_frames=B0)
    fb = p.frame_bytes

    # 1. append_batch against compress_batch, same frames
    raw = R.synth_ecg(0, B0, **SHAPE)
    out = p.alloc_output(B0)
    small = p.new_store(B0)

    def append(i):
        small.n_frames, small.stored_bytes = 0, 0
        p.append_batch(small, raw)

    arms = {"compress_batch": lambda i: p.compress_batch(raw, out=out), "append_batch": append}
    for fn in arms.values():
        timed(torch, fn, 3)
    assert torch.equal(small.stream[:small.stored_bytes], out.stream[:small.stored_bytes])
    ms = {a: [] for a in arms}
    for _ in range(3):
        for a, fn in arms.items():
            ms[a].append(window(torch, fn, args.window)[0])
    res["per_batch"] = {a: {"ms_median": float(np.median(v)), "ms_all": v, "raw_GBps": B0 * fb / (np.median(v) * 1e-3) / 1e9}
                        for a, v in ms.items()}
    print(json.dumps({"per_batch_ms": {a: round(float(np.median(v)), 4) for a, v in ms.items()}}), flush=True)
    del out, small
    torch.cuda.empty_cache()

    # 2. build the store
    first = p.compress_batch(raw)
    per_frame = int(first.offsets[-1].item()) / B0
    del first
    torch.cuda.empty_cache()
    free = torch.cuda.mem_get_info(dev)[0]
    cap = lambda n: int(n * per_frame * 1.02) + B0 * p.max_compressed_size
    n = args.frames - args.frames % B0
    while n > B0 and cap(n) + p.sidecar_used_bytes(n, cap(n)) > 0.75 * free - 8 * B0 * fb:
        n -= B0
    res["build"] = {"frames_target": args.frames, "frames": n, "free_bytes_before": free}
    store = p.new_store(n, bytes_capacity=cap(n))
    torch.cuda.synchronize()
    t_gen = 0.0
    t0 = time.perf_counter()
    for a in range(0, n, B0):
        g0 = time.perf_counter()
        R.synth_ecg(a, B0, out=raw, **SHAPE)
        torch.cuda.synchronize()
        t_gen += time.perf_counter() - g0
        p.append_batch(store, raw)
    torch.cuda.synchronize()
    t_build = time.perf_counter() - t0
    sb, ib = store.stored_bytes, store.sidecar_used_bytes()
    res["build"].update({"seconds": t_build, "synth_seconds": t_gen, "append_seconds": t_build - t_gen,
                         "raw_bytes": n * fb, "stream_bytes": sb, "index_bytes": ib, "index_bytes_per_frame": ib / n,
                         "cr": n * fb / sb, "cr_with_index": n * fb / (sb + ib)})
    print(json.dumps({"build": res["build"]}), flush=True)

    # 3. random minibatches from the store
    r06 = r06_rates(os.path.join(ROOT, "profiles", "r06_gather.json"))
    rng = np.random.default_rng(1)
    res["gather"] = []
    for B in [int(s) for s in args.sizes.split(",")]:
        pg = R.SignalPacker.new_xdelta_hzr(3, 12, 8192, 3, max_batch_frames=B)
        lists = [torch.from_numpy(rng.integers(0, n, B)).to(dev) for _ in range(64)]
        o = torch.empty(B * fb, dtype=torch.uint8, device=dev)
        status = torch.zeros(B, dtype=torch.int32, device=dev)
        want = torch.empty(B * fb, dtype=torch.uint8, device=dev)
        for j, g in enumerate(lists[0].tolist()):
            R.synth_ecg(g, 1, out=want[j * fb:(j + 1) * fb], **SHAPE)
        garms = {"gather_index": lambda i: pg.decompress_frames(store, lists[i % 64], out=o, status=status),
                 "gather_noindex": lambda i: pg.decompress_frames(store, lists[i % 64], out=o, status=status, use_sidecar=False)}
        checks = {}
        for a, fn in garms.items():
            fn(0)
            torch.cuda.synchronize()
            checks[a] = bool(torch.equal(o, want)) and not bool(status.any())
        assert all(checks.values()), (B, checks)
        for fn in garms.values():
            timed(torch, fn, 3)
        gms = {a: [] for a in garms}
        for _ in range(3):
            for a, fn in garms.items():
                gms[a].append(window(torch, fn, args.window)[0])
        row = {"B": B, "checks": checks}
        for a, v in gms.items():
            row[a] = {"ms_median": float(np.median(v)), "ms_all": v, "raw_GBps": B * fb / (np.median(v) * 1e-3) / 1e9}
        if B in r06:
            row["r06_from_4096_frame_batch"] = r06[B]
        res["gather"].append(row)
        print(json.dumps({"B": B, **{a: round(row[a]["raw_GBps"], 1) for a in garms}, "r06": r06.get(B)}), flush=True)
        pg.close()
        del lists, o, want
        torch.cuda.empty_cache()

    # 4. index_all over the same store, written without an index
    kept = store.sidecar
    store.sidecar = None
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    store.index_all(p)
    torch.cuda.synchronize()
    t_index = time.perf_counter() - t0
    a, b = store.sidecar.view(torch.int32), kept[:ib].view(torch.int32)
    differ = a != b
    res["index_all"] = {"seconds": t_index, "frames": n, "calls": -(-n // B0), "index_words": a.numel(),
                        "words_differing_from_appended_index": int(differ.sum()),
                        "of_them_unwritten_by_appends": int((differ & (b == 0)).sum())}
    # decoding with the rebuilt index: 4096 random frames against the regenerated ones
    pg = R.SignalPacker.new_xdelta_hzr(3, 12, 8192, 3, max_batch_frames=B0)
    ids = torch.from_numpy(rng.integers(0, n, B0)).to(dev)
    want = torch.empty(B0 * fb, dtype=torch.uint8, device=dev)
    for j, g in enumerate(ids.tolist()):
        R.synth_ecg(g, 1, out=want[j * fb:(j + 1) * fb], **SHAPE)
    status = torch.zeros(B0, dtype=torch.int32, device=dev)
    got = pg.decompress_frames(store, ids, status=status)
    torch.cuda.synchronize()
    res["index_all"]["gather_with_rebuilt_index_ok"] = bool(torch.equal(got, want)) and not bool(status.any())
    print(json.dumps({"index_all": res["index_all"]}), flush=True)
    assert res["index_all"]["gather_with_rebuilt_index_ok"]
    res["gpu_after"] = gpu_info(dev.index)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
