"""Which kernels each entry point of a handle launches, with grid, block and shared memory, as JSON.

A refactor of kernel selection can change which kernel runs without changing any output.  This drives a fixed
matrix of calls (every packer, the dct exact path, bps 1..4, several channel counts and lengths, 16-byte-aligned
and 4-byte-offset buffers, the native / int32 / host / debug / pre-filter / store / gather / index / verify entry
points) under torch.profiler and records, per call, the kernels of the library it launched and the handle's
kernel_launches count.  Run it once per library, each in its own process, and compare:

    python tools/launch_trace.py --lib rspt_b200/librspt_gpu.so --out new.json
    python tools/launch_trace.py --lib /path/to/other/librspt_gpu.so --out old.json
    python tools/launch_trace.py --compare old.json new.json
"""
from __future__ import annotations

import argparse
import json
import os
import re
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

LIB_KERNEL = re.compile(r"\bk_\w+")
SHAPES = [(ch, ns) for ch in (1, 3, 4, 12) for ns in (1, 300, 1024, 4096, 8192)] + [(3, 256)]
# packer variant -> (kind, nb for xdelta_hzr given bps, dct exact)
VARIANTS = {
    "xdelta_hzr": ("xdelta_hzr", lambda bps: bps, False),
    "xdelta_hzr_probe": ("xdelta_hzr", lambda bps: 1, False),  # nb < bps: the plane-count probe is on
    "hzr": ("hzr", None, False),
    "hadamard": ("hadamard", None, False),
    "dct": ("dct", None, False),
    "dct_exact": ("dct", None, True),
}
N_FRAMES = 2


def matrix():
    for var in VARIANTS:
        for bps in (1, 2, 3, 4):
            if var == "xdelta_hzr_probe" and bps == 1:
                continue
            for ch, ns in SHAPES:
                yield var, bps, ch, ns


def make_packer(R, var, bps, ch, ns):
    kind, nb, exact = VARIANTS[var]
    args = (kind, bps, ch, ns, nb(bps) if nb else 3)
    try:
        p = R.SignalPacker(*args, max_batch_frames=N_FRAMES)
    except R.RsptError:
        return None  # shape refused at create
    if exact:
        p.set_dct_exact(True)
    return p


def calls(torch, np, p, rng):
    """(id, thunk) per call on one handle; every thunk enqueues one entry point."""
    dev = torch.device("cuda", p.device)
    n, fb, words = N_FRAMES, p.frame_bytes, N_FRAMES * p.ch * p.ns
    raw = rng.integers(0, 256, n * fb, dtype=np.uint8)
    x32 = rng.integers(-(1 << (8 * p.bps - 1)), 1 << (8 * p.bps - 1), words, dtype=np.int64).astype(np.int32)

    def raw_view(off):  # the frames at a 16-byte-aligned address, or 4 bytes past one
        b = torch.from_numpy(np.concatenate([np.zeros(off, np.uint8), raw, np.zeros(16, np.uint8)])).to(dev)
        return b[off:off + n * fb]

    def words_view(off):
        b = torch.from_numpy(np.concatenate([np.zeros(off // 4, np.int32), x32])).to(dev)
        return b[off // 4:].view(n, p.ch, p.ns)

    st = {}

    def setup():  # what the decompress calls decode, and a store to append to
        st["batch"] = p.compress_batch(raw_view(0))
        st["one"] = p.compress(one)
        st["store"] = p.new_store(2 * n)

    one = raw[:fb].copy()
    out = [("setup", setup)]
    for off in (0, 4):
        a = "a16" if off == 0 else "off4"
        out += [
            (f"compress/{a}", lambda off=off: p.compress_batch(raw_view(off))),
            (f"decompress/{a}", lambda off=off: p.decompress_batch(st["batch"], out=raw_view(off))),
            (f"compress_i32/{a}", lambda off=off: p.compress_tensor(words_view(off))),
            (f"decompress_i32/{a}", lambda off=off: p.decompress_tensor(st["batch"], out=words_view(off))),
            (f"debug_planes/{a}", lambda off=off: p.debug_planes(raw_view(off))),
            (f"prefilter_iir/{a}", lambda off=off: p.prefilter_iir(raw_view(off), [1.0, -1.1429805, 0.4128016],
                                                                  [0.06745527, 0.13491055, 0.06745527], 10)),
            (f"prefilter_fir/{a}", lambda off=off: p.prefilter_fir(raw_view(off), np.full(9, 1 / 9))),
        ]
    host_dst = np.empty(n * p.max_compressed_size, np.uint8)
    host_off = np.zeros(n + 1, np.uint64)
    host_out = np.empty(n * fb, np.uint8)
    out += [
        ("compress_host", lambda: p.compress(one)),
        ("decompress_host", lambda: p.decompress(st["one"])),
        ("compress_batch_host", lambda: p.compress_batch_host(raw, host_dst, host_off)),
        ("decompress_batch_host", lambda: p.decompress_batch_host(host_dst, host_off, host_out)),
        ("append_batch", lambda: p.append_batch(st["store"], raw_view(0))),
        ("index_frames", lambda: p.index_frames(st["store"], [1, 0])),
        ("decompress_frames", lambda: p.decompress_frames(st["batch"], [1, 1])),
        ("decompress_frames_no_index", lambda: p.decompress_frames(st["batch"], [1, 1], use_sidecar=False)),
        ("build_index", lambda: p.build_index(st["batch"])),
        ("verify_batch", lambda: p.verify_batch(st["batch"])),
        ("debug_hzr_tables", lambda: p.debug_hzr_tables(raw[:min(fb, 65536)])),
    ]
    return out


def trace(lib_path: str, out_path: str) -> None:
    import numpy as np
    import torch
    from rspt_b200 import _lib
    _lib.LIB_PATH = os.path.abspath(lib_path)  # before the first call loads the library
    from rspt_b200 import packer as R
    from torch.profiler import ProfilerActivity, profile

    assert torch.cuda.is_available(), "launch_trace needs a CUDA device"
    torch.cuda.set_device(0)
    marker = torch.zeros(1, dtype=torch.int64, device="cuda")
    ids, launches = [], []
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for var, bps, ch, ns in matrix():
            p = make_packer(R, var, bps, ch, ns)
            if p is None:
                continue
            rng = np.random.default_rng(1000 * bps + 10 * ch + ns)
            for cid, thunk in calls(torch, np, p, rng):
                torch.cuda.synchronize()
                marker.add_(1)  # opens the call's window in the trace
                before = p.counters()["kernel_launches"]
                thunk()
                torch.cuda.synchronize()
                launches.append(p.counters()["kernel_launches"] - before)
                ids.append(f"{var}/bps{bps}/ch{ch}/ns{ns}/{cid}")
            p.close()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    kernels = sorted((e for e in events if e.get("cat") == "kernel"), key=lambda e: e["ts"])
    marker_name = kernels[0]["name"]  # the first kernel of the trace is a marker
    windows: list[dict[int, list]] = []
    for e in kernels:
        if e["name"] == marker_name:
            windows.append({})
            continue
        if not LIB_KERNEL.search(e["name"]):
            continue  # torch's own, such as debug_planes' header buffer fill
        a = e.get("args", {})
        k = [e["name"].split("(")[0], a.get("grid"), a.get("block"), a.get("shared memory")]
        windows[-1].setdefault(a.get("stream"), []).append(k)
    assert len(windows) == len(ids), f"{len(windows)} call windows in the trace for {len(ids)} calls"
    # per call: the kernel sequence of each stream, streams in a canonical order (stream ids are not stable)
    rows = [{"id": i, "launches": n, "kernels": sorted(w.values())} for i, n, w in zip(ids, launches, windows)]
    with open(out_path, "w") as f:
        json.dump({"lib": lib_path, "calls": rows}, f, indent=0)
    print(f"{len(rows)} calls, {sum(len(s) for r in rows for s in r['kernels'])} kernel launches traced -> {out_path}")


def compare(a_path: str, b_path: str) -> int:
    a, b = (json.load(open(x))["calls"] for x in (a_path, b_path))
    if [r["id"] for r in a] != [r["id"] for r in b]:
        print("the two traces ran different call lists")
        return 1
    diff = [(x, y) for x, y in zip(a, b) if x != y]
    for x, y in diff:
        print(x["id"], "launches", x["launches"], "->", y["launches"])
        print("   ", x["kernels"])
        print("   ", y["kernels"])
    print(f"{len(a)} calls, {len(diff)} differ")
    return 0


if __name__ == "__main__":
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--lib", help="librspt_gpu.so to trace")
    ap.add_argument("--out", help="JSON file to write")
    ap.add_argument("--compare", nargs=2, metavar=("A", "B"), help="print the calls whose launches differ")
    ap.add_argument("--list", action="store_true", help="print the (packer, bps, ch, ns) matrix and exit")
    args = ap.parse_args()
    if args.list:
        for m in matrix():
            print(*m)
    elif args.compare:
        sys.exit(compare(*args.compare))
    else:
        if not (args.lib and args.out):
            ap.error("--lib and --out are required to trace")
        trace(args.lib, args.out)
