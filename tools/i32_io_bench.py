"""What the int32 [F, ch, ns] entry points cost against the native ones, device resident, per 4096-frame batch.

    python tools/i32_io_bench.py [--frames 4096] [--batches 24] [--reps 5] [--out profiles/r04_i32_io.json]

Three arms per packer (xdelta_hzr and hzr on shape A, hadamard and dct on shape B: bench.py's shapes), timed with
CUDA events over `batches` distinct batches (each larger than the 126 MB L2), alternating arm by arm:
  i32     compress_tensor / decompress_tensor on int32 [F, ch, ns]
  native  compress_batch / decompress_batch on interleaved native bytes (no conversion: the lower bound)
  torch   what a torch caller without the new calls does: int32 [F, ch, ns] -> native bytes in torch, then
          compress_batch; decompress_batch, then native bytes -> int32 [F, ch, ns] in torch
Before timing, the i32 batch and decode are checked against the native ones.  Stage times (CUDA events inside the
library) come from a separate untimed pass.  The transform kernel's share of the copy rate is its bytes (4 B read +
nb_alloc B written per sample) over its stage time, against a device-to-device copy measured in the same run.
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
PACKERS = (("xdelta_hzr", "A"), ("hzr", "A"), ("hadamard", "B"), ("dct", "B"))


def native_to_words(torch, raw, F, bps, ch, ns, out=None):
    """uint8 [F * ns * ch * bps] interleaved -> int32 [F, ch, ns] sign-extended, in torch."""
    b = raw.view(F, ns, ch, bps)
    w = b[..., bps - 1].view(torch.int8).to(torch.int32) * (1 << (8 * (bps - 1)))
    for k in range(bps - 1):
        w += b[..., k].to(torch.int32) * (1 << (8 * k))
    w = w.permute(0, 2, 1)
    if out is None:
        return w.contiguous()
    return out.copy_(w)


def words_to_native(torch, words, F, bps, ch, ns, out):
    """int32 [F, ch, ns] -> the low bps bytes of every word, interleaved [F, ns, ch, bps], in torch (one copy)."""
    out.view(F, ns, ch, bps).copy_(words.view(torch.uint8).view(F, ch, ns, 4)[..., :bps].permute(0, 2, 1, 3))
    return out


def timed(torch, fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def copy_rate(torch, dev, nbytes):
    """Bytes moved (read + written) per second by a device-to-device copy of nbytes, best of 5 after a warm-up."""
    a = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    b = torch.empty_like(a)
    b.copy_(a)
    ms = min(timed(torch, lambda i: b.copy_(a), 4) for _ in range(5))
    return 2 * nbytes / (ms * 1e-3)


def gpu_info(dev: int) -> dict:
    q = subprocess.run(["nvidia-smi", "-i", str(dev), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip()
    name, power, clk = [s.strip() for s in q.split(",")]
    return {"name": name, "power_limit": power, "clocks_max_sm": clk}


def measure(R, torch, kind, sh, F, nbatch, reps):
    dev = torch.device("cuda", torch.cuda.current_device())
    bps, ch, ns = sh["bps"], sh["ch"], sh["ns"]
    fb = bps * ch * ns
    p = R.SignalPacker(kind, bps, ch, ns, 3, max_batch_frames=F)
    native = [R.synth_ecg(i * F, F, **sh) for i in range(nbatch)]
    words = [native_to_words(torch, x, F, **sh) for x in native]
    outs = [p.alloc_output(F, sidecar=True) for _ in range(2)]
    # the batches the decompress arms decode: the stream up to its last byte and the used part of the decode index
    comps = []
    for i in range(nbatch):
        b = p.compress_batch(native[i], out=outs[0])
        total = int(b.offsets[-1].item())
        comps.append(R.CompressedBatch(b.stream[: total + 64].clone(), b.offsets.clone(), b.frame_nb.clone(),
                                       b.sidecar[: p.sidecar_used_bytes(F, total)].clone(), F))
    # equality before timing
    bw = p.compress_tensor(words[0], out=outs[1])
    bn = p.compress_batch(native[0], out=outs[0])
    torch.cuda.synchronize()
    total = int(bn.offsets[-1].item())
    same_stream = bool(torch.equal(bw.offsets, bn.offsets) and torch.equal(bw.stream[:total], bn.stream[:total])
                       and torch.equal(bw.frame_nb, bn.frame_nb))
    dec_raw = torch.empty(F * fb, dtype=torch.uint8, device=dev)
    dec_w = torch.empty((F, ch, ns), dtype=torch.int32, device=dev)
    tmp_raw = torch.empty(F * fb, dtype=torch.uint8, device=dev)
    p.decompress_tensor(comps[0], out=dec_w)
    p.decompress_batch(comps[0], out=dec_raw)
    same_decode = bool(torch.equal(dec_w, native_to_words(torch, dec_raw, F, **sh)))
    lossless_ok = bool(torch.equal(dec_w, words[0])) if kind in ("xdelta_hzr", "hzr") else None
    assert same_stream and same_decode and lossless_ok in (True, None), (kind, same_stream, same_decode, lossless_ok)

    arms = {
        "i32": (lambda i: p.compress_tensor(words[i % nbatch], out=outs[i & 1]),
                lambda i: p.decompress_tensor(comps[i % nbatch], out=dec_w)),
        "native": (lambda i: p.compress_batch(native[i % nbatch], out=outs[i & 1]),
                   lambda i: p.decompress_batch(comps[i % nbatch], out=dec_raw)),
        "torch": (lambda i: p.compress_batch(words_to_native(torch, words[i % nbatch], F, bps, ch, ns, tmp_raw), out=outs[i & 1]),
                  lambda i: native_to_words(torch, p.decompress_batch(comps[i % nbatch], out=dec_raw), F, bps, ch, ns, out=dec_w)),
    }
    for c, d in arms.values():   # warm-up of every arm and shape
        timed(torch, c, 2)
        timed(torch, d, 2)
    res = {a: {"compress_ms": [], "decompress_ms": []} for a in arms}
    for _ in range(reps):
        for a, (c, d) in arms.items():
            res[a]["compress_ms"].append(timed(torch, c, nbatch))
            res[a]["decompress_ms"].append(timed(torch, d, nbatch))
    # stage times, separate untimed pass
    stages = {}
    for a in ("i32", "native"):
        c, d = arms[a]
        p.set_stage_timing(True)
        p.stage_times(reset=True)
        for i in range(nbatch):
            c(i)
            d(i)
        torch.cuda.synchronize()
        st = p.stage_times(reset=True)
        p.set_stage_timing(False)
        stages[a] = {k: st[k][0] / max(1, st[k][1]) for k in ("transform", "inverse")}
    out = {"kind": kind, "shape": sh, "frames_per_batch": F, "batches": nbatch, "reps": reps,
           "batch_bytes": {"native": F * fb, "int32": F * ch * ns * 4},
           "checks": {"stream_equal": same_stream, "decode_equal": same_decode, "lossless_round_trip": lossless_ok},
           "stage_ms_per_call": stages}
    for a in arms:
        for k in ("compress_ms", "decompress_ms"):
            v = res[a][k]
            out.setdefault(a, {})[k] = {"median": float(np.median(v)), "min": float(min(v)), "max": float(max(v)), "all": v}
    if kind in ("xdelta_hzr", "hzr"):
        nb_alloc = 3 if kind == "xdelta_hzr" else 4
        out["transform_bytes_i32"] = F * ch * ns * (4 + nb_alloc)
    p.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=4096)
    ap.add_argument("--batches", type=int, default=24)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_i32_io.json"))
    args = ap.parse_args()
    import torch
    from rspt_b200 import packer as R
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.cuda.current_device()
    info = gpu_info(dev)
    results = {"gpu": info, "packers": []}
    for kind, shape in PACKERS:
        r = measure(R, torch, kind, SHAPES[shape], args.frames, args.batches, args.reps)
        results["packers"].append(r)
        torch.cuda.empty_cache()
        print(json.dumps({k: r[k] for k in ("kind", "i32", "native", "torch", "stage_ms_per_call")}, default=str), flush=True)
    xd = results["packers"][0]
    cr = copy_rate(torch, torch.device("cuda", dev), xd["transform_bytes_i32"] // 2)
    t_ms = xd["stage_ms_per_call"]["i32"]["transform"]
    results["copy_rate_bytes_per_s"] = cr
    results["xdelta_i32_transform"] = {"bytes": xd["transform_bytes_i32"], "stage_ms": t_ms,
                                       "bytes_per_s": xd["transform_bytes_i32"] / (t_ms * 1e-3),
                                       "share_of_copy_rate": xd["transform_bytes_i32"] / (t_ms * 1e-3) / cr}
    results["gpu_after"] = gpu_info(dev)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(results, f, indent=1)
    print(json.dumps({"gpu": info, "copy_rate_TBps": cr / 1e12, "xdelta_i32_transform": results["xdelta_i32_transform"]}))


if __name__ == "__main__":
    main()
