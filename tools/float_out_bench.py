"""What float32 / bfloat16 output of decompress costs against int32 output and against converting in torch, device
resident, per 4096-frame batch.

    python tools/float_out_bench.py [--frames 4096] [--batches 24] [--reps 5] [--out profiles/r08_float_out.json]

Packers and shapes as tools/i32_io_bench.py (xdelta_hzr and hzr on shape A, hadamard and dct on shape B: bench.py's
shapes); `batches` distinct batches, each larger than the 126 MB L2, timed with CUDA events, arms alternating,
median of `reps`:
  i32         decompress_tensor
  f32, bf16   decompress_tensor(dtype=...) with a per-channel zero point and scale (dequantized in the kernels)
  torch_f32   decompress_tensor, then (x.long() - zp).float() * scale in torch
  torch_bf16  the same, then .to(torch.bfloat16)
Before timing, the fused outputs are checked against the torch arms bit for bit.  The INVERSE stage time of every arm
comes from a separate untimed pass.  Gather rows: a store of 16 batches, B = 256 and B = 4096 random ids,
decompress_frames_tensor bf16 against int32 + torch.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from i32_io_bench import PACKERS, SHAPES, gpu_info, timed  # noqa: E402


def stats(v):
    return {"median": float(np.median(v)), "min": float(min(v)), "max": float(max(v)), "all": v}


def params(torch, ch, dev):
    g = torch.Generator().manual_seed(7)
    zp = torch.randint(-2000, 2000, (ch,), dtype=torch.int32, generator=g).to(dev)
    scale = (torch.rand(ch, generator=g) * 4e-3 + 1e-4).to(dev)
    return zp, scale


def measure(R, torch, kind, sh, F, nbatch, reps):
    dev = torch.device("cuda", torch.cuda.current_device())
    bps, ch, ns = sh["bps"], sh["ch"], sh["ns"]
    p = R.SignalPacker(kind, bps, ch, ns, 3, max_batch_frames=F)
    out = p.alloc_output(F, sidecar=True)
    comps = []
    for i in range(nbatch):
        b = p.compress_batch(R.synth_ecg(i * F, F, **sh), out=out)
        total = int(b.offsets[-1].item())
        comps.append(R.CompressedBatch(b.stream[: total + 64].clone(), b.offsets.clone(), b.frame_nb.clone(),
                                       b.sidecar[: p.sidecar_used_bytes(F, total)].clone(), F))
    del out
    zp, scale = params(torch, ch, dev)
    zp3, sc3 = zp[None, :, None], scale[None, :, None]
    d_i32 = torch.empty((F, ch, ns), dtype=torch.int32, device=dev)
    d_f32 = torch.empty((F, ch, ns), dtype=torch.float32, device=dev)
    d_bf16 = torch.empty((F, ch, ns), dtype=torch.bfloat16, device=dev)
    kw = dict(zero_point=zp, scale=scale)
    arms = {
        "i32": lambda i: p.decompress_tensor(comps[i % nbatch], out=d_i32),
        "f32": lambda i: p.decompress_tensor(comps[i % nbatch], out=d_f32, dtype=torch.float32, **kw),
        "bf16": lambda i: p.decompress_tensor(comps[i % nbatch], out=d_bf16, dtype=torch.bfloat16, **kw),
        "torch_f32": lambda i: (p.decompress_tensor(comps[i % nbatch], out=d_i32).long() - zp3).float() * sc3,
        "torch_bf16": lambda i: ((p.decompress_tensor(comps[i % nbatch], out=d_i32).long() - zp3).float() * sc3).bfloat16(),
    }
    # bit-exact before timing
    ref = arms["torch_f32"](0)
    f = arms["f32"](0)
    eq_f32 = bool(torch.equal(f.view(torch.int32), ref.view(torch.int32)))
    bf = arms["bf16"](0)
    eq_bf16 = bool(torch.equal(bf.view(torch.int16), ref.bfloat16().view(torch.int16)))
    del ref
    assert eq_f32 and eq_bf16, (kind, eq_f32, eq_bf16)
    for a in arms.values():
        timed(torch, a, 2)
    res = {a: [] for a in arms}
    for _ in range(reps):
        for a, fn in arms.items():
            res[a].append(timed(torch, fn, nbatch))
    stages = {}
    for a, fn in arms.items():
        p.set_stage_timing(True)
        p.stage_times(reset=True)
        for i in range(nbatch):
            fn(i)
        torch.cuda.synchronize()
        st = p.stage_times(reset=True)
        p.set_stage_timing(False)
        stages[a] = {k: st[k][0] / max(1, st[k][1]) for k in ("parse", "decode", "inverse")}
    r = {"kind": kind, "shape": sh, "frames_per_batch": F, "batches": nbatch, "reps": reps,
         "checks": {"f32_equal_torch": eq_f32, "bf16_equal_torch": eq_bf16},
         "decompress_ms": {a: stats(v) for a, v in res.items()}, "stage_ms_per_call": stages}
    p.close()
    return r


def gather(R, torch, reps):
    """A store of 16 4096-frame batches (shape A, xdelta_hzr); B random ids: bf16 gather against int32 + torch."""
    dev = torch.device("cuda", torch.cuda.current_device())
    sh, F, nb = SHAPES["A"], 4096, 16
    p = R.SignalPacker("xdelta_hzr", sh["bps"], sh["ch"], sh["ns"], 3, max_batch_frames=F)
    store = p.new_store(nb * F, bytes_capacity=nb * F * sh["ch"] * sh["ns"] * 2)
    for i in range(nb):
        p.append_batch(store, R.synth_ecg(i * F, F, **sh))
    zp, scale = params(torch, sh["ch"], dev)
    zp3, sc3 = zp[None, :, None], scale[None, :, None]
    rows = []
    g = torch.Generator().manual_seed(11)
    for B in (256, 4096):
        ids = [torch.randint(0, store.n_frames, (B,), generator=g).to(dev) for _ in range(8)]
        arms = {
            "bf16": lambda i: p.decompress_frames_tensor(store, ids[i % 8], dtype=torch.bfloat16, zero_point=zp, scale=scale),
            "torch_bf16": lambda i: ((p.decompress_frames_tensor(store, ids[i % 8]).long() - zp3).float() * sc3).bfloat16(),
        }
        a, b = arms["bf16"](0), arms["torch_bf16"](0)
        assert torch.equal(a.view(torch.int16), b.view(torch.int16))
        for fn in arms.values():
            timed(torch, fn, 2)
        res = {k: [] for k in arms}
        for _ in range(reps):
            for k, fn in arms.items():
                res[k].append(timed(torch, fn, 16))
        rows.append({"B": B, "store_frames": store.n_frames, "ms": {k: stats(v) for k, v in res.items()}})
    p.close()
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=4096)
    ap.add_argument("--batches", type=int, default=24)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_float_out.json"))
    args = ap.parse_args()
    import torch
    from rspt_b200 import packer as R
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.cuda.current_device()
    results = {"gpu": gpu_info(dev), "packers": []}
    for kind, shape in PACKERS:
        r = measure(R, torch, kind, SHAPES[shape], args.frames, args.batches, args.reps)
        results["packers"].append(r)
        torch.cuda.empty_cache()
        print(json.dumps({"kind": kind, **{a: round(v["median"], 3) for a, v in r["decompress_ms"].items()},
                          "inverse_ms": {a: round(v["inverse"], 3) for a, v in r["stage_ms_per_call"].items()}}), flush=True)
    results["gather"] = gather(R, torch, args.reps)
    print(json.dumps([{"B": g["B"], **{k: round(v["median"], 3) for k, v in g["ms"].items()}} for g in results["gather"]]))
    results["gpu_after"] = gpu_info(dev)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
