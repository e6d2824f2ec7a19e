#!/usr/bin/env python
"""Benchmark of the signal-packer hot path (BASELINE.json: compress/decompress raw GB/s per packer, CR,
% HBM roofline).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Headline = BASELINE configs[1]: xdelta_hzr, 12 ch x 3 B x 8192 samples, synthetic ECG-like frames generated on
the device.  A STEP is one pass of the packer over `--batches` distinct batches of `--frames` frames per GPU
(24 x 4096 frames = 29 GB of raw input per step and GPU: every batch is far larger than the 126 MB L2 and no
batch repeats inside a step).  `value` is raw-input GB/s with the inputs resident in HBM; `e2e` is the same
metric through the host-buffer C-ABI call (pinned host memory, H2D + D2H inside the timed region).
`packers` carries, for each of the four packers and BOTH directions, the device-resident rate, its roofline
block (algorithmic bytes R + C resp. C + R + the decode-index bytes actually read), the host-buffer rate and a
single-core CPU baseline of the unmodified reference on a bounded sample of the same frames.
One JSON line on stdout (rank 0).

`--impl reference` times the reference's own CPU implementation (oracle/_ref/libref.so when it was built in
the container, else the oracle port) on this box's host cores.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SHAPES = {  # SURVEY.md section 8: A = config 2, B = configs 3/4, C = config 1
    "A": dict(bps=3, ch=12, ns=8192),
    "B": dict(bps=4, ch=12, ns=4096),
    "C": dict(bps=4, ch=1, ns=8192),
}
WORKLOAD = "xdelta_hzr batched: 12 ch x 3 B/sample x 8192 samples, synthetic ECG-like frames (BASELINE configs[1])"
PACKERS = (("xdelta_hzr", "A"), ("hzr", "A"), ("hadamard", "B"), ("dct", "B"))  # BASELINE configs[1..3] + hzr


def base_config(args, world):
    """The keys both arms report (the driver compares the two dicts)."""
    sh = SHAPES["A"]
    return {"workload": WORKLOAD, "packer": "xdelta_hzr", "bps": sh["bps"], "ch": sh["ch"], "ns": sh["ns"], "nb": 3,
            "data": "synthetic ECG-like, seed 42 (include/rspt_synth.h)"}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
            time.sleep(0.2)   # the first sample takes a moment
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.1)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU side: the unmodified reference (oracle/_ref/libref.so) or, without it, the oracle port
# ------------------------------------------------------------------------------------------------
def cpu_impl():
    from oracle import oracle as O
    impl = "reference" if O.ref_available() else "port"
    if impl == "port":
        O.build(ref=False)
    return O, impl


def run_reference(args):
    """The reference's CPU packer on the host cores: one packer instance per thread, each looping
    compress over its own frames (ctypes releases the GIL)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    O, impl = cpu_impl()
    sh = SHAPES["A"]
    fb = sh["bps"] * sh["ch"] * sh["ns"]
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    threads = max(1, min(cores, args.cpu_threads or cores))
    per = args.cpu_frames_per_thread
    frames = O.synth_ecg(0, threads * per, sh["bps"], sh["ch"], sh["ns"]).reshape(threads, per, fb)
    packers = [O.make_packer("xdelta_hzr", sh["bps"], sh["ch"], sh["ns"], 3, impl) for _ in range(threads)]
    sizes = [None] * threads

    def work(i):
        _, sz = packers[i].compress_many(frames[i])
        sizes[i] = sz

    def step():
        ts = [threading.Thread(target=work, args=(i,)) for i in range(threads)]
        t0 = time.perf_counter()
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        return time.perf_counter() - t0

    for _ in range(args.warmup):
        step()
    el = [step() for _ in range(args.steps)]
    total = sum(el)
    raw = args.steps * threads * per * fb
    gbs = raw / total / 1e9
    comp = sum(int(s.sum()) for s in sizes)
    cfg = base_config(args, 1)
    cfg.update({"frames_per_step": threads * per, "cr": threads * per * fb / comp})
    line = {
        "impl": "reference", "metric": "compress_raw_GBps", "value": gbs, "unit": "GB/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": cfg,
        "cpu_baseline": {"value": gbs, "unit": "GB/s", "cores": threads, "kind": impl,
                         "sample": f"{threads} threads x {per} frames x {args.steps} steps, compress only "
                                   f"(includes the reference's built-in verify-decode)"},
        "e2e": {"value": gbs, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


def cpu_baseline(kind: str, raw_frames: np.ndarray, sh: dict, budget_s: float) -> dict:
    """Reference CPU packer, single-threaded instances, on a bounded sample of the same frames (rank 0, N = 1).
    dct costs ~2 s per frame on one core, so its sample is one frame on each of up to 8 cores."""
    O, impl = cpu_impl()
    fb = sh["bps"] * sh["ch"] * sh["ns"]
    frames = raw_frames.reshape(-1, fb)
    if kind == "dct":
        cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
        nthr = max(1, min(8, cores, frames.shape[0]))
        packers = [O.make_packer(kind, sh["bps"], sh["ch"], sh["ns"], 3, impl) for _ in range(nthr)]
        outs = [None] * nthr
        tc = [0.0] * nthr
        td = [0.0] * nthr

        def work(i):
            t0 = time.perf_counter()
            dst, _ = packers[i].compress_many(frames[i:i + 1])
            tc[i] = time.perf_counter() - t0
            t0 = time.perf_counter()
            packers[i].decompress_many(dst, 1)
            td[i] = time.perf_counter() - t0

        ts = [threading.Thread(target=work, args=(i,)) for i in range(nthr)]
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        return {"value": fb / (sum(tc) / nthr) / 1e9, "decompress_value": fb / (sum(td) / nthr) / 1e9, "unit": "GB/s", "cores": 1,
                "kind": impl, "sample": f"{nthr} frames, one per host thread, per-core rate ({max(tc) + max(td):.1f} s)"}
    p = O.make_packer(kind, sh["bps"], sh["ch"], sh["ns"], 3, impl)
    t0 = time.perf_counter()
    p.compress_many(frames[:4])
    per = (time.perf_counter() - t0) / 4
    n = int(max(4, min(frames.shape[0], budget_s * 0.6 / per)))
    t0 = time.perf_counter()
    dst, sizes = p.compress_many(frames[:n])
    tc = time.perf_counter() - t0
    t0 = time.perf_counter()
    p.decompress_many(dst, n)
    td = time.perf_counter() - t0
    return {"value": n * fb / tc / 1e9, "decompress_value": n * fb / td / 1e9, "unit": "GB/s", "cores": 1, "kind": impl,
            "sample": f"{n} of the benchmark's frames, compress then decompress, 1 thread ({tc + td:.1f} s)"}


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
class Dist:
    """torch.distributed for rendezvous / barriers / max-reductions; the path's own collective (all-gather of the
    per-rank byte totals) goes through the C ABI on a communicator made from a broadcast NCCL unique id."""

    def __init__(self, torch, dev):
        import torch.distributed as dist
        from rspt_b200 import dist as RD
        from rspt_b200 import _lib
        self.torch, self.dist, self.dev = torch, dist, dev
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.comm = C.c_void_p()
        if self.world > 1:
            RD.init_process_group_quiet(dev)      # keeps NCCL's banner off stdout
            L = _lib.lib()
            uid = torch.zeros(128, dtype=torch.uint8)
            if self.rank == 0:
                buf = (C.c_uint8 * 128)()
                _lib.check(L.rspt_gpu_comm_unique_id(buf), None, "rspt_gpu_comm_unique_id")
                uid = torch.tensor(list(buf), dtype=torch.uint8)
            uid = uid.to(dev)
            dist.broadcast(uid, 0)
            host = (C.c_uint8 * 128)(*uid.cpu().tolist())
            sys.stdout.flush()
            saved = os.dup(1)
            os.dup2(2, 1)
            try:
                _lib.check(L.rspt_gpu_comm_init(self.world, host, self.rank, dev.index, C.byref(self.comm)), None, "rspt_gpu_comm_init")
                torch.cuda.synchronize(dev)
            finally:
                sys.stdout.flush()
                os.dup2(saved, 1)
                os.close(saved)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max(self, x: float) -> float:
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum(self, x: float) -> float:
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return float(t.item())

    def close(self):
        if self.world > 1:
            from rspt_b200 import _lib
            _lib.lib().rspt_gpu_comm_destroy(self.comm)
            self.dist.destroy_process_group()


def timed(torch, fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e-3


def copy_ceiling(torch, dev, h2d_bytes: int, d2h_bytes: int, reps: int = 3, barrier=None) -> float:
    """Seconds for plain pinned H2D + D2H copies of the same sizes, both directions at once (what the link gives
    a host-buffer call that does nothing else).  At N > 1 every repetition starts behind a barrier, so that all
    ranks copy at the same time as they do in the e2e legs; the mean of the repetitions after one warm-up."""
    hs = torch.empty(h2d_bytes, dtype=torch.uint8, pin_memory=True)
    hd = torch.empty(d2h_bytes, dtype=torch.uint8, pin_memory=True)
    ds = torch.empty(h2d_bytes, dtype=torch.uint8, device=dev)
    dd = torch.empty(d2h_bytes, dtype=torch.uint8, device=dev)
    s1, s2 = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    torch.cuda.synchronize()
    total = 0.0
    for r in range(reps + 1):
        if barrier is not None:
            barrier()
        t0 = time.perf_counter()
        with torch.cuda.stream(s1):
            ds.copy_(hs, non_blocking=True)
        with torch.cuda.stream(s2):
            hd.copy_(dd, non_blocking=True)
        torch.cuda.synchronize()
        if r > 0:
            total += time.perf_counter() - t0
    return total / reps


def measure_packer(R, torch, D, kind, sh, F, nbatch, reps, hbm_peak, e2e_frames, cpu_budget, want_cpu, stage_roofline=False):
    """Both directions of one packer: device resident (inputs in HBM) and through the host-buffer calls."""
    dev = D.dev
    fb = sh["bps"] * sh["ch"] * sh["ns"]
    raw_batch = F * fb
    p = R.SignalPacker(kind, sh["bps"], sh["ch"], sh["ns"], 3, max_batch_frames=F)
    first = D.rank * nbatch * F
    inputs = [R.synth_ecg(first + i * F, F, **sh) for i in range(nbatch)]
    outs = [p.alloc_output(F, sidecar=True) for _ in range(2)]
    dec = torch.empty(raw_batch, dtype=torch.uint8, device=dev)

    def comp(i):
        b = p.compress_batch(inputs[i % nbatch], out=outs[i & 1])
        if D.world > 1:   # the path's only collective, off the compute stream
            p.place_offsets_async(D.comm, b, D.rank, D.world)
        return b

    for i in range(2):
        comp(i)
    p.place_join()
    D.barrier()
    c0 = p.counters()["kernel_launches"]
    tc = D.max(timed(torch, comp, reps * nbatch))
    p.place_join()
    torch.cuda.synchronize()
    launches = p.counters()["kernel_launches"] - c0
    b = p.compress_batch(inputs[0], out=outs[0])
    torch.cuda.synchronize()
    comp_bytes = int(b.offsets[F].item()) - int(b.offsets[0].item())
    idx_bytes = p.sidecar_used_bytes(F, comp_bytes)
    for _ in range(2):
        p.decompress_batch(b, out=dec)
    D.barrier()
    nd = max(3, (reps * nbatch) // 2)
    td = D.max(timed(torch, lambda i: p.decompress_batch(b, out=dec), nd))
    r = {"shape": sh, "frames_per_batch_per_gpu": F, "batches": nbatch, "cr": raw_batch / comp_bytes,
         "index_bytes_per_frame": idx_bytes / F, "cr_including_index": raw_batch / (comp_bytes + idx_bytes)}
    if kind in ("hadamard", "dct"):
        r["prdn_percent"] = R.prdn(inputs[0], dec, F, sh["bps"], sh["ch"], sh["ns"])
    else:
        r["roundtrip_bit_exact"] = bool(torch.equal(inputs[0], dec))
    cgb = D.world * reps * nbatch * raw_batch / tc / 1e9
    dgb = D.world * nd * raw_batch / td / 1e9
    r["compress"] = {"raw_GBps": cgb, "ms_per_batch": 1e3 * tc / (reps * nbatch),
                     "roofline": {"bound": "hbm", "algorithmic_bytes_per_batch": raw_batch + comp_bytes,
                                  "achieved": (raw_batch + comp_bytes) * reps * nbatch / tc / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                  "frac": (raw_batch + comp_bytes) * reps * nbatch / tc / 1e9 / hbm_peak}}
    r["decompress"] = {"raw_GBps": dgb, "ms_per_batch": 1e3 * td / nd,
                       "roofline": {"bound": "hbm", "algorithmic_bytes_per_batch": raw_batch + comp_bytes + idx_bytes,
                                    "index_bytes_read_per_batch": idx_bytes,
                                    "achieved": (raw_batch + comp_bytes + idx_bytes) * nd / td / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                    "frac": (raw_batch + comp_bytes + idx_bytes) * nd / td / 1e9 / hbm_peak}}
    if stage_roofline:
        p.set_stage_timing(True)
        p.stage_times(reset=True)
        for i in range(4):
            p.compress_batch(inputs[i % nbatch], out=outs[i & 1])
        for _ in range(4):
            p.decompress_batch(b, out=dec)
        st = p.stage_times(reset=True)
        p.set_stage_timing(False)
        r["stage_ms"] = {k: (v[0] / v[1] if v[1] else 0.0) for k, v in st.items()}
    # ---- host buffers in, host buffers out (pinned), through the C-ABI host calls
    Fe = min(F, e2e_frames)
    h_raw = torch.empty(Fe * fb, dtype=torch.uint8, pin_memory=True)
    h_raw.copy_(inputs[0][: Fe * fb])
    h_cmp = torch.empty(Fe * p.max_compressed_size, dtype=torch.uint8, pin_memory=True)
    h_off = torch.empty(Fe + 1, dtype=torch.int64, pin_memory=True)
    h_back = torch.empty(Fe * fb, dtype=torch.uint8, pin_memory=True)
    pe = R.SignalPacker(kind, sh["bps"], sh["ch"], sh["ns"], 3, max_batch_frames=Fe)
    np_raw, np_cmp, np_off, np_back = h_raw.numpy(), h_cmp.numpy(), h_off.numpy().view(np.uint64), h_back.numpy()
    tot = pe.compress_batch_host(np_raw, np_cmp, np_off)
    pe.decompress_batch_host(np_cmp, np_off, np_back)
    D.barrier()
    ne = 3
    t0 = time.perf_counter()
    for _ in range(ne):
        tot = pe.compress_batch_host(np_raw, np_cmp, np_off)
    torch.cuda.synchronize()
    tec = D.max(time.perf_counter() - t0)
    D.barrier()
    t0 = time.perf_counter()
    for _ in range(ne):
        pe.decompress_batch_host(np_cmp, np_off, np_back)
    torch.cuda.synchronize()
    ted = D.max(time.perf_counter() - t0)
    if kind in ("xdelta_hzr", "hzr"):
        r["e2e_roundtrip_bit_exact"] = bool(np.array_equal(np_back, np_raw))
    ceil_c = D.max(copy_ceiling(torch, dev, Fe * fb, int(tot) + 8 * (Fe + 1), barrier=D.barrier))
    ceil_d = D.max(copy_ceiling(torch, dev, int(tot) + 8 * (Fe + 1), Fe * fb, barrier=D.barrier))
    r["compress"]["e2e"] = {"value": D.world * ne * Fe * fb / tec / 1e9, "unit": "GB/s", "h2d_bytes_per_step": Fe * fb,
                            "d2h_bytes_per_step": int(tot) + 8 * (Fe + 1), "frames_per_step": Fe,
                            "api": "rspt_gpu_compress_batch_host (pinned host buffers)",
                            "plain_copy_ceiling_GBps": D.world * Fe * fb / ceil_c / 1e9,
                            "frac_of_copy_ceiling": (ne * Fe * fb / tec) / (Fe * fb / ceil_c)}
    r["decompress"]["e2e"] = {"value": D.world * ne * Fe * fb / ted / 1e9, "unit": "GB/s", "h2d_bytes_per_step": int(tot) + 8 * (Fe + 1),
                              "d2h_bytes_per_step": Fe * fb, "frames_per_step": Fe,
                              "api": "rspt_gpu_decompress_batch_host (pinned host buffers, no decode index given)",
                              "plain_copy_ceiling_GBps": D.world * Fe * fb / ceil_d / 1e9,
                              "frac_of_copy_ceiling": (ne * Fe * fb / ted) / (Fe * fb / ceil_d)}
    pe.close()
    if want_cpu:
        nsample = 4096 if kind != "dct" else 8
        cb = cpu_baseline(kind, inputs[0][: min(F, nsample) * fb].cpu().numpy(), sh, cpu_budget)
        r["compress"]["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
        r["decompress"]["cpu_baseline"] = {"value": cb["decompress_value"], "unit": "GB/s", "cores": cb["cores"], "kind": cb["kind"],
                                           "sample": cb["sample"]}
    r["gpu_launches_timed_compress"] = int(launches)
    p.close()
    del inputs, outs, dec
    torch.cuda.empty_cache()
    return r


DUMP_FRAMES = 16          # frames per batch whose compressed bytes are dumped
DUMP_INDEX_BYTES = 1 << 19  # decode-index bytes dumped per batch


def dump_outputs(torch, p, outs, nb, F, out_dir):
    """What a caller of the timed path received in the last step, as .npy files: the batches still held in
    `outs` (the step's last two; the outputs alternate between two buffers).  Per batch the frame offsets and
    plane counts in full, the compressed bytes of a fixed sample of frames and a fixed sample of the decode
    index.  At most 2 x 16 x max_compressed_size x 4 B of stream plus 4 MB of index: under 64 MB."""
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(0)
    frames = np.sort(rng.choice(F, size=min(DUMP_FRAMES, F), replace=False))
    arrays = {"sample_frames": frames.astype(np.float64)}
    for i in range(max(0, nb - 2), nb):
        b = outs[i & 1]
        offs = b.offsets[: F + 1].cpu().numpy()
        stream = np.concatenate([b.stream[int(offs[f]):int(offs[f + 1])].cpu().numpy() for f in frames])
        used = p.sidecar_used_bytes(F, int(offs[F]))
        pos = np.sort(rng.choice(used, size=min(DUMP_INDEX_BYTES, used), replace=False))
        index = b.sidecar[torch.from_numpy(pos).to(b.sidecar.device)].cpu().numpy()
        arrays.update({f"batch{i}_offsets": offs.astype(np.float64), f"batch{i}_frame_nb": b.frame_nb[:F].cpu().numpy().astype(np.float32),
                       f"batch{i}_stream_sample": stream.astype(np.float32), f"batch{i}_index_sample": index.astype(np.float32)})
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_ours(args):
    import torch
    from rspt_b200 import packer as R

    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; this benchmark has no CPU path (use --impl reference)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    D = Dist(torch, dev)
    world, rank = D.world, D.rank
    sh = SHAPES["A"]
    fb = sh["bps"] * sh["ch"] * sh["ns"]
    F, NB = args.frames, args.batches
    hbm_peak, peak_src = peaks()

    # ---- headline: xdelta_hzr compress, device resident; a step = NB distinct batches of F frames
    p = R.SignalPacker.new_xdelta_hzr(sh["bps"], sh["ch"], sh["ns"], 3, max_batch_frames=F)
    first = rank * NB * F  # contiguous shard of the global frame index space per rank
    inputs = [R.synth_ecg(first + i * F, F, **sh) for i in range(NB)]
    outs = [p.alloc_output(F, sidecar=True) for _ in range(2)]

    no_place = os.environ.get("BENCH_NO_PLACE") == "1"   # diagnosis only: leaves the collective out

    def step(_):
        for i in range(NB):
            b = p.compress_batch(inputs[i], out=outs[i & 1])
            if world > 1 and not no_place:
                # the path's only collective: 8 bytes per rank, places this shard in the global stream;
                # issued on the handle's side stream so that the next batch's kernels start at once
                p.place_offsets_async(D.comm, b, rank, world)
        if world > 1:
            p.place_join()

    for i in range(args.warmup):
        step(i)
    D.barrier()
    c0 = p.counters()["kernel_launches"]
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    D.barrier()   # the sampler start takes 0.2 s on rank 0: without this the other ranks' timed region would hold that wait
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        step(i)
    e1.record()
    D.barrier()
    ms = D.max(e0.elapsed_time(e1))
    clocks = sampler.stop() if rank == 0 else None
    launches = p.counters()["kernel_launches"] - c0
    if args.dump_outputs and rank == 0:
        dump_outputs(torch, p, outs, NB, F, args.dump_outputs)
    raw_step = NB * F * fb
    value = world * args.steps * raw_step / (ms * 1e-3) / 1e9
    b = p.compress_batch(inputs[0], out=outs[0])
    torch.cuda.synchronize()
    comp_bytes = int(b.offsets[F].item()) - int(b.offsets[0].item())
    cr = F * fb / comp_bytes
    p.close()
    del inputs, outs, b
    torch.cuda.empty_cache()

    # ---- every packer, both directions (outside the headline's timed region)
    packers = {}
    for kind, shape in PACKERS:
        if args.quick and kind != "xdelta_hzr":
            continue
        packers[kind] = measure_packer(R, torch, D, kind, SHAPES[shape], args.packer_frames, 2, args.packer_reps, hbm_peak,
                                       args.e2e_frames, args.cpu_budget, rank == 0 and world == 1 and not args.no_cpu,
                                       stage_roofline=(kind == "xdelta_hzr"))
    x = packers["xdelta_hzr"]

    # roofline of the dominant kernel group of the headline (CUDA events around the stage on the handle's stream)
    stage_ms = x.get("stage_ms", {})
    comp_stages = {k: stage_ms.get(k, 0.0) for k in ("transform", "hist", "tree", "layout", "encode")}
    dom = max(comp_stages, key=comp_stages.get)
    Fp = args.packer_frames
    comp_p = Fp * fb / x["cr"]
    planes_bytes = Fp * 3 * sh["ch"] * sh["ns"]
    alg = {"transform": Fp * fb + planes_bytes, "hist": planes_bytes, "tree": 0, "layout": 0, "encode": planes_bytes / 3 + comp_p}
    achieved = alg[dom] / (comp_stages[dom] * 1e-3) / 1e9 if comp_stages[dom] > 0 else 0.0
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        try:
            tj = json.load(open(tpath))
            if tj.get("frames_per_launch"):
                traffic = tj["kernels"].get(dom, {}).get("dram_bytes_per_launch")
                if traffic is not None:
                    traffic = traffic * Fp / tj["frames_per_launch"]
        except Exception:
            traffic = None
    roofline = {"bound": "hbm", "kernel": {"transform": "k_xdelta_planes_tma", "hist": "k_hzr_hist", "tree": "k_hzr_tree",
                                           "layout": "k_scan_offsets", "encode": "k_hzr_encode_sparse + k_hzr_encode"}[dom],
                "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak, "traffic": traffic,
                "peak_source": peak_src, "ms_per_launch": comp_stages[dom],
                "algorithmic_bytes_per_launch": alg[dom],
                "pipeline": {"algorithmic_bytes_per_step": raw_step + raw_step / cr,
                             "achieved": (raw_step + raw_step / cr) * args.steps / (ms * 1e-3) / 1e9,
                             "frac": (raw_step + raw_step / cr) * args.steps / (ms * 1e-3) / 1e9 / hbm_peak},
                "stage_ms": stage_ms}

    if rank == 0:
        cfg = base_config(args, world)
        cfg.update({"frames_per_batch_per_gpu": F, "batches_per_step": NB, "raw_bytes_per_step_per_gpu": raw_step,
                    "l2": "every batch (%.2f GB) exceeds the 126 MB L2 and no batch repeats inside a step (%d distinct batches)" % (F * fb / 1e9, NB),
                    "sharding": ("contiguous frame ranges per rank; one NCCL all-gather of 8 B/rank per batch through the C ABI, "
                                 "on a side stream") if world > 1 else "single GPU",
                    "cr": cr})
        line = {
            "metric": "compress_raw_GBps", "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": cfg,
            "decompress_raw_GBps": x["decompress"]["raw_GBps"], "roundtrip_bit_exact": x.get("roundtrip_bit_exact"), "cr": cr,
            "roofline": roofline, "cpu_baseline": x["compress"].get("cpu_baseline"), "e2e": x["compress"]["e2e"],
            "e2e_decompress": x["decompress"]["e2e"], "gpu_launches": int(launches), "clocks": clocks, "packers": packers,
            "timed_region_s": ms * 1e-3,
        }
        print(json.dumps(line))
    D.close()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames", type=int, default=4096, help="frames per batch per GPU")
    ap.add_argument("--batches", type=int, default=24, help="distinct batches per step")
    ap.add_argument("--packer-frames", type=int, default=4096, help="frames per batch of the per-packer legs")
    ap.add_argument("--packer-reps", type=int, default=6)
    ap.add_argument("--e2e-frames", type=int, default=4096)
    ap.add_argument("--quick", action="store_true", help="xdelta_hzr only in the per-packer legs")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline legs")
    ap.add_argument("--cpu-budget", type=float, default=5.0)
    ap.add_argument("--cpu-threads", type=int, default=0)
    ap.add_argument("--cpu-frames-per-thread", type=int, default=64)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write a fixed sample of the last step's outputs to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's outputs; --impl reference has none")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
