"""A/B of the two builds of the sparse class in one process: a handle created with RSPT_SPARSE_LIST=1 (k_hzr_hist<3> +
one-pass k_hzr_encode_sparse) and one with RSPT_SPARSE_LIST=0 (k_hzr_hist<1> + two-pass encoder), the benchmark's
shape (xdelta_hzr 3 B x 12 ch x 8192, 4096 frames per batch).  Compress batches alternate between the two handles.

    python tools/sparse_ab.py [--rounds 24] [--batches 6] [--out DIR]            # ms per batch + stage times
    python tools/sparse_ab.py --profile [--out DIR]                               # per-kernel durations (torch.profiler)

Prints the GPU, its power limit and SM clock limit, then per arm the median / min / max ms per batch (CUDA events
around each batch), the per-stage CUDA-event times, and with --profile the mean device time of every kernel of the
sparse class and of the dense class beside it.  Results also go to DIR/sparse_ab*.json (default: a directory
under the system's temporary directory, so that the tree stays untouched)."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from rspt_b200 import packer as R

SH = dict(bps=3, ch=12, ns=8192)


def gpu_info():
    info = {"name": torch.cuda.get_device_name()}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.split(",")
        info.update(power_limit_w=float(q[0]), sm_max_mhz=float(q[1]))
    except Exception as e:  # the numbers are reported without them
        info["nvidia_smi"] = repr(e)
    return info


def make(arm, F):
    os.environ["RSPT_SPARSE_LIST"] = arm
    try:
        return R.SignalPacker.new_xdelta_hzr(SH["bps"], SH["ch"], SH["ns"], 3, max_batch_frames=F)
    finally:
        del os.environ["RSPT_SPARSE_LIST"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=4096)
    ap.add_argument("--batches", type=int, default=6, help="distinct input batches (each 1.2 GB at the default size)")
    ap.add_argument("--rounds", type=int, default=24, help="batches timed per arm")
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--out", default=os.path.join(tempfile.gettempdir(), "rspt_sparse_ab"))
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    F = a.frames
    arms = {"new": make("1", F), "old": make("0", F)}
    inputs = [R.synth_ecg(i * F, F, **SH) for i in range(a.batches)]
    outs = {k: p.alloc_output(F, sidecar=True) for k, p in arms.items()}
    res = {"gpu": gpu_info(), "shape": SH, "frames_per_batch": F}
    print(json.dumps(res["gpu"]))
    for _ in range(3):  # warm-up: every input through both arms
        for i in range(a.batches):
            for k, p in arms.items():
                p.compress_batch(inputs[i], out=outs[k])
    torch.cuda.synchronize()
    # the two arms' streams must agree byte for byte
    for i in range(a.batches):
        b = {k: p.compress_batch(inputs[i], out=outs[k]) for k, p in arms.items()}
        n = int(b["new"].offsets[F].item())
        assert n == int(b["old"].offsets[F].item()) and torch.equal(b["new"].stream[:n], b["old"].stream[:n]), i

    if a.profile:
        from torch.profiler import ProfilerActivity, profile
        per = {}
        for k, p in arms.items():
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for r in range(a.rounds):
                    p.compress_batch(inputs[r % a.batches], out=outs[k])
                torch.cuda.synchronize()
            prof.export_chrome_trace(os.path.join(a.out, "sparse_ab_%s.pt.trace.json" % k))
            d = {}
            for ev in prof.key_averages():
                if ev.device_type.name == "CUDA" or getattr(ev, "device_time_total", 0):
                    t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)
                    if t and ev.count:
                        d[ev.key] = {"us_per_launch": t / ev.count, "launches": ev.count}
            per[k] = d
            print(k)
            for name, v in sorted(d.items(), key=lambda kv: -kv[1]["us_per_launch"]):
                print("  %-70s %9.1f us  x%d" % (name[:70], v["us_per_launch"], v["launches"]))
        res["kernels"] = per
        with open(os.path.join(a.out, "sparse_ab_profile.json"), "w") as f:
            json.dump(res, f, indent=1)
        return

    ms = {k: [] for k in arms}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for r in range(a.rounds):
        for k in (("new", "old") if r % 2 == 0 else ("old", "new")):
            ev[0].record()
            arms[k].compress_batch(inputs[r % a.batches], out=outs[k])
            ev[1].record()
            ev[1].synchronize()
            ms[k].append(ev[0].elapsed_time(ev[1]))
    res["ms_per_batch"] = {k: {"median": statistics.median(v), "min": min(v), "max": max(v), "all": v} for k, v in ms.items()}
    gb = F * SH["bps"] * SH["ch"] * SH["ns"] / 1e9
    for k, v in res["ms_per_batch"].items():
        print("%s  ms/batch median %.3f  min %.3f  max %.3f  (%.0f GB/s at the median)" % (k, v["median"], v["min"], v["max"], gb / v["median"] * 1e3))
    # per-stage CUDA-event times, alternating again
    for p in arms.values():
        p.set_stage_timing(True)
        p.stage_times(reset=True)
    for r in range(a.rounds):
        for k, p in arms.items():
            p.compress_batch(inputs[r % a.batches], out=outs[k])
    torch.cuda.synchronize()
    res["stage_ms"] = {}
    for k, p in arms.items():
        st = p.stage_times(reset=True)
        res["stage_ms"][k] = {s: v[0] / v[1] for s, v in st.items() if v[1]}
        print(k, " ".join("%s=%.3f" % kv for kv in res["stage_ms"][k].items()))
    with open(os.path.join(a.out, "sparse_ab.json"), "w") as f:
        json.dump(res, f, indent=1)
    for p in arms.values():
        p.close()


if __name__ == "__main__":
    main()
