"""torch.profiler over xdelta_hzr compress (3 B x 12 ch x 8192, 4096 frames per batch, 8 batches): device time of
every k_hzr_tree launch and the mean per launch of every kernel.  The longer half of the tree launches is the dense
class, the shorter the sparse one (they run on two streams, so each is timed under the other's load).

    python tools/prof_tree.py <repository root to import rspt_b200 from> <out.json>
"""
import json, os, sys
root = sys.argv[1]
sys.path.insert(0, root)
import torch
from rspt_b200 import packer as R
F = 4096
p = R.SignalPacker("xdelta_hzr", 3, 12, 8192, 3, max_batch_frames=F)
xs = [R.synth_ecg(i * F, F, 3, 12, 8192) for i in range(2)]
out = p.alloc_output(F)
for i in range(4):
    p.compress_batch(xs[i & 1], out=out)
torch.cuda.synchronize()
from torch.profiler import profile, ProfilerActivity
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for i in range(8):
        p.compress_batch(xs[i & 1], out=out)
    torch.cuda.synchronize()
ev = [e for e in prof.events() if e.device_type.name == "CUDA"]
tree = [e.device_time for e in ev if "k_hzr_tree" in e.name]
per = {}
for e in ev:
    k = e.name.split("(")[0].replace("void ", "")
    per.setdefault(k, []).append(e.device_time)
res = {"tree_launches_us": tree, "dense_mean_us": sum(sorted(tree)[len(tree)//2:]) / (len(tree)//2),
       "sparse_mean_us": sum(sorted(tree)[:len(tree)//2]) / (len(tree)//2),
       "per_kernel_mean_us": {k: sum(v) / len(v) for k, v in per.items()}, "launches_per_kernel": {k: len(v) for k, v in per.items()}}
json.dump(res, open(sys.argv[2], "w"), indent=1)
print(sys.argv[2], "dense %.1f sparse %.1f us" % (res["dense_mean_us"], res["sparse_mean_us"]))
