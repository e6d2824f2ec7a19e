"""profiles/<name>: which Blackwell data-movement / synchronisation instructions the shipped cubin contains, per kernel,
with a short SASS excerpt.  usage: sass_features.py <out.txt>   (cuobjdump -sass rspt_b200/librspt_gpu.so)"""
import collections, os, re, subprocess, sys
root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
so = os.path.join(root, "rspt_b200", "librspt_gpu.so")
txt = subprocess.run(["cuobjdump", "-sass", so], capture_output=True, text=True).stdout.splitlines()
demangle = lambda n: subprocess.run(["c++filt", n], capture_output=True, text=True).stdout.strip().split("(")[0]
pat = re.compile(r"\b(UBLKCP[.\w]*|UTMA\w+[.\w]*|SYNCS[.\w]*|UCGABAR_\w+|LDGSTS[.\w]*|REDUX[.\w]*|MEMBAR[.\w]*\.CLUSTER|MAPA[.\w]*|S2UR\s+\w+, SR_CgaCtaId)")
per = collections.defaultdict(collections.Counter)
tot = collections.Counter()
lines_of = collections.defaultdict(list)
fn = None
arch = [l.strip() for l in txt if l.strip().startswith("arch =")]
for l in txt:
    m = re.search(r"Function : (\S+)", l)
    if m:
        fn = m.group(1)
        continue
    if fn is None or "/*" not in l:
        continue
    body = re.sub(r"/\* 0x[0-9a-f]+ \*/", "", l).rstrip()
    if re.match(r"\s+/\*[0-9a-f]{4,}\*/", body):
        lines_of[fn].append(body)
        for m in pat.finditer(body):
            key = m.group(1).split()[0] if not m.group(1).startswith("S2UR") else "S2UR SR_CgaCtaId"
            per[fn][key] += 1
            tot[key.split(".")[0]] += 1
out = []
out.append("cuobjdump -sass rspt_b200/librspt_gpu.so  (%s; %d kernels)" % (", ".join(sorted(set(arch))), len(lines_of)))
out.append("totals by mnemonic family: " + ", ".join(f"{k} {v}" for k, v in sorted(tot.items())))
out.append("  UBLKCP = cp.async.bulk (1-D bulk copy engine, global<->shared), SYNCS = mbarrier (arrive.expect_tx / try_wait),")
out.append("  UCGABAR_ARV/WAIT = barrier.cluster.arrive/wait (thread-block cluster), LDGSTS = cp.async (Ampere-style)")
out.append("")
out.append("per kernel (only kernels that have any of UBLKCP / SYNCS / UCGABAR):")
for f in sorted(per, key=demangle):
    c = per[f]
    if not any(k.startswith(("UBLKCP", "SYNCS", "UCGABAR")) for k in c):
        continue
    out.append("  %-60s %s" % (demangle(f)[:60], ", ".join(f"{k} x{v}" for k, v in sorted(c.items()) if k.startswith(("UBLKCP", "SYNCS", "UCGABAR", "LDGSTS")))))
def excerpt(name_part, needle, before, after, title):
    for f, ls in lines_of.items():
        if name_part in f:
            for i, l in enumerate(ls):
                if needle in l:
                    out.append("")
                    out.append(title + "  [" + demangle(f)[:70] + "]")
                    out.extend("    " + x.strip() for x in ls[max(0, i - before): i + after])
                    return
excerpt("k_hzr_decode", "UBLKCP", 14, 4, "payload staging of the decoder: mbarrier init, expect_tx, one bulk copy global -> shared")
excerpt("k_hzr_decode", "SYNCS.PHASECHK", 2, 6, "... and the wait on it (mbarrier.try_wait.parity loop)")
excerpt("k_hzr_encodeILi3", "UBLKCP", 10, 4, "dense encoder: header + payload leave the staging with one bulk store shared -> global (default path of xdelta_hzr and hadamard)")
open(sys.argv[1], "w").write("\n".join(out) + "\n")
print("\n".join(out[:12]))
