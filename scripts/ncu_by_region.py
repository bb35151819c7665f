"""Per-region table of an ncu capture of k_trace: share of warp-instructions, cycles per instruction and stall reasons
per instruction (scaled so that "selected" == 1 overall), active lanes per instruction.
Regions are ranges of source lines of torj_device.cuh found by marker strings, plus "kernel bookkeeping" (torj_kernels.cuh).
Capture with  --warp-sampling-interval 9 --warp-sampling-buffer-size 536870912  (the default buffer overflows on a 150 ms
kernel and the samples then cover only its first third).
usage: ncu_by_region.py report.ncu-rep libtorj_cuda.so kernel_mangled_substr"""
import collections, csv, os, re, subprocess, sys, tempfile

rep, so, kern = sys.argv[1:4]
root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
tmp = tempfile.mkdtemp()
subprocess.check_call(["cuobjdump", "-xelf", "all", os.path.abspath(so)], cwd=tmp, stdout=subprocess.DEVNULL)
cub = [f for f in os.listdir(tmp) if f.endswith(".cubin")][0]
dis = subprocess.run(["nvdisasm", "-g", "-c", os.path.join(tmp, cub)], capture_output=True, text=True).stdout.splitlines()
insts, cur, on = [], ("?", 0), False
for ln in dis:
    if ln.startswith(".text."):
        on = kern in ln
        continue
    if not on:
        continue
    m = re.match(r'\s*//## File "(.*)", line (\d+)', ln)
    if m:
        cur = (os.path.basename(m.group(1)), int(m.group(2)))
        continue
    if re.match(r"\s+/\*[0-9a-f]{4,}\*/", ln):
        insts.append(cur)
txt = subprocess.run(["ncu", "-i", rep, "--page", "source", "--csv", "--print-source", "sass"], capture_output=True, text=True).stdout
rows = list(csv.reader(txt.splitlines()))
hi = next(i for i, r in enumerate(rows) if "# Samples" in r)
hdr, data = rows[hi], rows[hi + 1:]
assert len(data) == len(insts), (len(data), len(insts))
ix = {h: i for i, h in enumerate(hdr)}
src = open(os.path.join(root, "torj_jl_b200", "csrc", "torj_device.cuh")).read().splitlines()
find = lambda s: next(i + 1 for i, l in enumerate(src) if s in l)
marks = [("rcp/rsqrt/sqrt", find("rcp_fast(double") - 8), ("bs_weights", find("bs_weights(") - 2), ("stencil", find("struct Fields")),
         ("fields misc", find("eval_field_ext(const DevTables T") - 8), ("dispersion", find("refractive_index_sq(") - 3),
         ("polarisation", find("struct Pol")), ("exp_fast", find("// exp(x), branch-free")),
         ("bessel+node loop", find("bessel_JD(double hz") - 8), ("harmonic_alpha", find("harmonic_sum_large(const HarmCoef c") - 2),
         ("abs_albajar", find("double abs_albajar(") - 8), ("rhs body", find("struct PointVals") - 4),
         ("deposition", find("struct DepoState") - 2)]


def region(loc):
    f, l = loc
    if f == "torj_kernels.cuh":
        return "kernel bookkeeping"
    if f == "torj_device.cuh":
        g = "head"
        for name, start in marks:
            if l >= start:
                g = name
        return g
    return f


names = ["stall_wait", "stall_no_inst", "stall_selected", "stall_math", "stall_short_sb", "stall_long_sb", "stall_branch_resolving",
         "stall_not_selected", "stall_dispatch", "stall_barrier"]
col = lambda r, n: int(r[ix[n]]) if r[ix[n]] else 0
agg = collections.defaultdict(collections.Counter)
for k, r in enumerate(data):
    g = region(insts[k])
    agg[g]["w"] += col(r, "Instructions Executed"); agg[g]["t"] += col(r, "Thread Instructions Executed"); agg[g]["s"] += col(r, "# Samples")
    for n in names:
        agg[g][n] += col(r, n)
tw = sum(a["w"] for a in agg.values()); ts = sum(a["s"] for a in agg.values()); tsel = sum(a["stall_selected"] for a in agg.values())
print(f"samples {ts}  warp-instructions {tw}  lanes/instr {sum(a['t'] for a in agg.values()) / tw:.2f}")
print("overall %:", {n[6:]: round(sum(a[n] for a in agg.values()) / ts * 100, 1) for n in names})
print(f"{'region':22s} inst%  samp%  cyc/inst lanes | " + " ".join(n[6:11] for n in names))
scale = tw / tsel
for g, a in sorted(agg.items(), key=lambda kv: -kv[1]["s"]):
    w = a["w"] or 1
    print(f"{g:22s} {a['w'] / tw * 100:5.1f} {a['s'] / ts * 100:6.1f} {a['s'] / w * scale:7.2f} {a['t'] / w:5.1f} | " +
          " ".join(f"{a[n] / w * scale:5.2f}" for n in names))
