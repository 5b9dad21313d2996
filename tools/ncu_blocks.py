"""Basic-block view of an ncu report: runs of consecutive SASS instructions with the same execution count.
    python tools/ncu_blocks.py report.ncu-rep [kernel-mangled-substring] [min_share_pct]
Prints per block: address, #instructions, executions per warp-iteration-equivalent, mean active threads, share of the kernel's
ISSUE CYCLES (one per instruction, two per FFMA2/FADD2/FMUL2 — the model that matches sm__cycles on B200), first source line and
the block's opcode mix.  The .so must be the build that was profiled."""
import collections, csv, io, os, re, subprocess, sys, tempfile

rep = sys.argv[1]
kern = sys.argv[2] if len(sys.argv) > 2 else "render_kernelIfLb1ELi256ELi3E"
min_share = float(sys.argv[3]) if len(sys.argv) > 3 else 0.3
root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
with tempfile.TemporaryDirectory() as td:
    subprocess.run(["cuobjdump", "-xelf", "all", os.path.join(root, "rtiow_b200/lib/librtiow_cuda.so")], cwd=td, capture_output=True)
    cub = [f for f in os.listdir(td) if f.startswith("capi.") and f.endswith(".cubin")][0]
    sass = subprocess.run(["nvdisasm", "-g", os.path.join(td, cub)], capture_output=True, text=True).stdout.splitlines()
start = next(i for i, l in enumerate(sass) if l.startswith(".text.") and kern in l and l.rstrip().endswith(":"))
lines, cur = [], ("?", 0)
for l in sass[start + 1:]:
    if l.startswith("//-----") or l.startswith("\t.section"):
        break
    m = re.match(r'\s*//## File "([^"]+)", line (\d+)', l)
    if m:
        cur = (os.path.basename(m.group(1)), int(m.group(2))); continue
    m = re.match(r"\s*/\*([0-9a-f]{4,})\*/\s+(.*?);", l)
    if m:
        lines.append((int(m.group(1), 16), cur, m.group(2)))
src = subprocess.run(["ncu", "-i", rep, "--page", "source", "--csv", "--print-source", "sass"], capture_output=True, text=True).stdout
rows = list(csv.reader(io.StringIO(src)))
hdr = rows[1]; data = [r for r in rows[2:] if len(r) == len(hdr)]
iex, ismp, iav = hdr.index("Instructions Executed"), hdr.index("# Samples"), hdr.index("Thread Instructions Executed")
# non-inlined callees (big_spheres_merge, big_spheres_best, filter_tail) follow the kernel in ncu's listing: keep them, without line info
lines += [(0, ("callee", 0), r[1].strip()) for r in data[len(lines):]]
assert len(data) == len(lines), (len(data), len(lines))
def cost(op): return 2 if op.split()[-1 if op.startswith("@") else 0].startswith(("FFMA2", "FADD2", "FMUL2")) or " FFMA2" in op[:14] else 1
recs = []
for r, (addr, loc, text) in zip(data, lines):
    op = text.split()[1] if text.startswith("@") else text.split()[0]
    recs.append((addr, loc, op, int(r[iex]), int(r[ismp]), int(r[iav]), 2 if op in ("FFMA2", "FADD2", "FMUL2") else 1))
tot_cycles = sum(x[3] * x[6] for x in recs); tot_s = sum(x[4] for x in recs)
scan_exec = max(x[3] for x in recs if x[2].split(".")[0] in ("FFMA2", "SHF"))    # executions of the scan's inner instructions (FFMA2 filter / SHF sign collection)
n_ffma2 = sum(1 for x in recs if x[2] == "FFMA2" and x[3] > scan_exec // 2)
words = 1
print(f"# {rep}: {len(recs)} SASS instructions, issue-cycle model total {tot_cycles/1e9:.2f} G; per-'scan word' counts = executions / {scan_exec}")
blocks = []
i = 0
while i < len(recs):
    j = i
    while j + 1 < len(recs) and recs[j + 1][3] == recs[i][3] and recs[j][2] not in ("BRA", "EXIT", "BSYNC", "RET"):
        j += 1
    blocks.append(recs[i:j + 1]); i = j + 1
print(f"{'addr':>6} {'n':>4} {'exec/word':>9} {'thr':>5} {'cyc%':>6} {'smp%':>6}  first line; ops")
for b in blocks:
    cyc = sum(x[3] * x[6] for x in b); share = 100 * cyc / tot_cycles
    if share < min_share: continue
    ops = collections.Counter(x[2] for x in b).most_common(5)
    thr = sum(x[5] for x in b) / max(1, sum(x[3] for x in b))
    print(f"{b[0][0]:6x} {len(b):4d} {b[0][3]/scan_exec:9.3f} {thr:5.1f} {share:6.2f} {100*sum(x[4] for x in b)/tot_s:6.2f}  {b[0][1][0]}:{b[0][1][1]}; " + " ".join(f"{o}x{c}" for o, c in ops))
