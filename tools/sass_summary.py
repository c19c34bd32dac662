"""SASS evidence for profiles/: per kernel of the built library, the counts of the instructions that prove the data path
(TMA-engine bulk copies / prefetches, mbarrier ops, 256-bit loads, FP64 FMAs, FP64 tensor ops, shuffles, barriers), plus
registers / shared memory / stack per kernel.  Runs in the build container (cuobjdump only, no GPU).

    python tools/sass_summary.py > profiles/r02_sass_summary.txt

--fingerprint: one line per function instead -- the name without namespaces, registers, stack, instruction count and a
hash of the instruction text (addresses, encodings and mangled symbol names removed), sorted.  Two builds that differ in
translation units or namespaces but compile the same machine code print the same lines:

    diff <(python tools/sass_summary.py --fingerprint old.so) <(python tools/sass_summary.py --fingerprint new.so)"""
import collections
import hashlib
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ARGS = [a for a in sys.argv[1:] if a != "--fingerprint"]
FINGERPRINT = "--fingerprint" in sys.argv
LIB = ARGS[0] if ARGS else os.path.join(ROOT, "ccqppy_b200", "csrc", "libccqp_b200.so")
PATTERNS = [("UBLKCP", r"\bUBLKCP"), ("UBLKPF", r"\bUBLKPF"), ("SYNCS(mbarrier)", r"\bSYNCS"), ("LDG.*.256", r"\bLDG\S*\.256"),
            ("LDG.*.128", r"\bLDG\S*\.128"), ("LDS.128", r"\bLDS\S*\.128"), ("DFMA", r"\bDFMA"), ("DADD", r"\bDADD"), ("DMUL", r"\bDMUL"),
            ("DMMA", r"\bDMMA"), ("SHFL", r"\bSHFL"), ("BAR", r"\bBAR\."), ("MUFU.RCP64H", r"MUFU\.RCP64H"), ("ATOM/RED", r"\b(ATOMG|REDG|ATOM|RED)\b"),
            ("LDL/STL(local: spills + SPG window ring)", r"\b(LDL|STL)"), ("UTC*MMA/LDTM(none expected)", r"\b(UTCMMA|UTCHMMA|UTCQMMA|LDTM|UTMALDG)")]

sass = subprocess.run(["cuobjdump", "-sass", LIB], capture_output=True, text=True, check=True).stdout
res = subprocess.run(["cuobjdump", "--dump-resource-usage", LIB], capture_output=True, text=True, check=True).stdout
usage = {}
for m in re.finditer(r"Function (\S+):\n\s*(.*)", res):
    usage[m.group(1)] = m.group(2)
kern = None
counts = collections.OrderedDict()
text = collections.defaultdict(hashlib.sha256)
arch = set(re.findall(r"arch = (sm_\w+)", sass))
for line in sass.splitlines():
    m = re.search(r"Function : (\S+)", line)
    if m:
        kern = m.group(1)
        counts[kern] = collections.Counter(total=0)
        continue
    if kern and re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+\S", line):
        counts[kern]["total"] += 1
        ins = re.sub(r"/\*.*?\*/", "", line)
        text[kern].update((re.sub(r"\b_Z\w+", "_Z", ins).strip() + "\n").encode())
        for name, pat in PATTERNS:
            if re.search(pat, line):
                counts[kern][name] += 1
dem = subprocess.run(["c++filt"] + list(counts), capture_output=True, text=True).stdout.splitlines()
if FINGERPRINT:
    lines = []
    for (k, c), d in zip(counts.items(), dem):
        d = re.sub(r"\b(ccqp\w*|\(anonymous namespace\))::", "", d)
        u = usage.get(k, "")
        regs = re.search(r"REG:(\d+)", u); st = re.search(r"STACK:(\d+)", u)
        lines.append("%s | regs %s stack %s | %d | %s" % (d, regs.group(1) if regs else "?", st.group(1) if st else "?",
                                                        c["total"], text[k].hexdigest()[:16]))
    print("\n".join(sorted(lines)))
    sys.exit(0)
print("# %s\n# arch: %s ; %d kernels" % (os.path.relpath(LIB, ROOT), ", ".join(sorted(arch)), len(counts)))
print("# columns: instructions, then " + ", ".join(n for n, _ in PATTERNS))
tot = collections.Counter()
for (k, c), d in zip(counts.items(), dem):
    d = d.replace("ccqp::", "").replace("void ", "").replace("(anonymous namespace)::", "")
    d = re.sub(r"\(.*\)$", "", d)
    u = usage.get(k, "")
    regs = re.search(r"REG:(\d+)", u); sh = re.search(r"SHARED:(\d+)", u); st = re.search(r"STACK:(\d+)", u)
    print("%-34s regs %3s smem %6s stack %4s | %6d | %s" % (d, regs.group(1) if regs else "?", sh.group(1) if sh else "?",
          st.group(1) if st else "?", c["total"], " ".join("%s=%d" % (n, c[n]) for n, _ in PATTERNS if c[n])))
    tot.update(c)
print("# library total: %d instructions | %s" % (tot["total"], " ".join("%s=%d" % (n, tot[n]) for n, _ in PATTERNS)))
