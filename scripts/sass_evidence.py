"""cuobjdump -sass of libfenix_knn.so -> profiles/r02_sass_evidence.txt: per kernel the Blackwell-specific mnemonics it
contains (tcgen05.mma = UTCHMMA / UTCIMMA (kind::i8) / UTCQMMA, TMEM loads = LDTM, TMA = UTMALDG / UBLKCP, tcgen05.commit = UTCBAR, cluster
barriers) with counts, and the head of the listing of the dominant kernels."""
import collections, os, re, subprocess
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
so = os.path.join(ROOT, "fenix_b200", "libfenix_knn.so")
txt = subprocess.run(["cuobjdump", "-sass", so], capture_output=True, text=True, check=True).stdout
kernels, name = collections.OrderedDict(), None
for line in txt.splitlines():
    m = re.match(r"\s*Function : (\S+)", line)
    if m:
        name = subprocess.run(["c++filt", m.group(1)], capture_output=True, text=True).stdout.strip()
        kernels[name] = []
    elif name and re.match(r"\s+/\*[0-9a-f]{4,}\*/", line):
        kernels[name].append(line.rstrip())
KEY = ("UTCHMMA", "UTCIMMA", "UTCQMMA", "UTCOMMA", "LDTM", "STTM", "UTMALDG", "UTMAPF", "UBLKCP", "UTCBAR", "UTCCP", "SYNCS", "UCGABAR", "DFMA", "F2F.F64.F32", "SHFL", "ATOMG", "MEMBAR")
out = [f"# {so} ({os.path.getsize(so)} bytes): {len(kernels)} kernels; counts of the instructions that matter per kernel\n"]
for k, lines in kernels.items():
    ops = collections.Counter()
    for l in lines:
        m = re.search(r"\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", l)
        if m:
            for key in KEY:
                if m.group(1).startswith(key):
                    ops[key] += 1
    short = k if len(k) < 150 else k[:147] + "..."
    out.append(f"{short}\n    {len(lines)} instructions; " + ", ".join(f"{a} x{b}" for a, b in ops.items()) + "\n")
for pat, n in (("knn_tc_filter_kernel<2, 1, 0, 1>", 70), ("knn_tc_filter_kernel<2, 2, 0, 1>", 70), ("knn_rq_filter_kernel<2, 0>", 50), ("knn_direct_kernel<1, 1, false, false>", 60)):
    for k, lines in kernels.items():
        if pat in k.replace("(int)", "").replace("(bool)", ""):
            mma = [i for i, l in enumerate(lines) if "UTCHMMA" in l or "UTCIMMA" in l or "DFMA" in l]
            lo = max(0, (mma[0] if mma else 0) - 12)
            out.append(f"\n## {k[:160]}\n## listing around the first MMA / DFMA (instructions {lo}..{lo + n} of {len(lines)})\n" + "\n".join(lines[lo: lo + n]) + "\n")
            break
open(os.path.join(ROOT, "profiles", "r02_sass_evidence.txt"), "w").write("".join(out))
print("".join(out)[:3000])
