"""Per-kernel SASS extract of the built library: instruction count, code size and the mnemonics that show how data
moves (UBLKCP = cp.async.bulk / TMA bulk copy, SYNCS = mbarrier, LDGSTS = cp.async, REDUX = warp reduce, ATOM/RED).
    python tools/sass_summary.py [lib.so] > profiles/r2_sass_summary.txt
    python tools/sass_summary.py --fingerprint [lib.so]
--fingerprint prints one line per kernel: a hash of its instructions (without the function name and the addresses),
the instruction count and the demangled name.  Two builds whose sorted hash lists are equal run the same machine code,
whatever the kernels are called."""
import collections
import hashlib
import re
import subprocess
import sys

args = [a for a in sys.argv[1:] if a != "--fingerprint"]
lib = args[0] if args else "hironaka_b200/_lib/libhironaka_b200.so"
out = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout

if "--fingerprint" in sys.argv:
    code = []  # (mangled name, instructions) per kernel, in library order; a name that appears twice is kept twice
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            code.append((m.group(1), []))
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,6}\*/\s+(.*?)\s*;", line)
        if m and code:
            code[-1][1].append(m.group(1))
    demangled = subprocess.run(["c++filt"], input="\n".join(n for n, _ in code), capture_output=True,
                               text=True).stdout.splitlines()
    for (mangled, ins), nice in zip(code, demangled):
        print(f"{hashlib.sha256(chr(10).join(ins).encode()).hexdigest()[:16]} {len(ins):6d} {nice}")
    sys.exit(0)

WATCH = ["UBLKCP", "SYNCS", "LDGSTS", "REDUX", "UTMALDG", "UTMASTG", "ATOMG", "RED.", "LDS", "STS", "LDG", "STG", "SHFL", "VOTE",
         "LOP3", "IADD3", "IMAD", "ISETP", "VIMNMX", "POPC", "FLO", "BAR", "MUFU"]
kernels = collections.OrderedDict()
name, arch = None, None
for line in out.splitlines():
    m = re.search(r"Function : (\S+)", line)
    if m:
        name = m.group(1)
        kernels[name] = collections.Counter()
        continue
    m = re.match(r"\s+/\*([0-9a-f]{4,6})\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", line)
    if m and name:
        op = m.group(2)
        kernels[name]["_n"] += 1
        for w in WATCH:
            if op.startswith(w):
                kernels[name][w] += 1
demangle = subprocess.run(["c++filt"], input="\n".join(kernels), capture_output=True, text=True).stdout.splitlines()
print(f"# cuobjdump -sass {lib}: {len(kernels)} sm_100a kernels; columns: instructions, code KiB, then mnemonic counts")
tot = collections.Counter()
rows = []
for (mangled, c), nice in zip(kernels.items(), demangle):
    tot.update(c)
    rows.append((nice.replace("void ", "").replace("hk::", "").replace("(hk::StepParams)", "").replace("(hk::StepParams, int, int)", ""), c))
keep = [r for r in rows if any(k in r[0] for k in ("<int, 20, 3", "<int, 5, false, 2", "<int, 5, 8", "hk_exp", "hk_value", "hk_overflow",
                                                   "hk_random", "hk_pack"))]
for nice, c in keep:
    print(f"{nice[:78]:78s} {c['_n']:6d} {c['_n'] * 16 / 1024:7.1f}  " +
          " ".join(f"{w}={c[w]}" for w in ("UBLKCP", "SYNCS", "LDGSTS", "REDUX", "ATOMG", "RED.", "VOTE", "SHFL", "LOP3", "IADD3", "IMAD") if c[w]))
print(f"# whole library: {tot['_n']} instructions ({tot['_n'] * 16 / 2 ** 20:.1f} MiB of SASS), " +
      ", ".join(f"{w} {tot[w]}" for w in ("UBLKCP", "SYNCS", "LDGSTS", "REDUX", "UTMALDG", "UTMASTG")))
