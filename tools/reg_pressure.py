"""Register pressure of compiled kernels: where the registers of a kernel are live at once.

usage: python tools/reg_pressure.py OBJ [OBJ ...] [--kernel SUBSTR ...] [--top N]

OBJ is a .o, .so or .cubin built for sm_100a with -lineinfo (csrc/Makefile builds that way); several OBJs (e.g. the parent's build and
this one's) give a before / after table.  For every kernel whose mangled name contains one of the --kernel substrings (default: the
4-wide sphere instantiations of k_mega) it prints
  - registers and stack frame (cuobjdump -res-usage), spill stores / loads (the ptxas -v log: the Makefile writes build/kernels.ptxas.log
    next to build/kernels.o, which is the default);
  - the source lines with the highest live-register counts: nvdisasm --print-life-ranges (-lrm count) gives the live general registers
    before each instruction, nvdisasm -gi the source line of each instruction (innermost project line of its inlining chain); the two
    listings are joined on the instruction offset.
Runs on the CPU; needs cuobjdump and nvdisasm from the CUDA toolkit.
"""
import argparse, collections, os, re, shutil, struct, subprocess, sys, tempfile

CUDA_BIN = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin")
DEFAULT_KERNELS = ["k_megaILb0ELi5ELb0ELj1ELb0ELb1E", "k_megaILb0ELi5ELb0ELj3ELb0ELb1E", "k_megaILb0ELi5ELb0ELj5ELb0ELb1E",
                   "k_megaILb0ELi6ELb0ELj1ELb0ELb1E", "k_megaILb0ELi6ELb0ELj3ELb0ELb1E", "k_megaILb0ELi6ELb0ELj5ELb0ELb1E"]


def tool(name):
    p = shutil.which(name) or os.path.join(CUDA_BIN, name)
    if not os.path.exists(p):
        sys.exit(f"reg_pressure: {name} not found (set CUDA_HOME)")
    return p


def run(*cmd):
    return subprocess.run(cmd, capture_output=True, text=True, check=True).stdout


def cubins(obj, tmp):
    if obj.endswith(".cubin"):
        return [obj]
    subprocess.run([tool("cuobjdump"), "-xelf", "all", os.path.abspath(obj)], cwd=tmp, capture_output=True, check=True)
    return sorted(os.path.join(tmp, f) for f in os.listdir(tmp) if f.endswith(".cubin"))


def global_functions(cubin):
    """{mangled name: symbol index} of the kernels (global FUNC symbols) in an ELF64 cubin."""
    data = open(cubin, "rb").read()
    shoff, = struct.unpack_from("<Q", data, 0x28)
    shentsize, shnum = struct.unpack_from("<HH", data, 0x3A)
    secs = [struct.unpack_from("<IIQQQQIIQQ", data, shoff + i * shentsize) for i in range(shnum)]
    out = {}
    for s in secs:
        if s[1] != 2:  # SHT_SYMTAB
            continue
        strtab = secs[s[6]]
        for i in range(s[5] // s[9]):
            name_off, info, _, _, _, _ = struct.unpack_from("<IBBHQQ", data, s[4] + i * s[9])
            if (info >> 4) == 1 and (info & 0xF) == 2:  # GLOBAL FUNC
                end = data.index(b"\0", strtab[4] + name_off)
                out[data[strtab[4] + name_off:end].decode()] = i
    return out


def res_usage(obj):
    """{mangled name: (registers, stack bytes)} from cuobjdump -res-usage."""
    out, name = {}, None
    for l in run(tool("cuobjdump"), "-res-usage", obj).splitlines():
        m = re.match(r"\s*Function (\S+):", l)
        if m:
            name = m.group(1)
            continue
        m = re.search(r"REG:(\d+) STACK:(\d+)", l)
        if m and name:
            out[name] = (int(m.group(1)), int(m.group(2)))
    return out


def ptxas_spills(log):
    """{mangled name: (stack frame, spill stores, spill loads)} from a ptxas -v log."""
    out = {}
    if not log or not os.path.exists(log):
        return out
    name = None
    for l in open(log):
        m = re.search(r"Function properties for (\S+)", l)
        if m:
            name = m.group(1)
            continue
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", l)
        if m and name:
            out[name] = tuple(int(x) for x in m.groups())
            name = None
    return out


INSN = re.compile(r"^\s*/\*([0-9a-f]{4,})\*/\s+(.*?);")


def live_counts(cubin, idx):
    """{offset: live general registers} for the function with symbol index idx."""
    out = {}
    for l in run(tool("nvdisasm"), "-fun", str(idx), "-lrm", "count", cubin).splitlines():
        m = INSN.match(l)
        if not m or "// |" not in l:
            continue
        cols = l.split("// |")[1].split("|")
        if cols and cols[0].strip().isdigit():
            out[int(m.group(1), 16)] = int(cols[0])
    return out


def line_map(cubin, idx):
    """{offset: (file, line)}: the innermost line of the inlining chain that lies outside the CUDA headers."""
    out, where, chain = {}, None, []
    for l in run(tool("nvdisasm"), "-fun", str(idx), "-gi", cubin).splitlines():
        m = re.match(r'\s*//## File "([^"]+)", line (\d+)(?: inlined at "([^"]+)", line (\d+))?', l)
        if m:
            chain.append((m.group(1), int(m.group(2))))
            continue
        m = INSN.match(l)
        if not m:
            continue
        if chain:  # a new annotation block: innermost entry first, the kernel's own line last
            own = [c for c in chain if "/targets/" not in c[0] and "/include/crt/" not in c[0]]
            where = (own or chain)[0]
            chain = []
        out[int(m.group(1), 16)] = where
    return out


def source_line(path, line, cache={}):
    if path not in cache:
        cache[path] = open(path).read().split("\n") if os.path.exists(path) else []
    text = cache[path]
    return text[line - 1].strip() if 0 < line <= len(text) else ""


def short_name(mangled):
    try:
        d = run(tool("cu++filt"), mangled).strip()
    except (subprocess.CalledProcessError, SystemExit):
        return mangled
    d = d[:d.rfind(">(") + 1] if ">(" in d else d  # drop the parameter list
    d = re.sub(r"^void |\((unsigned )?int\)", "", d).replace("rtb::", "")
    return d.replace("(bool)0", "false").replace("(bool)1", "true")


def ptxas_log_for(obj):
    d = os.path.dirname(os.path.abspath(obj))
    for cand in (os.path.join(d, "build", "kernels.ptxas.log"), os.path.join(d, "csrc", "build", "kernels.ptxas.log")):
        if os.path.exists(cand):
            return cand
    logs = [os.path.join(d, f) for f in sorted(os.listdir(d)) if f.endswith(".ptxas.log")]
    return logs[0] if logs else None


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("obj", nargs="+")
    ap.add_argument("--kernel", action="append", help="substring of the mangled kernel name (repeatable)")
    ap.add_argument("--top", type=int, default=10, help="source lines to list per kernel (0: the table only)")
    a = ap.parse_args()
    pats = a.kernel or DEFAULT_KERNELS
    table, details = [], []
    for obj in a.obj:
        spills = ptxas_spills(ptxas_log_for(obj))
        usage = res_usage(obj)
        found = 0
        with tempfile.TemporaryDirectory() as tmp:
            for cub in cubins(obj, tmp):
                for name, idx in sorted(global_functions(cub).items()):
                    if not any(p in name for p in pats):
                        continue
                    found += 1
                    regs, stack = usage.get(name, (None, None))
                    frame, sst, sld = spills.get(name, (stack, None, None))
                    live, lines = live_counts(cub, idx), line_map(cub, idx)
                    peak = max(live.values()) if live else 0
                    table.append((obj, short_name(name), regs, frame, sst, sld, peak))
                    if a.top <= 0:
                        continue
                    per_line = collections.defaultdict(list)
                    for off, n in live.items():
                        per_line[lines.get(off)].append(n)
                    out = [f"{obj}: {short_name(name)}", f"  {'max':>4} {'mean':>5} {'insns':>5}  line"]
                    for where, ns in sorted(per_line.items(), key=lambda kv: (-max(kv[1]), -len(kv[1])))[:a.top]:
                        f, ln = where if where else ("?", 0)
                        out.append(f"  {max(ns):4d} {sum(ns) / len(ns):5.1f} {len(ns):5d}  {os.path.basename(f)}:{ln}  {source_line(f, ln)[:90]}")
                    details.append("\n".join(out))
        if not found:
            sys.exit(f"reg_pressure: no kernel matching {pats} in {obj}")
    na = lambda v: "n/a" if v is None else str(v)
    w = max(len(t[1]) for t in table)
    print(f"{'kernel':<{w}}  {'regs':>4}  {'stack B':>7}  {'spill st B':>10}  {'spill ld B':>10}  {'peak live':>9}  object")
    for obj, k, regs, frame, sst, sld, peak in table:
        print(f"{k:<{w}}  {na(regs):>4}  {na(frame):>7}  {na(sst):>10}  {na(sld):>10}  {peak:>9}  {obj}")
    for d in details:
        print("\n" + d)


if __name__ == "__main__":
    main()
