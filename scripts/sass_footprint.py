"""Instruction footprint of the bs = 1 GEMV kernel image, read from the built library (CPU only, no GPU needed).

For every kernel whose name matches --kernel (default: gemv1_kernel) it prints the SASS instruction count, registers,
stack (spills) and a breakdown of the instructions by the source region they come from.  Regions are found from
`nvdisasm --print-line-info`: each instruction carries the innermost file and line it was generated from, and that line
is mapped to the function of the source file that encloses it.  Out-of-line device functions of the same cubin (cold
paths the kernel calls) are listed separately.

    python scripts/sass_footprint.py [--lib llama2-accessory_b200/libb200decode.so] [--kernel gemv1_kernel]
"""
import argparse
import collections
import os
import re
import shutil
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "llama2-accessory_b200", "csrc")

# (region, file basename, function names or None for the whole file); the first match wins
REGIONS = [
    ("producer: L2 prefetch helpers", "common.cuh", {"l2_prefetch", "prefetch_next_stream"}),
    ("producer body (gemv1.cu)", "gemv1.cu", {"<producer>"}),
    ("epilogue (g1_epilogue_phase)", "gemv1_core.cuh", {"g1_epilogue_phase"}),
    ("cuda_fp16.hpp (inlined)", "cuda_fp16.hpp", None),
    ("load_delta8 / rank_sum8", "gemv_core.cuh", {"load_delta8", "rank_sum8"}),
    ("LL poll (ll.cuh)", "ll.cuh", None),
    ("digit split (split8)", "gemv1_core.cuh", {"split8"}),
    ("x staging", "gemv1_core.cuh", {"stage_own_slice", "stage_own_slice_pass", "stage_piece", "g1_delta8"}),
    ("x staging", "gemv_core.cuh", {"hsum8"}),
    ("main loop (g1_mma_tiles)", "gemv1_core.cuh", {"g1_mma_tiles", "imma16832"}),
    ("timeline stamps", "gemv1_core.cuh", {"g1_stamp"}),
    ("timeline stamps", "common.cuh", {"tl_min", "tl_max", "tl_cta", "gtime_ns"}),
]

FUNC_RE = re.compile(r"^(?:template\s*<[^>]*>\s*)?(?:static\s+)?__(?:device|global)__\b.*?\b(\w+)\s*\(")


def tool(name):
    p = os.path.join("/usr/local/cuda/bin", name)
    return p if os.path.isfile(p) else (shutil.which(name) or name)


def function_map(path):
    """line number (1-based) -> enclosing function name, by brace matching from each __device__/__global__ definition.
    In gemv1.cu the producer branch of the kernel is reported as '<producer>'."""
    lines = open(path).read().split("\n")
    owner = {}
    i = 0
    while i < len(lines):
        m = FUNC_RE.match(lines[i].strip())
        if not m:
            i += 1
            continue
        name, depth, started, j = m.group(1), 0, False, i
        while j < len(lines):
            code = lines[j].split("//")[0]
            depth += code.count("{") - code.count("}")
            started = started or "{" in code
            owner[j + 1] = name
            if started and depth <= 0:
                break
            j += 1
        i = j + 1
    if os.path.basename(path) == "gemv1.cu":
        inside = False
        for n, text in enumerate(lines, 1):
            if "if (warp == kConsumerWarps)" in text:
                inside = True
            elif "if (warp > kConsumerWarps)" in text:
                inside = False
            if inside:
                owner[n] = "<producer>"
    return owner


def region_of(path, line, maps):
    base = os.path.basename(path)
    for name, fbase, funcs in REGIONS:
        if base != fbase:
            continue
        if funcs is None:
            return name
        src = path if os.path.isfile(path) else os.path.join(CSRC, base)
        if src not in maps:
            maps[src] = function_map(src) if os.path.isfile(src) else {}
        if maps[src].get(line) in funcs:
            return name
    return "other (setup, barriers, mbarrier and bulk-copy helpers, ...)"


def parse_text_sections(dis):
    """{section: {function: [(file, line, opcode text)]}} for every .text section of the disassembly.  A kernel's
    section also holds the out-of-line functions it calls (its __noinline__ helpers, the runtime's slow paths)."""
    out, cur, fn, loc = {}, None, None, ("?", 0)
    for raw in dis.split("\n"):
        m = re.match(r"\s*\.section\s+\.text\.(\S+?),", raw)
        if m:
            cur = fn = m.group(1)
            out[cur] = {fn: []}
            continue
        if raw.startswith("\t.section"):
            cur = None
            continue
        if cur is None:
            continue
        m = re.match(r"\s*\.type\s+(\S+),@function", raw)
        if m:
            fn = m.group(1)
            out[cur].setdefault(fn, [])
            continue
        m = re.match(r'\s*//## File "([^"]+)", line (\d+)', raw)
        if m:
            loc = (m.group(1), int(m.group(2)))
            continue
        m = re.match(r"\s*/\*[0-9a-f]+\*/\s+(.*?)\s*;", raw)
        if m:
            out[cur][fn].append((loc[0], loc[1], m.group(1)))
    return out


def opcode(op):
    words = op.split()
    return (words[1] if words[0].startswith("@") else words[0]).split(".")[0]


def res_usage(cubin):
    txt = subprocess.run([tool("cuobjdump"), "-res-usage", cubin], capture_output=True, text=True, check=True).stdout
    res, fn = {}, None
    for line in txt.split("\n"):
        m = re.match(r"\s*Function (\S+):", line)
        if m:
            fn = m.group(1)
            continue
        if fn and "REG:" in line:
            res[fn] = dict(re.findall(r"(\w+(?:\[\d+\])?):(\d+)", line))
            fn = None
    return res


def demangle(names):
    try:
        r = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True, check=True)
        return dict(zip(names, r.stdout.split("\n")))
    except (OSError, subprocess.CalledProcessError):
        return {n: n for n in names}


def analyse(lib, member="gemv1.sm_100a.cubin", kernel="gemv1_kernel"):
    """[{name, body, total, registers, stack, regions: Counter, split_copies, out_of_line: [(name, n)]}] per kernel."""
    with tempfile.TemporaryDirectory() as tmp:
        subprocess.run([tool("cuobjdump"), "-xelf", member, os.path.abspath(lib)], cwd=tmp, capture_output=True, check=True)
        cubin = os.path.join(tmp, member)
        dis = subprocess.run([tool("nvdisasm"), "--print-line-info", cubin], capture_output=True, text=True,
                             check=True).stdout
        res = res_usage(cubin)
    secs = parse_text_sections(dis)
    maps, out = {}, []
    for k in [k for k in secs if re.search(kernel, k)]:
        ins = secs[k][k]
        split_prmt = sum(1 for f, l, op in ins if opcode(op) == "PRMT" and region_of(f, l, maps) == "digit split (split8)")
        ool = []
        for fn, fins in secs[k].items():
            if fn != k:
                short = re.sub(r"^\$" + re.escape(k) + r"\$", "", fn)
                name = demangle([short])[short] if short.startswith("_Z") else short
                ool.append((re.sub(r"_INTERNAL_\w+?_cu_[0-9a-f]+::", "", name), len(fins)))
        out.append(dict(name=demangle([k])[k], body=len(ins), total=sum(len(v) for v in secs[k].values()),
                        registers=int(res.get(k, {}).get("REG", -1)), stack=int(res.get(k, {}).get("STACK", -1)),
                        regions=collections.Counter(region_of(f, l, maps) for f, l, _ in ins),
                        split_copies=split_prmt / 12, out_of_line=ool))
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--lib", default=os.path.join(ROOT, "llama2-accessory_b200", "libb200decode.so"))
    ap.add_argument("--cubin", default="gemv1.sm_100a.cubin", help="ELF member of the library to read")
    ap.add_argument("--kernel", default="gemv1_kernel", help="regex on the mangled kernel name")
    a = ap.parse_args()
    kernels = analyse(a.lib, a.cubin, a.kernel)
    if not kernels:
        sys.exit(f"no kernel matching {a.kernel!r} in {a.cubin}")
    print(f"library: {os.path.relpath(os.path.abspath(a.lib), ROOT)}  member: {a.cubin}")
    for k in kernels:
        print(f"\n== {k['name']}")
        print(f"   SASS instructions: {k['body']} in the kernel body, {k['total']} with its out-of-line functions   "
              f"registers: {k['registers']}   stack (spills): {k['stack']} B")
        for name, n in sorted(k["regions"].items(), key=lambda kv: -kv[1]):
            print(f"   {n:6d}  {name}")
        print(f"   inlined copies of the digit split: {k['split_copies']:g}  (PRMT in split8 / 12 per copy)")
        for name, n in k["out_of_line"]:
            print(f"   out of line: {n:5d}  {name}")


if __name__ == "__main__":
    main()
