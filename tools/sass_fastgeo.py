"""Static SASS summary of the register-resident STFT / mask-iSTFT kernels (csrc/fastgeo.cu).

Compiles fastgeo.cu alone for sm_100a with ``-Xptxas -v`` into a temporary directory and prints, for every instantiation of
``stft_run_kernel`` (K1) and ``mask_istft_run_kernel`` (K3) without the trace hook, its registers and spills next to its SASS
opcode counts.  The counts are of the whole kernel and static (each instruction once, whatever its trip count); the frame
loop is most of every kernel, so a change of the per-frame instruction stream shows in them one to one.

    python tools/sass_fastgeo.py [--root REPO] > profiles/<name>.txt
"""
import argparse
import collections
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# opcodes printed as columns (the rest only enter the total); LDS / STS keep their width, every other opcode its base name
COLUMNS = ["FFMA2", "FADD2", "FMUL2", "FFMA", "FADD", "FMUL", "MOV", "FSEL", "SHFL", "LDS", "LDS.64", "LDS.128", "STS.64",
           "STS.128", "LDGSTS", "IMAD", "IADD3", "LEA", "ISETP", "BSSY", "BRA", "VOTE"]


def nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    return "nvcc"


def compile_fastgeo(root, tmp):
    pkg = os.path.join(root, "speech_enhancement_by_s3prl_b200")
    cubin = os.path.join(tmp, "fastgeo.cubin")
    cmd = [nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas=-v", "-cubin",
           "-I", os.path.join(root, "include"), os.path.join(pkg, "csrc", "fastgeo.cu"), "-o", cubin]
    log = subprocess.run(cmd, capture_output=True, text=True, check=True).stderr
    return cubin, log


def ptxas_resources(log):
    """mangled name -> (registers, spill store bytes, spill load bytes)"""
    res, cur, spill = {}, None, (0, 0)
    for line in log.splitlines():
        m = re.search(r"Function properties for (\S+)", line)
        if m:
            cur = m.group(1)
            continue
        m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and cur:
            spill = (int(m.group(1)), int(m.group(2)))
            continue
        m = re.search(r"Used (\d+) registers", line)
        if m and cur:
            res[cur] = (int(m.group(1)),) + spill
            cur = None
    return res


def opcode_counts(cubin):
    txt = subprocess.run(["cuobjdump", "-sass", cubin], capture_output=True, text=True, check=True).stdout
    counts, cur = collections.OrderedDict(), None
    for line in txt.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            counts[cur] = collections.Counter()
            continue
        m = re.match(r"\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\w+\s+)?([A-Z0-9_]+)((?:\.[A-Z0-9_]+)*)", line)
        if m and cur:
            op, mods = m.group(1), m.group(2)
            if op == "NOP":
                continue
            if op in ("LDS", "STS"):
                width = [w for w in (".64", ".128") if w in mods]
                op += width[0] if width else ""
            counts[cur][op] += 1
    return counts


def short_name(demangled):
    name = re.sub(r"\(anonymous namespace\)::", "", demangled)
    return re.sub(r"\(sekern::\w+, GeoRunPlan\)", "", name).replace("void ", "")


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--root", default=ROOT, help="repository tree whose fastgeo.cu is compiled (default: this one)")
    args = ap.parse_args()
    with tempfile.TemporaryDirectory() as tmp:
        cubin, log = compile_fastgeo(args.root, tmp)
        res = ptxas_resources(log)
        counts = opcode_counts(cubin)
    mangled = list(counts)
    names = subprocess.run(["c++filt"], input="\n".join(mangled), capture_output=True, text=True).stdout.splitlines()
    rows = []
    for mg, dm in zip(mangled, names):
        name = short_name(dm)
        m = re.match(r"(stft_run_kernel|mask_istft_run_kernel)<(Geo\w+), (.*)>$", name)
        if not m:
            continue
        targs = [t.strip() for t in m.group(3).split(",")]
        trace = targs[2] if m.group(1) == "stft_run_kernel" else targs[1]
        if trace == "true":
            continue
        rows.append((name, res.get(mg, (0, 0, 0)), counts[mg]))
    print("Static SASS of csrc/fastgeo.cu (nvcc -gencode arch=compute_100a,code=sm_100a -O3, cuobjdump -sass), "
          "instantiations without the trace hook.")
    print("regs / spill = -Xptxas -v registers and spill store+load bytes; total = all instructions but NOP; "
          "LDS = 32-bit loads, LDS.64 / LDS.128 wider ones.\n")
    for name, (regs, sst, sld), c in rows:
        print(f"{name}")
        print(f"    regs {regs}, spill {sst + sld} B, total {sum(c.values())}")
        print("    " + ", ".join(f"{k} {c.get(k, 0)}" for k in COLUMNS))
    return 0


if __name__ == "__main__":
    sys.exit(main())
