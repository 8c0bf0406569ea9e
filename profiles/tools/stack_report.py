"""Stack frame, spills and local-memory instructions of the fused RRT kernel, without a GPU:
    python profiles/tools/stack_report.py [--kernel NAME] [--json OUT]
Compiles theta_rrt_b200/csrc/thetarrt.cu to a cubin with the flags of theta_rrt_b200/build.py plus -Xptxas -v, once as
shipped and once with -DTRRT_CHECKED, and prints for the kernel (default rrt_kernel_spec<32>): registers, stack frame,
spill stores / loads (ptxas), and the LDL / STL instructions in its SASS (cuobjdump -sass), in total and per device
function it calls (nvdisasm labels every callee inside the kernel's section)."""
import argparse, json, os, re, subprocess, sys, tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from theta_rrt_b200 import build as B  # noqa: E402

KERNEL = "_ZN4trrt15rrt_kernel_specILi32EEEvNS_6RrtDevE"
ADDR = re.compile(r"/\*[0-9a-f]{4,}\*/")


def tool(name):
    return os.path.join(os.path.dirname(B.nvcc_path()), name)


def compile_cubin(cubin, flags):
    # the device flags of build.py: host-compiler options and -shared do not reach a cubin
    base, skip = [], False
    for f in B.NVCC_FLAGS:
        if skip or f == "-shared":
            skip = False
            continue
        if f == "-Xcompiler":
            skip = True
            continue
        base.append(f)
    cmd = [B.nvcc_path(), *base, *flags, "-Xptxas", "-v", "-cubin", "-o", cubin, os.path.join(B.CSRC, "thetarrt.cu")]
    out = subprocess.run(cmd, capture_output=True, text=True)
    if out.returncode:
        sys.exit(out.stderr[-3000:])
    return out.stderr.splitlines()


def ptxas_numbers(lines, kernel):
    for i, l in enumerate(lines):
        if "Function properties for " + kernel in l:
            m1 = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", lines[i + 1])
            m2 = re.search(r"Used (\d+) registers", lines[i + 2])
            return dict(registers=int(m2.group(1)), stack_frame=int(m1.group(1)), spill_stores=int(m1.group(2)),
                        spill_loads=int(m1.group(3)))
    sys.exit("kernel %s not in the ptxas output" % kernel)


def sass_counts(cubin, kernel):
    sass = subprocess.run([tool("cuobjdump"), "-sass", "-fun", kernel, cubin], capture_output=True, text=True, check=True).stdout
    ins = [l for l in sass.splitlines() if ADDR.search(l)]
    total = dict(LDL=sum(1 for l in ins if re.search(r"\bLDL\b", l)), STL=sum(1 for l in ins if re.search(r"\bSTL\b", l)),
                 instructions=len(ins))
    # per callee: nvdisasm names the device functions of the kernel's section "$<kernel>$<function>"
    dis = subprocess.run([tool("nvdisasm"), "-c", cubin], capture_output=True, text=True, check=True).stdout
    per, cur = {}, None
    for l in dis.splitlines():
        m = re.match(r"^(\$?[\w$]+):\s*$", l)
        if m and not m.group(1).startswith(".L"):
            label = m.group(1)
            if label == kernel: cur = "(kernel body)"
            elif label.startswith("$" + kernel + "$"): cur = label.split("$")[-1]
            elif not label.startswith("$__internal"): cur = None  # another kernel's section
            continue
        if cur and ADDR.search(l):
            c = per.setdefault(cur, [0, 0])
            c[0] += bool(re.search(r"\bLDL\b", l))
            c[1] += bool(re.search(r"\bSTL\b", l))
    return total, {k: v for k, v in per.items() if v[0] or v[1]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--kernel", default=KERNEL)
    ap.add_argument("--json", help="also write the numbers to this file")
    args = ap.parse_args()
    report = {}
    with tempfile.TemporaryDirectory() as tmp:
        for name, flags in (("default", []), ("checked", ["-DTRRT_CHECKED"])):
            cubin = os.path.join(tmp, name + ".cubin")
            r = ptxas_numbers(compile_cubin(cubin, flags), args.kernel)
            total, per = sass_counts(cubin, args.kernel)
            r.update(total)
            r["per_function"] = {k: dict(LDL=v[0], STL=v[1]) for k, v in sorted(per.items(), key=lambda kv: -sum(kv[1]))}
            report[name] = r
            print(f"{name:8s} {args.kernel}: {r['registers']} registers, {r['stack_frame']} B stack frame, "
                  f"{r['spill_stores']} B spill stores, {r['spill_loads']} B spill loads, "
                  f"{r['LDL']} LDL + {r['STL']} STL = {r['LDL'] + r['STL']} of {r['instructions']} SASS instructions")
            for k, v in r["per_function"].items():
                print(f"         {v['LDL']:4d} LDL {v['STL']:4d} STL  {k}")
    if args.json:
        with open(args.json, "w") as f:
            json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
