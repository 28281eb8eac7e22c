"""Compile evidence for the hyper-parameter sweep instantiations (no GPU needed).

Builds csrc/rlrm_b200.cu of this tree and of a parent revision (git archive into a temporary directory) for sm_100a with
-Xptxas -v, then writes:
  r05_ptxas_sweep.txt     registers / stack / spills of every SWEEP = true training-kernel instantiation, next to its uniform twin
  r05_uniform_check.txt   every uniform training-kernel instantiation against the parent (registers, stack, spills), and a
                          diff of `cuobjdump -sass` of train_qrm4_kernel<FrozenLake, STOCH=1, LEARN=1, TRACE=0, MINB=7>

usage: python profiles/r05/compile_evidence.py [parent-rev]   (default HEAD)
"""
import os
import re
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
CUOBJDUMP = os.path.join(os.path.dirname(NVCC), "cuobjdump")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-shared", "-Xcompiler", "-fPIC", "-Xptxas", "-v"]
TRAIN = ("train_kernel", "train_qrm4_kernel", "train_ql_fast_kernel", "train_qrmn_kernel", "train_qrm_block_kernel",
         "train_qlambda_kernel", "train_qlambda_sparse_kernel")


def build(src_root, out):
    r = subprocess.run([NVCC, *FLAGS, "-o", out, os.path.join(src_root, "multiagent-rl-rm_b200", "csrc", "rlrm_b200.cu")],
                       capture_output=True, text=True, check=True)
    return r.stdout + r.stderr


def parse(log):
    """mangled entry name -> (registers, stack bytes, spill store bytes, spill load bytes)"""
    out, cur, frame = {}, None, None
    for line in log.splitlines():
        m = re.search(r"Compiling entry function '(\w+)'", line)
        if m:
            cur, frame = m.group(1), None
            continue
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and cur:
            frame = tuple(int(x) for x in m.groups())
        m = re.search(r"Used (\d+) registers", line)
        if m and cur:
            out[cur] = (int(m.group(1)),) + (frame or (0, 0, 0))
            cur = None
    return out


def demangle(names):
    r = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True, check=True).stdout.split("\n")
    return dict(zip(names, r))


def sass(lib, mangled):
    return subprocess.run([CUOBJDUMP, "-sass", "-fun", mangled, lib], capture_output=True, text=True, check=True).stdout


def main():
    parent = sys.argv[1] if len(sys.argv) > 1 else "HEAD"
    with tempfile.TemporaryDirectory() as tmp:
        src = os.path.join(tmp, "parent")
        os.makedirs(src)
        subprocess.run(f"git -C {ROOT} archive {parent} | tar -x -C {src}", shell=True, check=True)
        base_lib, new_lib = os.path.join(tmp, "parent.so"), os.path.join(tmp, "new.so")
        base, new = parse(build(src, base_lib)), parse(build(ROOT, new_lib))
        dn, db = demangle(list(new)), demangle(list(base))
        base_by_name = {db[k]: (k, v) for k, v in base.items()}

        def kind(name):
            return name.split("<")[0].replace("void ", "")

        sweep_lines, uni_lines, changed = [], [], 0
        for mangled, v in sorted(new.items(), key=lambda kv: dn[kv[0]]):
            name = dn[mangled]
            if kind(name) not in TRAIN:
                continue
            # the SWEEP flag is the last template argument, Sweep the last parameter
            uniform_name = re.sub(r", (true|false)>\(", ">(", name, count=1).replace(", Sweep)", ")")
            twin = base_by_name.get(uniform_name)
            fmt = "regs %3d  stack %4d  spill st %4d ld %4d"
            if ", true>(" in name:
                ref = ("uniform twin " + fmt % twin[1]) if twin else "no uniform twin"
                sweep_lines.append(f"{uniform_name.split('(')[0]} +SWEEP   {fmt % v}   | {ref}")
            else:
                same = twin is not None and twin[1] == v
                changed += not same
                uni_lines.append(f"{'same' if same else 'CHANGED'}  {name.split('(')[0]}   {fmt % v}" +
                                 ("" if same else f"   parent: {fmt % twin[1] if twin else 'missing'}"))
        with open(os.path.join(HERE, "r05_ptxas_sweep.txt"), "w") as f:
            f.write(f"# sm_100a, nvcc {NVCC}; SWEEP = true instantiations of the training kernels and their uniform twins\n")
            f.write("\n".join(sweep_lines) + "\n")
        headline = "void train_qrm4_kernel<0, true, true, false, 7>(KP, DState, unsigned long long, int, unsigned int*)"
        hb = base_by_name[headline][0]
        hn = next(k for k, n in dn.items() if n.startswith("void train_qrm4_kernel<0, true, true, false, 7, false>"))
        sb, sn = sass(base_lib, hb), sass(new_lib, hn)
        body = lambda s: [ln for ln in s.splitlines() if re.match(r"\s+/\*[0-9a-f]{4}\*/", ln)]  # instruction lines only
        identical = body(sb) == body(sn)
        with open(os.path.join(HERE, "r05_uniform_check.txt"), "w") as f:
            f.write(f"# uniform training-kernel instantiations of this tree against {parent}: {len(uni_lines)} kernels, "
                    f"{changed} with different registers / stack / spills\n")
            f.write("\n".join(uni_lines) + "\n")
            f.write(f"\n# cuobjdump -sass of train_qrm4_kernel<FrozenLake, 1, 1, 0, 7> ({len(body(sn))} instruction lines): "
                    f"{'IDENTICAL to the parent' if identical else 'DIFFERENT from the parent'}\n")
        print(f"uniform kernels changed: {changed}; headline SASS identical: {identical}")


if __name__ == "__main__":
    main()
