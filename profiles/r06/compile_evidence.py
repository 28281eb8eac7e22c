"""Compile evidence for the softmax-exploration instantiations (no GPU needed).

Builds csrc/rlrm_b200.cu of this tree and of a parent revision (git archive into a temporary directory) for sm_100a with
-Xptxas -v, then writes:
  r06_ptxas_softmax.txt    registers / stack / spills of every SOFTMAX = true instantiation next to its epsilon-greedy twin
  r06_uniform_check.txt    every kernel of the parent against the same (epsilon-greedy) instantiation of this tree (registers,
                           stack, spills), and a diff of `cuobjdump -sass` of train_qrm4_kernel<FrozenLake, 1, 1, 0, 7, false>

The kernels that gained the flag (train_kernel, train_qlambda_kernel, train_qlambda_sparse_kernel, select_kernel,
update_list_kernel) take beta as their last parameter and the flag as their last template argument (train_kernel: an optional
sixth one, absent in its epsilon-greedy instantiations); an epsilon-greedy instantiation is matched to the parent's kernel of
the same name with both removed.

Result (nvcc 12.9): the headline train_qrm4_kernel, every specialised kernel, the Q(lambda), select and update-list kernels are
unchanged (the latter four instruction for instruction). The 32 epsilon-greedy train_kernel instantiations differ in SASS and 22
of them in registers / spills: 21 use fewer registers or spill less, train_kernel<FrozenLake, QRM, per-agent, double, false>
uses 2 more (96, no spills). Their PTX is the parent's up to the numbering of virtual registers (cicc numbers them in another
order once the module also holds the softmax instantiations; compared for train_kernel<0, 1, true, double, false>), and ptxas
allocates from that numbering.

usage: python profiles/r06/compile_evidence.py [parent-rev]   (default HEAD)
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
FLAGGED = ("train_kernel", "train_qlambda_kernel", "train_qlambda_sparse_kernel", "select_kernel", "update_list_kernel")
FMT = "regs %3d  stack %4d  spill st %4d ld %4d"


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


def nvcc_release():
    out = subprocess.run([NVCC, "--version"], capture_output=True, text=True).stdout
    return next((ln.strip() for ln in out.splitlines() if "release" in ln), "nvcc")


def kind(name):
    return name.split("<")[0].replace("void ", "")


def strip_flag(name):
    """(the epsilon-greedy instantiation's name as the parent spells it, SOFTMAX value)"""
    if kind(name) == "train_kernel" and name.split(">")[0].count(",") == 4:  # no SOFTMAX argument: epsilon-greedy
        return name.replace(", double)", ")"), False
    if kind(name) not in FLAGGED:
        return name, False
    m = re.match(r"(.*), (true|false)>\((.*), double\)$", name)
    return f"{m.group(1)}>({m.group(3)})", m.group(2) == "true"


def main():
    parent = sys.argv[1] if len(sys.argv) > 1 else "HEAD"
    with tempfile.TemporaryDirectory() as tmp:
        src = os.path.join(tmp, "parent")
        os.makedirs(src)
        subprocess.run(f"git -C {ROOT} archive {parent} | tar -x -C {src}", shell=True, check=True)
        base_lib, new_lib = os.path.join(tmp, "parent.so"), os.path.join(tmp, "new.so")
        base, new = parse(build(src, base_lib)), parse(build(ROOT, new_lib))
        dn, db = demangle(list(new)), demangle(list(base))
        new_by_name = {}
        for mangled, v in new.items():
            name = dn[mangled]
            key, soft = strip_flag(name)
            new_by_name[(key, soft)] = (mangled, v)

        uni_lines, changed, missing = [], 0, 0
        for mangled, v in sorted(base.items(), key=lambda kv: db[kv[0]]):
            name = db[mangled]
            twin = new_by_name.get((name, False))
            same = twin is not None and twin[1] == v
            changed += twin is not None and not same
            missing += twin is None
            uni_lines.append(f"{'same' if same else ('MISSING' if twin is None else 'CHANGED')}  {name.split('(')[0]}   {FMT % v}" +
                             ("" if same or twin is None else f"   now: {FMT % twin[1]}"))
        soft_lines = []
        for (key, soft), (_m, v) in sorted(new_by_name.items()):
            if soft:
                twin = new_by_name.get((key, False))
                soft_lines.append(f"{key.split('(')[0]} +SOFTMAX   {FMT % v}   | epsilon-greedy " + (FMT % twin[1] if twin else "missing"))
        with open(os.path.join(HERE, "r06_ptxas_softmax.txt"), "w") as f:
            f.write(f"# sm_100a, {nvcc_release()}; SOFTMAX = true instantiations and their epsilon-greedy twins ({len(soft_lines)} kernels)\n")
            f.write("\n".join(soft_lines) + "\n")
        headline = "void train_qrm4_kernel<0, true, true, false, 7, false>(KP, DState, unsigned long long, int, unsigned int*, Sweep)"
        hb = next(k for k, n in db.items() if n == headline)
        hn = new_by_name[(headline, False)][0]
        sb, sn = sass(base_lib, hb), sass(new_lib, hn)
        body = lambda s: [ln for ln in s.splitlines() if re.match(r"\s+/\*[0-9a-f]{4}\*/", ln)]  # instruction lines only
        identical = body(sb) == body(sn)
        # the epsilon-greedy instantiations of every kernel the change touched: instruction for instruction as in the parent?
        sass_lines, sass_same = [], 0
        for mangled in sorted(base, key=lambda m: db[m]):
            name = db[mangled]
            if kind(name) in FLAGGED:
                same = body(sass(base_lib, mangled)) == body(sass(new_lib, new_by_name[(name, False)][0]))
                sass_same += same
                sass_lines.append(f"{'same SASS' if same else 'DIFFERENT SASS'}  {name.split('(')[0]}")
        with open(os.path.join(HERE, "r06_uniform_check.txt"), "w") as f:
            f.write(f"# every kernel of {parent} against its epsilon-greedy instantiation in this tree: {len(uni_lines)} kernels, "
                    f"{changed} with different registers / stack / spills, {missing} missing\n")
            f.write("\n".join(uni_lines) + "\n")
            f.write(f"\n# cuobjdump -sass of train_qrm4_kernel<FrozenLake, 1, 1, 0, 7, false> ({len(body(sn))} instruction lines): "
                    f"{'IDENTICAL to the parent' if identical else 'DIFFERENT from the parent'}\n")
            f.write(f"\n# cuobjdump -sass of the epsilon-greedy instantiations of the kernels with a softmax variant: {sass_same} of "
                    f"{len(sass_lines)} identical to the parent\n")
            f.write("\n".join(sass_lines) + "\n")
        print(f"epsilon-greedy SASS identical: {sass_same} / {len(sass_lines)}")
        print(f"kernels changed: {changed}; missing: {missing}; softmax instantiations: {len(soft_lines)}; headline SASS identical: {identical}")


if __name__ == "__main__":
    main()
