#!/bin/bash
# Round-4 measurement of train_qrm4_kernel (block fetch overlapped with the next iteration's draws and the episode-end
# reduction) against the parent build, in one run: card, timed A/B of build/variants/*.so through RLRM_LIB_PATH (alternating
# builds, default --steps 50 --warmup 3), bit-identity of the dumped engine state at the timed sizes, the GPU test suite,
# smoke(), and the default bench line.
# Expects build/variants/librlrm_parent.so (parent commit) and build/variants/librlrm_r04.so (this tree). Results go to $OUT.
set -u
OUT=${OUT:-build/r04_out}
export OUT
mkdir -p $OUT
# the library loader rebuilds a library older than its sources: keep the variants as built
touch build/variants/*.so
md5sum build/variants/*.so > $OUT/variants_md5_before.txt
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $OUT/card.txt

WL=${WL:-"cfg3 cfg5_tables cfg3_ql cfg2_batch ow_exp6_qrm cfg3_f64"}
REP=${REP:-3}
for rep in $(seq 1 $REP); do
  for v in build/variants/librlrm_parent.so build/variants/librlrm_r04.so; do
    for w in $WL; do
      RLRM_LIB_PATH=$PWD/$v timeout 300 python bench.py --no-cpu-baseline --no-configs --no-call-by-call --workload $w 2>>$OUT/ab_stderr.txt | \
        python -c "import json,sys; d=json.loads(sys.stdin.read()); print('$(basename $v) $w rep$rep', '%.4e' % d['value'], '%.3f ms' % d['ms_per_step'])"
    done
  done
done | tee $OUT/ab_r04.txt
python - <<'PY' | tee -a $OUT/ab_r04.txt

# workload: mean (min..max spread) per build, new / parent
import collections, os
v = collections.defaultdict(list)
for line in open(os.environ["OUT"] + "/ab_r04.txt"):
    f = line.split()
    if len(f) >= 4 and f[0].endswith(".so"):
        v[(f[0], f[1])].append(float(f[3]))
for w in dict.fromkeys(k[1] for k in v):
    a, b = v[("librlrm_parent.so", w)], v[("librlrm_r04.so", w)]
    sp = lambda x: 100 * (max(x) - min(x)) / (sum(x) / len(x))
    print(f"{w:12s} parent {sum(a)/len(a):.4e} ({sp(a):.2f} %)  new {sum(b)/len(b):.4e} ({sp(b):.2f} %)  ratio {sum(b)/len(b) / (sum(a)/len(a)):.4f}")
PY

for w in cfg3 cfg5_tables; do
  for v in parent r04; do
    RLRM_LIB_PATH=$PWD/build/variants/librlrm_$v.so timeout 300 python bench.py --dump-outputs $OUT/dump_${w}_$v \
      --no-cpu-baseline --no-configs --no-call-by-call --workload $w > $OUT/dump_${w}_$v.json 2>>$OUT/dump_stderr.txt
  done
done
python - <<'PY' | tee $OUT/dump_compare.txt
import filecmp, os
root = os.environ["OUT"]
for w in ("cfg3", "cfg5_tables"):
    a, b = f"{root}/dump_{w}_parent", f"{root}/dump_{w}_r04"
    names = sorted(os.listdir(a))
    same = [n for n in names if os.path.exists(f"{b}/{n}") and filecmp.cmp(f"{a}/{n}", f"{b}/{n}", shallow=False)]
    print(w, f"{len(same)}/{len(names)} .npy byte-identical", "OK" if names and len(same) == len(names) == len(os.listdir(b)) else "DIFFER", names)
PY
rm -rf $OUT/dump_*_parent/ $OUT/dump_*_r04/  # the comparison is the result; the arrays are large
md5sum build/variants/*.so > $OUT/variants_md5_after.txt
cmp -s $OUT/variants_md5_before.txt $OUT/variants_md5_after.txt && echo "variants unchanged" || echo "VARIANTS CHANGED"

timeout 900 python -m pytest -m gpu -q -p no:cacheprovider tests 2>&1 | tail -15 | tee $OUT/pytest_gpu.txt
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -8 | tee $OUT/smoke.txt
timeout 1200 python bench.py > $OUT/bench_default.json 2> $OUT/bench_default_stderr.txt; echo "bench rc=$?"
tail -c 600 $OUT/bench_default.json
