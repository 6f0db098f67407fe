#!/bin/bash
# Same-box A/B of library builds: the in-tree library (arm "new") against tools/gpu/ab/lib*.so (built from another commit or
# with -D switches), alternated, so that both arms share the box, its clocks and its neighbours.   bash tools/gpu/ab.sh TAG OUTDIR
#   AB_REPS=5        alternations of the Test_03 kernel-time run (bench.py --no-cpu --no-sweep --no-configs --no-policy --episodes 0)
#   AB_CFGS="..."    further configurations per alternation, each "name[:envs]" (e.g. "Test_08 Test_14 Test_02:8192")
#   AB_TEST=1        the GPU tests of the in-tree library first
#   AB_DUMP="..."    bench.py --dump-outputs of every arm per "name[:envs]", compared byte for byte against the in-tree library
#   AB_PHASES=1      tools/phase_times.py per arm (Test_03)
#   AB_BENCH=1       the default `python bench.py` once per arm
# Everything goes to OUTDIR/TAG_*; TAG_ab.jsonl holds one bench line per run with its arm and configuration.
TAG=${1:-ab}
O=${2:?usage: ab.sh TAG OUTDIR}
mkdir -p $O
LIB=flatland-marl_b200/csrc/libflatland_b200.so
W=$(mktemp -d)
cp $LIB $W/libnew.so
ARMS="new"; for f in tools/gpu/ab/lib*.so; do [ -f $f ] && { a=$(basename $f .so); a=${a#lib}; cp $f $W/lib$a.so; ARMS="$ARMS $a"; }; done
use() { cp $W/lib$1.so $LIB; }
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $O/${TAG}_gpu.txt
if [ "${AB_TEST:-0}" = 1 ]; then
  use new
  timeout 1500 python -m pytest tests/test_gpu_parity.py tests/test_gpu_deep.py tests/test_gpu_fullsize.py tests/test_fork.py \
    tests/test_gpu_rollout.py tests/test_gpu_conflict_check.py -m gpu -q -x > $O/${TAG}_pytest.log 2>&1; tail -3 $O/${TAG}_pytest.log
fi
for spec in $AB_DUMP; do
  cfg=${spec%%:*}; env=$([ "$spec" != "$cfg" ] && echo "--envs ${spec#*:}")
  for a in $ARMS; do
    use $a
    timeout 600 python bench.py --config $cfg $env --steps 20 --warmup 5 --no-cpu --no-sweep --no-configs --no-policy --episodes 0 \
      --dump-outputs $W/dump_${a}_$cfg > /dev/null 2>> $O/${TAG}_dump.err
  done
  for a in $ARMS; do
    [ $a = new ] && continue
    if diff -r -q $W/dump_new_$cfg $W/dump_${a}_$cfg > /dev/null && [ -n "$(ls $W/dump_new_$cfg 2>/dev/null)" ]; then r=identical; else r=DIFFERENT; fi
    echo "dump $spec new vs $a: $r ($(ls $W/dump_new_$cfg | wc -l) files)" | tee -a $O/${TAG}_dump.txt
  done
done
OUT=$O/${TAG}_ab.jsonl; : > $OUT
run() { a=$1; spec=$2; cfg=${spec%%:*}; env=$([ "$spec" != "$cfg" ] && echo "--envs ${spec#*:}")
  use $a
  timeout 300 python bench.py --config $cfg $env --no-cpu --no-sweep --no-configs --no-policy --episodes 0 2>> $O/${TAG}_ab.err |
    python -c "import sys,json; d=json.loads(sys.stdin.read()); print(json.dumps({'arm': '$a', 'config': '$spec', 'value': d['value'], 'ms_per_step': d['ms_per_step'], 'kernels': {k: v['ms_per_launch'] for k, v in d['kernels'].items()}, 'clocks': d.get('clocks')}))" >> $OUT; }
for r in $(seq ${AB_REPS:-5}); do
  for a in $ARMS; do run $a Test_03; for spec in $AB_CFGS; do run $a $spec; done; done
done
python - $OUT <<'EOF' | tee $O/${TAG}_ab.txt
import json, sys, collections, statistics as st
rows = [json.loads(l) for l in open(sys.argv[1]) if l.strip()]
g = collections.defaultdict(list)
for r in rows:
    g[(r["config"], r["arm"])].append(r)
for (cfg, arm), rs in sorted(g.items()):
    ks = sorted(rs[0]["kernels"])
    ker = "  ".join("%s %.4f [%.4f..%.4f]" % (k, st.median(x["kernels"][k] for x in rs), min(x["kernels"][k] for x in rs), max(x["kernels"][k] for x in rs)) for k in ks)
    v = [x["value"] / 1e6 for x in rs]
    print("%-14s %-5s n=%d  value %.1f M [%.1f..%.1f]  ms/step %.4f  %s" % (cfg, arm, len(rs), st.median(v), min(v), max(v), st.median(x["ms_per_step"] for x in rs), ker))
EOF
if [ "${AB_PHASES:-0}" = 1 ]; then
  for a in $ARMS; do use $a; echo "== phase_times Test_03 arm $a"; timeout 300 python tools/phase_times.py Test_03 2>&1 | tail -14; done | tee $O/${TAG}_phases.txt
fi
if [ "${AB_BENCH:-0}" = 1 ]; then
  for a in $ARMS; do use $a; timeout 1500 python bench.py > $O/${TAG}_bench_$a.json 2> $O/${TAG}_bench_$a.err; echo "bench $a: $(head -c 200 $O/${TAG}_bench_$a.json)"; done
fi
use new
rm -rf $W
