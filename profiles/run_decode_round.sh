#!/bin/bash
# A/B of the flat crop decode's measure pass (profiles/decode_round_r01.md), run from the repository root:
#   profiles/run_decode_round.sh PARENT_TREE OUT_DIR
# PARENT_TREE is a built checkout of the parent commit; the JSON lines and logs go to OUT_DIR.  bench.py is
# alternated between the two trees in one call (C2 defaults five times each; C1, C3 and C4 three times each), then
# profiles/bench_intervals.py runs once in each tree for the per-launch kernel times.  The CPU arm of bench.py
# (--no-cpu) runs after the GPU measurements and does not change them; it is left out to save time.
P=${1:?usage: $0 PARENT_TREE OUT_DIR}
mkdir -p "${2:?usage: $0 PARENT_TREE OUT_DIR}"
out=$(cd "$2" && pwd)
gpu() { nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader; }
gpu | tee $out/gpu.txt
run() {  # run ARM TAG ARGS...: bench.py in the parent tree or in this one, the JSON line to $out/TAG_ARM.json
    local arm=$1 tag=$2; shift 2
    local d=.; [ $arm = parent ] && d=$P
    (cd $d && timeout 900 python bench.py "$@" > /tmp/dr_$$.json 2> /tmp/dr_$$.err) || tail -3 /tmp/dr_$$.err
    tail -n 1 /tmp/dr_$$.json > $out/${tag}_${arm}.json
}
for i in 1 2 3 4 5; do
    for arm in parent branch; do run $arm c2_$i --no-cpu; done
done
for i in 1 2 3; do
    for arm in parent branch; do
        run $arm c1_$i --config c1_powder_example --no-cpu --no-e2e --no-api --no-span
        run $arm c3_$i --config c3_satellites --no-cpu --no-e2e --no-api --no-span
        run $arm c4_$i --config c4_spheroidite --images 40 --sparse --no-cpu --no-e2e --no-api --no-span
    done
done
for arm in parent branch; do
    d=.; [ $arm = parent ] && d=$P
    (cd $d && timeout 900 python profiles/bench_intervals.py --rounds 3 --reps 20 --out /tmp/bi_$arm > $out/intervals_$arm.log 2>&1)
    cp /tmp/bi_$arm/intervals.json $out/intervals_$arm.json
done
gpu | tee -a $out/gpu.txt
OUT=$out python - <<'PY'
import glob, json, os, statistics as S
out = os.environ['OUT']
def load(tag, arm):
    r = []
    for f in sorted(glob.glob('%s/%s_*_%s.json' % (out, tag, arm))):
        try:
            r.append(json.loads(open(f).read()))
        except ValueError:
            pass
    return r
for tag in ('c2', 'c1', 'c3', 'c4'):
    for arm in ('parent', 'branch'):
        r = load(tag, arm)
        if not r:
            print(tag, arm, 'no runs'); continue
        ms = [d['ms_per_step'] for d in r]
        line = '%s %-6s ms_per_step median %.4f [%.4f, %.4f] n=%d' % (tag, arm, S.median(ms), min(ms), max(ms), len(ms))
        if tag == 'c2':
            c5 = [d['c5_strong']['ms_per_pass'] for d in r if 'c5_strong' in d]
            e2e = [d['e2e']['ms_per_step'] for d in r if 'e2e' in d]
            line += '  c5 %.3f [%.3f, %.3f]  e2e %.3f [%.3f, %.3f]' % (S.median(c5), min(c5), max(c5), S.median(e2e), min(e2e), max(e2e))
        print(line)
for arm in ('parent', 'branch'):
    d = json.load(open('%s/intervals_%s.json' % (out, arm)))
    for c in ('c2', 'c1', 'c3', 'c4'):
        print(arm, c, 'kernels on', json.dumps(d[c]['kernels_on']), 'off', json.dumps(d[c]['kernels_off']),
              'ms on', ['%.4f' % x for x in d[c]['ms_on']], 'off', ['%.4f' % x for x in d[c]['ms_off']])
PY
