#!/bin/bash
# The int8 filter pass (DESIGN.md section 4, K1f8) with its side data staged through the ring, two rows per consumer
# warp and the query split once per CTA, against the previous build of that pass, in one run (profiles/r07_filter8_ring.txt):
# the card, both libraries built, bench.py --only alternating old / new three times each, one full bench.py line of each,
# scripts/filter_roofline.py --c4 of each, and --dump-outputs compared file by file: old against new (automatic route),
# and SVSB_FILTER=0 against automatic (new).
#   scripts/gpu_r07_filter8_ring.sh OUT OLD_TREE
# OLD_TREE: a checkout of the previous commit (e.g. git worktree add /tmp/old HEAD~1); its library is built there.
set -u
OUT=${1:?output directory}
OLD=$(cd "${2:?checkout of the previous commit}" && pwd)
NEW=$(cd "$(dirname "$0")/.." && pwd)
mkdir -p "$OUT"
OUT=$(cd "$OUT" && pwd)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv
for t in "$OLD" "$NEW"; do (cd "$t" && python -m svs_b200.build > /dev/null) || { echo "build failed in $t"; exit 1; }; done
summ() {
    python3 - "$1" <<'EOF'
import json, sys
j = json.loads(open(sys.argv[1]).read().strip().splitlines()[-1])
def leg(x):
    r = x.get("roofline", {})
    return (f"value {x['value']:.1f} e2e {x['e2e']['value']:.1f} (1 in flight {x['e2e'].get('one_query_in_flight', 0):.1f}) "
            f"roofline achieved {r.get('achieved', 0):.0f} {r.get('unit', '')} frac {r.get('frac', 0):.3f} parity {json.dumps(x.get('parity'))[:90]}")
print("  c2:", leg(j), "| clocks", json.dumps(j.get("clocks")))
for name, x in sorted(j.get("configs", {}).items()):
    print(f"  {name}:", leg(x))
EOF
}
run() {                            # run <tree> <SVSB_FILTER value or "auto"> <output stem> <bench.py arguments...>
    local tree=$1 f=$2 stem=$3; shift 3
    if [ "$f" = auto ]; then (cd "$tree" && env -u SVSB_FILTER python bench.py --gpus 1 --steps 20 --warmup 3 "$@") > "$OUT/$stem.json" 2> "$OUT/$stem.err"
    else (cd "$tree" && SVSB_FILTER=$f python bench.py --gpus 1 --steps 20 --warmup 3 "$@") > "$OUT/$stem.json" 2> "$OUT/$stem.err"; fi
}
for rep in 1 2 3; do
    for v in old new; do
        if [ $v = old ]; then t=$OLD; else t=$NEW; fi
        run "$t" auto only_${v}_r$rep --only
        echo "--only $v repeat $rep (rc=$?):"; summ "$OUT/only_${v}_r$rep.json"
    done
done
for v in old new; do
    if [ $v = old ]; then t=$OLD; else t=$NEW; fi
    run "$t" auto full_$v
    echo "full bench.py $v (rc=$?):"; summ "$OUT/full_$v.json"
done
rm -rf "$OUT"/dump_*
run "$OLD" auto dump_run_old --dump-outputs "$OUT/dump_old"
run "$NEW" auto dump_run_new --dump-outputs "$OUT/dump_new"
run "$NEW" 0 dump_run_new_f0 --dump-outputs "$OUT/dump_new_f0"
cmpdir() {
    echo "dump-outputs, $3:"
    for p in "$1"/*; do
        b=$(basename "$p")
        if cmp -s "$p" "$2/$b"; then echo "  $b identical"; else echo "  $b DIFFERS"; fi
    done
}
cmpdir "$OUT/dump_old" "$OUT/dump_new" "old against new (automatic route)"
cmpdir "$OUT/dump_new_f0" "$OUT/dump_new" "new, SVSB_FILTER=0 against automatic"
for v in old new; do
    if [ $v = old ]; then t=$OLD; else t=$NEW; fi
    echo "filter_roofline.py --c4, $v:"
    (cd "$t" && python scripts/filter_roofline.py --c4)
done
