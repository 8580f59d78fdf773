#!/bin/bash
# A/B of the single-query int8 filter (DESIGN.md section 4, K1f8) against the fp16 filter in one run
# (profiles/r06_filter8_ab.txt): the card, bench.py --only alternating SVSB_FILTER=16 / automatic three times each, one
# full bench.py line of each, --dump-outputs under SVSB_FILTER=0 (K1) and automatic compared file by file, and
# scripts/filter_roofline.py (real bytes and rows re-scored per route, C4 included).
set -u
OUT=${1:-$(mktemp -d)}             # output directory (first argument; default: a fresh temporary one)
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv
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
run() {                            # run <SVSB_FILTER value or "auto"> <output stem> <bench.py arguments...>
    local f=$1 stem=$2; shift 2
    if [ "$f" = auto ]; then env -u SVSB_FILTER python bench.py --gpus 1 --steps 20 --warmup 3 "$@" > "$OUT/$stem.json" 2> "$OUT/$stem.err"
    else SVSB_FILTER=$f python bench.py --gpus 1 --steps 20 --warmup 3 "$@" > "$OUT/$stem.json" 2> "$OUT/$stem.err"; fi
}
for rep in 1 2 3; do
    for f in 16 auto; do
        run $f only_f${f}_r$rep --only
        echo "--only SVSB_FILTER=$f repeat $rep (rc=$?):"; summ "$OUT/only_f${f}_r$rep.json"
    done
done
for f in 16 auto; do
    run $f full_f$f
    echo "full bench.py SVSB_FILTER=$f (rc=$?):"; summ "$OUT/full_f$f.json"
done
for f in 0 auto; do
    rm -rf "$OUT/dump_f$f"
    run $f dump_run_f$f --dump-outputs "$OUT/dump_f$f"
done
echo "dump-outputs, SVSB_FILTER=0 against automatic:"
for p in "$OUT"/dump_f0/*; do
    b=$(basename "$p")
    if cmp -s "$p" "$OUT/dump_fauto/$b"; then echo "  $b identical"; else echo "  $b DIFFERS"; fi
done
python scripts/filter_roofline.py --c4
