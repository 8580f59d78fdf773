#!/bin/bash
# A/B of the single-query filter against K1 in one run (profiles/r05_filter_ab.txt): the card, bench.py --only
# alternating SVSB_FILTER=0 / 1 three times each, one full bench.py line of each, --dump-outputs of both compared file
# by file, and scripts/filter_roofline.py (real bytes, candidates, size cut-off).
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
if "incremental_update" in j:
    print("  incremental_update:", json.dumps(j["incremental_update"])[:200])
for name, x in sorted(j.get("configs", {}).items()):
    print(f"  {name}:", leg(x))
EOF
}
for rep in 1 2 3; do
    for f in 0 1; do
        SVSB_FILTER=$f python bench.py --gpus 1 --steps 20 --warmup 3 --only > "$OUT/only_f${f}_r$rep.json" 2> "$OUT/only_f${f}_r$rep.err"
        echo "--only SVSB_FILTER=$f repeat $rep (rc=$?):"; summ "$OUT/only_f${f}_r$rep.json"
    done
done
for f in 0 1; do
    rm -rf "$OUT/dump_f$f"
    SVSB_FILTER=$f python bench.py --gpus 1 --steps 20 --warmup 3 --dump-outputs "$OUT/dump_f$f" > "$OUT/full_f$f.json" 2> "$OUT/full_f$f.err"
    echo "full bench.py SVSB_FILTER=$f (rc=$?):"; summ "$OUT/full_f$f.json"
done
echo "dump-outputs, SVSB_FILTER=0 against =1:"
for p in "$OUT"/dump_f0/*; do
    b=$(basename "$p")
    if cmp -s "$p" "$OUT/dump_f1/$b"; then echo "  $b identical"; else echo "  $b DIFFERS"; fi
done
python scripts/filter_roofline.py
python scripts/filter_roofline.py --sweep
