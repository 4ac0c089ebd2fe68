#!/bin/bash
# A/B of K1s's launch hand-over (two static first tiles per CTA, pre-wait prefetch of both): a build of the
# parent version against this tree, alternated in one session on one GPU.
#
#   bash tools/span_handover_ab.sh OLD_TREE [OUT_DIR]
#
# OLD_TREE: a checkout of the parent version built in place (python __graft_entry__.py).  Its timeline is taken only if
# it carries tools/span_timeline.py and the BSQ_SPAN_TRACE probe in bsq_span.cu (the probe compiles to nothing without
# the switch).  Writes OUT_DIR (default: a new temporary directory, printed first): bench JSON lines, both timelines.
set -u
OLD=$(cd "$1" && pwd)
NEW=$(pwd)
O=${2:-$(mktemp -d -t span_handover.XXXXXX)}
mkdir -p "$O"
echo "output: $O"
O=$(cd "$O" && pwd)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$O/gpu.txt"

ext() {
    python -c "
import sys, json
d = json.loads(sys.stdin.read().strip().splitlines()[-1])
r = d['roofline']
out = ['launch_us %.3f' % r['launch_us'], 'frac %.3f' % r['frac'], 'value %.1f' % d['value']]
x = d.get('extra', {})
for k in ('c1_dna_4096x1000_bf_u8_streamed', 'c1_dna_4096x1000_bf_u8_many_16_per_launch', 'c1x64_dna_262144x1000_bf_u8_one_launch',
          'c2x4_protein_bf_u8', 'c2x4_protein_bf_u8_padlen1026'):
    if k in x:
        out.append('%s %.2f' % (k, x[k]['us_per_call']))
print(' | '.join(out))"
}

run() {  # side, sections, steps
    local d=$OLD
    [ "$1" = new ] && d=$NEW
    (cd "$d" && timeout 600 python bench.py --sections "$2" --steps "$3" --warmup 20 2>>"$O/bench_$1.err") | tee -a "$O/bench_$1.jsonl" | ext
}

echo "== headline: value, 200 steps, A/B x 3"
for r in 1 2 3; do
    for side in old new; do echo -n "$side: "; run $side value 200; done
done
echo "== extra entries, A/B x 2"
for r in 1 2; do
    for side in old new; do echo -n "$side: "; run $side value,extra 200; done
done
echo "== C2, C2x4, P = 1026, P = 652 in one process per build (median of 5 windows), A/B x 2"
for r in 1 2; do
    for side in old new; do
        d=$OLD; [ $side = new ] && d=$NEW
        echo "$side:"; timeout 600 python "$NEW/tools/sweep_span_head.py" --root "$d" --rounds 5 2>&1 | tee -a "$O/sweep_$side.txt"
    done
done
echo "== outputs of the last timed step"
for side in old new; do
    d=$OLD; [ $side = new ] && d=$NEW
    (cd "$d" && timeout 600 python bench.py --sections value --steps 20 --warmup 2 --dump-outputs "$O/dump_$side" > "$O/dump_$side.json" 2>>"$O/bench_$side.err")
done
python - "$O" <<'EOF'
import json, os, sys
o = sys.argv[1]
for f in ("tokens.npy", "rows.npy"):
    a = open(os.path.join(o, "dump_old", f), "rb").read()
    b = open(os.path.join(o, "dump_new", f), "rb").read()
    print(f, "byte-identical" if a == b else "DIFFERENT", len(a), "bytes")
for side in ("old", "new"):
    d = json.loads(open(os.path.join(o, f"dump_{side}.json")).read().strip().splitlines()[-1])
    print(side, "parity_every_rank", d.get("parity_every_rank"))
EOF
rm -rf "$O/dump_old" "$O/dump_new"
echo "== timelines"
if [ -f "$OLD/tools/span_timeline.py" ]; then
    (cd "$OLD" && timeout 600 python tools/span_timeline.py --out "$O/timeline_old.txt" > /dev/null 2>"$O/timeline_old.err") && tail -1 "$O/timeline_old.txt"
fi
timeout 600 python tools/span_timeline.py --out "$O/timeline_new.txt" > /dev/null 2>"$O/timeline_new.err" && tail -1 "$O/timeline_new.txt"
