#!/usr/bin/env bash
# r07: the class-token tail against the build before it (profiles/r07_cls_tail.md).
#
#   git archive <parent> | tar -x -C _parent      # the build to compare against, untracked, next to this tree
#   bash profiles/r07_cls_tail.sh _parent OUT      # run from the repository root on a B200
#
# Builds both trees, dumps the logits of both at ViT-B/16 (both 16-bit formats) and ViT-H/14 (batch 64), then
# alternates quick c2 runs of the two builds ROUNDS times, one quick c5 pair and one full c2 run per build (kernels_ms).
# Every bench.py JSON line lands in OUT/runs.jsonl, tagged with the build and the round.
set -euo pipefail
PARENT=${1:?parent tree}
OUT=${2:?output directory}
ROUNDS=${ROUNDS:-3}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT/gpu.csv"
python -c "import __graft_entry__ as g; g.build()"
(cd "$PARENT" && python -c "import __graft_entry__ as g; g.build()")

run() {   # run TAG ROUND bench-args...: one bench.py of build TAG (new | parent), its JSON line tagged
  local tag=$1 round=$2; shift 2
  local dir=.
  [ "$tag" = parent ] && dir=$PARENT
  python "$dir/bench.py" "$@" > "$OUT/last.txt" 2> "$OUT/last.err" || { cat "$OUT/last.err"; return 1; }
  python - "$OUT/last.txt" "$tag" "$round" "$*" >> "$OUT/runs.jsonl" <<'EOF'
import json, sys
line = [l for l in open(sys.argv[1]) if l.startswith("{")][-1]
d = json.loads(line)
d.update(build=sys.argv[2], round=sys.argv[3], args=sys.argv[4])
print(json.dumps(d))
EOF
  tail -c 400 "$OUT/last.txt"; echo
}

# same results: the logits of both builds on the same seeded weights and images
for tag in parent new; do
  run "$tag" full --gpus 1 --no-cpu-baseline --no-train --dump-outputs "$OUT/dump_c2_$tag"
  run "$tag" dump --config c4 --quick --batch 64 --dump-outputs "$OUT/dump_c4_$tag"
done
python - "$OUT" <<'EOF'
import sys
from pathlib import Path
import numpy as np
out = Path(sys.argv[1])
for cfg, names in (("c2", ("logits_bf16.npy", "logits_fp16.npy")), ("c4", None)):
    a_dir, b_dir = out / f"dump_{cfg}_parent", out / f"dump_{cfg}_new"
    for name in names or sorted(p.name for p in a_dir.glob("*.npy")):
        a, b = np.load(a_dir / name), np.load(b_dir / name)
        print(f"{cfg} {name}: shape {a.shape}, array_equal {np.array_equal(a, b)}, max |diff| {float(np.abs(a - b).max()):.3e}")
EOF

# faster: alternated quick runs
for r in $(seq 1 "$ROUNDS"); do
  run parent "$r" --quick --steps 40
  run new "$r" --quick --steps 40
done
run parent c5 --config c5 --quick
run new c5 --config c5 --quick
