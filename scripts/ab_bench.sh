#!/bin/bash
# A/B of builds of libogs_b200 on one GPU, in one call so that both see the same card and the same neighbours:
#   ab_bench.sh <out_dir> <rounds> <name>=<lib.so>[,VAR=value...] ...
# Each round runs `bench.py $BENCH_ARGS` (default `--no-kmeans --no-configs --no-cpu-baseline`; without `--no-kmeans`
# the bench also times the k-means and Stage-1 step legs) once per build, in the order given (the builds alternate),
# selecting the library with OGS_LIB_PATH and setting the listed environment variables.  Before the rounds every
# build writes `--dump-outputs` from a short headline-only run into a temporary directory; the first build's outputs are
# compared with the others'.  The card's name, power limit and SM clocks are recorded in <out_dir>/gpu.txt.  Bench lines
# go to <out_dir>/<name>.jsonl, one per round; medians, ranges and the output comparison to <out_dir>/summary.txt.
set -e
out=$1; rounds=$2; shift 2
ROOT=$(cd "$(dirname "$0")/.." && pwd)
cd "$ROOT"
mkdir -p "$out"
dumps=$(mktemp -d)
trap 'rm -rf "$dumps"' EXIT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm --format=csv > "$out/gpu.txt"
cat "$out/gpu.txt"

run() {   # run <spec> <extra bench args...>
    local spec=$1; shift
    local name=${spec%%=*} rest=${spec#*=}
    local lib=${rest%%,*} envs=()
    [ "$rest" != "$lib" ] && IFS=, read -ra envs <<< "${rest#*,}"
    env OGS_LIB_PATH="$(realpath "$lib")" "${envs[@]}" python bench.py ${BENCH_ARGS:---no-kmeans --no-configs --no-cpu-baseline} "$@"
}

for spec in "$@"; do
    name=${spec%%=*}
    BENCH_ARGS="--no-kmeans --no-configs --no-cpu-baseline" run "$spec" --steps 4 --warmup 2 --repeats 1 \
        --dump-outputs "$dumps/$name" > /dev/null
done
for r in $(seq "$rounds"); do
    for spec in "$@"; do
        name=${spec%%=*}
        run "$spec" | grep '^{' | tail -1 | tee -a "$out/$name.jsonl" | cut -c1-160
    done
done

python - "$out" "$dumps" "$@" <<'EOF'
import glob, json, os, statistics, sys
import numpy as np
out, dumps, specs = sys.argv[1], sys.argv[2], sys.argv[3:]
names = [s.split("=", 1)[0] for s in specs]
lines = []
for n in names:
    rs = [json.loads(l) for l in open(os.path.join(out, n + ".jsonl"))]
    v = [r["value"] for r in rs]
    bd = {k: statistics.median(r["breakdown"][k]["ms_per_launch"] for r in rs) for k in rs[0].get("breakdown", {})}
    lo, hi = min(r["repeat"]["value_min"] for r in rs), max(r["repeat"]["value_max"] for r in rs)
    lines.append(f"{n}: value median {statistics.median(v):.1f} over {len(v)} runs {[round(x, 1) for x in v]}, "
                 f"value_min..value_max over all runs {lo:.1f}..{hi:.1f}, "
                 f"ms_per_launch medians {json.dumps({k: round(x, 4) for k, x in bd.items()})}")
    st = {k: round(statistics.median(r[k]["ms_per_step"] for r in rs), 4) for k in rs[0] if k.startswith("stage1_step")}
    if st:
        lines.append(f"{n}: Stage-1 ms_per_step medians {json.dumps(st)}")
ref = os.path.join(dumps, names[0])
for n in names[1:]:
    worst = {}
    for f in sorted(glob.glob(os.path.join(ref, "*.npy"))):
        a, b = np.load(f), np.load(os.path.join(dumps, n, os.path.basename(f)))
        d = np.abs(a.astype(np.float64) - b)
        worst[os.path.basename(f)[:-4]] = "equal" if np.array_equal(a, b) else \
            f"max abs {d.max():.3g} (rel to max |ref| {d.max() / max(np.abs(a).max(), 1e-30):.3g})"
    lines.append(f"outputs {names[0]} vs {n}: " + json.dumps(worst))
open(os.path.join(out, "summary.txt"), "w").write("\n".join(lines) + "\n")
print("\n".join(lines))
EOF
