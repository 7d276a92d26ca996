# usage: bash tools/ab_run.sh [--cats "cat1 cat2 ..."] name1 name2 ...   (libhitsir_<name>.so built by tools/ab_build.py)
# prints step time + the named breakdown categories (default: the six largest)
mkdir -p gpurun_out
PKG=single-image-super-resolution-application_b200
CATS=""
if [ "$1" = "--cats" ]; then CATS="$2"; shift 2; fi
for rep in 1 2; do
for n in "$@"; do
  HITSIR_B200_LIB=$PWD/$PKG/libhitsir_$n.so timeout 90 python bench.py --steps 6 --warmup 3 --no-extras --no-cpu-baseline > gpurun_out/ab_$n.log 2> gpurun_out/ab_$n.err || { echo "$n FAILED"; tail -5 gpurun_out/ab_$n.err; continue; }
  python - "$n" "$CATS" <<'PY'
import json, sys
n, cats = sys.argv[1], sys.argv[2].split()
d = json.loads(open(f"gpurun_out/ab_{n}.log").read().strip().split("\n")[-1])
b = d["breakdown"]
top = ", ".join(f"{k} {b[k]['ms_per_step']:.3f}" for k in (cats or list(b)[:6]) if k in b)
print(f"{n:12s} {d['ms_per_step']:8.2f} ms/step {d['value']:7.1f} MP/s  clk {d['clocks']['sm_mhz']}  | {top}")
PY
done
done
