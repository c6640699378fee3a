#!/bin/bash
# Round 6, all-frozen 8-leaf halves of SUB16 (profiles/r6/README.md), on ONE box in one call:
#   r3   = gpu_variants/libpolar_b200_r3.so, the library of round 3 (489bc16, the parent of round 4)
#   base = gpu_variants/libpolar_b200_base.so, the library of the parent of this round (rounds 4 and 5 in); `base2` is
#          the same library run with POLAR_B200_KDEBUG=2 (identity exit of the fork off, i.e. round 4 alone)
#   new  = the library build() made from this tree
# r3 and base are built beforehand (build() in a checkout of each commit) and swapped into place in turn.
# Usage: tools/gpu_jobs/r6.sh [OUTDIR] from the repository root; the bench JSON lines go to OUTDIR (default: a fresh
# temporary directory).
set -x
O=${1:-$(mktemp -d)}
mkdir -p "$O"
LIB=quantized_decoder_polar_codes_b200/libpolar_b200.so
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm --format=csv
cp $LIB /tmp/lib_new.so
cp gpu_variants/libpolar_b200_base.so /tmp/lib_base.so
cp gpu_variants/libpolar_b200_r3.so /tmp/lib_r3.so
P='import sys,json; d=json.loads(sys.stdin.read()); print(sys.argv[1], "value=%.5g e2e=%.4g kernel_ms=%.3f F=%d wave=%d clocks=%s" % (d["value"], d["e2e"]["value"], d["roofline"]["kernel_ms"], d["run"]["frames_per_step_per_gpu"], d["run"]["wave_frames"], json.dumps(d.get("clocks"))))'
use() { cp /tmp/lib_${1%2}.so $LIB; }
dbg() { [ "$1" = base2 ] && echo 2 || echo 0; }
for r in 1 2 3; do
  for v in r3 base new; do
    use $v
    timeout 300 python bench.py --steps 20 --warmup 3 --no-cpu-baseline 2>/dev/null | tee $O/ns_${v}_$r.json | python -c "$P" "NS $v $r"
  done
done
use base
POLAR_B200_KDEBUG=2 timeout 300 python bench.py --steps 20 --warmup 3 --no-cpu-baseline 2>/dev/null | tee $O/ns_base2.json | python -c "$P" "NS base2 1"
for c in C2 C3 C4; do
  for v in base new; do
    use $v
    timeout 300 python bench.py --config $c --steps 20 --warmup 3 --no-cpu-baseline 2>/dev/null | tee $O/${c}_${v}.json | python -c "$P" "$c $v"
  done
done
for c in NS C2 C3 C4; do
  for v in base new; do
    use $v
    timeout 300 python bench.py --config $c --steps 2 --warmup 1 --no-cpu-baseline --dump-outputs $O/dump_${c}_$v > /dev/null 2>&1
  done
  for f in $O/dump_${c}_base/*.npy; do cmp "$f" "$O/dump_${c}_new/$(basename $f)" && echo "$c $(basename $f) equal"; done
  rm -rf $O/dump_${c}_base $O/dump_${c}_new   # (too large to keep: the comparison is the result)
done
use new
timeout 1800 python -m pytest -m gpu -q -x tests 2>&1 | tail -n 15
timeout 600 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -n 8
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm --format=csv
