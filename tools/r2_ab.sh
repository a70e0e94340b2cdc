#!/bin/bash
# A/B of library BUILDS on ONE box (box-to-box spread is +-5 %, so only same-box comparisons count):
#   neural-photo-editor_b200/_variants/libian_b200_<tag>.so are earlier builds of the same sources (git-ignored, shipped by
#   gpurun), selected with IAN_B200_LIB; "new" is the in-tree build.  Usage: bash tools/r2_ab.sh "head st128 new" [rounds]
mkdir -p gpurun_out
V=$PWD/neural-photo-editor_b200/_variants
TAGS=${1:-"head new"}
# a tag is <build>[+opt...]: +nopdl runs that build with IAN_PDL=0 (plain launches)
setvar() {
  local b=${1%%+*}
  if [ "$b" = new ]; then unset IAN_B200_LIB; else export IAN_B200_LIB=$V/libian_b200_$b.so; fi
  unset IAN_PDL
  case "$1" in *+nopdl*) export IAN_PDL=0;; esac
}
ROUNDS=${2:-2}
for r in $(seq 1 $ROUNDS); do
  for t in $TAGS; do
    setvar $t
    python bench.py --steps 30 --warmup 5 --no-cpu-baseline --no-full --no-config5 $AB_BENCH_ARGS > gpurun_out/ab_${t}_$r.json 2> gpurun_out/ab_${t}_$r.err
    python tools/bench_brief.py ${t}_$r gpurun_out/ab_${t}_$r.json
  done
done
[ -n "$AB_NO_FULL" ] && TAGS=""
for t in $TAGS; do
  setvar $t
  python bench.py --steps 10 --warmup 3 --no-cpu-baseline --no-edit --no-config5 > gpurun_out/ab_full_${t}.json 2> gpurun_out/ab_full_${t}.err
  python tools/bench_brief.py full_${t} gpurun_out/ab_full_${t}.json
done
unset IAN_B200_LIB IAN_PDL
