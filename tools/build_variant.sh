#!/bin/bash
# developer tool: build libaai_b200 variants with extra -D flags into csrc/gpurun_variants/<name>.so
# usage: tools/build_variant.sh <name> [-DAAI_TILE_W=16 -DAAI_TILE_H=8 ...]
# Sources and nvcc flags are the ones __graft_entry__.build() uses (build_library), plus the given flags.
set -e
name=$1; shift
root=$(cd "$(dirname "$0")/.." && pwd)
csrc=$root/area_average_interpolation_b200/csrc
out=$csrc/gpurun_variants; tmp=$out/obj_$name; mkdir -p $tmp
python3 -c 'import sys; sys.path.insert(0, sys.argv[1]); import __graft_entry__ as g; g.build_library(sys.argv[2], sys.argv[3], sys.argv[4:])' \
    "$root" "$out/$name.so" "$tmp" "$@"
rm -rf $tmp
echo built $out/$name.so
