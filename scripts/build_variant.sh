#!/bin/bash
# usage: scripts/build_variant.sh <tag> [-DFLAG=..]...   -> build_dbg/libpda_<tag>.so (A/B builds for scripts/fast_path_probe.py)
set -e
ROOT=$(cd "$(dirname "$0")/.." && pwd)
TAG=$1; shift
OBJ=/tmp/variant_$TAG; mkdir -p $OBJ $ROOT/build_dbg
cd $ROOT/probabilisticsemslam_b200/csrc
for f in pda_capi murty_kernel murty_cta_kernel murty_ladder_kernel weights_kernel permanent_kernel permanent_approx_kernel permprob_device_kernel association_kernel association_perm_kernel bbox_kernel quadric_kernel; do
  if [ $f = murty_kernel ] || [ $f = murty_ladder_kernel ] || [ ! -f $OBJ/$f.o ]; then
    nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -fmad=false -Xcompiler -fPIC -I$ROOT/include -I. "$@" -c $f.cu -o $OBJ/$f.o 2>/dev/null &
  fi
done
wait
nvcc -shared -cudart static -o $ROOT/build_dbg/libpda_$TAG.so $OBJ/*.o 2>/dev/null
ls -la $ROOT/build_dbg/libpda_$TAG.so
