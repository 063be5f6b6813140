#!/bin/bash
# Development helper: build/variants/<name>.so for each "name=NVCC_FLAGS" argument (separate object dirs), e.g.
#   scripts/build_variants.sh base= trace=-DBALF_TC_TRACE
set -e
for spec in "$@"; do
  name=${spec%%=*}; flags=${spec#*=}
  ( BALF_OBJ_DIR=$PWD/build/obj_$name BALF_LIB_OUT=$PWD/build/variants/$name.so NVCC_FLAGS="$flags" python balf_b200/build.py > /dev/null && echo "built $name" ) &
done
wait
