#!/bin/bash
# Build libjt_vm.so for sm_100a (B200) in-tree: one object per .cu (compiled in parallel, rebuilt only when the
# source or a header is newer), then one link. Usage: build.sh [extra nvcc flags]   (extra flags force a rebuild)
set -e
cd "$(dirname "$0")"
mkdir -p _obj
FLAGS="-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC -Xptxas -v $*"
echo "$FLAGS" > _obj/.flags.new
if ! cmp -s _obj/.flags.new _obj/.flags 2>/dev/null; then rm -f _obj/*.o; mv _obj/.flags.new _obj/.flags; fi
NEWEST_HDR=$(ls -t *.cuh ../../include/jt_vm.h | head -1)
TODO=""
OBJS=""    # the objects of the current sources only: one left behind by a renamed or deleted .cu is not linked
for f in *.cu; do
  o=_obj/${f%.cu}.o
  OBJS="$OBJS $o"
  if [ ! -f "$o" ] || [ "$f" -nt "$o" ] || [ "$NEWEST_HDR" -nt "$o" ]; then TODO="$TODO $f"; fi
done
if [ -n "$TODO" ]; then
  printf '%s\n' $TODO | xargs -P "$(nproc)" -I{} sh -c "nvcc $FLAGS -c {} -o _obj/\$(basename {} .cu).o 2> _obj/\$(basename {} .cu).log || { cat _obj/\$(basename {} .cu).log >&2; exit 255; }"
fi
nvcc -gencode arch=compute_100a,code=sm_100a -shared -o libjt_vm.so $OBJS
