#!/bin/bash
# tools/build_variant.sh NAME "-DWIN_TH=384 ..." : a tuning build of the library under variants/ (git-ignored;
# it travels to the GPU box).  Use with DBAT_LIB=variants/libdbatgpu_NAME.so.
set -e
cd "$(dirname "$0")/.."
name=$1; shift
mkdir -p variants/obj_$name
objs=""
for f in eval schur schur_win chol tilechol tilesym plan general_io covstats api startval order; do
  o=dbat_b200/csrc/$f.o
  if grep -q "$VARIANT_FILES_PLACEHOLDER" /dev/null 2>/dev/null; then :; fi
  case " $VARIANT_FILES " in
    *" $f "*) o=variants/obj_$name/$f.o
       nvcc $@ -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC -c dbat_b200/csrc/$f.cu -o $o ;;
  esac
  objs="$objs $o"
done
nvcc -shared -o variants/libdbatgpu_$name.so $objs -ldl
echo variants/libdbatgpu_$name.so
