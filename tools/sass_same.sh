#!/bin/bash
# Do two builds of the fused kernel's instantiations compile to the same code? For each key, compares the opcode
# sequence of k_fused_mfcc (cuobjdump -sass, addresses, encodings and operands stripped, so constant-bank offsets and
# register numbers do not count; a different register allocation still shows in the register / spill line) and the
# register / spill / shared-memory figures of ptxas -v. No GPU needed.
# Usage: tools/sass_same.sh <old package dir> <new package dir> [keys...]   (default keys 0..23)
# Each package dir is an asr-featext-opencl_b200 tree after `make` (build/afe_fused_inst_<key>.o).
set -u
old=$1; new=$2; shift 2
keys=${*:-$(seq 0 23)}
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
CUOBJDUMP=${CUOBJDUMP:-/usr/local/cuda/bin/cuobjdump}
ops() { "$CUOBJDUMP" -sass "$1" | sed -n 's@^ *\/\*[0-9a-f]\{4,\}\*\/ *\([A-Z][A-Z0-9._]*\).*@\1@p'; }
ptxas() {
  (cd "$1" && "$NVCC" -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo -Xcompiler -fPIC -I../include -Icsrc \
     -Xptxas -v -DAFE_INST_KEY="$2" -x cu -c -o /dev/null csrc/afe_fused_inst.cu 2>&1) |
    grep -A3 "Compiling entry.*k_fused" | grep -oE "[0-9]+ bytes (stack frame|spill stores|spill loads)|Used [0-9]+ registers" | tr '\n' ' '
}
fail=0
for k in $keys; do
  a=$(ops "$old/build/afe_fused_inst_$k.o" | md5sum | cut -c1-12); na=$(ops "$old/build/afe_fused_inst_$k.o" | wc -l)
  b=$(ops "$new/build/afe_fused_inst_$k.o" | md5sum | cut -c1-12); nb=$(ops "$new/build/afe_fused_inst_$k.o" | wc -l)
  pa=$(ptxas "$old" "$k"); pb=$(ptxas "$new" "$k")
  same=same; [ "$a" = "$b" ] && [ "$pa" = "$pb" ] || { same=DIFFERENT; fail=1; }
  printf "key %2s  %-9s  opcodes %s (%s) / %s (%s)  ptxas: %s| %s\n" "$k" "$same" "$a" "$na" "$b" "$nb" "$pa" "$pb"
done
exit $fail
