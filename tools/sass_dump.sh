#!/usr/bin/env bash
# SASS evidence for profiles/sass/ (CPU only: cuobjdump on the built library).  One compact summary per hot kernel: the
# instruction-class histogram and the lines that prove what the kernel is built from (128-bit stores/loads, LDGSTS, UBLKCP,
# packed FP32, MUFU.EX2, RED).  Full listings are large (0.3-1 MB each); they are regenerated on demand with
#   cuobjdump -sass -fun <mangled name> rag_b200/librag_b200.so
set -euo pipefail
cd "$(dirname "$0")/.."
LIB=rag_b200/librag_b200.so
OUT=profiles/sass
mkdir -p $OUT
names=$(cuobjdump -sass $LIB | grep -oE "Function : \S+" | awk '{print $3}')
summ() {  # $1 = regex on the mangled name, $2 = output stem
  for f in $(echo "$names" | grep -E "$1" | head -${3:-1}); do
    dem=$(echo $f | c++filt | cut -c1-160)
    lst=$(cuobjdump -sass -fun "$f" $LIB | grep -E "^\s+/\*[0-9a-f]{4}\*/" | sed 's#/\*[0-9a-f]*\*/##g' | awk '{$1=$1};1')
    {
      echo "# $dem"
      echo "# $(echo "$lst" | wc -l) SASS instructions; opcode histogram (static):"
      echo "$lst" | awk '{op=$1; if (op ~ /^@/) op=$2; sub(/;$/,"",op); print op}' | sort | uniq -c | sort -rn | head -24
      echo "# evidence lines:"
      echo "$lst" | grep -E "STG\.E\.(EF\.)?128|LDG\.E\.(EF\.|CONSTANT\.)?128|LDGSTS|UBLKCP|FFMA2|FMUL2|MUFU\.EX2|RED\.|ATOMG|LDS\.128|STS\.128|BAR\.SYNC" | sort | uniq -c | sort -rn | head -16
      echo
    } >> $OUT/$2.txt
  done
}
rm -f $OUT/r2_*.txt
summ "cv_fwd_lean_kernelILi256ELi2ELb1ELi0" r2_cv_fwd_lean
summ "cv_fwd_tma_kernel" r2_cv_fwd_tma
summ "cv_bwd_v4_kernel" r2_cv_bwd_v4
summ "cv_bwd_v4_persistent" r2_cv_bwd_v4
summ "head_fwd_x3r_kernelILi4ELi4ELi16ELi2ELi2ELb0" r2_head_fwd_x3r
summ "head_bwd_x3w_kernelILb1ELb1" r2_head_bwd_x3w
summ "stem_bwd_maps_kernelILi8" r2_stem_train
summ "stem_bwd_inputs_kernel" r2_stem_train
summ "stem_bwd_weight_kernel" r2_stem_train
summ "bn3d_bwd_rows_kernel" r2_stem_train
summ "conv3d_c1_bwd_data" r2_tail
summ "conv3d_c1_bwd_weight_kernel" r2_tail
summ "trilinear_fwd_kernelILb1" r2_tail
summ "trilinear_bwd_kernelILb1" r2_tail
ls -la $OUT | tail -8
