#!/bin/sh
# Parity guard: NVVM turns `x / constant` into a multiplication by the reciprocal when -ftz=true is given, which
# is 1 ulp off the IEEE quotient the reference computes.  Compile the device code with -ftz=false (where the
# rewrite does not happen) and with the product flags, and require the same number of IEEE divisions in both.
set -e
cd "$(dirname "$0")/../pearray_b200"
T=$(mktemp -d)
trap 'rm -rf "$T"' EXIT
F="-std=c++17 -O3 -gencode arch=compute_100a,code=sm_100a -fmad=false -prec-div=true -prec-sqrt=true --expt-relaxed-constexpr -w"
nvcc $F -ftz=false -ptx csrc/prb_api.cu -o "$T/prb_ftz0.ptx" &
nvcc $F -ftz=true -ptx csrc/prb_api.cu -o "$T/prb_ftz1.ptx"
wait
# (divPositive writes its division as inline PTX, `div.rn.ftz.f32` in both builds: count both spellings in both files)
A=$(grep -c "div\.rn\(\.ftz\)\?\.f32" "$T/prb_ftz0.ptx")
B=$(grep -c "div\.rn\(\.ftz\)\?\.f32" "$T/prb_ftz1.ptx")
echo "IEEE divisions: -ftz=false $A, -ftz=true $B"
test "$A" = "$B"
