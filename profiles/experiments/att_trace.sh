#!/bin/bash
# Debug build of the library with per-phase clock stamps in the tcgen05 attention kernel (-DPNP_ATT_TRACE), written next to the
# shipped one as gpurun_libtrace.so; profiles/experiments/att_trace.py loads it and prints the stamps of one CTA.
set -e
cd "$(dirname "$0")/../../pnp_ovss_b200/csrc"
mkdir -p build_trace
for f in lib tf32x3 attention xattn gradcam upsample_blur lattice crf confusion; do
  /usr/local/cuda/bin/nvcc -O3 -std=c++17 -lineinfo -gencode arch=compute_100a,code=sm_100a -Xcompiler -fPIC --fmad=true -DPNP_ATT_TRACE -c $f.cu -o build_trace/$f.o &
done
wait
/usr/local/cuda/bin/nvcc -gencode arch=compute_100a,code=sm_100a -shared -cudart static -o ../../gpurun_libtrace.so build_trace/*.o
