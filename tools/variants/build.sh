#!/bin/bash
# DEV ONLY: builds the candidate shells (libvariants.so) and the timeline-probe build of the shipped shell (libtrace.so).
# CSRC=<dir> builds libtrace.so against another copy of the sources (e.g. a parent commit with the probe hooks added).
cd "$(dirname "$0")"
CSRC=${CSRC:-../../pypose_b200/csrc}
FLAGS="-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 --expt-relaxed-constexpr -Xcompiler -fPIC -shared -I ../../include"
nvcc $FLAGS -I ../../pypose_b200/csrc variants.cu -o libvariants.so & a=$!
nvcc $FLAGS -I "$CSRC" trace.cu -o "${TRACE_OUT:-libtrace.so}" & b=$!
wait $a && wait $b
