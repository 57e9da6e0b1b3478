#!/usr/bin/env bash
# Builds libbadba_b200.so of the current tree into tools/ab/<name>.so, so that an edited tree can be A/B-compared against it:
#   python -m badslam_b200.build && tools/ab_build.sh base        # before the edit
#   python -m badslam_b200.build && python tools/ab_fast.py tools/ab/base.so
# kernels.cu is compiled afresh (with any extra nvcc flags given after the name); the other units are linked from badslam_b200/_obj.
set -euo pipefail
cd "$(dirname "${BASH_SOURCE[0]}")/.."
name="$1"; shift
mkdir -p tools/ab
C=badslam_b200/csrc
nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -Xcompiler -fPIC --expt-relaxed-constexpr -use_fast_math "$@" \
     -c $C/kernels.cu -o tools/ab/$name.kernels.o
nvcc -gencode arch=compute_100a,code=sm_100a -shared -o tools/ab/$name.so tools/ab/$name.kernels.o \
     badslam_b200/_obj/intrinsics.cu.o badslam_b200/_obj/pcg.cu.o badslam_b200/_obj/lifecycle.cu.o badslam_b200/_obj/preprocess.cu.o badslam_b200/_obj/odometry.cu.o badslam_b200/_obj/pose_solve.cu.o badslam_b200/_obj/badba.cu.o -cudart static
echo tools/ab/$name.so
