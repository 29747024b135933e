#!/bin/bash
# build a tuning variant of the scan solver: tools/build_scan_variant.sh NAME "-DIBS_SCAN_BLK=2 ..."  -> lib/variants/libibs_NAME.so
# (select it at run time with IBS_LIB=.../lib/variants/libibs_NAME.so)
set -e
cd "$(dirname "$0")/../ideal-ballooning-solver_b200"
mkdir -p lib/variants
F="-O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo -Xcompiler -fPIC -DIBS_BUILD -fmad=true"
nvcc $F $2 -Xptxas=-v -c csrc/ibs_scan_solver.cu -o lib/variants/scan_$1.o 2> lib/variants/ptxas_scan_$1.log
nvcc -shared -o lib/variants/libibs_$1.so lib/ibs_api.o lib/ibs_solver.o lib/variants/scan_$1.o lib/ibs_geometry.o lib/ibs_geometry_full.o lib/ibs_geometry_adjoint.o lib/ibs_adjoint.o -gencode arch=compute_100a,code=sm_100a -cudart static
grep -A2 -E "scan2?_solve_kernelENS" lib/variants/ptxas_scan_$1.log | grep -v "^--"
