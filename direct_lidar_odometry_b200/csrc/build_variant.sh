#!/bin/sh
# A/B builds of the kNN/covariance translation unit: ./build_variant.sh <name> "<-D flags>" -> variants/libnanogicp_<name>.so
# (all other objects are the regular ones; pick a variant at run time with NGICP_LIB_PATH=<path>)
set -e
cd "$(dirname "$0")"
mkdir -p variants
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
ARCH="-gencode arch=compute_100a,code=sm_100a"
$NVCC -O3 -std=c++17 $ARCH -lineinfo -Xcompiler -fPIC --expt-relaxed-constexpr -ccbin /usr/bin/g++ -fmad=false $2 -c knn_cov.cu -o variants/knn_cov_$1.o
$NVCC $ARCH -shared -cudart static -o variants/libnanogicp_$1.so sort_scan.o cloud_index.o variants/knn_cov_$1.o align.o voxel.o fitness.o api.o submap_select.o
rm -f variants/knn_cov_$1.o
echo built variants/libnanogicp_$1.so
