# Build an A/B variant of the library: benchmarks/bin/libssp_NAME.so from the sources of the tree this script is in (further
# arguments are passed to every nvcc call).  Edit a constant in a copy of the tree, build it there and point SSP_B200_LIB at it:
#   bash COPY/benchmarks/build_variant.sh NAME && SSP_B200_LIB=COPY/benchmarks/bin/libssp_NAME.so python bench.py ...
set -e
cd "$(dirname "$0")/.."
name=$1; shift
out=benchmarks/bin/libssp_$name.so
tmp=$(mktemp -d)
for f in speech_signal_processing_b200/csrc/*.cu; do
  nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo -Xcompiler -fPIC -DSSP_BUILD "$@" -c $f -o $tmp/$(basename $f .cu).o &
done
wait
nvcc -shared -o $out $tmp/*.o -gencode arch=compute_100a,code=sm_100a
rm -rf $tmp
echo $out
