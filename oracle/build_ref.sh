#!/usr/bin/env bash
# TEST INFRASTRUCTURE -- builds oracle/_ref/ (git-ignored, NOT gpurun-ignored).
#
# Compiles the UNMODIFIED reference library sources where they lie under /root/reference
# (the list in the reference's CMakeLists.txt:149-164) with g++ directly -- the reference's own
# CMake build is not run (it needs find_package(BLAS) and cannot see the wheel-bundled OpenBLAS).
# BLAS/LAPACK = OpenBLAS inside the scipy wheel (symbols prefixed scipy_), reached through
# oracle/ref_shim/cblas.h.  -ffast-math (reference Release flag, CMakeLists.txt:211) is NOT used:
# the oracle should be the cleanest IEEE evaluation of the reference algorithm.
#
# Outputs:  oracle/_ref/libcals_ref.so   the reference library
#           oracle/_ref/cals_ref         oracle/ref_tool.cpp linked against it
#           oracle/_ref/libcals_ref_rel{3,4}.so + cals_ref_rel{3,4}
#                                        the same sources with the reference's RELEASE flags (CMake Release adds
#                                        -O3 -DNDEBUG; CMakeLists.txt:210-211 adds -ffast-math -march=native) for the
#                                        timed CPU arm of bench.py only.  -march=native cannot travel (this container
#                                        builds, another host of the pool runs), so two portable levels are built and
#                                        caseio.ref_binary(release=True) picks x86-64-v4 when the running CPU has
#                                        AVX-512, x86-64-v3 otherwise.  Golden vectors and parity tests keep the
#                                        no-fast-math build above.
# No reference source is copied into the repo.
set -euo pipefail
HERE="$(cd "$(dirname "${BASH_SOURCE[0]}")" && pwd)"
REF="${CALS_REFERENCE_DIR:-/root/reference}"
OUT="$HERE/_ref"
if [ ! -d "$REF/src" ]; then
  echo "build_ref: no reference sources in $REF (set CALS_REFERENCE_DIR) -- keeping whatever $OUT holds" >&2
  exit 0
fi
SP="$(python -c 'import scipy, os; print(os.path.join(os.path.dirname(os.path.dirname(scipy.__file__)), "scipy.libs"))')"
BLAS="$(ls "$SP"/libscipy_openblas-*.so | head -1)"
mkdir -p "$OUT"
SRCS=(src/als.cpp src/cals.cpp src/tensor.cpp src/matrix.cpp src/ktensor.cpp src/cals_blas.cpp src/cuda_utils.cpp
      src/utils/utils.cpp src/utils/error.cpp src/utils/mttkrp.cpp src/utils/update.cpp src/multi_ktensor.cpp
      src/utils/line_search.cpp extern/rectangular_lsap/rectangular_lsap.cpp)
CXXFLAGS=(-std=c++17 -O2 -march=x86-64-v3 -fopenmp -fPIC -w -DCALS_OPENBLAS=1 -DWITH_TIME=1 -DNDEBUG
          "-DSOURCE_DIR=\"$REF\"" -I"$HERE/ref_shim" -I"$REF/include" -I"$REF/include/utils" -I"$REF/extern")
OBJS=()
for s in "${SRCS[@]}"; do
  o="$OUT/$(echo "$s" | tr '/' '_').o"
  g++ "${CXXFLAGS[@]}" -c "$REF/$s" -o "$o" &
  OBJS+=("$o")
done
wait
g++ -shared -fopenmp -o "$OUT/libcals_ref.so" "${OBJS[@]}" "$BLAS" -Wl,-rpath,"$SP"
g++ "${CXXFLAGS[@]}" "$HERE/ref_tool.cpp" -o "$OUT/cals_ref" -L"$OUT" -lcals_ref "$BLAS" \
    -Wl,-rpath,'$ORIGIN' -Wl,-rpath,"$SP"
rm -f "${OBJS[@]}"
for lvl in 3 4; do
  RFLAGS=(-std=c++17 -O3 -ffast-math -march=x86-64-v$lvl -fopenmp -fPIC -w -DCALS_OPENBLAS=1 -DWITH_TIME=1 -DNDEBUG
          "-DSOURCE_DIR=\"$REF\"" -I"$HERE/ref_shim" -I"$REF/include" -I"$REF/include/utils" -I"$REF/extern")
  OBJS=()
  for s in "${SRCS[@]}"; do
    o="$OUT/rel${lvl}_$(echo "$s" | tr '/' '_').o"
    g++ "${RFLAGS[@]}" -c "$REF/$s" -o "$o" &
    OBJS+=("$o")
  done
  wait
  g++ -shared -fopenmp -o "$OUT/libcals_ref_rel$lvl.so" "${OBJS[@]}" "$BLAS" -Wl,-rpath,"$SP"
  g++ "${RFLAGS[@]}" "$HERE/ref_tool.cpp" -o "$OUT/cals_ref_rel$lvl" -L"$OUT" -lcals_ref_rel$lvl "$BLAS" \
      -Wl,-rpath,'$ORIGIN' -Wl,-rpath,"$SP"
  rm -f "${OBJS[@]}"
done
echo "build_ref: built $OUT/cals_ref (+ cals_ref_rel3, cals_ref_rel4 with the reference's Release flags) against $BLAS"
