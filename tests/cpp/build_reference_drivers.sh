#!/bin/bash
# Builds the reference's own hot-path programs, UNCHANGED, against the seal/seal.h shim and
# libckks_b200.so.  The reference's sources are not part of this repository: pass a checkout of them
# as $1 or in CKKS_REFERENCE_DIR.  The binaries land in tests/cpp/_build/ (git-ignored), where the GPU
# tests run them.
set -e
ROOT="$(cd "$(dirname "$0")/../.." && pwd)"
PKG="$ROOT/seal-fyp-logistic-regression_b200"
REF="${1:-$CKKS_REFERENCE_DIR}"
[ -d "$REF" ] || { echo "usage: $0 REFERENCE_DIR (or set CKKS_REFERENCE_DIR)" >&2; exit 2; }
OUT="$ROOT/tests/cpp/_build"
mkdir -p "$OUT"
for f in 4_ckks matrix_mult_benchmark matrix_multiplication linear_transformation2 linear_transformation polynomial matrix_transpose benchmark logistic_regression_ckks; do
  g++ -std=c++17 -O2 -w -I "$ROOT/include" -I "$PKG/include" -I "$REF" "$REF/$f.cpp" -o "$OUT/$f" \
      "$PKG/libckks_b200.so" -Wl,-rpath,"$PKG" -Wl,-rpath,'$ORIGIN/../../../seal-fyp-logistic-regression_b200'
  echo "built $f"
done
# the reference's helper.h functions vs the batched b200:: drop-ins (bit-identity driver)
g++ -std=c++17 -O2 -w -I "$ROOT/include" -I "$PKG/include" -I "$REF" "$ROOT/tests/cpp/helper_driver.cpp" -o "$OUT/helper_driver" \
    "$PKG/libckks_b200.so" -Wl,-rpath,"$PKG" -Wl,-rpath,'$ORIGIN/../../../seal-fyp-logistic-regression_b200'
echo "built helper_driver"
g++ -std=c++17 -O2 -w -I "$ROOT/include" -I "$PKG/include" -I "$REF" "$ROOT/tests/cpp/matmul_driver.cpp" -o "$OUT/matmul_driver" \
    "$PKG/libckks_b200.so" -Wl,-rpath,"$PKG" -Wl,-rpath,'$ORIGIN/../../../seal-fyp-logistic-regression_b200'
echo "built matmul_driver"
g++ -std=c++17 -O2 -Wall -I "$ROOT/include" -I "$PKG/include" "$ROOT/tests/cpp/lr_driver.cpp" -o "$OUT/lr_driver" \
    "$PKG/libckks_b200.so" -Wl,-rpath,"$PKG" -Wl,-rpath,'$ORIGIN/../../../seal-fyp-logistic-regression_b200'
echo "built lr_driver"
g++ -std=c++17 -O2 -Wall -I "$ROOT/include" -I "$PKG/include" "$ROOT/tests/cpp/epoch_driver.cpp" -o "$OUT/epoch_driver" \
    "$PKG/libckks_b200.so" -Wl,-rpath,"$PKG" -Wl,-rpath,'$ORIGIN/../../../seal-fyp-logistic-regression_b200'
echo "built epoch_driver"
