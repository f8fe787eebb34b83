#!/bin/bash
# usage: oracle/install_ref.sh <reference checkout>
# Build from the UNMODIFIED reference (intel/MLSL; its checkout may be read-only) into oracle/_ref (git-ignored):
#   1. _ref/tests/{mlsl_test,cmlsl_test,mlsl_sample,mlsl_example}, _ref/tests/python/   tests/test_reference_sources_cpu.py
#      (the reference's own test programs, compiled against THIS repository's headers and linked to its library, which
#      must be built first)
#   2. _ref/intel64/{lib/libmlsl.so*,bin/ep_server}  _ref/include/  _ref/mpirt/  _ref/bin/ref_*   bench.py --impl reference
#      (the reference library itself; the pip route does not apply: the reference ships no setup.py/pyproject.toml, it
#      is a Makefile project, SURVEY 6.2)
set -e
HERE="$(cd "$(dirname "$0")" && pwd)"
ROOT="$(dirname "$HERE")"
SRC="$(cd "${1:?usage: $0 <reference checkout>}" && pwd)"
DST="$HERE/_ref"
TMP="$(mktemp -d)"
trap 'rm -rf "$TMP"' EXIT
rm -rf "$DST"
mkdir -p "$DST/tests/python"
# 1. the rpath is relative so that the tree can move
ours=(-I"$ROOT/include" -L"$ROOT/mlsl_b200/lib" -lmlsl_b200 -Wl,-rpath,'$ORIGIN/../../../mlsl_b200/lib')
g++ -std=c++11 -O1 -w "$SRC/tests/examples/mlsl_test/mlsl_test.cpp" -o "$DST/tests/mlsl_test" "${ours[@]}"
g++ -std=c++11 -O1 -w "$SRC/mlsl_to_oneccl/mlsl_sample.cpp" -o "$DST/tests/mlsl_sample" "${ours[@]}"
g++ -std=c++11 -O1 -w "$SRC/tests/examples/mlsl_example/mlsl_example.cpp" -o "$DST/tests/mlsl_example" "${ours[@]}"
gcc -std=gnu99 -O1 -w "$SRC/tests/examples/mlsl_test/cmlsl_test.c" -o "$DST/tests/cmlsl_test" "${ours[@]}" -lm
# its Python binding and the Python test that drives it
cp -r "$SRC/include/mlsl" "$DST/tests/python/mlsl"
cp "$SRC/tests/examples/mlsl_test/mlsl_test.py" "$DST/tests/python/"
# 2.
cp -r "$SRC"/. "$TMP"/
chmod -R u+w "$TMP"
cd "$TMP"
make libep MLSL_MODE=process EXTRA_CFLAGS=-w > build_ep.log 2>&1
make libmlsl MLSL_MODE=process EXTRA_CFLAGS=-w > build_mlsl.log 2>&1
mkdir -p "$DST/intel64/lib" "$DST/intel64/bin" "$DST/include" "$DST/bin"
cp src/process/libmlsl.so.1.0 "$DST/intel64/lib/"
ln -sf libmlsl.so.1.0 "$DST/intel64/lib/libmlsl.so.1"
ln -sf libmlsl.so.1.0 "$DST/intel64/lib/libmlsl.so"
cp eplib/ep_server "$DST/intel64/bin/"
cp include/mlsl.hpp include/mlsl.h "$DST/include/"
cp -r mpirt "$DST/mpirt"
[ -e "$DST/mpirt/lib/libmpi.so" ] || ln -sf libmpi.so.12 "$DST/mpirt/lib/libmpi.so"
# the harness is OUR source, but it only uses API that exists in the reference and is compiled against the
# reference's own header and library
g++ -O2 -std=c++11 -I"$DST/include" "$ROOT/csrc/tests/mlsl_allreduce_bench.cpp" -o "$DST/bin/ref_allreduce_bench" \
    -L"$DST/intel64/lib" -lmlsl -L"$DST/mpirt/lib" -lmpi -ldl -lrt -lpthread \
    -Wl,-rpath,'$ORIGIN/../intel64/lib' -Wl,-rpath,'$ORIGIN/../mpirt/lib'
g++ -O2 -std=c++11 -I"$DST/include" "$ROOT/csrc/tests/mlsl_sample.cpp" -o "$DST/bin/ref_mlsl_sample" \
    -L"$DST/intel64/lib" -lmlsl -L"$DST/mpirt/lib" -lmpi -ldl -lrt -lpthread \
    -Wl,-rpath,'$ORIGIN/../intel64/lib' -Wl,-rpath,'$ORIGIN/../mpirt/lib'
echo "reference installed into $DST"
