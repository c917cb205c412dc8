#!/bin/bash
# TEST INFRASTRUCTURE ONLY — builds oracle/_ref/libdso_ref_select.so: oracle/ref_select.cpp (a C harness around the reference's own
# PixelSelector) linked against oracle/_ref/libdso_ref.so, which oracle/ref_build.sh compiles from the reference's sources where they lie.
# Same flags and include path as ref_build.sh.  Output goes to oracle/_ref/ only (git-ignored).
set -e
HERE="$(cd "$(dirname "$0")" && pwd)"
# the reference's sources: $REF_ROOT, else where oracle/ref_build.sh looks for them
REF=${REF_ROOT:-$(sed -n 's/^REF=\${REF_ROOT:-\(.*\)}$/\1/p' "$HERE/ref_build.sh")}
if [ ! -d "$REF/src/dso" ]; then echo "ref_select_build: $REF/src/dso not present: keeping the prebuilt oracle/_ref"; exit 0; fi
OUT="$HERE/_ref"
CXX=${CXX:-g++}
if [ ! -f "$OUT/libdso_ref.so" ]; then bash "$HERE/ref_build.sh"; fi
$CXX -std=c++17 -O3 -fPIC -w -I"$HERE/shim" -I"$REF/src/dso" -I"$REF/src" -shared -o "$OUT/libdso_ref_select.so" "$HERE/ref_select.cpp" \
     -L"$OUT" -ldso_ref -Wl,-rpath,'$ORIGIN'
echo "ref_select_build: $OUT/libdso_ref_select.so"
