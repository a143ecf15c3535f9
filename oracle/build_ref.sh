#!/usr/bin/env bash
# TEST INFRASTRUCTURE ONLY -- builds the *unmodified* reference (ShadenSmith/splatt)
# from the sources where they lie under /root/reference into oracle/_ref/.
# Nothing under oracle/ is ever linked, imported or executed by the product
# (splatt_b200/, libsplatt_b200.so); only tests/, __graft_entry__.smoke() and
# bench.py's cpu_baseline / --impl reference legs use it, as the checker.
#
# The reference's own build system (configure + cmake) is NOT run: cmake would
# write include/splatt/types.h into the read-only source tree
# (cmake/types.cmake:48-49).  We generate that one header into oracle/_ref/gen/
# with the default widths (idx 64, val 64, blas-int 32; cmake/types.cmake:3-4)
# and compile src/*.c directly with the reference's release flags
# (cmake/flags.cmake:5-16) minus -march=native (the GPU box host CPU may differ
# from the build container; x86-64-v3 = AVX2+FMA is used instead).
#
# Outputs (git-ignored, shipped to the GPU box by gpurun):
#   oracle/_ref/libsplatt_ref.so   reference library (all of src/*.c, OpenMP) + ref_driver.c
#   oracle/_ref/splatt             reference CLI (src/cmds/*.c), BASELINE config #1
#   oracle/_ref/splatt_gpu         the same CLI linked against libsplatt_b200.so for the
#                                  MTTKRP symbols (drop-in proof, needs a GPU to run)
#   oracle/_ref/gen/splatt/types.h generated type-width header
set -euo pipefail
HERE="$(cd "$(dirname "${BASH_SOURCE[0]}")" && pwd)"
REF="${SPLATT_REFERENCE:-/root/reference}"
OUT="$HERE/_ref"
if [ ! -d "$REF/src" ]; then
  echo "build_ref: $REF not present; keeping prebuilt $OUT (if any)" >&2
  exit 0
fi
mkdir -p "$OUT/gen/splatt" "$OUT/obj"
sed -e 's/@CONFIG_IDX_WIDTH@/64/' -e 's/@CONFIG_VAL_WIDTH@/64/' \
    -e 's/@CONFIG_BLAS_INT@/32/' "$REF/include/splatt/types_config.h" \
    > "$OUT/gen/splatt/types.h"

# LP64 BLAS/LAPACK (dsyrk_/dpotrf_/dpotrs_/dgelss_): the image has no system
# BLAS; the OpenBLAS 0.3.15 bundled with opencv-python-headless exports them.
SITE="$(python - <<'PY'
import sysconfig; print(sysconfig.get_paths()["purelib"])
PY
)"
BLASDIR="$SITE/opencv_python_headless.libs"
BLASLIB="$(ls "$BLASDIR"/libopenblasp-*.so 2>/dev/null | head -1 || true)"
if [ -z "$BLASLIB" ]; then
  echo "build_ref: no OpenBLAS found under $BLASDIR" >&2; exit 1
fi

CFLAGS="-O3 -std=c99 -fgnu89-inline -fstrict-aliasing -fPIC -funroll-loops \
 -march=x86-64-v3 -ftree-vectorize -fopenmp -D_GNU_SOURCE -DNDEBUG -w \
 -I$OUT/gen -I$REF/include"

objs=()
for f in "$REF"/src/*.c; do
  o="$OUT/obj/$(basename "${f%.c}").o"
  gcc $CFLAGS -c "$f" -o "$o" &
  objs+=("$o")
done
wait
# flat ctypes-facing driver (oracle/ref_driver.c, ours) compiled against the
# reference's internal headers and linked into the same library
gcc $CFLAGS -I"$REF/src" -c "$HERE/ref_driver.c" -o "$OUT/obj/ref_driver.o"
gcc -shared -fopenmp -o "$OUT/libsplatt_ref.so" "${objs[@]}" "$OUT/obj/ref_driver.o" \
    "$BLASLIB" -Wl,--disable-new-dtags,-rpath,"$BLASDIR" -lm -lrt

cmdobjs=()
for f in "$REF"/src/cmds/*.c; do
  case "$f" in *mpi_cmd_cpd.c) continue;; esac
  o="$OUT/obj/cmd_$(basename "${f%.c}").o"
  gcc $CFLAGS -I"$REF/src" -c "$f" -o "$o" &
  cmdobjs+=("$o")
done
wait
gcc -fopenmp -o "$OUT/splatt" "${cmdobjs[@]}" "${objs[@]}" \
    "$BLASLIB" -Wl,--disable-new-dtags,-rpath,"$BLASDIR" -lm -lrt
# The drop-in proof: the SAME unmodified reference CLI, but with the four MTTKRP
# symbols of src/mttkrp.c renamed out of the way (objcopy, no source edits) so that
# cpd.c / bench.c / the tests resolve splatt_mttkrp_csf, splatt_mttkrp_alloc_ws,
# splatt_mttkrp_free_ws and splatt_mttkrp from libsplatt_b200.so (INTEGRATION.md,
# option A).  `splatt_gpu cpd ...` = reference host code + B200 MTTKRP.
B200LIB="$HERE/../splatt_b200/libsplatt_b200.so"
# linked by name, not path: the library has no soname, so a path on the link line would be
# recorded as the dependency and the binaries would break once the tree moves; the
# $ORIGIN-relative rpath below finds it in whatever directory the tree lands in
B200LINK=(-L"$HERE/../splatt_b200" -l:libsplatt_b200.so)
if [ -f "$B200LIB" ]; then
  objcopy --redefine-sym splatt_mttkrp_csf=splatt_mttkrp_csf_cpu \
          --redefine-sym splatt_mttkrp=splatt_mttkrp_cpu \
          --redefine-sym splatt_mttkrp_alloc_ws=splatt_mttkrp_alloc_ws_cpu \
          --redefine-sym splatt_mttkrp_free_ws=splatt_mttkrp_free_ws_cpu \
          "$OUT/obj/mttkrp.o" "$OUT/obj/mttkrp_cpu.o"
  gpuobjs=()
  for o in "${objs[@]}"; do
    case "$o" in */mttkrp.o) gpuobjs+=("$OUT/obj/mttkrp_cpu.o");; *) gpuobjs+=("$o");; esac
  done
  gcc -fopenmp -o "$OUT/splatt_gpu" "${cmdobjs[@]}" "${gpuobjs[@]}" "${B200LINK[@]}" \
      "$BLASLIB" -Wl,--disable-new-dtags,-rpath,"$BLASDIR" -Wl,-rpath,'$ORIGIN/../../splatt_b200' -lm -lrt
fi
# The reference's OWN MTTKRP unit tests (tests/mttkrp_test.c: every fixture x every mode x
# ONEMODE/TWOMODE/ALLMODE x NOTILE/DENSETILE levels, gold = mttkrp_stream, abs tol 1e-10),
# built twice: against the reference's kernels (reftest_mttkrp_cpu) and against
# libsplatt_b200.so through the same symbol rename (reftest_mttkrp_gpu).  The fixture
# directory is relative to the working directory: tests/test_reference_unit_tests.py writes
# it from tests/golden/*.npz into a temporary directory and runs the binaries there.
FIX='"splatt_b200_fixtures/"'
tobjs=()
for f in main.c mttkrp_test.c; do
  o="$OUT/obj/t_${f%.c}.o"
  gcc $CFLAGS -I"$REF/src" -DSPLATT_TEST_DATASETS="$FIX" -DSPLATT_TEST_GRAPHS="$FIX" \
      -c "$REF/tests/$f" -o "$o"
  tobjs+=("$o")
done
gcc -fopenmp -o "$OUT/reftest_mttkrp_cpu" "${tobjs[@]}" "${objs[@]}" \
    "$BLASLIB" -Wl,--disable-new-dtags,-rpath,"$BLASDIR" -lm -lrt
if [ -f "$B200LIB" ]; then
  gcc -fopenmp -o "$OUT/reftest_mttkrp_gpu" "${tobjs[@]}" "${gpuobjs[@]}" "${B200LINK[@]}" \
      "$BLASLIB" -Wl,--disable-new-dtags,-rpath,"$BLASDIR" -Wl,-rpath,'$ORIGIN/../../splatt_b200' -lm -lrt
fi
rm -rf "$OUT/obj"
echo "build_ref: built $OUT/libsplatt_ref.so and $OUT/splatt"
