#!/bin/bash
# Compiles the drop-in C++ adapter (include/CPhotoconsistencyOdometryCuda.h) against the reference's
# abstract class and matrix types, with OpenCV / Eigen replaced by the stand-ins of oracle/shim, and
# links programs against the in-tree libphovo_b200.so:
#   _build/frame_alignment_app      the headless mirror of both apps' main() (tests/cpp/frame_alignment_app.cpp)
# Where REF names a checkout of the original project, the adapter is compiled against its own
# phovo/include/CPhotoconsistencyOdometry.h + Matrix.h, unmodified, and two more programs are built:
#   _build/reference_frame_alignment  a copy of the reference's apps/PhotoconsistencyFrameAlignment/
#                                   PhotoconsistencyFrameAlignment.cpp with exactly the INTEGRATION.md patch
#                                   applied (USE_PHOTOCONSISTENCY_ODOMETRY_METHOD == 3); the patched copy
#                                   lives only under _build/ (git-ignored), never in the repository.
#   _build/reference_visual_odometry  the same for apps/PhotoconsistencyVisualOdometry/PhotoconsistencyVisualOdometry.cpp
#                                   (with the reference's own CCameraRecord / CMultiSensorDataSource / CImageReader
#                                   headers; Boost.Filesystem is std::filesystem behind oracle/shim/boost).
# Without REF the base class comes from tests/cpp/shim/CPhotoconsistencyOdometry.h, which declares the
# same interface.
set -e
HERE="$(cd "$(dirname "$0")" && pwd)"
ROOT="$(cd "$HERE/../.." && pwd)"
PKG="$ROOT/photoconsistency-visual-odometry_b200"
REF="${REF:-}"
OUT="$HERE/_build"
mkdir -p "$OUT"
if [ -n "$REF" ] && [ ! -d "$REF/phovo/include" ]; then
  echo "REF=$REF is not a checkout of the original project (no phovo/include)" >&2
  exit 1
fi
BASE="$HERE/shim"
[ -n "$REF" ] && BASE="$REF/phovo/include"
INC=(-I "$ROOT/include" -I "$BASE" -I "$ROOT/oracle/shim" -I "$ROOT/oracle/shim/eigen3")
LINK=(-L "$PKG" -lphovo_b200 -Wl,-rpath,"\$ORIGIN/../../../photoconsistency-visual-odometry_b200"
      -L /usr/local/cuda/lib64 -Wl,-rpath,/usr/local/cuda/lib64 -lcudart)
g++ -std=c++11 -O2 -Wall -Wextra -Wno-unused-parameter "${INC[@]}" "$HERE/frame_alignment_app.cpp" -o "$OUT/frame_alignment_app" "${LINK[@]}"
echo "built $OUT/frame_alignment_app"
if [ -z "$REF" ]; then
  rm -f "$OUT"/reference_* "$OUT"/Photoconsistency*_method3.cpp
  echo "REF not set: the reference apps are not built"
  exit 0
fi

# the reference apps themselves + the INTEGRATION.md patch
patch_app() {   # <reference source> <patched copy> <what the object-definition branch declares>
python3 - "$1" "$2" "$3" <<'PY'
import sys
src = open(sys.argv[1]).read()
def once(text, old, new):
    assert text.count(old) == 1, old
    return text.replace(old, new)
src = once(src, "#define USE_PHOTOCONSISTENCY_ODOMETRY_METHOD 0", "#define USE_PHOTOCONSISTENCY_ODOMETRY_METHOD 3")
src = once(src, '  #include "CPhotoconsistencyOdometryBiObjective.h"\n#endif',
           '  #include "CPhotoconsistencyOdometryBiObjective.h"\n'
           '#elif USE_PHOTOCONSISTENCY_ODOMETRY_METHOD == 3\n  #include "CPhotoconsistencyOdometryCuda.h"\n#endif')
tail = sys.argv[3]
src = once(src, "phovo::Analytic::CPhotoconsistencyOdometryBiObjective< PixelType, CoordinateType > " + tail + ";\n#endif",
           "phovo::Analytic::CPhotoconsistencyOdometryBiObjective< PixelType, CoordinateType > " + tail + ";\n"
           "#elif USE_PHOTOCONSISTENCY_ODOMETRY_METHOD == 3\n"
           "  " + ("typedef " if tail[0].isupper() else "") + "phovo::Cuda::CPhotoconsistencyOdometryCuda< PixelType, CoordinateType > " + tail + ";\n#endif")
open(sys.argv[2], "w").write(src)
PY
}
patch_app "$REF/apps/PhotoconsistencyFrameAlignment/PhotoconsistencyFrameAlignment.cpp" "$OUT/PhotoconsistencyFrameAlignment_method3.cpp" photoconsistencyOdometry
g++ -std=c++17 -O2 -w "${INC[@]}" "$OUT/PhotoconsistencyFrameAlignment_method3.cpp" -o "$OUT/reference_frame_alignment" "${LINK[@]}"
echo "built $OUT/reference_frame_alignment (reference app + METHOD == 3)"
patch_app "$REF/apps/PhotoconsistencyVisualOdometry/PhotoconsistencyVisualOdometry.cpp" "$OUT/PhotoconsistencyVisualOdometry_method3.cpp" PhotoconsistencyVisualOdometryType
g++ -std=c++17 -O2 -w "${INC[@]}" "$OUT/PhotoconsistencyVisualOdometry_method3.cpp" -o "$OUT/reference_visual_odometry" "${LINK[@]}"
echo "built $OUT/reference_visual_odometry (reference app + METHOD == 3)"
