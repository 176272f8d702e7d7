#!/bin/bash
# Builds tests/host/host_boundary: the four host translation units + the test driver, against the REFERENCE's own headers
# (ORBextractor.h, ORBmatcher.h, Optimizer.h under $REF/include) with the skeleton map and the miniature third-party headers of
# orb_slam3_detailed_comments_b200/host/refshim.  Without a reference checkout the same units compile against the reduced
# declarations of host/refshim/decl, so every checkout builds the binary (__graft_entry__.build()); it is git-ignored.
set -e
ROOT="$(cd "$(dirname "$0")/../.." && pwd)"
REF="${ORB_REFERENCE_ROOT:-/root/reference}"
H="$ROOT/orb_slam3_detailed_comments_b200/host"
if [ -f "$REF/include/ORBmatcher.h" ]; then DECL=(-I "$REF/include" -I "$REF"); else DECL=(-I "$H/refshim/decl"); fi
g++ -std=c++14 -O1 -Wall -Wno-unused-function -Wno-comment -include "$H/refshim/ref_skeleton.h" -I "$H/refshim" "${DECL[@]}" \
    -I "$ROOT/include" -I "$H" "$ROOT/tests/host/host_boundary.cc" "$H/ORBextractor_b200.cc" "$H/Frame_stereo_b200.cc" \
    "$H/ORBmatcher_b200.cc" "$H/Optimizer_lba_b200.cc" -L "$ROOT/orb_slam3_detailed_comments_b200/lib" -lorbslam3_b200 \
    -Wl,-rpath,'$ORIGIN/../../orb_slam3_detailed_comments_b200/lib' -lpthread -o "$ROOT/tests/host/host_boundary"
