// refshim/decl/Frame.h -- stands in for ORB-SLAM3 include/Frame.h: the Frame class itself is declared by the pre-included
// refshim/ref_skeleton.h.  Used by tests/host/build.sh only when no reference checkout is given.
#pragma once
#include "ref_skeleton.h"
