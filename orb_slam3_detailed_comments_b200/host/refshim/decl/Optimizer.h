// refshim/decl/Optimizer.h -- the declaration of ORB_SLAM3::Optimizer (ORB-SLAM3 include/Optimizer.h), reduced to the members the
// host units define.  Frame / KeyFrame / Map come from the pre-included refshim/ref_skeleton.h.  Used only where no reference checkout
// is given (tests/host/build.sh, tests/test_host_shim.py).  Lines between //@ref and //@end are the reference's text (checked by
// tests/test_host_shim.py where a checkout is given); the others carry the parameter types of the units' own definitions, without the
// reference's default arguments.
#ifndef OPTIMIZER_H
#define OPTIMIZER_H

namespace ORB_SLAM3 {

class Optimizer {
   public:
//@ref Optimizer.h
    void static LocalBundleAdjustment(KeyFrame* pKF, bool *pbStopFlag, Map *pMap, int& num_fixedKF, int& num_OptKF, int& num_MPs, int& num_edges);
//@end
    void static LocalInertialBA(KeyFrame* pKF, bool* pbStopFlag, Map* pMap, int& num_fixedKF, int& num_OptKF, int& num_MPs, int& num_edges,
                                bool bLarge, bool bRecInit);
    int static PoseOptimization(Frame* pFrame);
};

}  // namespace ORB_SLAM3

#endif
