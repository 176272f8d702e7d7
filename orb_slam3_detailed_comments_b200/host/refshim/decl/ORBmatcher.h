// refshim/decl/ORBmatcher.h -- the declaration of ORB_SLAM3::ORBmatcher (ORB-SLAM3 include/ORBmatcher.h), reduced to the members
// the host units define.  Frame / KeyFrame / MapPoint come from the pre-included refshim/ref_skeleton.h.  Used only where no reference
// checkout is given (tests/host/build.sh, tests/test_host_shim.py).  Lines between //@ref and //@end are the reference's text
// (tests/test_host_shim.py checks them against the header where a checkout is given); the remaining members are declared with the
// parameter types of the units' own definitions, without the reference's default arguments.
#ifndef ORBMATCHER_H
#define ORBMATCHER_H

#include <set>
#include <utility>
#include <vector>

#include <opencv2/opencv.hpp>

namespace ORB_SLAM3 {

class ORBmatcher {
   public:
//@ref ORBmatcher.h
    ORBmatcher(float nnratio=0.6, bool checkOri=true);
    static int DescriptorDistance(const cv::Mat &a, const cv::Mat &b);
    int SearchByProjection(Frame &F, const std::vector<MapPoint*> &vpMapPoints, const float th=3, const bool bFarPoints = false, const float thFarPoints = 50.0f);
    int SearchByProjection(Frame &CurrentFrame, const Frame &LastFrame, const float th, const bool bMono);
//@end

    int SearchByProjection(Frame& CurrentFrame, KeyFrame* pKF, const std::set<MapPoint*>& sAlreadyFound, const float th, const int ORBdist);
    int SearchByProjection(KeyFrame* pKF, Sophus::Sim3f& Scw, const std::vector<MapPoint*>& vpPoints, std::vector<MapPoint*>& vpMatched, int th,
                           float ratioHamming);
    int SearchByProjection(KeyFrame* pKF, Sophus::Sim3<float>& Scw, const std::vector<MapPoint*>& vpPoints, const std::vector<KeyFrame*>& vpPointsKFs,
                           std::vector<MapPoint*>& vpMatched, std::vector<KeyFrame*>& vpMatchedKF, int th, float ratioHamming);
    int SearchByBoW(KeyFrame* pKF, Frame& F, std::vector<MapPoint*>& vpMapPointMatches);
    int SearchByBoW(KeyFrame* pKF1, KeyFrame* pKF2, std::vector<MapPoint*>& vpMatches12);
    int SearchForInitialization(Frame& F1, Frame& F2, std::vector<cv::Point2f>& vbPrevMatched, std::vector<int>& vnMatches12, int windowSize);
    int SearchForTriangulation(KeyFrame* pKF1, KeyFrame* pKF2, std::vector<std::pair<size_t, size_t> >& vMatchedPairs, const bool bOnlyStereo,
                               const bool bCoarse);
    int Fuse(KeyFrame* pKF, const std::vector<MapPoint*>& vpMapPoints, const float th, const bool bRight);
    int Fuse(KeyFrame* pKF, Sophus::Sim3f& Scw, const std::vector<MapPoint*>& vpPoints, float th, std::vector<MapPoint*>& vpReplacePoint);

   public:
//@ref ORBmatcher.h
    static const int TH_LOW;
    static const int TH_HIGH;
    static const int HISTO_LENGTH;
//@end

   protected:
//@ref ORBmatcher.h
    float RadiusByViewingCos(const float &viewCos);
    void ComputeThreeMaxima(std::vector<int>* histo, const int L, int &ind1, int &ind2, int &ind3);
    float mfNNratio;
    bool mbCheckOrientation;
//@end
};

}  // namespace ORB_SLAM3

#endif
