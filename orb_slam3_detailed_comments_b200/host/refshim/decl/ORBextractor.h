// refshim/decl/ORBextractor.h -- the declaration of ORB_SLAM3::ORBextractor (ORB-SLAM3 include/ORBextractor.h), reduced to the
// members host/ORBextractor_b200.cc defines and its callers use.  Used only where no reference checkout is given (tests/host/build.sh,
// tests/test_host_shim.py); with one, the units compile against the reference's own header.  Lines between //@ref and //@end are the
// reference's text (tests/test_host_shim.py checks them against the header where a checkout is given).
#ifndef ORBEXTRACTOR_H
#define ORBEXTRACTOR_H

#include <list>
#include <vector>

#include <opencv2/opencv.hpp>

namespace ORB_SLAM3 {

class ORBextractor {
   public:
//@ref ORBextractor.h
    ORBextractor(int nfeatures, float scaleFactor, int nlevels,
                 int iniThFAST, int minThFAST);
    ~ORBextractor(){}
    int operator()( cv::InputArray _image, cv::InputArray _mask,
                    std::vector<cv::KeyPoint>& _keypoints,
                    cv::OutputArray _descriptors, std::vector<int> &vLappingArea);
    int inline GetLevels(){
        return nlevels;}
    float inline GetScaleFactor(){
        return scaleFactor;}
    std::vector<float> inline GetScaleFactors(){
        return mvScaleFactor;
    }
    std::vector<float> inline GetInverseScaleFactors(){
        return mvInvScaleFactor;
    }
    std::vector<float> inline GetScaleSigmaSquares(){
        return mvLevelSigma2;
    }
    std::vector<float> inline GetInverseScaleSigmaSquares(){
        return mvInvLevelSigma2;
    }
    std::vector<cv::Mat> mvImagePyramid;
//@end

   protected:
//@ref ORBextractor.h
    std::vector<cv::Point> pattern;
    int nfeatures;
    double scaleFactor;
    int nlevels;
    int iniThFAST;
    int minThFAST;
    std::vector<int> mnFeaturesPerLevel;
    std::vector<int> umax;
    std::vector<float> mvScaleFactor;
    std::vector<float> mvInvScaleFactor;
    std::vector<float> mvLevelSigma2;
    std::vector<float> mvInvLevelSigma2;
//@end
};

}  // namespace ORB_SLAM3

#endif
