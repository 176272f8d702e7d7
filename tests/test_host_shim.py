"""CPU tier: the C++ drop-ins (orb_slam3_detailed_comments_b200/host/*.cc) compile against the REFERENCE'S OWN class declarations --
include/ORBextractor.h, include/ORBmatcher.h, include/Optimizer.h, unchanged -- and define exactly the members they replace.
Frame / KeyFrame / MapPoint / Map come from host/refshim/ref_skeleton.h (their real headers pull in Sophus, g2o, DBoW2, boost and
Pangolin, none of which exist here); every skeleton member is checked, line by line, against the text of the reference header it
claims to restate.  Without a reference checkout the units compile against host/refshim/decl (the three class declarations reduced
to the members the units define) and every check but the two that read the reference's own files still runs;
tests/test_zz_host_boundary_gpu.py RUNS the same translation units on a B200."""
import os
import re
import subprocess

import pytest

from oracle import pyoracle as po

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = po.REFERENCE_ROOT      # ORB_REFERENCE_ROOT, as tests/host/build.sh reads it
HOST = os.path.join(ROOT, "orb_slam3_detailed_comments_b200", "host")
HAVE_REF = os.path.exists(os.path.join(REF, "include", "ORBmatcher.h"))
needs_ref = pytest.mark.skipif(not HAVE_REF, reason="reference checkout not present")
DECL = ["-I", os.path.join(REF, "include"), "-I", REF] if HAVE_REF else ["-I", os.path.join(HOST, "refshim", "decl")]


def _compile(tmp_path, name, *defines):
    obj = str(tmp_path / (name + ".o"))
    subprocess.check_call(["g++", "-std=c++14", "-Wall", "-Wno-comment", *defines, "-c", os.path.join(HOST, name + ".cc"),
                           "-include", os.path.join(HOST, "refshim", "ref_skeleton.h"), "-I", os.path.join(HOST, "refshim"),
                           *DECL, "-I", os.path.join(ROOT, "include"), "-I", HOST, "-o", obj])
    return subprocess.check_output(["nm", "-C", obj], text=True)


def test_extractor_unit_defines_the_reference_class(tmp_path):
    syms = _compile(tmp_path, "ORBextractor_b200")
    assert "T ORB_SLAM3::ORBextractor::ORBextractor(int, float, int, int, int)" in syms
    assert "T ORB_SLAM3::ORBextractor::operator()(" in syms
    for used in ("orbx_create", "orbx_extract", "orbx_get_tables", "orbx_download_pyramid", "orbx_destroy"):
        assert f"U {used}" in syms
    assert "orbx_download_level" not in syms          # one batched pyramid download, not eight synchronous ones
    assert "abort" not in syms                        # failures throw orb_b200::Error


def test_matcher_unit_defines_the_per_frame_searches(tmp_path):
    syms = _compile(tmp_path, "ORBmatcher_b200")
    assert "T ORB_SLAM3::ORBmatcher::ORBmatcher(float, bool)" in syms
    assert "T ORB_SLAM3::ORBmatcher::DescriptorDistance(cv::Mat const&, cv::Mat const&)" in syms
    assert re.search(r"T ORB_SLAM3::ORBmatcher::SearchByProjection\(ORB_SLAM3::Frame&, std::vector<ORB_SLAM3::MapPoint\*.*> const&, float, bool, float\)", syms)
    assert "T ORB_SLAM3::ORBmatcher::SearchByProjection(ORB_SLAM3::Frame&, ORB_SLAM3::Frame const&, float, bool)" in syms
    for c in ("TH_HIGH", "TH_LOW", "HISTO_LENGTH"):
        assert f"ORB_SLAM3::ORBmatcher::{c}" in syms
    assert "U orbm_search_local_points" in syms and "U orbm_search_last_frame" in syms


def test_stereo_and_lba_units(tmp_path):
    syms = _compile(tmp_path, "Frame_stereo_b200")
    assert "T ORB_SLAM3::Frame::ComputeStereoMatches()" in syms and "U orbm_stereo_pair" in syms
    syms = _compile(tmp_path, "Optimizer_lba_b200")
    assert "T ORB_SLAM3::Optimizer::LocalBundleAdjustment(ORB_SLAM3::KeyFrame*, bool*, ORB_SLAM3::Map*, int&, int&, int&, int&)" in syms
    assert "U lba_solve_bool" in syms and "g2o" not in syms


def test_inertial_ba_unit(tmp_path):
    """host/Optimizer_liba_b200.cc against the reference's Optimizer.h; the skeleton's IMU members are behind ORB_REFSHIM_LIBA so that the
    other units' translation (the binary validated on the B200) does not change."""
    syms = _compile(tmp_path, "Optimizer_liba_b200", "-DORB_REFSHIM_LIBA")
    assert "T ORB_SLAM3::Optimizer::LocalInertialBA(ORB_SLAM3::KeyFrame*, bool*, ORB_SLAM3::Map*, int&, int&, int&, int&, bool, bool)" in syms
    assert "U liba_solve" in syms and "U liba_link_information" in syms and "g2o" not in syms and "abort" not in syms


def test_bow_search_unit(tmp_path):
    syms = _compile(tmp_path, "ORBmatcher_bow_b200", "-DORB_REFSHIM_BOW")
    assert re.search(r"T ORB_SLAM3::ORBmatcher::SearchByBoW\(ORB_SLAM3::KeyFrame\*, ORB_SLAM3::Frame&, std::vector<ORB_SLAM3::MapPoint\*.*>&\)", syms)
    assert re.search(r"T ORB_SLAM3::ORBmatcher::SearchByBoW\(ORB_SLAM3::KeyFrame\*, ORB_SLAM3::KeyFrame\*, std::vector<ORB_SLAM3::MapPoint\*.*>&\)", syms)
    assert "U orbm_search_bow" in syms and "U orbm_search_bow_keyframes" in syms and "abort" not in syms


def test_triangulation_search_unit(tmp_path):
    syms = _compile(tmp_path, "ORBmatcher_triangulation_b200", "-DORB_REFSHIM_BOW", "-DORB_REFSHIM_TRI")
    assert re.search(r"T ORB_SLAM3::ORBmatcher::SearchForTriangulation\(ORB_SLAM3::KeyFrame\*, ORB_SLAM3::KeyFrame\*, std::vector<std::pair<unsigned long, unsigned long>.*>&, bool, bool\)", syms)
    assert "U orbm_search_triangulation" in syms and "abort" not in syms


def test_initialization_search_unit(tmp_path):
    syms = _compile(tmp_path, "ORBmatcher_init_b200")
    assert re.search(r"T ORB_SLAM3::ORBmatcher::SearchForInitialization\(ORB_SLAM3::Frame&, ORB_SLAM3::Frame&, std::vector<cv::Point_<float>.*>&, std::vector<int.*>&, int\)", syms)
    assert "U orbm_search_initialization" in syms and "abort" not in syms


@needs_ref
def test_compute_bow_unit_and_its_vocabulary_access(tmp_path):
    """Frame_bow_b200.cc against the skeleton (with a mock vocabulary whose nodes are protected, as in DBoW2), and the same access pattern
    against the reference's REAL DBoW2 headers (over the boost / OpenCV miniatures of oracle/ref_shim)."""
    syms = _compile(tmp_path, "Frame_bow_b200", "-DORB_REFSHIM_VOC")
    assert "T ORB_SLAM3::Frame::ComputeBoW()" in syms and "U orbv_transform" in syms and "U orbv_create" in syms and "abort" not in syms
    dbow = os.path.join(REF, "Thirdparty", "DBoW2")
    shim = os.path.join(ROOT, "oracle", "ref_shim")
    subprocess.check_call(["g++", "-std=c++14", "-Wall", "-Wno-comment", "-Wno-sign-compare", "-Wno-unused-variable", "-c", os.path.join(ROOT, "tests", "host", "voc_access_probe.cc"),
                           "-I", os.path.join(shim, "dbow"), "-I", shim, "-I", dbow, "-I", os.path.join(dbow, "DBoW2"), "-o", str(tmp_path / "probe.o")])


def test_fuse_unit(tmp_path):
    syms = _compile(tmp_path, "ORBmatcher_fuse_b200", "-DORB_REFSHIM_FUSE", "-Wno-reorder")
    assert re.search(r"T ORB_SLAM3::ORBmatcher::Fuse\(ORB_SLAM3::KeyFrame\*, std::vector<ORB_SLAM3::MapPoint\*.*> const&, float, bool\)", syms)
    assert "U orbm_search_keyframe" in syms and "abort" not in syms


def test_relocalisation_search_unit(tmp_path):
    syms = _compile(tmp_path, "ORBmatcher_reloc_b200", "-DORB_REFSHIM_FUSE", "-Wno-reorder")
    assert re.search(r"T ORB_SLAM3::ORBmatcher::SearchByProjection\(ORB_SLAM3::Frame&, ORB_SLAM3::KeyFrame\*, std::set<ORB_SLAM3::MapPoint\*.*> const&, float, int\)", syms)
    assert "U orbm_search_keyframe" in syms and "abort" not in syms


def test_sim3_searches_unit(tmp_path):
    syms = _compile(tmp_path, "ORBmatcher_sim3_b200", "-DORB_REFSHIM_FUSE", "-Wno-reorder")
    assert re.search(r"T ORB_SLAM3::ORBmatcher::SearchByProjection\(ORB_SLAM3::KeyFrame\*, Sophus::Sim3<float>&, std::vector<ORB_SLAM3::MapPoint\*.*> const&, std::vector<ORB_SLAM3::MapPoint\*.*>&, int, float\)", syms)
    assert re.search(r"T ORB_SLAM3::ORBmatcher::Fuse\(ORB_SLAM3::KeyFrame\*, Sophus::Sim3<float>&, std::vector<ORB_SLAM3::MapPoint\*.*> const&, float, std::vector<ORB_SLAM3::MapPoint\*.*>&\)", syms)
    assert re.search(r"T ORB_SLAM3::ORBmatcher::SearchByProjection\(ORB_SLAM3::KeyFrame\*, Sophus::Sim3<float>&, std::vector<ORB_SLAM3::MapPoint\*.*> const&, std::vector<ORB_SLAM3::KeyFrame\*.*> const&, std::vector<ORB_SLAM3::MapPoint\*.*>&, std::vector<ORB_SLAM3::KeyFrame\*.*>&, int, float\)", syms)
    assert "U orbm_search_keyframe" in syms and "abort" not in syms


def test_pose_optimization_unit(tmp_path):
    syms = _compile(tmp_path, "Optimizer_pose_b200", "-DORB_REFSHIM_POSE")
    assert "T ORB_SLAM3::Optimizer::PoseOptimization(ORB_SLAM3::Frame*)" in syms
    assert "U orbo_pose_optimization" in syms and "U orb_b200_handle_of" in syms and "g2o" not in syms and "abort" not in syms


def _norm(s):
    return re.sub(r"\s+", "", re.sub(r"//.*", "", s))


@needs_ref
def test_skeleton_members_are_the_reference_declarations():
    """Every line between //@ref <header> and //@end in ref_skeleton.h and decl/*.h appears verbatim (whitespace and comments aside) in
    that header."""
    text = []
    for f in ["ref_skeleton.h"] + sorted(os.path.join("decl", h) for h in os.listdir(os.path.join(HOST, "refshim", "decl"))):
        text += open(os.path.join(HOST, "refshim", f)).read().splitlines()
    cur, checked = None, 0
    cache = {}
    for line in text:
        m = re.match(r"\s*//@ref (\S+)", line)
        if m:
            cur = m.group(1)
            cache.setdefault(cur, _norm(open(os.path.join(REF, "include", cur)).read()))
            continue
        if re.match(r"\s*//@end", line):
            cur = None
            continue
        if cur and _norm(line):
            assert _norm(line) in cache[cur], f"{cur}: no such declaration: {line.strip()}"
            checked += 1
    assert checked >= 116
