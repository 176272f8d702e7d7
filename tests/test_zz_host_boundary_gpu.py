"""GPU tier: the host translation units (orb_slam3_detailed_comments_b200/host/*.cc) LINKED AND RUN through the reference's own
class declarations -- ORB_SLAM3::ORBextractor::operator(), Frame::ComputeStereoMatches, the two per-frame
ORBmatcher::SearchByProjection overloads and Optimizer::LocalBundleAdjustment (window selection, flattening, outlier removal,
write-back: Optimizer.cc:1744-1855, 1873-2091, 2107-2187) over a mock map -- against the oracle.
tests/host/host_boundary is built by __graft_entry__.build() (tests/host/build.sh)."""
import os
import subprocess

import numpy as np
import pytest

from oracle import pyoracle as po
from orb_slam3_detailed_comments_b200 import synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "tests", "host", "host_boundary")
W, H, NF = 640, 480, 1200
FX, FY, CX, CY, BF, B = 435.2, 435.2, 320.0, 240.0, 47.9, 0.11
CAM6 = np.array([FX, FY, CX, CY, BF, B], np.float32)
BOUNDS = np.array([0, W, 0, H], np.float32)
KP = po.KP_DTYPE


def _binary():
    assert os.path.exists(BIN), "tests/host/host_boundary is not built (run __graft_entry__.build())"
    return BIN


def _run(d, meta):
    with open(os.path.join(d, "meta.txt"), "w") as f:
        for k, v in meta.items():
            f.write(f"{k} {float(v)!r}\n")
    r = subprocess.run([_binary(), d], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    return lambda name, dt: np.fromfile(os.path.join(d, name), dt)


def _quat_pose(yaw_deg, t):
    a = np.deg2rad(yaw_deg) / 2
    return np.array([0, np.sin(a), 0, np.cos(a), *t], np.float32)


@pytest.fixture(scope="module")
def frame(tmp_path_factory):
    """One stereo frame through the C++ classes, plus the oracle's view of the same frame."""
    d = str(tmp_path_factory.mktemp("host"))
    l, r, _ = synth.stereo_pair(W, H, seed=321)
    l.tofile(os.path.join(d, "left.u8")); r.tofile(os.path.join(d, "right.u8"))
    eL, eR = po.OracleExtractor(NF, 1.2, 8, 20, 7), po.OracleExtractor(NF, 1.2, 8, 20, 7)
    monoL, kL, dL = eL(l)
    monoR, kR, dR = eR(r)
    uR, dep, _ = po.stereo_matches(eL, eR, kL, dL, kR, dR, np.float32(BF), np.float32(B))
    rng = np.random.default_rng(5)
    N = len(kL)
    meta = dict(W=W, H=H, nfeatures=NF, fx=FX, fy=FY, cx=CX, cy=CY, bf=BF, b=B)

    # ---- queries of SearchByProjection(F, vpMapPoints): the frame's own stereo points, jittered, 4x over-subscribed ----
    sel = np.nonzero(dep > 0)[0]
    sel = np.concatenate([sel, rng.choice(sel, 3 * len(sel))])
    jit = rng.normal(0, 1.5, (len(sel), 2)).astype(np.float32)
    loc = dict(px=(kL["x"][sel] + jit[:, 0]).astype(np.float32), py=(kL["y"][sel] + jit[:, 1]).astype(np.float32))
    loc["pxr"] = (loc["px"] - np.float32(BF) / dep[sel]).astype(np.float32)
    loc["level"] = np.clip(kL["octave"][sel] + rng.integers(-1, 2, len(sel)), 0, 7).astype(np.int32)
    loc["vcos"] = rng.uniform(0.99, 1.0, len(sel)).astype(np.float32)
    loc["depth"] = dep[sel].astype(np.float32)
    loc["inview"] = (rng.random(len(sel)) < 0.9).astype(np.uint8)
    loc["bad"] = (rng.random(len(sel)) < 0.05).astype(np.uint8)
    qd = dL[sel].copy()
    flip = rng.random(qd.shape) < 0.02
    qd[flip] ^= (1 << rng.integers(0, 8, int(flip.sum()))).astype(np.uint8)
    loc["desc"] = qd
    claimed = np.zeros(N, np.uint8)
    claimed[rng.random(N) < 0.15] = 1          # already holds a map point with observations (Tracking's motion-model matches)
    claimed[(rng.random(N) < 0.05) & (claimed == 0)] = 2   # holds a point WITHOUT observations: may be overwritten (:101-103)
    loc["claimed"] = claimed
    th_far = float(np.percentile(dep[sel], 80))
    for k, v in loc.items():
        v.tofile(os.path.join(d, f"loc_{k}." + {"float32": "f32", "int32": "i32", "uint8": "u8"}[str(v.dtype)]))
    meta.update(loc_n=len(sel), loc_th=3.0, loc_nnratio=0.8, loc_far=1, loc_thfar=th_far)

    # ---- LastFrame of SearchByProjection(CurrentFrame, LastFrame): the same points seen from a camera 30 cm behind ----
    has = (dep > 0).astype(np.uint8)
    outl = ((rng.random(N) < 0.1) & (has == 1)).astype(np.uint8)
    z = np.where(dep > 0, dep, 1.0).astype(np.float32)
    xw = np.stack([(kL["x"] - np.float32(CX)) * z / np.float32(FX), (kL["y"] - np.float32(CY)) * z / np.float32(FY), z], 1).astype(np.float32)
    zmid = float(np.median(dep[dep > 0]))
    Tcw = _quat_pose(0.05, [2.0 * zmid / FX, 1.0 * zmid / FY, -0.15])     # the current camera is 0.15 m AHEAD (> mb): bForward
    Tlw = _quat_pose(0.0, [0, 0, 0])
    last = dict(has=has, outlier=outl, obspos=(rng.random(N) < 0.7).astype(np.uint8), desc=dL, xw=xw, angle=kL["angle"].astype(np.float32),
                octave=kL["octave"].astype(np.int32), Tcw=Tcw, Tlw=Tlw)
    for k, v in last.items():
        np.ascontiguousarray(v).tofile(os.path.join(d, f"last_{k}." + {"float32": "f32", "int32": "i32", "uint8": "u8"}[str(v.dtype)]))
    meta.update(last_n=N, last_th=15.0, last_mono=0, last_checkori=1)
    out = _run(d, meta)
    return dict(out=out, l=l, r=r, eL=eL, kL=kL, dL=dL, kR=kR, monoL=monoL, monoR=monoR, uR=uR, dep=dep, loc=loc, sel=sel, th_far=th_far,
                last=last, N=N)


def test_extractor_class_matches_oracle(frame):
    out = frame["out"]
    kps = out("out_kpsL.bin", KP)
    assert len(kps) == len(frame["kL"]) and (kps.view(np.uint8) == frame["kL"].view(np.uint8)).all()
    assert (out("out_descL.bin", np.uint8).reshape(-1, 32) == frame["dL"]).all()
    assert (out("out_kpsR.bin", KP).view(np.uint8) == frame["kR"].view(np.uint8)).all()
    assert list(out("out_mono.i32", np.int32)) == [frame["monoL"], frame["monoR"], len(frame["kL"]), len(frame["kR"])]
    pyr = np.concatenate([frame["eL"].level_pyramid(l).ravel() for l in range(8)])
    assert (out("out_pyramidL.u8", np.uint8) == pyr).all()                       # mvImagePyramid, one batched download
    assert (out("out_scale.f32", np.float32).view(np.uint32) == frame["eL"].scale_factors.view(np.uint32)).all()
    # the monocular call site {0, 1000} and the empty-image return value
    e = po.OracleExtractor(NF, 1.2, 8, 20, 7)
    mono, k, _ = e(frame["l"], (0, 1000))
    assert list(out("out_monoM.i32", np.int32)) == [mono, len(k)] and (out("out_kpsM.bin", KP).view(np.uint8) == k.view(np.uint8)).all()
    assert list(out("out_empty.i32", np.int32)) == [-1]


def test_compute_stereo_matches_member(frame):
    out = frame["out"]
    assert (out("out_uright.f32", np.float32).view(np.uint32) == frame["uR"].view(np.uint32)).all()
    assert (out("out_depth.f32", np.float32).view(np.uint32) == frame["dep"].view(np.uint32)).all()
    assert (frame["dep"] > 0).sum() > 300


def test_search_by_projection_local_map_member(frame):
    loc, N = frame["loc"], frame["N"]
    res = frame["out"]("out_local.i32", np.int32)
    ok = np.nonzero((loc["inview"] == 1) & (loc["bad"] == 0))[0]          # :52-58 skips; the far gate is inside the search
    sf = frame["eL"].scale_factors
    rmatch, rnm = po.search_local(frame["kL"], frame["dL"], frame["uR"], BOUNDS, sf, loc["px"][ok], loc["py"][ok], loc["pxr"][ok],
                                  loc["level"][ok], loc["vcos"][ok], loc["desc"][ok], 3.0, np.float32(0.8), claimed=(loc["claimed"] == 1),
                                  trackdepth=loc["depth"][ok], far=True, th_far=np.float32(frame["th_far"]))
    want = np.where(loc["claimed"] == 1, -2, np.where(loc["claimed"] == 2, -3, -1)).astype(np.int32)
    for q, f in enumerate(rmatch):
        if f >= 0:
            want[f] = ok[q]
    assert res[N] == rnm and rnm > 100
    assert (res[:N] == want).all()
    assert (want[loc["claimed"] == 2] >= 0).any()          # a point without observations was overwritten


def test_search_by_projection_last_frame_member(frame):
    last, N = frame["last"], frame["N"]
    res = frame["out"]("out_last.i32", np.int32)
    src = np.nonzero((last["has"] == 1) & (last["outlier"] == 0))[0]
    sf = frame["eL"].scale_factors
    rfm, rnm = po.search_last(frame["kL"], frame["dL"], frame["uR"], BOUNDS, sf, CAM6, last["Tcw"], 1, last["xw"][src], last["octave"][src],
                              last["angle"][src], last["desc"][src], last["obspos"][src], 15.0, True)
    want = np.where(rfm >= 0, src[np.clip(rfm, 0, None)], -1).astype(np.int32)
    assert res[N] == rnm and rnm > 100
    assert (res[:N] == want).all()


# ---------------------------------------------------------------------------------------------------------------------------
# Optimizer::LocalBundleAdjustment
# ---------------------------------------------------------------------------------------------------------------------------
def _window(pr, role, badmp, init_id):
    """Python restatement of the window selection + flattening (Optimizer.cc:1744-1855, 1873-2091) over the mock map the binary builds:
    keyframe k has id 100 + k; its features are its edges in edge order; observation maps iterate in keyframe order."""
    nKF, nMP = len(pr["pose"]), len(pr["point"])
    ekf, emp = pr["edge_kf"], pr["edge_mp"]
    pkf = int(np.nonzero(role == 0)[0][0])
    local = [pkf] + [k for k in range(nKF) if role[k] == 1]            # role 3 (bad) neighbours are skipped
    seen, points = set(), []
    for k in local:
        for e in np.nonzero(ekf == k)[0]:
            p = int(emp[e])
            if not badmp[p] and p not in seen:
                seen.add(p); points.append(p)
    fixed, inl = [], set(local)
    for p in points:
        for e in sorted(np.nonzero(emp == p)[0], key=lambda e: ekf[e]):
            k = int(ekf[e])
            if k not in inl and k not in fixed:
                if role[k] != 3:
                    fixed.append(k)
                else:
                    inl.add(k)       # marked mnBAFixedForKF but bad: never added, never revisited
    fixed = [k for k in fixed if role[k] != 3]
    order = local + fixed
    kidx = {k: i for i, k in enumerate(order)}
    fl = dict(kf=order, n_local=len(local), points=points, edges=[])
    for pi, p in enumerate(points):
        for e in sorted(np.nonzero(emp == p)[0], key=lambda e: ekf[e]):
            if role[ekf[e]] != 3:
                fl["edges"].append((int(e), kidx[int(ekf[e])], pi))
    fl["fixed_flags"] = np.array([1 if (i >= len(local) or 100 + k == init_id) else 0 for i, k in enumerate(order)], np.uint8)
    fl["n_fixed"] = len(fixed) + (1 if any(100 + k == init_id for k in local) else 0)
    return fl


def _norm_pose32(p):
    q = p[:, :4].astype(np.float32)
    n = np.sqrt((q[:, 0] * q[:, 0] + q[:, 1] * q[:, 1] + q[:, 2] * q[:, 2] + q[:, 3] * q[:, 3]).astype(np.float32)).astype(np.float32)
    return np.concatenate([(q / n[:, None]).astype(np.float32), p[:, 4:].astype(np.float32)], 1)


@pytest.mark.parametrize("case", ["plain", "init_kf_in_window", "inertial_lambda", "stop_flag"])
def test_local_bundle_adjustment_member(tmp_path, case):
    d = str(tmp_path)
    l, r, _ = synth.stereo_pair(W, H, seed=9)
    l.tofile(os.path.join(d, "left.u8")); r.tofile(os.path.join(d, "right.u8"))
    pr = synth.lba_problem(n_kf=12, n_fixed=3, n_mp=500, seed=31)
    nKF, nMP = len(pr["pose"]), len(pr["point"])
    rng = np.random.default_rng(2)
    role = np.array([2] * 3 + [0] + [1] * (nKF - 4), np.int32)      # keyframe 3 runs the BA; 4.. are its covisible neighbours; 0-2 only observe
    role[nKF - 1] = 3                                               # one covisible neighbour has been culled (isBad)
    badmp = (rng.random(nMP) < 0.03).astype(np.uint8)
    init_id = 100 + 5 if case == "init_kf_in_window" else 0
    pose32 = pr["pose"].astype(np.float32)
    for name, a in [("lba_pose.f32", pose32), ("lba_role.i32", role), ("lba_point.f32", pr["point"].astype(np.float32)),
                    ("lba_edge_kf.i32", pr["edge_kf"]), ("lba_edge_mp.i32", pr["edge_mp"]), ("lba_obs.f32", pr["obs"].astype(np.float32)),
                    ("lba_inv_sigma2.f32", pr["inv_sigma2"].astype(np.float32)), ("lba_badmp.u8", badmp)]:
        np.ascontiguousarray(a).tofile(os.path.join(d, name))
    meta = dict(W=W, H=H, nfeatures=NF, fx=FX, fy=FY, cx=CX, cy=CY, bf=BF, b=B, lba_nkf=nKF, lba_nmp=nMP, lba_init_kf_id=init_id,
                lba_inertial=1 if case == "inertial_lambda" else 0, lba_stop=1 if case == "stop_flag" else 0)
    out = _run(d, meta)
    fl = _window(pr, role, badmp, init_id)
    cnt = out("out_lba_counters.i32", np.int32)
    pose_out = out("out_lba_pose.f32", np.float32).reshape(nKF, 7)
    pt_out = out("out_lba_point.f32", np.float32).reshape(nMP, 3)
    alive = out("out_lba_alive.i32", np.int32)
    updates = out("out_lba_updates.i32", np.int32)
    n_local = fl["n_local"]
    assert cnt[0] == fl["n_fixed"] and cnt[1] == n_local and cnt[2] == len(fl["edges"])
    in_pose = _norm_pose32(pr["pose"])
    if case == "stop_flag":                                       # :2093-2095: nothing solved, nothing written
        assert cnt[3] == 0 and (cnt[6:] == 0).all() and (updates == 0).all() and (alive == 3).all()
        assert np.abs(pose_out - in_pose).max() < 1e-6
        return
    assert cnt[3] == 1 and cnt[4] == n_local and cnt[5] == len(fl["kf"]) - n_local
    sets = cnt[6:6 + nKF]
    assert all(sets[k] == (1 if k in fl["kf"][:n_local] else 0) for k in range(nKF))      # SetPose on the local keyframes only
    assert all(updates[p] == (1 if p in fl["points"] else 0) for p in range(nMP))          # SetWorldPos + UpdateNormalAndDepth
    # the oracle on the flattened problem (inputs rounded to float32 like the map's members)
    E = fl["edges"]
    eidx = np.array([e for e, _, _ in E])
    o = po.lba(in_pose[fl["kf"]].astype(np.float64), fl["fixed_flags"], pr["point"].astype(np.float32)[fl["points"]].astype(np.float64),
               np.array([k for _, k, _ in E], np.int32), np.array([p for _, _, p in E], np.int32), pr["obs"].astype(np.float32)[eidx].astype(np.float64),
               pr["inv_sigma2"].astype(np.float32)[eidx].astype(np.float64), pr["cam5"], 100.0 if case == "inertial_lambda" else 0.0, 10)
    assert o["iterations"] >= 3
    for i, k in enumerate(fl["kf"][:n_local]):
        want = o["pose"][i]
        got = pose_out[k].astype(np.float64)
        if np.dot(want[:4], got[:4]) < 0:
            got[:4] = -got[:4]
        assert np.abs(got - want).max() < 1e-4, (k, got, want)
    for k in fl["kf"][n_local:]:
        assert np.abs(pose_out[k] - in_pose[k]).max() < 1e-6                                  # fixed cameras are not written
    assert np.abs(pt_out[fl["points"]] - o["point"]).max() < 1e-3                             # metres, float32 map points 2-15 m away
    others = [p for p in range(nMP) if p not in fl["points"]]
    assert (pt_out[others] == pr["point"].astype(np.float32)[others]).all()
    # outliers (:2107-2150): chi2 above the 95 % quantile of its edge type or a point behind the camera -> both links erased
    mono = pr["obs"][eidx, 2] < 0
    thr = np.where(mono, 5.991, 7.815)
    erase = (o["edge_chi2"] > thr) | (o["edge_depth_pos"] == 0)
    clear = np.abs(o["edge_chi2"] - thr) > 1e-3 * thr                                        # away from the threshold: rounding cannot flip it
    want_alive = np.where(erase, 0, 3)
    assert (alive[eidx][clear] == want_alive[clear]).all() and erase.sum() > 5
    untouched = np.setdiff1d(np.arange(len(alive)), eidx)
    assert (alive[untouched] == 3).all()
