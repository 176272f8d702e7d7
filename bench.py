#!/usr/bin/env python3
"""bench.py -- tracking-thread frames/s on synthetic 640x480 stereo, 1200 features (BASELINE.json metric).

One "step" = BPS batches of B synthetic stereo frames (default 16 x 64 = 1024 frames per GPU) through the tracking-thread hot
path: both eyes through ORBextractor, Frame::ComputeStereoMatches, ORBmatcher::SearchByProjection(cur, last) (motion model) and
ORBmatcher::SearchByProjection(F, local map points) (TrackLocalMap).  A step is long enough (~28 ms) for the timed region of the
default run to last > 0.5 s.

  value     frames resident in HBM, every batch one CUDA-graph replay, NH handles / streams in flight, CUDA events
  e2e       host buffers in, host buffers out through orbr_submit / orbr_collect (H2D of the images and query arrays, D2H of
            keypoints / descriptors / mvuRight / mvDepth / matches inside the timed region), ONE host thread, 5 repeats
  latency   B = 1: one stereo frame per step (graph replay, device-resident; and end to end through orbr_*), p50 / p99
  parity    the first frames of the run against the CPU oracle, before anything is timed (the run aborts on a mismatch)

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 3|5] [--dump-outputs DIR]

N > 1 is launched by torchrun (one rank per GPU); frames shard across ranks with no data-path collective (weak scaling).  The
`config5` section (1280x720 stereo, 2000 features, one sequence per rank) adds the one exchange the design has: the NCCL
all-gather of new-keyframe state.  --impl reference times the CPU oracle (test infrastructure; `oracle/_ref` holds the
reference's own ORBextractor.cc, the rest of the reference needs OpenCV / Eigen / g2o and cannot be built here) on the host cores.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "tracking-thread frames/sec (640x480 stereo, 1200 feat)"
UNIT = "frames/s"
CONFIGS = {
    3: dict(W=640, H=480, NFEAT=1200, B=64, cam=(435.2, 435.2, 320.0, 240.0, 47.9, 0.11),
            name="config 3: stereo 640x480, 1200 features per eye"),
    5: dict(W=1280, H=720, NFEAT=2000, B=16, cam=(870.4, 870.4, 640.0, 360.0, 95.8, 0.11),
            name="config 5: stereo 1280x720, 2000 features per eye, one sequence per GPU"),
}
TH_LAST, TH_LOCAL = 15.0, 3.0


def config_dict(cid, B, bps):
    """The workload description BOTH arms print (identical strings => same_config)."""
    c = CONFIGS[cid]
    return {"workload": f"{c['name']}; per frame: ORBextractor L+R, ComputeStereoMatches, SearchByProjection(cur,last,th={TH_LAST:g}), "
                        f"SearchByProjection(F,local map points,th={TH_LOCAL:g})",
            "frames_per_step_per_gpu": B * bps, "frames_per_batch": B, "batches_per_step": bps,
            "image": f"{c['W']}x{c['H']} u8", "features": c["NFEAT"], "levels": 8, "scale_factor": 1.2}


# algorithmic bytes per IMAGE (SURVEY.md 8d): read each input once, write each output once
def issue_table(stage_ms, nimg, sm_mhz, counts):
    """Second roofline of the extractor stages: executed warp instructions per clock per SM (counts from the committed ncu captures,
    stage times and SM clock of THIS run) against the 4 per clock an SM can issue -- and against the 2.0 at which the multiply /
    byte-permute instructions these kernels are made of issue (profiles/r02_idp_rate.txt).  Pure function: unit-tested on the CPU."""
    out = {}
    scale = nimg / float(counts["images_per_launch"])
    for k, n in counts["warp_instructions_per_launch"].items():
        ms = stage_ms.get(k)
        if not ms or not sm_mhz:
            continue
        ipc = n * scale / (ms * 1e-3 * sm_mhz * 1e6 * counts["n_sms"])
        out[k] = {"warp_inst_per_clk_per_sm": ipc, "frac_of_issue_peak_4": ipc / 4.0}
    return {"stages": out, "peak_warp_inst_per_clk_per_sm": 4.0, "half_rate_pipe": 2.0,
            "note": "IMAD / IDP / PRMT / SHF / VIMNMX3 issue at 2.0 per clock per SM, IADD3 and two-input packed min / max at 3.9 (measured)",
            "source": counts.get("source")}


def algorithmic_bytes(n_kp, n_cand, level_px):
    p_all = sum(level_px)
    pyramid = (p_all - level_px[-1]) + (p_all - level_px[0])
    fast = p_all + 12 * n_cand
    blur = 2 * p_all
    angle = n_kp * 749 + 4 * n_kp
    desc = n_kp * 512 + n_kp * 60
    tree = 12 * n_cand + 28 * n_kp
    return {"pyramid": pyramid, "fast": fast, "quadtree": tree, "blur": blur, "orient_desc": angle + desc}


def make_pairs(n_pairs, W, H, base=8, sigma=1.5, nrect=60):
    """n_pairs distinct stereo pairs: `base` generated pairs + cheap deterministic variants."""
    from orb_slam3_detailed_comments_b200 import synth
    gen = [synth.stereo_pair(W, H, seed=100 + i, sigma=sigma, nrect=nrect)[:2] for i in range(min(base, n_pairs))]
    out = np.empty((n_pairs, 2, H, W), np.uint8)
    for i in range(n_pairs):
        l, r = gen[i % len(gen)]
        k = i // len(gen)
        if k % 4 == 1:
            l, r = 255 - l, 255 - r
        elif k % 4 == 2:
            l, r = l[::-1], r[::-1]
        elif k % 4 == 3:
            l, r = 255 - l[::-1], 255 - r[::-1]
        sh = (k // 4) * 7
        out[i, 0] = np.roll(l, sh, axis=0)
        out[i, 1] = np.roll(r, sh, axis=0)
    return out


def local_map_queries(k, d, z, rng, cam, W, H):
    """Local-map query set of one frame (SearchLocalPoints shape): one map point per feature of the frame (its own
    descriptor, projection jittered by 1.5 px, stereo coordinate from its depth or 5 m) plus as many unrelated points
    (random positions, random descriptors) -- roughly the matched / unmatched mix of a real local map."""
    fx, fy, cx, cy, bf, _ = cam
    n = len(k)
    jit = rng.normal(0, 1.5, (n, 2)).astype(np.float32)
    zz = np.where(z > 0, z, 5.0).astype(np.float32)
    x = np.concatenate([k["x"] + jit[:, 0], rng.uniform(20, W - 20, n)]).astype(np.float32)
    y = np.concatenate([k["y"] + jit[:, 1], rng.uniform(20, H - 20, n)]).astype(np.float32)
    zq = np.concatenate([zz, rng.uniform(2, 15, n)]).astype(np.float32)
    lvl = np.concatenate([k["octave"], rng.integers(0, 8, n)]).astype(np.int32)
    vc = rng.uniform(0.99, 1.0, 2 * n).astype(np.float32)
    desc = np.concatenate([d, rng.integers(0, 256, (n, 32), dtype=np.uint8)])
    # world position of every map point, in the frame's own camera frame (the synthetic map is anchored there): the matched
    # half sits where the feature was triangulated, so its projection differs from the query's by the 1.5 px jitter
    xs = np.concatenate([k["x"], x[n:]]).astype(np.float32)
    ys = np.concatenate([k["y"], y[n:]]).astype(np.float32)
    xw = np.stack([(xs - cx) * zq / fx, (ys - cy) * zq / fy, zq], 1).astype(np.float32)
    return x, y, (x - np.float32(bf) / zq).astype(np.float32), lvl, vc, desc, xw


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    def __init__(self, gpu):
        self.rows, self.proc, self.gpu = [], None, gpu

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def wait_first(self, timeout=5.0):
        t0 = time.time()
        while not self.rows and time.time() - t0 < timeout:
            time.sleep(0.01)

    def stop(self, t_begin=None, t_end=None):
        if self.proc:
            self.proc.terminate()
        sm, mx, reasons = [], [], set()
        rows = [r for (t, r) in self.rows if (t_begin is None or t >= t_begin) and (t_end is None or t <= t_end + 0.05)]
        if not rows:
            rows = [r for (_, r) in self.rows][-3:]
        for r in rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------------------------
# CPU oracle (test infrastructure): the checker of the in-run parity assertion, the cpu_baseline leg and the reference arm
# ------------------------------------------------------------------------------------------------------------------------------
def oracle_frame(l, r, eL, eR, cam, W, H, pool2=None, queries=None, with_pose_opt=False):
    """One stereo frame through the CPU oracle: both eyes through the extractor (on two threads like Frame.cc:136-141 when pool2 is
    given), ComputeStereoMatches, then the two projection searches.  queries = (last dict, local dict) of host arrays for this frame
    (the GPU arm's own query set: parity check); None builds them from the frame's own stereo points (same shape as the GPU arm).
    Returns dict(kL, dL, kR, dR, uR, dep, fm, mt)."""
    from oracle import pyoracle as po
    FX, FY, CX, CY, BF, BL = cam
    bounds = np.array([0, W, 0, H], np.float32)
    cam6 = np.array([FX, FY, CX, CY, BF, BL], np.float32)
    T = np.array([0, 0, 0, 1, 0.002, 0.001, 0], np.float32)
    if pool2 is not None:
        fr = pool2.submit(eR, r)
        _, kL, dL = eL(l)
        _, kR, dR = fr.result()
    else:
        _, kL, dL = eL(l)
        _, kR, dR = eR(r)
    uR, dep, _ = po.stereo_matches(eL, eR, kL, dL, kR, dR, BF, BL)
    out = dict(kL=kL, dL=dL, kR=kR, dR=dR, uR=uR, dep=dep, fm=None, mt=None)
    sf = eL.scale_factors
    isg = (1.0 / (sf * sf)).astype(np.float32)
    cam5 = np.float32([FX, FY, CX, CY, BF])

    def pose_opt(feat, xw):        # Optimizer::PoseOptimization over the features that hold a map point (feature order)
        obs = np.stack([kL["x"][feat], kL["y"][feat], uR[feat]], 1)
        return po.pose_optimization(T, xw, obs, isg[kL["octave"][feat]], cam5)
    if queries is None:
        sel = np.nonzero(dep > 0)[0]
        if len(sel) == 0:
            return out
        z = dep[sel]
        pts = np.stack([(kL["x"][sel] - CX) * z / FX, (kL["y"][sel] - CY) * z / FY, z], 1).astype(np.float32)
        ql = dict(xw=pts, oct=kL["octave"][sel], ang=kL["angle"][sel], desc=dL[sel], obs=np.ones(len(sel), np.uint8), Tcw=T, dir=0)
        x, y, xr, lvl, vc, dq, xwl = local_map_queries(kL, dL, dep, np.random.default_rng(7), cam, W, H)
        qc = dict(px=x, py=y, pxr=xr, lvl=lvl, vc=vc, desc=dq, xw=xwl)
    else:
        ql, qc = queries
    fm, _ = po.search_last(kL, dL, uR, bounds, sf, cam6, np.asarray(ql["Tcw"], np.float32), int(ql["dir"]), ql["xw"], ql["oct"], ql["ang"], ql["desc"],
                           ql["obs"], TH_LAST, True)
    out["fm"] = fm
    if with_pose_opt:
        feat = np.nonzero(fm >= 0)[0]
        pose_opt(feat, ql["xw"][fm[feat]])
    mt, _ = po.search_local(kL, dL, uR, bounds, sf, qc["px"], qc["py"], qc["pxr"], qc["lvl"], qc["vc"], qc["desc"], TH_LOCAL, 0.8)
    out["mt"] = mt
    if with_pose_opt:
        qs = np.nonzero(mt >= 0)[0]
        order = np.argsort(mt[qs], kind="stable")
        pose_opt(mt[qs][order], qc["xw"][qs][order])
    return out


def reference_frame(l, r, eL, eR, cam, W, H, pool2=None):
    """One stereo frame through the REFERENCE'S OWN SOURCE as far as it compiles here (oracle/_ref): the unmodified ORBextractor.cc for both
    eyes, then Frame::ComputeStereoMatches and the two ORBmatcher::SearchByProjection overloads cut out of the reference and compiled
    verbatim over skeleton classes.  Same work and the same synthetic query sets as oracle_frame(queries=None)."""
    from oracle import pyoracle as po
    FX, FY, CX, CY, BF, BL = cam
    bounds = np.array([0, W, 0, H], np.float32)
    cam6 = np.array([FX, FY, CX, CY, BF, BL], np.float32)
    T = np.array([0, 0, 0, 1, 0.002, 0.001, 0], np.float32)
    if pool2 is not None:
        fr = pool2.submit(eR, r)
        _, kL, dL = eL(l)
        _, kR, dR = fr.result()
    else:
        _, kL, dL = eL(l)
        _, kR, dR = eR(r)
    F = po.RefFrame(kL, dL, None, bounds, eL.scale_factors, cam6, T)
    uR, dep = F.stereo_matches(eL, eR, kR, dR)               # writes mvuRight / mvDepth of the frame the searches then read
    sel = np.nonzero(dep > 0)[0]
    if len(sel) == 0:
        return 0
    z = dep[sel]
    pts = np.stack([(kL["x"][sel] - CX) * z / FX, (kL["y"][sel] - CY) * z / FY, z], 1).astype(np.float32)
    fm, n1, _ = F.search_last(T, T, pts, kL["octave"][sel], kL["angle"][sel], dL[sel], np.ones(len(sel), np.uint8), TH_LAST, True)
    x, y, xr, lvl, vc, dq, _ = local_map_queries(kL, dL, dep, np.random.default_rng(7), cam, W, H)
    mt, n2 = F.search_local(x, y, xr, lvl, vc, dq, TH_LOCAL, 0.8)
    return n1 + n2


def reference_source_available():
    try:
        from oracle import pyoracle as po
        po.ref_lib()
        po.ref2_lib()
        return True
    except Exception:
        return False


def cpu_reference_frames(pairs, threads, cid=3):
    """cpu_oracle_frames with reference_frame: `pairs` stereo frames through oracle/_ref on `threads` host threads.  (frames/s, seconds)"""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import pyoracle as po
    c = CONFIGS[cid]
    nthr = max(1, threads)
    nworkers = max(1, nthr // 2)
    exs = [(po.RefExtractor(c["NFEAT"], 1.2, 8, 20, 7), po.RefExtractor(c["NFEAT"], 1.2, 8, 20, 7)) for _ in range(nworkers)]
    pools2 = [ThreadPoolExecutor(1) if nthr >= 2 else None for _ in range(nworkers)]
    t0 = time.perf_counter()
    chunks = [[(pairs[i, 0], pairs[i, 1], exs[wk][0], exs[wk][1], pools2[wk]) for i in range(wk, len(pairs), nworkers)] for wk in range(nworkers)]
    run = lambda a: reference_frame(a[0], a[1], a[2], a[3], c["cam"], c["W"], c["H"], a[4])
    if nworkers == 1:
        for a in chunks[0]:
            run(a)
    else:
        with ThreadPoolExecutor(nworkers) as pool:
            list(pool.map(lambda ch: [run(a) for a in ch], chunks))
    dt = time.perf_counter() - t0
    for p2 in pools2:
        if p2 is not None:
            p2.shutdown()
    return len(pairs) / dt, dt


def cpu_oracle_frames(pairs, threads, cid=3, with_pose_opt=False):
    """`pairs` stereo frames through the CPU oracle on `threads` host threads (two per frame: the eyes run in parallel like
    Frame.cc:136-141).  Returns (frames/s, seconds)."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import pyoracle as po
    c = CONFIGS[cid]
    nthr = max(1, threads)
    nworkers = max(1, nthr // 2)
    exs = [(po.OracleExtractor(c["NFEAT"], 1.2, 8, 20, 7), po.OracleExtractor(c["NFEAT"], 1.2, 8, 20, 7)) for _ in range(nworkers)]
    pools2 = [ThreadPoolExecutor(1) if nthr >= 2 else None for _ in range(nworkers)]
    t0 = time.perf_counter()
    chunks = [[(pairs[i, 0], pairs[i, 1], exs[wk][0], exs[wk][1], pools2[wk]) for i in range(wk, len(pairs), nworkers)]
              for wk in range(nworkers)]
    run = lambda a: oracle_frame(a[0], a[1], a[2], a[3], c["cam"], c["W"], c["H"], a[4], None, with_pose_opt)
    if nworkers == 1:
        for a in chunks[0]:
            run(a)
    else:
        with ThreadPoolExecutor(nworkers) as pool:
            list(pool.map(lambda ch: [run(a) for a in ch], chunks))
    dt = time.perf_counter() - t0
    for p2 in pools2:
        if p2 is not None:
            p2.shutdown()
    return len(pairs) / dt, dt


def _straw_man_guard(pair, cid=3):
    """BASELINE.md section 3: the oracle's OpenCV-equivalent stages are scalar restatements; cv2 (one thread) runs the same stages with
    SIMD.  Times both on one image of the workload and returns the factor by which a frame of the CPU arm gets cheaper when every
    such stage is charged at min(oracle, cv2): ratio = frame_ms_with_cv2_stages / frame_ms_oracle (<= 1).
    cv2's FAST is charged as ONE whole-level detect at iniThFAST per pyramid level -- a lower bound on what the reference does
    (577 per-cell cv::FAST calls over windows that overlap by 6 px, empty cells again at minThFAST; ORBextractor.cc:1098-1166)."""
    try:
        import cv2
    except ImportError:
        return None
    from oracle import pyoracle as po
    cv2.setNumThreads(1)
    nf = CONFIGS[cid]["NFEAT"]
    img = np.ascontiguousarray(pair[0])
    ex, ex2 = po.OracleExtractor(nf, 1.2, 8, 20, 7), po.OracleExtractor(nf, 1.2, 8, 20, 7)

    def best(f, n=5):
        f()
        ts = []
        for _ in range(n):
            t0 = time.perf_counter()
            f()
            ts.append(time.perf_counter() - t0)
        return 1e3 * min(ts)
    t_img = best(lambda: ex(img), 3)
    stage = {k: 1e3 * v for k, v in ex.timings().items()}
    img_r = np.ascontiguousarray(pair[1])
    t_img_r = best(lambda: ex2(img_r), 3)
    sizes = [ex.level_size(l) for l in range(8)]

    def pyr():
        lv = [img]
        for l in range(1, 8):
            lv.append(cv2.resize(lv[-1], sizes[l], interpolation=cv2.INTER_LINEAR))
        for x in lv:
            cv2.copyMakeBorder(x, 19, 19, 19, 19, cv2.BORDER_REFLECT_101)
        return lv
    lv = pyr()
    fd = cv2.FastFeatureDetector_create(20, True)
    cv = {"pyramid": best(pyr), "fast": best(lambda: [fd.detect(x) for x in lv]),
          "blur": best(lambda: [cv2.GaussianBlur(x, (7, 7), 2, 2, borderType=cv2.BORDER_REFLECT_101) for x in lv])}
    delta = sum(max(0.0, stage[k] - cv[k]) for k in cv)
    # the rest of a frame (ComputeStereoMatches + both searches), isolated and single-threaded: one whole frame minus two extractions
    one = np.ascontiguousarray(pair)[None]
    cpu_oracle_frames(one, 1, cid)
    t_frame_seq = 1e3 * min(cpu_oracle_frames(one, 1, cid)[1] for _ in range(3))
    t_rest = max(0.0, t_frame_seq - t_img - t_img_r)
    t_eye = max(t_img, t_img_r)                                          # the two eyes run in parallel (Frame.cc:136-141)
    f_or, f_cv = t_eye + t_rest, max(t_eye - delta, 0.0) + t_rest
    return {"oracle_stage_ms_per_image": stage, "cv2_stage_ms_per_image": cv, "image_ms_oracle": t_img, "rest_of_frame_ms_oracle": t_rest, "delta_ms_per_image": delta,
            "frame_ms_oracle": f_or, "frame_ms_with_cv2_stages": f_cv, "ratio": f_cv / f_or if f_or > 0 else 1.0,
            "note": "value = oracle-measured frames/s / ratio; cv2 4.x single-threaded; FAST charged as one whole-level detect per level"}


def straw_man_guard(pair, cid=3):
    try:
        return _straw_man_guard(pair, cid)
    except Exception as exc:      # the guard must never cost the bench line
        return {"error": repr(exc), "ratio": 1.0}


def run_reference(args, rank, world):
    """Reference arm: the CPU oracle with every host thread on the GPU arm's workload.  A step of the workload is
    frames_per_step frames; the arm times a bounded SAMPLE of each step (sized in the warm-up for ~2 s of CPU work) and reports the
    step time scaled to the whole step -- frames/s is the measured rate either way."""
    if rank != 0:
        return
    cid = args.config
    c = CONFIGS[cid]
    B, bps = args.batch or c["B"], args.batches_per_step
    fps_step = B * bps
    cores = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
    unit = max(cores // 2, 1)                                  # frames in flight: two threads per frame
    pool = make_pairs(min(fps_step, max(4 * unit, 64)), c["W"], c["H"], base=4)
    rate, _ = cpu_oracle_frames(pool[:unit * 2], cores, cid)   # calibration (also page-in / thread-pool warm-up)
    n_s = int(min(fps_step, max(unit, round(rate * 2.0 / unit) * unit)))
    idx = lambda s: np.arange(s * n_s, (s + 1) * n_s) % len(pool)
    for s in range(args.warmup):
        cpu_oracle_frames(pool[idx(s)], cores, cid)
    t0 = time.perf_counter()
    frames = 0
    for s in range(args.steps):
        cpu_oracle_frames(pool[idx(args.warmup + s)], cores, cid)
        frames += n_s
    dt = time.perf_counter() - t0
    v_oracle = frames / dt
    guard = straw_man_guard(pool[0], cid)
    v_port = v_oracle / guard["ratio"] if guard else v_oracle
    # the same sample through the reference's own source as far as it compiles here (oracle/_ref); the arm reports the FASTER of the two
    ref_src = None
    if reference_source_available():
        cpu_reference_frames(pool[:unit * 2], cores, cid)                       # page-in
        t0 = time.perf_counter()
        fr = 0
        for s in range(args.steps):
            cpu_reference_frames(pool[idx(args.warmup + s)], cores, cid)
            fr += n_s
        dtr = time.perf_counter() - t0
        ref_src = {"value": fr / dtr, "seconds": dtr, "frames": fr,
                   "what": "the reference's unmodified ORBextractor.cc (over the cv2-pinned pixel models) + Frame::ComputeStereoMatches and both "
                           "ORBmatcher::SearchByProjection overloads cut out of the reference and compiled verbatim (oracle/_ref)"}
    use_ref = ref_src is not None and ref_src["value"] > v_port
    v = ref_src["value"] if use_ref else v_port
    line = {"metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * fps_step / v, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic", "impl": "reference",
            "config": config_dict(cid, B, bps),
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "reference" if use_ref else "port",
                             "sample": f"{n_s} of the step's {fps_step} stereo frames per step on {cores} threads ({dt:.1f} s for {args.steps} steps); "
                                       "ms_per_step is that rate scaled to the whole step",
                             "value_oracle_only": v_oracle, "straw_man_guard": guard, "value_port_with_guard": v_port, "reference_source": ref_src,
                             "note": "two CPU implementations are timed on the same sample and the FASTER one is the arm's value: the oracle port "
                                     "(oracle/, SIMD FAST, charged at cv2's stage times where cv2 is faster: straw_man_guard) and the reference's own "
                                     "source as far as it compiles in this image (oracle/_ref).  g2o / the rest of the reference need OpenCV / Eigen "
                                     "and cannot be built here"},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------------------------------
class Workload:
    """Handles, input pool (> L2), per-batch query sets, captured graphs and host staging of one configuration on one GPU."""

    def __init__(self, cid, B, NH, local, rank, sigma=1.5, nrect=60, pool_bytes=140e6):
        import torch
        from orb_slam3_detailed_comments_b200 import ORBextractor, ORBmatcher, camera
        self.torch = torch
        c = CONFIGS[cid]
        self.cid, self.c, self.B, self.NH, self.local = cid, c, B, NH, local
        self.W, self.H, self.NF = c["W"], c["H"], c["NFEAT"]
        self.cam_t = c["cam"]
        FX, FY, CX, CY, BF, BL = c["cam"]
        self.nimg = 2 * B
        self.dev = torch.device("cuda", local)
        self.cam = camera(FX, FY, CX, CY, BF, BL, self.W, self.H)
        mk = lambda: ORBextractor(self.NF, 1.2, 8, 20, 7, max_width=self.W, max_height=self.H, max_batch=self.nimg, device=local)
        self.exs = [mk() for _ in range(NH)]
        self.ex = self.exs[0]
        self.streams = [torch.cuda.ExternalStream(e.cuda_stream(), device=self.dev) for e in self.exs]
        self.m_last, self.m_local = ORBmatcher(0.9, True), ORBmatcher(0.8, True)
        # input pool larger than L2 (126 MB), cycled through the timed steps
        self.pool_batches = max(2, int(np.ceil(pool_bytes / (self.nimg * self.W * self.H))))
        self.pairs = make_pairs(B * self.pool_batches, self.W, self.H, base=8, sigma=sigma, nrect=nrect)
        self.host_pool = torch.from_numpy(self.pairs.reshape(self.pool_batches, self.nimg, self.H, self.W)).pin_memory()
        self.dev_pool = self.host_pool.cuda(non_blocking=False)
        self._build_queries(rank)
        self.graphs = {}

    def _build_queries(self, rank):
        """Map state for the matchers, one query set per pool batch: the "last frame" of every sequence is the frame itself one
        step earlier (its stereo points, unprojected), the local map holds one map point per feature plus as many unrelated points."""
        torch, ex, B, nimg = self.torch, self.ex, self.B, self.nimg
        FX, FY, CX, CY, BF, BL = self.cam_t
        rng = np.random.default_rng(1234 + rank)
        T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(self.dev)
        cat = lambda xs, dt: np.concatenate(xs).astype(dt) if len(xs) else np.zeros(0, dt)
        pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()
        self.H_LAST, self.H_LOC, self.D_LAST, self.D_LOC, self.P_LAST, self.P_LOC, self.P_CHAIN = [], [], [], [], [], [], []
        sfac = ex.GetScaleFactors()
        for pb in range(self.pool_batches):
            ex.extract_batch_device(self.dev_pool[pb].data_ptr(), nimg, self.W, self.H)
            ex.stereo_batch(B, BF, BL)
            n0, _, off0, kps0, desc0 = ex.download(nimg)
            uR0, dep0 = ex.stereo_download(int(off0[-1]))
            q_last = dict(off=[0], xw=[], oct=[], ang=[], desc=[], obs=[])
            q_loc = dict(off=[0], px=[], py=[], pxr=[], lvl=[], vc=[], desc=[], xw=[])
            q_ch = dict(off=[0], xw=[], normal=[], max_dist=[], min_dist=[], desc=[], last_query=[])
            for p in range(B):
                a, b = int(off0[2 * p]), int(off0[2 * p + 1])
                k, d, z = kps0[a:b], desc0[a:b], dep0[a:b]
                sel = np.nonzero(z > 0)[0]
                pts = np.stack([(k["x"][sel] - CX) * z[sel] / FX, (k["y"][sel] - CY) * z[sel] / FY, z[sel]], 1).astype(np.float32)
                q_last["xw"].append(pts); q_last["oct"].append(k["octave"][sel].astype(np.int32))
                q_last["ang"].append(k["angle"][sel].astype(np.float32)); q_last["desc"].append(d[sel])
                q_last["obs"].append(np.ones(len(sel), np.uint8)); q_last["off"].append(q_last["off"][-1] + len(sel))
                x, y, xr, lvl, vc, dq, xwl = local_map_queries(k, d, z, rng, self.cam_t, self.W, self.H)
                q_loc["px"].append(x); q_loc["py"].append(y); q_loc["pxr"].append(xr); q_loc["lvl"].append(lvl)
                q_loc["vc"].append(vc); q_loc["desc"].append(dq); q_loc["xw"].append(xwl)
                q_loc["off"].append(q_loc["off"][-1] + len(x))
                # chained flow (orbr_chain): the local map = the LastFrame map points themselves + one point per remaining feature + as many
                # unrelated ones, as world positions with normals and distance ranges (the device projects them with the optimised pose)
                nl = len(sel)
                lq = np.full(len(xwl), -1, np.int32)
                lq[sel] = np.arange(nl, dtype=np.int32)
                octs = np.concatenate([k["octave"], rng.integers(0, 8, len(k))])
                dist = np.linalg.norm(xwl, axis=1).astype(np.float32)
                maxd = (dist * sfac[octs]).astype(np.float32)
                q_ch["xw"].append(xwl); q_ch["normal"].append((xwl / np.maximum(dist[:, None], 1e-6)).astype(np.float32)); q_ch["max_dist"].append(maxd)
                q_ch["min_dist"].append((maxd / sfac[7]).astype(np.float32)); q_ch["desc"].append(dq); q_ch["last_query"].append(lq)
                q_ch["off"].append(q_ch["off"][-1] + len(xwl))
            h_last = dict(fimg=np.arange(0, nimg, 2, dtype=np.int32), off=np.array(q_last["off"], np.int32),
                          Tcw=np.tile(np.array([0, 0, 0, 1, 0.002, 0.001, 0], np.float32), (B, 1)), dir=np.zeros(B, np.int32),
                          xw=cat(q_last["xw"], np.float32).reshape(-1, 3), oct=cat(q_last["oct"], np.int32), ang=cat(q_last["ang"], np.float32),
                          desc=cat(q_last["desc"], np.uint8).reshape(-1, 32), obs=cat(q_last["obs"], np.uint8))
            h_loc = dict(fimg=h_last["fimg"], off=np.array(q_loc["off"], np.int32), px=cat(q_loc["px"], np.float32),
                         py=cat(q_loc["py"], np.float32), pxr=cat(q_loc["pxr"], np.float32), lvl=cat(q_loc["lvl"], np.int32),
                         vc=cat(q_loc["vc"], np.float32), desc=cat(q_loc["desc"], np.uint8).reshape(-1, 32), xw=cat(q_loc["xw"], np.float32).reshape(-1, 3))
            self.H_LAST.append(h_last); self.H_LOC.append(h_loc)
            self.D_LAST.append({k: T(v) for k, v in h_last.items()}); self.D_LOC.append({k: T(v) for k, v in h_loc.items()})
            self.P_LAST.append({k: pin(v) for k, v in h_last.items()}); self.P_LOC.append({k: pin(v) for k, v in h_loc.items()})
            self.P_CHAIN.append(dict(off=pin(np.array(q_ch["off"], np.int32)), xw=pin(cat(q_ch["xw"], np.float32).reshape(-1, 3)),
                                     normal=pin(cat(q_ch["normal"], np.float32).reshape(-1, 3)), max_dist=pin(cat(q_ch["max_dist"], np.float32)),
                                     min_dist=pin(cat(q_ch["min_dist"], np.float32)), desc=pin(cat(q_ch["desc"], np.uint8).reshape(-1, 32)),
                                     last_query=pin(cat(q_ch["last_query"], np.int32))))
        dev, NH = self.dev, self.NH
        self.rows_cap = nimg * (self.ex._L.orbx_max_features(self.ex._h))
        self.max_last = max(int(h["off"][-1]) for h in self.H_LAST)
        self.max_loc = max(int(h["off"][-1]) for h in self.H_LOC)
        self.maxq_frame = max(max(int(np.diff(h["off"]).max()) for h in self.H_LAST), max(int(np.diff(h["off"]).max()) for h in self.H_LOC))
        self.nq_last = float(np.mean([int(h["off"][-1]) for h in self.H_LAST]))
        self.nq_loc = float(np.mean([int(h["off"][-1]) for h in self.H_LOC]))
        self.d_fm = [torch.full((self.rows_cap,), -1, dtype=torch.int32, device=dev) for _ in range(NH)]
        self.d_nm = [torch.zeros(2 * B, dtype=torch.int32, device=dev) for _ in range(NH)]
        self.d_match = [torch.full((max(self.max_loc, 1),), -1, dtype=torch.int32, device=dev) for _ in range(NH)]
        zi = lambda n, dt: torch.zeros(n, dtype=dt, device=dev)
        rc = self.rows_cap
        self.d_po = [dict(off=zi(B + 1, torch.int32), feat=zi(rc, torch.int32), xw=zi((rc, 3), torch.float32), obs=zi((rc, 3), torch.float32),
                          w=zi(rc, torch.float32), pose=zi((2, B, 7), torch.float64), out=zi(rc, torch.uint8), inl=zi((2, B), torch.int32))
                     for _ in range(NH)]
        for e in self.exs:      # sync-free device-pointer searches (capturable)
            e.set_device_query_bounds(max(self.max_last, self.max_loc, 1), max(self.maxq_frame, 1), rc)

    # ---- device-resident step ----
    def step_device(self, i, with_po=False, k=None, pb=None):
        from orb_slam3_detailed_comments_b200 import PoseOptimizationDevice, PoseEdgesDevice
        k, pb, B = i % self.NH if k is None else k, i % self.pool_batches if pb is None else pb, self.B
        e = self.exs[k]
        FX, FY, CX, CY, BF, BL = self.cam_t
        d_last, d_loc = self.D_LAST[pb], self.D_LOC[pb]
        e.extract_batch_device(self.dev_pool[pb].data_ptr(), self.nimg, self.W, self.H)
        e.stereo_batch(B, BF, BL)
        self.m_last.SearchByProjectionLastFrameDevice(e, self.cam, B, d_last["fimg"], d_last["off"], d_last["Tcw"], d_last["dir"],
                                                      d_last["xw"], d_last["oct"], d_last["ang"], d_last["desc"], d_last["obs"],
                                                      TH_LAST, self.d_fm[k], self.d_nm[k][:B])
        po_ = self.d_po[k]
        CAM5 = [FX, FY, CX, CY, BF]
        if with_po:
            PoseEdgesDevice(e, B, d_last["fimg"], d_last["xw"], po_["off"], po_["feat"], po_["xw"], po_["obs"], po_["w"], feature_match=self.d_fm[k])
            PoseOptimizationDevice(e, B, po_["off"], d_last["Tcw"], po_["xw"], po_["obs"], po_["w"], CAM5, po_["pose"][0], po_["out"], po_["inl"][0])
        self.m_local.SearchByProjectionDevice(e, self.cam, B, d_loc["fimg"], d_loc["off"], d_loc["px"], d_loc["py"], d_loc["pxr"],
                                              d_loc["lvl"], d_loc["vc"], d_loc["desc"], self.d_match[k], self.d_nm[k][B:], th=TH_LOCAL)
        if with_po:
            PoseEdgesDevice(e, B, d_loc["fimg"], d_loc["xw"], po_["off"], po_["feat"], po_["xw"], po_["obs"], po_["w"],
                            query_offset=d_loc["off"], query_match=self.d_match[k])
            PoseOptimizationDevice(e, B, po_["off"], d_last["Tcw"], po_["xw"], po_["obs"], po_["w"], CAM5, po_["pose"][1], po_["out"], po_["inl"][1])

    def launch(self, i, with_po=False, use_graph=True):
        """Batch i on handle i % NH: one CUDA-graph replay (captured on first use, after one eager run sized the scratch)."""
        if not use_graph:
            return self.step_device(i, with_po)
        k, pb = i % self.NH, i % self.pool_batches
        key = (k, pb, with_po)
        g = self.graphs.get(key)
        if g is None:
            self.step_device(i, with_po)
            self.torch.cuda.synchronize()
            g = self.exs[k].graph_capture(lambda: self.step_device(i, with_po))
            self.graphs[key] = g
        self.exs[k].graph_launch(g)

    def timed_device_loop(self, first, count, with_po, barrier, use_graph=True):
        """count batches starting at batch index `first`, round-robin over the handles' streams; returns device milliseconds
        (events on stream 0, the other streams fork from / join into it)."""
        torch, streams = self.torch, self.streams
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(streams[0])
        for st in streams[1:]:
            st.wait_event(e0)
        for i in range(count):
            self.launch(first + i, with_po, use_graph)
        for st in streams[1:]:
            ev = torch.cuda.Event()
            ev.record(st)
            streams[0].wait_event(ev)
        e1.record(streams[0])
        barrier()
        return e0.elapsed_time(e1)

    # ---- end to end: host buffers through orbr_submit / orbr_collect, one host thread, NH handles in flight ----
    def e2e_setup(self):
        from orb_slam3_detailed_comments_b200.replay import TrackingStep
        from orb_slam3_detailed_comments_b200._native import KP_DTYPE
        torch, B, rc = self.torch, self.B, self.rows_cap
        FX, FY, CX, CY, BF, BL = self.cam_t
        pz = lambda shape, dt: torch.zeros(shape, dtype=dt).pin_memory().numpy()
        self.steps_e2e = [TrackingStep(e, self.cam, BF, BL, TH_LAST, TH_LOCAL, 0.8, True) for e in self.exs]
        self.OUT = [dict(kps=torch.zeros(rc * 28, dtype=torch.uint8).pin_memory().numpy().view(KP_DTYPE), desc=pz((rc, 32), torch.uint8),
                         ur=pz(rc, torch.float32), dep=pz(rc, torch.float32), n=pz(self.nimg, torch.int32), offsets=pz(self.nimg + 1, torch.int32),
                         fm=pz(rc, torch.int32), nm1=pz(B, torch.int32), mt=pz(max(self.max_loc, 1), torch.int32), nm2=pz(B, torch.int32),
                         pose=pz((2, B, 7), torch.float64), inl=pz((2, B), torch.int32), eoff=pz((2, B + 1), torch.int32),
                         efeat=pz((2, rc), torch.int32), outl=pz((2, rc), torch.uint8)) for _ in range(self.NH)]

    def e2e_submit(self, i, with_po=False):
        k, pb = i % self.NH, i % self.pool_batches
        pl, pc = self.P_LAST[pb], self.P_LOC[pb]
        if with_po == "chain":       # the chained flow: the local map as world points, projected on the device with the optimised pose
            self.steps_e2e[k].submit(self.host_pool[pb].numpy(), last=pl, pose=pl["Tcw"], chain=self.P_CHAIN[pb])
            return
        self.steps_e2e[k].submit(self.host_pool[pb].numpy(), last=pl, local=pc, pose=pl["Tcw"] if with_po else None,
                                 local_world_pos=pc["xw"] if with_po else None)

    def e2e_collect(self, i, with_po=False):
        k = i % self.NH
        o = self.OUT[k]
        if not with_po:
            o = {kk: v for kk, v in o.items() if kk not in ("pose", "inl", "eoff", "efeat", "outl")}
        rows = self.steps_e2e[k].collect(o)
        nq = int(self.H_LOC[i % self.pool_batches]["off"][-1])
        d2h = rows * (28 + 32 + 4 + 4 + 4) + 4 * (2 * self.nimg + 1) + 4 * nq + 8 * self.B
        if with_po:
            d2h += 2 * self.B * (56 + 4) + int(self.OUT[k]["eoff"][0][-1] + self.OUT[k]["eoff"][1][-1]) * 5 + 8 * (self.B + 1)
        return rows, d2h

    def e2e_loop(self, first, count, with_po=False):
        """count batches, one host thread: batch i + NH - 1 is submitted before batch i is collected.  Returns (seconds, D2H bytes)."""
        NH = self.NH
        self.torch.cuda.synchronize()
        t0 = time.perf_counter()
        d2h = 0
        for j in range(min(NH - 1, count)):
            self.e2e_submit(first + j, with_po)
        for i in range(count):
            if i + NH - 1 < count:
                self.e2e_submit(first + i + NH - 1, with_po)
            d2h += self.e2e_collect(first + i, with_po)[1]
        dt = time.perf_counter() - t0
        return dt, d2h

    def chain_stats(self):
        """what the last chained batch on handle 0 produced (sanity numbers for the bench line)"""
        o = self.OUT[0]
        return {"local_matches_per_frame": float(o["nm2"].mean()), "motion_model_matches_per_frame": float(o["nm1"].mean()),
                "inliers_after_motion_model": float(o["inl"][0].mean()), "inliers_after_local_map": float(o["inl"][1].mean()),
                "local_map_points_per_frame": float(self.P_CHAIN[0]["off"][-1]) / self.B}

    def h2d_bytes_per_batch(self, with_po=False):
        skip = () if with_po else ("xw",)
        n = self.nimg * self.W * self.H + sum(v.nbytes for v in self.H_LAST[0].values())
        n += sum(v.nbytes for k, v in self.H_LOC[0].items() if k not in skip)
        return n + (28 * self.B if with_po else 0)

    # ---- parity: the first frames of the run against the CPU oracle (outside every timed region) ----
    def parity_check(self, n_frames=2):
        """Frames 0 .. n_frames-1 of pool batch 0 through the END-TO-END path (orbr_submit / orbr_collect, the same call the e2e leg
        times) against the CPU oracle on the same images and the same query sets: keypoint records, descriptor bytes, mvuRight /
        mvDepth float bits and both match arrays must be identical."""
        from oracle import pyoracle as po
        self.e2e_submit(0)
        rows, _ = self.e2e_collect(0)
        o = self.OUT[0]
        off = o["offsets"]
        hl, hc = self.H_LAST[0], self.H_LOC[0]
        eL, eR = po.OracleExtractor(self.NF, 1.2, 8, 20, 7), po.OracleExtractor(self.NF, 1.2, 8, 20, 7)
        checked = dict(frames=n_frames, keypoints=0, last_queries=0, local_queries=0)
        for p in range(n_frames):
            a, b, c2 = int(off[2 * p]), int(off[2 * p + 1]), int(off[2 * p + 2])
            l0, l1, c0, c1 = int(hl["off"][p]), int(hl["off"][p + 1]), int(hc["off"][p]), int(hc["off"][p + 1])
            ql = dict(xw=hl["xw"][l0:l1], oct=hl["oct"][l0:l1], ang=hl["ang"][l0:l1], desc=hl["desc"][l0:l1], obs=hl["obs"][l0:l1], Tcw=hl["Tcw"][p], dir=hl["dir"][p])
            qc = dict(px=hc["px"][c0:c1], py=hc["py"][c0:c1], pxr=hc["pxr"][c0:c1], lvl=hc["lvl"][c0:c1], vc=hc["vc"][c0:c1], desc=hc["desc"][c0:c1])
            want = oracle_frame(self.pairs[p, 0], self.pairs[p, 1], eL, eR, self.cam_t, self.W, self.H, None, (ql, qc))
            got_fm = o["fm"][a:b].copy()
            got_fm[got_fm >= 0] -= l0          # query index inside the frame's own list
            pairs_ = [("left keypoints", o["kps"][a:b].view(np.uint8), want["kL"].view(np.uint8)), ("left descriptors", o["desc"][a:b], want["dL"]),
                      ("right keypoints", o["kps"][b:c2].view(np.uint8), want["kR"].view(np.uint8)), ("right descriptors", o["desc"][b:c2], want["dR"]),
                      ("mvuRight", o["ur"][a:b].view(np.uint32), want["uR"].view(np.uint32)), ("mvDepth", o["dep"][a:b].view(np.uint32), want["dep"].view(np.uint32)),
                      ("SearchByProjection(cur,last)", got_fm, want["fm"]), ("SearchByProjection(F,local)", o["mt"][c0:c1], want["mt"])]
            for name, g_, w_ in pairs_:
                if g_.shape != w_.shape or not (g_ == w_).all():
                    raise SystemExit(f"PARITY FAILURE (frame {p}, {name}): the GPU path differs from the CPU oracle -- no number is reported")
            checked["keypoints"] += (b - a) + (c2 - b)
            checked["last_queries"] += l1 - l0
            checked["local_queries"] += c1 - c0
        return {"ok": True, "against": "CPU oracle (oracle/), same images and query sets, through orbr_submit / orbr_collect", **checked,
                "compared": "keypoint records (28 B), descriptors, mvuRight / mvDepth float bits, both match arrays: identical"}

    def dump_batch(self, i, out_dir, budget=64 << 20):
        """Writes what batch i returned to its caller as out_dir/<name>.npy, read back from the handle that ran it -- valid until that
        handle runs another batch.  Stereo pairs p = 0, 1, ... are kept while the files fit in `budget` bytes.  All float32 but
        image_offsets (float64); integers are exact in both.
          keypoints (rows, 7)         x, y, size, angle, response, octave, class_id of every keypoint, images L0 R0 L1 R1 ...
          image_offsets (2P + 1)      first row of each image in keypoints / descriptors
          descriptors (rows, 32)      descriptor bytes, one row per keypoint
          uright_left, depth_left     mvuRight / mvDepth, one per LEFT-image keypoint (left images' rows in pair order; -1: none)
          last_frame_match_left       one per left-image keypoint: the matched query of SearchByProjection(cur, last), as an index
                                      into the batch's whole last-frame query list (pair p's queries follow pair p-1's); -1: none
          local_map_match             one per local-map query (the batch's list, pairs in order): the matched keypoint of
                                      SearchByProjection(F, local points), as an index into that pair's left image; -1: none
          matches_per_frame (P, 2)    matches of the last-frame and of the local-map search per stereo pair"""
        self.torch.cuda.synchronize()
        k, pb, B = i % self.NH, i % self.pool_batches, self.B
        e = self.exs[k]
        _, _, off, kps, desc = e.download(self.nimg)
        uR, dep = e.stereo_download(int(off[-1]))
        fm, nm, mt = self.d_fm[k].cpu().numpy(), self.d_nm[k].cpu().numpy(), self.d_match[k].cpu().numpy()
        loff = self.H_LOC[pb]["off"]
        n_pairs, used = 0, 0
        while n_pairs < B:
            rows, left = int(off[2 * n_pairs + 2] - off[2 * n_pairs]), int(off[2 * n_pairs + 1] - off[2 * n_pairs])
            need = rows * (7 + 32) * 4 + left * 3 * 4 + int(loff[n_pairs + 1] - loff[n_pairs]) * 4 + 2 * 4 + 2 * 8
            if used + need > budget - (1 << 16):
                break
            used += need
            n_pairs += 1
        if n_pairs == 0:
            raise SystemExit(f"--dump-outputs: one stereo pair of batch {i} does not fit in {budget} bytes")
        rows, left = int(off[2 * n_pairs]), np.concatenate([np.arange(off[2 * p], off[2 * p + 1]) for p in range(n_pairs)]).astype(np.int64)
        kp = kps[:rows]
        out = {"keypoints": np.stack([kp["x"], kp["y"], kp["size"], kp["angle"], kp["response"], kp["octave"], kp["class_id"]], 1).astype(np.float32),
               "image_offsets": off[:2 * n_pairs + 1].astype(np.float64), "descriptors": desc[:rows].astype(np.float32),
               "uright_left": uR[left].astype(np.float32), "depth_left": dep[left].astype(np.float32),
               "last_frame_match_left": fm[left].astype(np.float32), "local_map_match": mt[:int(loff[n_pairs])].astype(np.float32),
               "matches_per_frame": np.stack([nm[:n_pairs], nm[B:B + n_pairs]], 1).astype(np.float32)}
        os.makedirs(out_dir, exist_ok=True)
        for name, a in out.items():
            np.save(os.path.join(out_dir, name + ".npy"), a)
        return {"dir": out_dir, "batch": i, "stereo_pairs": n_pairs, "of": B, "bytes": int(sum(a.nbytes for a in out.values())),
                "sample": "the last batch of the last timed step (one of --batches-per-step batches), first stereo_pairs pairs"}

    def close(self):
        for (k, _, _), g in self.graphs.items():
            self.exs[k].graph_destroy(g)
        self.graphs = {}
        for e in self.exs:
            e.close()


def percentile_ms(xs):
    a = np.sort(np.asarray(xs, np.float64))
    return {"p50_ms": float(np.percentile(a, 50)), "p99_ms": float(np.percentile(a, 99)), "min_ms": float(a[0]), "max_ms": float(a[-1]), "n": int(len(a))}


def latency_section(wl_cfg, local, n_iter):
    """B = 1: one stereo frame per step on a 2-image handle.  Device-resident: one CUDA-graph replay per frame, CUDA events around
    every replay.  End to end: orbr_submit + orbr_collect per frame (images and queries from pinned host memory, every result back),
    host clock around the pair of calls."""
    import torch
    w1 = Workload(wl_cfg, 1, 1, local, 0, pool_bytes=8 * 2 * CONFIGS[wl_cfg]["W"] * CONFIGS[wl_cfg]["H"])
    out = {}
    for with_po in (False, True):
        for i in range(2 * w1.pool_batches):     # captures the graph of every pool batch before anything is timed
            w1.launch(i, with_po)
        torch.cuda.synchronize()
        ts = []
        st = w1.streams[0]
        for i in range(n_iter):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            w1.launch(i, with_po)      # one handle; the pool batch cycles
            e1.record(st)
            e1.synchronize()
            ts.append(e0.elapsed_time(e1))
        key = "with_pose_optimization" if with_po else "headline_step"
        out[key] = {"graph_replay_device_resident": percentile_ms(ts),
                    "kernels_per_frame": w1.exs[0].graph_kernels(w1.graphs[(0, 0, with_po)])}
    w1.e2e_setup()
    for with_po in (False, True):
        for i in range(5):
            w1.e2e_submit(i, with_po); w1.e2e_collect(i, with_po)
        ts = []
        for i in range(n_iter):
            t0 = time.perf_counter()
            w1.e2e_submit(i, with_po)
            w1.e2e_collect(i, with_po)
            ts.append(1e3 * (time.perf_counter() - t0))
        out["with_pose_optimization" if with_po else "headline_step"]["e2e_host_buffers"] = percentile_ms(ts)
    out["workload"] = "one stereo frame per step (2 images), same per-frame work as the headline step; ~%d last-frame and ~%d local-map queries" % (
        int(w1.nq_last), int(w1.nq_loc))
    w1.close()
    return out


def config5_section(args, local, rank, world, barrier):
    """BASELINE.json config 5: 1280x720 stereo, 2000 features, one sequence per GPU, with the design's one exchange: every
    `kf_every` batches each rank inserts a keyframe and all ranks all-gather its state (pose, keypoints, mvuRight, descriptors; one
    fixed-capacity block per rank, packed on the device by orbx_pack_keyframe_device) with ONE all_gather_into_tensor over NCCL on a
    side stream, overlapping the next batches.  Reports frames/s with and without the exchange and the collective's own time."""
    import torch
    import torch.distributed as dist
    c = CONFIGS[5]
    B, NH = c["B"], max(2, args.handles)
    w5 = Workload(5, B, NH, local, rank, pool_bytes=70e6)
    nb = max(8 * NH, 48)
    for i in range(2 * NH * w5.pool_batches):       # every (handle, pool batch) graph is captured here
        w5.launch(i)
    ms_plain = w5.timed_device_loop(0, nb, False, barrier)
    res = {"workload": config_dict(5, B, nb), "batches": nb, "frames_per_batch": B}
    t = torch.tensor([ms_plain], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    res["frames_per_s_no_exchange"] = world * B * nb / (float(t.item()) * 1e-3)
    blk = w5.ex.keyframe_block_bytes()
    blk = (blk + 255) // 256 * 256
    kf_every = 4
    mine = [torch.zeros(blk, dtype=torch.uint8, device=w5.dev) for _ in range(NH)]
    gathered = [torch.zeros(world * blk, dtype=torch.uint8, device=w5.dev) for _ in range(NH)]
    pose = torch.tensor([0, 0, 0, 1, 0.1 * rank, 0, 0], dtype=torch.float32, device=w5.dev)
    comm = torch.cuda.Stream(device=w5.dev)

    def exchange(i):
        k = i % NH
        w5.exs[k].pack_keyframe_device(0, pose, mine[k])           # on the handle's stream, after the batch's kernels
        ev = torch.cuda.Event()
        ev.record(w5.streams[k])
        comm.wait_event(ev)
        with torch.cuda.stream(comm):
            if world > 1:
                dist.all_gather_into_tensor(gathered[k], mine[k])
            else:
                gathered[k].copy_(mine[k])
        ev2 = torch.cuda.Event()
        ev2.record(comm)
        w5.streams[k].wait_event(ev2)                               # the handle's next batch may overwrite mine[k] only after the gather read it

    def loop_with_exchange():
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(w5.streams[0])
        for st in w5.streams[1:]:
            st.wait_event(e0)
        comm.wait_event(e0)
        nkf = 0
        for i in range(nb):
            w5.launch(i)
            if i % kf_every == kf_every - 1:
                exchange(i)
                nkf += 1
        for st in list(w5.streams[1:]) + [comm]:
            ev = torch.cuda.Event()
            ev.record(st)
            w5.streams[0].wait_event(ev)
        e1.record(w5.streams[0])
        barrier()
        return e0.elapsed_time(e1), nkf
    loop_with_exchange()
    ms_x, nkf = loop_with_exchange()
    t = torch.tensor([ms_x], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    res["frames_per_s_with_exchange"] = world * B * nb / (float(t.item()) * 1e-3)
    # the collective alone: pack + all-gather, back to back on the comm stream
    reps = 50
    for _ in range(5):
        exchange(0)
    torch.cuda.synchronize()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(w5.streams[0])
    for _ in range(reps):
        exchange(0)
    e1.record(w5.streams[0])
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / reps], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    # check: every rank's block arrives intact (first words: n and the pose the rank packed)
    g = gathered[0].cpu().numpy()
    ok = True
    for r in range(world):
        b = g[r * blk:(r + 1) * blk]
        n = int(b[:4].view(np.int32)[0])
        ok = ok and 0 < n <= 5000 and abs(float(b[4:32].view(np.float32)[4]) - 0.1 * r) < 1e-6
    res.update({"keyframe_exchange": {"every_batches": kf_every, "keyframes_per_rank": nkf, "block_bytes_per_rank": int(blk),
                                      "collective": "one torch.distributed all_gather_into_tensor (NCCL) of fixed-capacity device blocks on a side stream" if world > 1
                                                    else "single rank: device copy (no peer)",
                                      "us_per_keyframe_pack_plus_gather": 1e3 * float(t.item()), "blocks_intact": bool(ok)}})
    w5.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", type=int, default=3, choices=[3, 5])
    ap.add_argument("--batch", type=int, default=0, help="stereo frames per batch per GPU (default: 64 for config 3, 16 for config 5)")
    ap.add_argument("--batches-per-step", type=int, default=16)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--extract-only", action="store_true", help="headline step only: skip the latency / config 5 / LBA / inertial / knn / PoseOptimization sections")
    ap.add_argument("--handles", type=int, default=4, help="extractor handles (CUDA streams) the batches are pipelined over")
    ap.add_argument("--no-graph", action="store_true", help="eager launches instead of CUDA-graph replays in the value leg")
    ap.add_argument("--e2e-repeats", type=int, default=5)
    ap.add_argument("--latency-frames", type=int, default=200)
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last batch of the last step returned (a "
                    "one-batch sample of the step: keypoints, descriptors, mvuRight, mvDepth, both match arrays) as DIR/<name>.npy, "
                    "to compare two builds on the same seeded inputs (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from orb_slam3_detailed_comments_b200 import _native
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() in ("VERSION", "WARN"):
            os.environ["NCCL_DEBUG"] = "NONE"       # NCCL prints its version banner on stdout from VERSION up: rank 0 prints ONE JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    cid = args.config
    c = CONFIGS[cid]
    B, BPS, NH = args.batch or c["B"], args.batches_per_step, max(2, args.handles)
    W, H, NFEAT = c["W"], c["H"], c["NFEAT"]
    use_graph = not args.no_graph
    wl = Workload(cid, B, NH, local, rank)
    ex, nimg = wl.ex, wl.nimg

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_ranks(x):
        t = torch.tensor([x], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- parity gate (rank 0; every rank runs the same code on the same kind of data) ----
    wl.e2e_setup()
    parity = wl.parity_check(2) if rank == 0 else None

    # ---- value: inputs resident in HBM; every batch one graph replay, NH handles in flight ----
    sampler = ClockSampler(local)
    sampler.start()
    nwarm = max(args.warmup, 1) * BPS
    for i in range(max(nwarm, wl.NH * wl.pool_batches)):       # also captures every (handle, pool batch) graph
        wl.launch(i, False, use_graph)
    barrier()
    sampler.wait_first()
    launches0 = _native.lib().orb_kernel_launches()
    t_begin = time.time()
    ms = wl.timed_device_loop(nwarm, args.steps * BPS, False, barrier, use_graph)
    t_end = time.time()
    clocks = sampler.stop(t_begin, t_end)
    launches = _native.lib().orb_kernel_launches() - launches0
    ms_max = max_ranks(ms)
    value = world * B * BPS * args.steps / (ms_max * 1e-3)
    nm_host = wl.d_nm[0].cpu().numpy()
    dumped = wl.dump_batch(nwarm + args.steps * BPS - 1, args.dump_outputs) if args.dump_outputs and rank == 0 else None
    kernels_per_batch = wl.exs[0].graph_kernels(wl.graphs[(0, 0, False)]) if use_graph else launches // (args.steps * BPS)

    # ---- per-stage times for the roofline: a serial (un-overlapped, eager) pass over the same batches, CUDA events per stage ----
    def serial_profile(w):
        w.ex.set_profiling(True)
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        nser = 16
        torch.cuda.synchronize()
        s0.record(w.streams[0])
        for i in range(nser):
            w.step_device(i, False, k=0, pb=i % w.pool_batches)      # handle 0 is the profiled one; the pool batch cycles
        s1.record(w.streams[0])
        torch.cuda.synchronize()
        serial = s0.elapsed_time(s1) / nser
        st = w.ex.last_timings()
        w.ex.set_profiling(False)
        n, _, _ = w.ex.counts(w.nimg)
        n_cand = float(np.mean([sum(len(w.ex.candidates(b, l)) for l in range(8)) for b in range(2)]))
        return serial, st, float(n.mean()), n_cand
    serial_ms, stage_ms, n_kp, n_cand = serial_profile(wl)

    # ---- e2e: host buffers through orbr_submit / orbr_collect, H2D + D2H inside the timed region, one host thread ----
    wl.e2e_loop(0, max(2 * NH, BPS))        # warm-up (sizes the replay buffers)
    barrier()
    reps, d2h_tot = [], 0
    for r in range(max(1, args.e2e_repeats)):
        barrier()
        dt, d2h_tot = wl.e2e_loop(nwarm + r, args.steps * BPS)
        reps.append(max_ranks(dt))
    e2e_rates = [world * B * BPS * args.steps / t for t in reps]
    e2e_value = float(np.median(e2e_rates))
    # the same steps with PoseOptimization after each search (SURVEY 8f N1): resident and end to end
    in_step = None
    if not args.extract_only:
        n_po = max(NH, (args.steps * BPS) // 4)
        for i in range(wl.NH * wl.pool_batches):
            wl.launch(i, True, use_graph)
        ms_po = max_ranks(wl.timed_device_loop(0, n_po, True, barrier, use_graph))
        wl.e2e_loop(0, 2 * NH, True)
        barrier()
        dt_po = max_ranks(wl.e2e_loop(NH, n_po, True)[0])
        in_step = {"batches": n_po, "value_frames_per_s": world * B * n_po / (ms_po * 1e-3), "e2e_frames_per_s": world * B * n_po / dt_po,
                   "note": "the headline step plus PoseOptimization after each search (device correspondence walk + optimiser in the same graph; "
                           "pose_optimization = 1 in orbr_submit for the e2e leg)"}

    # ---- the chained per-frame data flow (orbr_chain): pose -> isInFrustum -> search -> PoseOptimization on the device, end to end ----
    chained = None
    if not args.extract_only:
        try:
            n_ch = max(NH, (args.steps * BPS) // 4)
            wl.e2e_loop(0, 2 * NH, "chain")
            barrier()
            dt_ch = max_ranks(wl.e2e_loop(NH, n_ch, "chain")[0])
            chained = {"batches": n_ch, "e2e_frames_per_s": world * B * n_ch / dt_ch, **wl.chain_stats(),
                       "note": "TrackWithMotionModel + TrackLocalMap as one device flow per batch (Tracking.cc:3389-3522, 4010-4062): motion-model search, "
                               "PoseOptimization, outlier release, Sophus::SE3f, isInFrustum of the local map, local-map search against the remaining "
                               "claims, PoseOptimization over every map point of the frame; host buffers in and out (orbr_submit with orbr_chain)"}
        except Exception as exc:
            chained = {"error": repr(exc)}

    # ---- a real-texture-like input (SURVEY 2.1 K2: 5-10 k FAST candidates per image) beside the corner-rich default ----
    natural = None
    if not args.extract_only and cid == 3:
        try:
            wn = Workload(cid, B, 2, local, rank, sigma=3.5, nrect=40)
            for i in range(wn.NH * wn.pool_batches):
                wn.launch(i)
            nb_n = max(4 * BPS, 32)
            ms_n = max_ranks(wn.timed_device_loop(0, nb_n, False, barrier))
            ser_n, st_n, kp_n, cand_n = serial_profile(wn)
            natural = dict(w=wn, ms=ms_n, nb=nb_n, serial=ser_n, stage=st_n, n_kp=kp_n, n_cand=cand_n)
        except Exception as exc:
            natural = {"error": repr(exc)}

    cfg5 = None
    if not args.extract_only and cid == 3:
        try:
            cfg5 = config5_section(args, local, rank, world, barrier)
        except Exception as exc:
            cfg5 = {"error": repr(exc)}

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        level_px = [ex.level_size(l)[0] * ex.level_size(l)[1] for l in range(8)]

        def stage_table(stage, serial, n_kp_, n_cand_):
            ab = algorithmic_bytes(n_kp_, n_cand_, level_px)
            ext = {k: stage[k] for k in ["pyramid", "fast", "quadtree", "blur", "orient_desc"]}
            stages = dict(ext)
            stages["stereo+search"] = max(serial - stage["total"], 0.0)
            stages["serial_step_total"] = serial
            gbs = {k: ab[k] * nimg / (ext[k] * 1e-3) / 1e9 for k in ext}
            fr = ab["fast"] + ab["blur"] + ab["orient_desc"]
            fr_ms = ext["fast"] + ext["blur"] + ext["orient_desc"]
            return ab, ext, stages, gbs, {"achieved": fr * nimg / (fr_ms * 1e-3) / 1e9, "frac": fr * nimg / (fr_ms * 1e-3) / 1e9 / peak, "ms": fr_ms}
        ab, ext, stages, gbs, frb = stage_table(stage_ms, serial_ms, n_kp, n_cand)
        top = max(ext, key=ext.get)
        achieved = ab[top] * nimg / (ext[top] * 1e-3) / 1e9
        traffic, tsrc = None, None      # DRAM bytes per launch of the dominant kernel from the committed ncu --set full capture
        for fn in ("r02_fast_traffic.json", "r01_fast_traffic.json"):
            try:
                tr = json.load(open(os.path.join(ROOT, "profiles", fn)))
            except Exception:
                continue
            if top == "fast":
                traffic = (tr["dram_bytes_read"] + tr["dram_bytes_write"]) * nimg / tr["images_per_launch"]
                tsrc = f"profiles/{fn} (ncu --set full, bytes per launch scaled to {nimg} images)"
            break
        roofline = {"bound": "hbm", "kernel": top, "achieved": achieved, "peak": peak, "unit": "GB/s",
                    "frac": achieved / peak, "traffic": traffic,
                    "peak_source": "MEASURED_PEAKS.json (of measured)" if peaks else "fallback 6650 GB/s (of fallback)",
                    "stage_ms_per_batch": stages, "stage_gbs": gbs, "algorithmic_bytes_per_image": ab,
                    "fast_blur_orient_describe": frb, "traffic_source": tsrc,
                    "images_per_launch": nimg, "fast_candidates_per_image": n_cand,
                    "note": "stage times from a serial eager pass (one stream) right after the timed region; the timed region itself replays "
                            "one graph per batch on the handles' streams.  FAST is bound by integer issue and shared-memory latency (profiles/), "
                            "not by HBM; see DESIGN.md"}
        try:        # the integer-pipe roofline (see issue_table); never allowed to break the line
            cnt = json.load(open(os.path.join(ROOT, "profiles", "r02_inst_counts.json")))
            roofline["integer_issue"] = issue_table(ext, nimg, (clocks or {}).get("sm_mhz"), cnt)
        except Exception:
            roofline["integer_issue"] = None
        if isinstance(natural, dict) and "w" in natural:
            abn, extn, stn, gbn, frn = stage_table(natural["stage"], natural["serial"], natural["n_kp"], natural["n_cand"])
            roofline["real_texture_like_input"] = {
                "input": "synth.stereo_pair(sigma=3.5, nrect=40): 5-10 k FAST candidates per image (SURVEY 2.1 K2) instead of ~24 k",
                "fast_candidates_per_image": natural["n_cand"], "keypoints_per_image": natural["n_kp"],
                "value_frames_per_s": world * B * natural["nb"] / (natural["ms"] * 1e-3), "stage_ms_per_batch": stn, "stage_gbs": gbn,
                "fast": {"achieved": gbn["fast"], "frac": gbn["fast"] / peak}, "fast_blur_orient_describe": frn}
            natural["w"].close()
        elif natural is not None:
            roofline["real_texture_like_input"] = natural
        cpu = None
        if not args.no_cpu_baseline and world == 1:      # rank 0 at N = 1 only
            # faithful threading (Frame.cc:136-141): the two eyes on two threads, bounded sample
            n_cpu = min(len(wl.pairs), 96)
            cpu_oracle_frames(wl.pairs[:2], 2, cid)     # warm-up (page-in, thread pools)
            v_oracle, secs = cpu_oracle_frames(wl.pairs[:n_cpu], 2, cid)
            guard = straw_man_guard(wl.pairs[0], cid)
            v = v_oracle / guard["ratio"] if guard else v_oracle
            cpu = {"value": v, "unit": UNIT, "cores": 2, "kind": "port",
                   "sample": f"{n_cpu} stereo frames (extraction + stereo matching + both projection searches), "
                             f"L/R eyes on 2 threads (Frame.cc:136-141), {secs:.1f} s",
                   "value_oracle_only": v_oracle, "straw_man_guard": guard}
        latency = None
        if not args.extract_only:
            try:
                latency = latency_section(cid, local, args.latency_frames)
            except Exception as exc:
                latency = {"error": repr(exc)}
        side = {} if args.extract_only else side_benchmarks(args, wl, local)
        if side.get("pose_optimization") is not None and in_step is not None and "error" not in side["pose_optimization"]:
            side["pose_optimization"]["in_step"] = in_step
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "config": config_dict(cid, B, BPS),
                "detail": {"pipeline": f"{NH} extractor handles / CUDA streams, one CUDA-graph replay per batch ({kernels_per_batch} kernels); one host thread in both legs"
                                       if use_graph else f"{NH} extractor handles / CUDA streams, eager launches",
                           "timed_region_s": ms_max * 1e-3,
                           "queries_per_frame": {"last_frame": wl.nq_last / B, "local_map": wl.nq_loc / B},
                           "matches_per_frame": {"last_frame": float(nm_host[:B].mean()), "local_map": float(nm_host[B:].mean())},
                           "l2": f"input pool of {wl.pool_batches} batches = {wl.pool_batches * nimg * W * H / 1e6:.0f} MB > 126 MB L2, "
                                 "intermediates rewritten every batch",
                           "keypoints_per_image": n_kp, "fast_candidates_per_image": n_cand,
                           "kernel_variants": {"quadtree": int(os.environ.get("ORB_QT_VARIANT", "1") != "0"),
                                               "stereo": int(os.environ.get("ORB_STEREO_VARIANT", "1") != "0"),
                                               "fast": int(os.environ.get("ORB_FAST_VARIANT", "1"))}},
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(wl.h2d_bytes_per_batch() * BPS),
                        "d2h_bytes_per_step": int(d2h_tot // args.steps),
                        "repeats_frames_per_s": e2e_rates, "spread": (max(e2e_rates) - min(e2e_rates)) / e2e_value if e2e_value else None,
                        "api": "orbr_submit / orbr_collect (pinned host buffers in and out), one host thread, median of the repeats"},
                "gpu_launches": int(launches), "graph_launches": int(args.steps * BPS) if use_graph else 0, "kernels_per_batch": int(kernels_per_batch),
                "clocks": clocks, "parity": parity, "dumped_outputs": dumped, "roofline": roofline, "cpu_baseline": cpu, "latency_b1": latency, "chained_flow": chained, "config5": cfg5, **side}
        print(json.dumps(line))
    wl.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def side_benchmarks(args, wl, local):
    """LBA (config 4), LocalInertialBA, brute-force Hamming 2-NN and PoseOptimization, each timed alone (rank 0)."""
    import torch
    from orb_slam3_detailed_comments_b200 import Optimizer, synth
    FX, FY, CX, CY, BF, BL = wl.cam_t
    B, dev, ex, streams = wl.B, wl.dev, wl.ex, wl.streams
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    # ---- local BA (config 4): 20 KF / 3000 MP, one problem and a batch of 8 -------------------------
    try:
        from oracle import pyoracle as po
        opt = Optimizer(local)
        prs = [synth.lba_problem(seed=s) for s in range(8)]
        for _ in range(2):
            opt.LocalBundleAdjustment(prs[0], lambda_init=100.0)
        opt.LocalBundleAdjustmentBatch(prs, lambda_init=100.0)      # warm-up: sizes the pinned / device workspaces
        t0 = time.perf_counter()
        for s in range(5):
            g = opt.LocalBundleAdjustment(prs[s], lambda_init=100.0)
        t_one = (time.perf_counter() - t0) / 5
        t0 = time.perf_counter()
        opt.LocalBundleAdjustmentBatch(prs, lambda_init=100.0)
        t_batch = (time.perf_counter() - t0) / 8
        t0 = time.perf_counter()
        for s in range(3):
            po.lba(prs[s]["pose"], prs[s]["fixed"], prs[s]["point"], prs[s]["edge_kf"], prs[s]["edge_mp"], prs[s]["obs"],
                   prs[s]["inv_sigma2"], prs[s]["cam5"], 100.0, 10)
        t_cpu = (time.perf_counter() - t0) / 3
        lba = {"workload": "config 4: LocalBundleAdjustment 20 KF (2 fixed) / 3000 MP / ~18k edges, lambda_init 100",
               "ms_per_solve_e2e": 1e3 * t_one, "ms_per_solve_batch8_e2e": 1e3 * t_batch, "cpu_oracle_ms": 1e3 * t_cpu,
               "cpu_cores": 1, "iterations": int(g["iterations"]), "trials": int(g.get("trials", -1)), "edges": int(len(prs[0]["edge_kf"]))}
        opt.close()
    except Exception as exc:   # never lose the headline line because the side benchmark failed
        lba = {"error": repr(exc)}
    # ---- LocalInertialBA (SURVEY 8f N2) ---------------------------------------------------------------------------
    try:
        from oracle import pyoracle as po
        from orb_slam3_detailed_comments_b200 import InertialOptimizer
        iopt = InertialOptimizer(local)
        wins = [synth.inertial_window(seed=s) for s in range(8)]
        for _ in range(2):
            iopt.LocalInertialBA(wins[0], 1.0, 10)
        iopt.LocalInertialBABatch(wins, 1.0, 10)
        t0 = time.perf_counter()
        for s in range(5):
            gi = iopt.LocalInertialBA(wins[s], 1.0, 10)
        ti_one = (time.perf_counter() - t0) / 5
        t0 = time.perf_counter()
        iopt.LocalInertialBABatch(wins, 1.0, 10)
        ti_batch = (time.perf_counter() - t0) / 8
        t0 = time.perf_counter()
        w4 = wins[4]
        ri = po.liba(w4["state"], w4["fixed"], w4["point"], w4["edge_kf"], w4["edge_mp"], w4["obs"], w4["inv_sigma2"], w4["Tcb"],
                     w4["cam5"], w4["links"].view(po.LIBA_LINK), 1.0, 10)
        ti_cpu = time.perf_counter() - t0
        liba = {"workload": "LocalInertialBA window: 10 optimisable + 4 fixed keyframes, 10 inertial links, 2000 points, "
                            f"{len(w4['edge_kf'])} edges, lambda 1e0, 10 iterations",
                "ms_per_solve_e2e": 1e3 * ti_one, "ms_per_solve_batch8_e2e": 1e3 * ti_batch, "cpu_oracle_ms": 1e3 * ti_cpu, "cpu_cores": 1,
                "iterations": int(gi["iterations"]), "oracle_iterations": int(ri["iterations"]),
                "max_abs_state_diff_vs_oracle": float(np.abs(gi["state"] - ri["state"]).max()),
                "max_abs_point_diff_vs_oracle": float(np.abs(gi["point"] - ri["point"]).max())}
        iopt.close()
    except Exception as exc:
        liba = {"error": repr(exc)}
    # ---- K9 brute-force Hamming 2-NN (BFMatcher.knnMatch of ComputeStereoFishEyeMatches) ----------------------------------
    try:
        from orb_slam3_detailed_comments_b200 import knnMatch2
        krng = np.random.default_rng(5)
        qs = [krng.integers(0, 256, (1200, 32), dtype=np.uint8) for _ in range(64)]
        ts = [krng.integers(0, 256, (1200, 32), dtype=np.uint8) for _ in range(64)]
        for _ in range(3):
            knnMatch2(ex, qs, ts)
        t0 = time.perf_counter()
        for _ in range(5):
            got = knnMatch2(ex, qs, ts)
        t_knn = (time.perf_counter() - t0) / 5
        t_cv = None
        try:
            import cv2
            cv2.setNumThreads(1)
            bfm = cv2.BFMatcher(cv2.NORM_HAMMING)
            t0 = time.perf_counter()
            ref = bfm.knnMatch(qs[0], ts[0], 2)
            t_cv = time.perf_counter() - t0
            same = all(got[0][0][i, 0] == m[0].trainIdx and got[0][0][i, 1] == m[1].trainIdx for i, m in enumerate(ref))
        except ImportError:
            same = None
        knn = {"workload": "64 pairs of 1200 x 1200 descriptors, knnMatch k = 2, host pointers", "ms_per_call_e2e": 1e3 * t_knn,
               "pairs_per_s": 64 / t_knn, "cv2_bfmatcher_ms_per_pair_1_thread": None if t_cv is None else 1e3 * t_cv,
               "first_pair_equals_cv2": same}
    except Exception as exc:
        knn = {"error": repr(exc)}
    # ---- PoseOptimization (SURVEY 8f N1, twice per frame on the tracking thread): a batch of B frames --------------
    try:
        from oracle import pyoracle as po
        from orb_slam3_detailed_comments_b200 import PoseOptimization, PoseOptimizationDevice
        prng = np.random.default_rng(99)

        def po_frame(n):
            Xc = np.stack([prng.uniform(-3, 3, n), prng.uniform(-2, 2, n), prng.uniform(2, 12, n)], 1)
            ax = prng.normal(size=3); ax /= np.linalg.norm(ax)
            q = np.concatenate([ax * np.sin(0.015), [np.cos(0.015)]]); tt = prng.normal(0, 0.05, 3)
            x, y, z, w = q
            R = np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                          [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                          [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])
            Xw = (Xc - tt) @ R
            u, v = FX * Xc[:, 0] / Xc[:, 2] + CX, FY * Xc[:, 1] / Xc[:, 2] + CY
            obs = np.stack([u, v, u - BF / Xc[:, 2]], 1) + prng.normal(0, 0.7, (n, 3))
            obs[prng.random(n) < 0.2, 2] = -1
            bad = prng.random(n) < 0.1
            obs[bad, :2] += prng.normal(0, 30, (int(bad.sum()), 2))
            return dict(pose=np.array([0, 0, 0, 1, 0, 0, 0], np.float32), world_pos=Xw.astype(np.float32), obs=obs.astype(np.float32),
                        inv_sigma2=(1 / (1.2 ** prng.integers(0, 8, n)) ** 2).astype(np.float32))
        cam5 = [FX, FY, CX, CY, BF]
        res = {}
        for tag, n_e in (("after_motion_model_550_edges", 550), ("after_local_map_1200_edges", 1200)):
            frames = [po_frame(n_e) for _ in range(B)]
            PoseOptimization(ex, frames, cam5)
            t0 = time.perf_counter()
            for _ in range(5):
                got = PoseOptimization(ex, frames, cam5)
            t_e2e = (time.perf_counter() - t0) / 5
            eoff = torch.tensor(np.arange(B + 1, dtype=np.int32) * n_e, device=dev)
            d_pose = T(np.stack([f["pose"] for f in frames])); d_xw = T(np.concatenate([f["world_pos"] for f in frames]))
            d_obs = T(np.concatenate([f["obs"] for f in frames])); d_w = T(np.concatenate([f["inv_sigma2"] for f in frames]))
            o_pose = torch.zeros((B, 7), dtype=torch.float64, device=dev); o_out = torch.zeros(B * n_e, dtype=torch.uint8, device=dev)
            o_inl = torch.zeros(B, dtype=torch.int32, device=dev)
            ea, eb2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            PoseOptimizationDevice(ex, B, eoff, d_pose, d_xw, d_obs, d_w, cam5, o_pose, o_out, o_inl)
            torch.cuda.synchronize()
            ea.record(streams[0])
            for _ in range(10):
                PoseOptimizationDevice(ex, B, eoff, d_pose, d_xw, d_obs, d_w, cam5, o_pose, o_out, o_inl)
            eb2.record(streams[0])
            torch.cuda.synchronize()
            t_dev = ea.elapsed_time(eb2) / 10
            t0 = time.perf_counter()
            for f in frames[:8]:
                po.pose_optimization(f["pose"], f["world_pos"], f["obs"], f["inv_sigma2"], np.float32(cam5))
            t_cpu = (time.perf_counter() - t0) / 8
            res[tag] = {"frames_per_call": B, "ms_per_call_device_resident": t_dev, "ms_per_call_e2e": 1e3 * t_e2e,
                        "cpu_oracle_ms_per_frame": 1e3 * t_cpu, "lm_iterations_per_frame": float(np.mean([g["iterations"] for g in got])),
                        "inliers_per_frame": float(np.mean([g["inliers"] for g in got]))}
        pose_opt = {"workload": "Optimizer::PoseOptimization, one CTA per frame, 80 % stereo / 20 % monocular edges, 10 % outliers", **res}
    except Exception as exc:
        pose_opt = {"error": repr(exc)}
    return {"lba": lba, "inertial_ba": liba, "hamming_knn": knn, "pose_optimization": pose_opt}


if __name__ == "__main__":
    main()
