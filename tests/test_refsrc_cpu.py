"""Pins the CPU oracle (oracle/*.cpp restatement) to the REFERENCE'S OWN SOURCES: oracle/_ref/librefsrc.so is
src/ORBextractor.cc, src/ORBmatcher.cc, src/Frame.cc, src/KeyFrame.cc, src/MapPoint.cc and src/Map.cc of
the reference compiled unmodified against the OpenCV / DBoW2 stand-in headers of oracle/standin/ (oracle/Makefile,
target `ref`).  Every assertion below is restatement == reference sources, bit for bit, on the same inputs.

The reference's outputs are recorded (tests/reference_outputs.py): the comparisons run everywhere against the record,
and also live where oracle/_ref/librefsrc.so exists."""
import glob
import os

import numpy as np
import pytest

from orb_slam2_ssd_semantic_b200 import synth
from orb_slam2_ssd_semantic_b200._abi import BowView, FrameView, LastView, TrackPointsView
from tests.reference_outputs import Reference

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
SF = np.cumprod(np.concatenate([[np.float32(1.0)], np.full(7, np.float32(1.2), np.float32)])).astype(np.float32)


@pytest.fixture(scope="module")
def src(oracle):
    return oracle


@pytest.fixture
def ref_out(request, oracle):
    return Reference(request.node.originalname, oracle.refsrc_available())


TABLES = ("mvScaleFactor", "mvInvScaleFactor", "mvLevelSigma2", "mvInvLevelSigma2", "mnFeaturesPerLevel", "umax")


def _extract(E, img, nlevels):
    """Scale tables, keypoints, descriptors and the pyramid (plain and bordered) of extractor E on img."""
    K, D = E(img)
    return [getattr(E, name) for name in TABLES], K, D, [(E.level(l), E.level(l, bordered=True)) for l in range(nlevels)]


def test_oracle_equals_reference_sources(src, ref_out):
    """THE pin: ORBextractor::operator() of the reference (ComputePyramid, per-cell FAST + retry, DistributeOctTree,
    IC_Angle, GaussianBlur, computeOrbDescriptor) == oracle/orb_ref.cpp on every golden image, the adversarial set,
    other geometries / parameters, and the scale tables / pyramid read-back."""
    cases = []
    for path in sorted(glob.glob(os.path.join(G, "extract_*.npz"))):
        z = np.load(path)
        cases.append((os.path.basename(path), z["image"], tuple(z["params"].tolist())))
    for name, img in synth.adversarial_frames().items():
        cases.append(("adv_" + name, img, (1000, 1.2, 8, 20, 7)))
    for t in range(3):
        cases.append(("synth%d" % t, synth.synth_frame(1234, t), (1000, 1.2, 8, 20, 7)))
    cases.append(("n2000", synth.synth_frame(1234, 3), (2000, 1.2, 8, 20, 7)))
    for shape, prm in [((240, 320), (500, 1.2, 8, 20, 7)), ((480, 752), (1200, 1.2, 8, 20, 7)),
                       ((376, 1241), (2000, 1.2, 8, 20, 7)), ((300, 300), (300, 1.5, 4, 30, 10)),
                       ((480, 640), (50, 1.2, 8, 20, 7)), ((480, 640), (1000, 1.2, 1, 20, 7))]:
        cases.append((str(shape), synth.synth_frame(77, 3, h=shape[0], w=shape[1]), prm))
    total = 0
    for tag, img, prm in cases:
        prm = (int(prm[0]), float(prm[1]), int(prm[2]), int(prm[3]), int(prm[4]))
        mine = _extract(src.RefExtractor(*prm), img, prm[2])
        ref_out.same((tag, prm), mine, lambda: _extract(src.SrcExtractor(*prm), img, prm[2]))
        total += len(mine[1])
    assert total > 15000
    # strided input (cv::Mat with step > cols)
    big = synth.synth_frame(5, 0, h=500, w=700)
    view = big[10:490, 30:670]
    K, D = src.RefExtractor(1000, 1.2, 8, 20, 7)(np.ascontiguousarray(view))
    ref_out.same("strided", (K, D), lambda: src.SrcExtractor(1000, 1.2, 8, 20, 7)(view))


def test_distribute_oct_tree_equals_reference_sources(src, ref_out):
    """DistributeOctTree alone (src/ORBextractor.cc:540-765) on random candidate sets: dense clusters, many equal-size
    nodes (the (size, pointer) ties), N above and below the candidate count, non-4:3 regions (nIni = 2, 3)."""
    rng = np.random.default_rng(11)
    n_ties = 0
    for case in range(40):
        w, h = [(602, 442), (300, 300), (1203, 338), (640, 200)][case % 4]
        n = int(rng.integers(1, 4000))
        k = np.zeros(n, src.KP_DTYPE)
        if case % 3 == 0:   # clustered
            c = rng.integers(0, [w, h], size=(8, 2))
            p = c[rng.integers(0, 8, n)] + rng.normal(0, 12, size=(n, 2))
        else:
            p = rng.uniform(0, [w, h], size=(n, 2))
        k["x"] = np.clip(np.floor(p[:, 0]), 0, w - 1)
        k["y"] = np.clip(np.floor(p[:, 1]), 0, h - 1)
        k["response"] = rng.integers(1, 40 if case % 2 else 250, n)
        k["size"] = 7
        k["angle"] = -1
        k["class_id"] = -1
        N = int(rng.integers(1, 900))
        a = src.distribute(k, 0, w, 0, h, N)
        ref_out.same(case, a, lambda: src.src_distribute(k, 0, w, 0, h, N))
        n_ties += len(a)
    assert n_ties > 5000


def _mapbin_views(z):
    fx, fy, cx, cy, bf = [float(v) for v in z["cam"]]
    cur = FrameView(z["cur_x"], z["cur_y"], z["cur_oct"], z["cur_angle"], z["cur_uright"], z["cur_desc"], z["cur_Tcw"], fx,
                    fy, cx, cy, bf, 0.0, 640.0, 0.0, 480.0, z["sf"])
    last = LastView(z["last_xw"], z["last_valid"], z["last_oct"], z["last_angle"], z["last_desc"], z["last_Tcw"],
                    mp_obs=np.ones(len(z["last_valid"]), np.int32))
    return cur, last


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(G, "match_mapbin_*.npz"))))
def test_projection_last_on_mapbin_keyframes(src, ref_out, path):
    """SearchByProjection(Frame&, const Frame&, th, bMono) of the reference on real keyframes of its map.bin."""
    z = np.load(path)
    cur, last = _mapbin_views(z)
    for th in (float(z["th"]), 7.0, 30.0):
        for mono in (False, True):
            a = src.search_by_projection_last(cur, last, th, mono, 0.9, True)
            ref_out.same((os.path.basename(path), th, mono), a,
                         lambda: src.src_search_by_projection_last(cur, last, th, mono, 0.9, True))
    assert a[0] > 100


def _random_frame(rng, n, with_obs):
    x = rng.uniform(5, 635, n).astype(np.float32)
    y = rng.uniform(5, 475, n).astype(np.float32)
    octv = rng.integers(0, 8, n).astype(np.int32)
    desc = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    z = rng.uniform(0.5, 4.0, n).astype(np.float32)
    ur = np.where(rng.random(n) < 0.7, x - synth.BF / z, -1).astype(np.float32)
    T = np.eye(4, dtype=np.float32)
    F = FrameView(x, y, octv, rng.uniform(0, 360, n).astype(np.float32), ur, desc, T, synth.FX, synth.FY, synth.CX,
                  synth.CY, synth.BF, 0, 640, 0, 480, SF)
    if with_obs:
        F.mp_obs = rng.integers(-1, 2, n).astype(np.int32)
    return F, z


def test_projection_last_random(src, ref_out):
    """Random frames: pre-existing points (Observations 0 / >0), double claims, forward / backward / lateral motion,
    mono, orientation check off, points behind the camera and outside the image."""
    rng = np.random.default_rng(5)
    tot = 0
    for case in range(24):
        n = int(rng.integers(40, 400))
        cur, z = _random_frame(rng, n, case % 3 == 0)
        T = np.eye(4, dtype=np.float32)
        T[:3, 3] = rng.normal(0, 0.02, 3)
        if case % 4 == 1:
            T[2, 3] = 0.3
        if case % 4 == 2:
            T[2, 3] = -0.3
        cur.Tcw = np.ascontiguousarray(T, np.float32).reshape(16)
        m = int(rng.integers(40, 400))
        sel = rng.integers(0, n, m)
        zz = z[sel] * rng.uniform(0.98, 1.02, m).astype(np.float32)
        if case % 5 == 0:
            zz[: m // 10] *= -1          # behind the camera
        xw = np.stack([(cur.x[sel] + rng.normal(0, 3, m) - synth.CX) * zz / synth.FX,
                       (cur.y[sel] + rng.normal(0, 3, m) - synth.CY) * zz / synth.FY, zz], 1).astype(np.float32)
        d2 = cur.desc[sel].copy()
        d2[:, :4] ^= rng.integers(0, 256, size=(m, 4), dtype=np.uint8)
        last = LastView(xw, (rng.random(m) < 0.9).astype(np.uint8), np.clip(cur.octave[sel] + rng.integers(-1, 2, m), 0, 7),
                        rng.uniform(0, 360, m).astype(np.float32), d2, np.eye(4, dtype=np.float32),
                        mp_obs=rng.integers(0, 2, m).astype(np.int32))
        chk = case % 5 != 4
        mono = case % 8 == 7
        a = src.search_by_projection_last(cur, last, 15.0, mono, 0.9, chk)
        ref_out.same(case, a, lambda: src.src_search_by_projection_last(cur, last, 15.0, mono, 0.9, chk))
        tot += a[0]
    assert tot > 800


def test_other_searches_random(src, ref_out):
    """SearchByProjection(Frame&, vector<MapPoint*>&, th), SearchByBoW(KF, F), SearchByBoW(KF, KF) and
    SearchForInitialization of the reference on random frames."""
    rng = np.random.default_rng(21)
    tot = [0, 0, 0, 0]
    for case in range(10):
        n = int(rng.integers(80, 300))
        F, z = _random_frame(rng, n, case % 2 == 0)
        m = int(rng.integers(80, 300))
        sel = rng.integers(0, n, m)
        d2 = F.desc[sel].copy()
        d2[:, :3] ^= rng.integers(0, 256, size=(m, 3), dtype=np.uint8)
        px = (F.x[sel] + rng.normal(0, 4, m)).astype(np.float32)
        py = (F.y[sel] + rng.normal(0, 4, m)).astype(np.float32)
        pts = TrackPointsView((rng.random(m) < 0.9).astype(np.uint8), px, py, (px - synth.BF / z[sel]).astype(np.float32),
                              np.clip(F.octave[sel] + rng.integers(0, 2, m), 0, 7),
                              rng.uniform(0.99, 1.0, m).astype(np.float32), d2, mp_obs=rng.integers(0, 2, m).astype(np.int32))
        for th in (1.0, 3.0):
            a = src.search_by_projection_points(F, pts, th, 0.8)
            ref_out.same(("points", case, th), a, lambda: src.src_search_by_projection_points(F, pts, th, 0.8))
            tot[0] += a[0]
        nw = int(rng.integers(4, 40))
        fv1, fv2 = {}, {}
        for i, w in enumerate(rng.integers(0, nw, n)):
            fv1.setdefault(int(w) * 3, []).append(i)
        for i, w in enumerate(rng.integers(0, nw, m)):
            fv2.setdefault(int(w) * 3 + (0 if rng.random() < 0.8 else 1), []).append(i)
        ang2 = rng.uniform(0, 360, m).astype(np.float32)
        K = BowView(F.desc, F.angle, fv1, valid=(rng.random(n) < 0.85).astype(np.uint8))
        Fr = BowView(d2, ang2, fv2)
        K2 = BowView(d2, ang2, fv2, valid=(rng.random(m) < 0.85).astype(np.uint8))
        for ori in (True, False):
            a = src.search_by_bow(K, Fr, 0.7, ori)
            ref_out.same(("bow", case, ori), a, lambda: src.src_search_by_bow(K, Fr, 0.7, ori))
            tot[1] += a[0]
            a = src.search_by_bow_kf(K, K2, 0.75, ori)
            ref_out.same(("bow_kf", case, ori), a, lambda: src.src_search_by_bow_kf(K, K2, 0.75, ori))
            tot[2] += a[0]
        # SearchForInitialization: level-0 keypoints, contested F2 keypoints (near-duplicate descriptors)
        octv = rng.integers(0, 3, n).astype(np.int32)
        mk = lambda xx, yy, dd, aa: FrameView(xx, yy, octv, aa, np.full(n, -1, np.float32), dd, np.eye(4, dtype=np.float32),
                                              synth.FX, synth.FY, synth.CX, synth.CY, synth.BF, 0, 640, 0, 480, SF)
        F1 = mk(F.x, F.y, F.desc, F.angle)
        d3 = F.desc.copy()
        d3[:, :2] ^= rng.integers(0, 256, size=(n, 2), dtype=np.uint8)
        dup = rng.integers(0, n, n // 6)
        d3[dup] = d3[(dup + 1) % n]
        F2 = mk((F.x + rng.normal(0, 6, n)).astype(np.float32), (F.y + rng.normal(0, 6, n)).astype(np.float32), d3,
                (F.angle + rng.normal(0, 4, n)).astype(np.float32) % np.float32(360))
        prev = np.stack([F.x, F.y], 1)
        for window, ori in ((100, True), (30, False)):
            a = src.search_for_initialization(F1, F2, prev, window, 0.9, ori)
            ref_out.same(("init", case, window), a, lambda: src.src_search_for_initialization(F1, F2, prev, window, 0.9, ori))
            tot[3] += a[0]
    assert min(tot) > 50, tot


def test_hamming_equals_reference_sources(src, ref_out):
    rng = np.random.default_rng(0)
    pairs = [rng.integers(0, 256, size=(2, 32), dtype=np.uint8) for _ in range(200)]
    mine = [src.hamming(a, b) for a, b in pairs]
    assert mine == [int(np.unpackbits(a ^ b).sum()) for a, b in pairs]
    ref_out.same("pairs", mine, lambda: [src.src_hamming(a, b) for a, b in pairs])


def test_rgbd_frame_constructor_equals_reference_sources(src, ref_out):
    """The reference's RGB-D Frame constructor (src/Frame.cc:176-240: ExtractORB, UndistortKeyPoints with zero
    distortion, ComputeStereoFromRGBD, AssignFeaturesToGrid) + UnprojectStereo per keypoint against the oracle's
    extractor + frame_ref_stereo_unproject, on frames with depth holes."""
    ws = synth.WallStream(seed=4, n=2)
    rng = np.random.default_rng(2)
    for t in range(2):
        gray, depth, rgb, T = ws.frame(t * 9)
        depth = depth.copy()
        depth[rng.random(depth.shape) < 0.3] = 0
        K, D = src.RefExtractor(500, 1.2, 8, 20, 7)(gray)
        ur, dp, xw, va = src.stereo_unproject(K, depth, T, synth.FX, synth.FY, synth.CX, synth.CY, synth.BF)
        assert 0.5 * len(K) < va.sum() < 0.9 * len(K)

        def ref():
            K2, D2, ur2, dp2, xw2, va2 = src.src_frame_rgbd(gray, depth, T, synth.FX, synth.FY, synth.CX, synth.CY, synth.BF,
                                                            nfeatures=500)
            return K2, D2, ur2, dp2, va2, xw2[va2 > 0]
        ref_out.same("frame %d" % t, (K, D, ur, dp, va, xw[va > 0]), ref)


def test_tracking_pipeline_equals_reference_sources(src, ref_out):
    """The CPU-baseline drivers agree: oracle/pipeline_ref.cpp (port) and refsrc_pipeline_run (the reference's own Frame
    constructor + SearchByProjection(cur, last) over a non-planar RGB-D stream) give the same keypoint and match counts
    per frame -- so `bench.py --impl reference` may time either as the same work."""
    rs = synth.RoomStream(seed=3, n=40)
    fr = [rs.frame(3 * t) for t in range(6)]
    gray, depth, T = np.stack([f[0] for f in fr]), np.stack([f[1] for f in fr]), np.stack([f[3] for f in fr])
    kw = dict(fx=synth.FX, fy=synth.FY, cx=synth.CX, cy=synth.CY, bf=synth.BF)
    a = src.pipeline_run(gray, depth, T, 2, 1000, **kw)
    ref_out.same("counts", a[1:], lambda: src.src_pipeline_run(gray, depth, T, 2, 1000, **kw)[1:])
    assert a[2][1:].min() > 100


# ---- the remaining ORBmatcher members -------------------------------------------------------------------------------
def test_best_search_equals_reference_sources(src, ref_out):
    """match_ref_best (the candidate loop Fuse x2 / SearchBySim3 share, no gate) against the reference's own
    KeyFrame::GetFeaturesInArea + DescriptorDistance walked in the same order."""
    from tests import members_gen as G
    rng = np.random.default_rng(71)
    M = src.SrcMembers("refsrc") if ref_out.live else None
    hits = 0
    for case in range(6):
        F, _ = _random_frame(rng, int(rng.integers(150, 600)), False)
        q = G.best_queries(rng, F)
        a = src.search_best(F, q, 0)
        ref_out.same(case, a, lambda: M.kf_best(F, q))
        hits += int((a[0] >= 0).sum())
    assert hits > 500


def test_triangulation_equals_reference_sources(src, ref_out):
    """match_ref_triangulation against ORBmatcher::SearchForTriangulation of the reference on two real KeyFrames
    (mono / stereo mixes, occupied keypoints, bOnlyStereo, orientation check on / off)."""
    from tests import members_gen as G
    rng = np.random.default_rng(73)
    M = src.SrcMembers("refsrc") if ref_out.live else None
    tot = 0
    for case in range(8):
        k1, k2, T1, T2, cam, F12 = G.tri_pair(rng, mono_frac=[0.6, 0.0, 1.0, 0.3][case % 4])
        only_stereo, ori = case % 4 == 1, case % 3 != 2
        ref = lambda: M.triangulation(k1, k2, T1, T2, cam, F12, only_stereo, 0.6, ori)
        # the epipole (kf1's camera centre projected into kf2) is computed by the reference and is an input of the oracle
        ep = np.array(ref_out.value(("epipole", case), lambda: ref()[2].tolist()), np.float32)
        n_or, m_or = src.search_for_triangulation(k1, k2, F12, ep, G.SF, G.SF * G.SF, only_stereo, ori)
        ref_out.same(case, (n_or, m_or), lambda: ref()[:2])
        assert n_or == (m_or >= 0).sum()
        tot += n_or
    assert tot > 300


def test_reference_members_run_on_synthetic_graphs(src, ref_out):
    """The harness around Fuse / Fuse(Sim3) / SearchBySim3 / the relocalisation and loop-closing projections produces
    non-trivial results on the synthetic graphs the GPU suite compares the shims on (sanity of the generator).  The
    graphs are pinned to the recorded ones, so that the recorded results of the reference still apply to them."""
    from tests import members_gen as G
    rng = np.random.default_rng(79)
    M = src.SrcMembers("refsrc") if ref_out.live else None
    count = lambda *arrays: [int(a.sum()) for a in arrays]
    n = 500
    X = G.world_points(rng, n)
    desc = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    T = G.pose(rng)
    octs = rng.integers(0, 4, n)
    KF, owner = G.frame_of(rng, T, X, desc, octaves=octs)
    # the keyframe's own MapPoints: the world point behind each keypoint (60 % of them)
    has = (owner >= 0) & (rng.random(KF.n) < 0.6)
    Xk = np.where(has[:, None], X[np.maximum(owner, 0)], 0.0)
    kf_mps = G.map_points(rng, Xk, KF.desc, G.camera_centre(T), src, octaves=KF.octave)
    kf_mps.valid = has.astype(np.uint8)
    pts = G.map_points(rng, X + rng.normal(0, 0.004, X.shape), desc, G.camera_centre(T), src, octaves=octs)
    in_kf = (rng.random(n) < 0.05).astype(np.uint8)

    def fuse():
        nf, slot, rep, krep = M.fuse(KF, kf_mps, pts, in_kf, 3.0)
        return [nf] + count(rep >= 0, krep >= 0, (slot >= 0) & (slot < 1000000))
    nf, n_rep, n_krep, n_slot = ref_out.value("fuse", fuse)
    assert nf > 50 and n_rep > 5 and n_krep > 5 and n_slot > 10
    S = T.copy()
    S[:3, :] *= np.float32(1.3)
    nf2, n_rep2 = ref_out.value("fuse_sim3", lambda: (lambda r: [r[0]] + count(r[2] >= 1000000))(M.fuse_sim3(KF, kf_mps, S, pts, 4.0)))
    assert nf2 > 50 and n_rep2 > 10
    matched = np.where(rng.random(KF.n) < 0.1, -2, -1).astype(np.int32)
    nm = ref_out.value("projection_sim3", lambda: M.projection_sim3(KF, S, pts, matched, 10)[0])
    assert nm > 50
    cur, _ = G.frame_of(rng, G.pose(rng), X, desc, octaves=octs)
    cur.mp_obs = np.where(rng.random(cur.n) < 0.1, 1, -1).astype(np.int32)
    found = (rng.random(KF.n) < 0.1).astype(np.uint8)
    nm2 = ref_out.value("projection_kf", lambda: M.projection_kf(cur, KF, kf_mps, found, 15.0, 100)[0])
    assert nm2 > 30
    T2 = G.pose(rng, 0.2, 3.0)
    KF2, owner2 = G.frame_of(rng, T2, X, desc, octaves=octs)
    has2 = (owner2 >= 0) & (rng.random(KF2.n) < 0.6)
    mp2 = G.map_points(rng, np.where(has2[:, None], X[np.maximum(owner2, 0)], 0.0), KF2.desc, G.camera_centre(T2), src,
                       octaves=KF2.octave)
    mp2.valid = has2.astype(np.uint8)
    T12 = T.astype(np.float64) @ np.linalg.inv(T2.astype(np.float64))
    nf3, n_m12 = ref_out.value("search_by_sim3", lambda: (lambda r: [r[0]] + count(r[1] >= 0))(
        M.search_by_sim3(KF, KF2, kf_mps, mp2, np.full(KF.n, -1, np.int32), 1.0, T12[:3, :3], T12[:3, 3], 7.5)))
    assert nf3 > 20 and n_m12 == nf3
    ref_out.same("graphs", (KF, kf_mps, pts, in_kf, S, matched, cur, found, KF2, mp2, T12))


def test_frame_glue_equals_reference_sources(src, ref_out):
    """Frame::isInFrustum + MapPoint::PredictScale and Frame::UndistortKeyPoints: the flat oracles against the reference's
    own Frame.cc / MapPoint.cc (isInFrustum per point on a real Frame; UndistortKeyPoints through the real RGB-D Frame
    constructor with a distorted camera)."""
    from tests import members_gen as G
    rng = np.random.default_rng(91)
    for case in range(4):
        n = 3000
        X = G.world_points(rng, n)
        X[: n // 10, 2] *= -1                       # behind the camera
        T = G.pose(rng, 0.3, 8.0)
        F, _ = _random_frame(rng, 50, False)
        F.Tcw = T.reshape(16)
        PO = X - G.camera_centre(T)
        dist = np.linalg.norm(PO, axis=1)
        normal = PO / dist[:, None] + rng.normal(0, 0.5, (n, 3))
        normal /= np.linalg.norm(normal, axis=1)[:, None]
        lvl = rng.integers(0, 9, n)
        maxd = (dist * 1.2 ** lvl * rng.uniform(0.97, 1.03, n)).astype(np.float32)   # ratios close to the level boundaries
        mind = (maxd / 1.2 ** 7 * rng.uniform(0.5, 1.4, n)).astype(np.float32)
        a = src.is_in_frustum(F, X, normal, mind, maxd, 0.5, np.log(np.float32(1.2)), "oracle")
        assert 0.15 * n < a[0].sum() < 0.9 * n
        m = a[0] > 0
        in_view = lambda r: [r[0]] + [x[r[0] > 0] for x in r[1:]]    # the outputs of points outside the view are unset
        ref_out.same(case, in_view(a), lambda: in_view(src.is_in_frustum(F, X, normal, mind, maxd, 0.5, np.log(np.float32(1.2)),
                                                                          "refsrc")))
        assert len(np.unique(a[4][m])) >= 6
    # UndistortKeyPoints through the real Frame constructor
    rs = synth.RoomStream(seed=9, n=4)
    gray, depth, rgb, T = rs.frame(2)
    dist4 = np.array([-0.28, 0.07, 0.0002, 0.0001], np.float32)
    K, D = src.RefExtractor(800, 1.2, 8, 20, 7)(gray)
    Kmat = np.array([synth.FX, 0, synth.CX, 0, synth.FY, synth.CY, 0, 0, 1], np.float32)
    un = src.undistort(np.stack([K["x"], K["y"]], 1), Kmat, dist4)

    def ref():
        Kun, D2, ur, dp, xw, va = src.src_frame_rgbd(gray, depth, T, synth.FX, synth.FY, synth.CX, synth.CY, synth.BF,
                                                     nfeatures=800, dist=dist4)
        return D2, Kun["x"], Kun["y"]
    ref_out.same("undistort", (D, np.ascontiguousarray(un[:, 0]), np.ascontiguousarray(un[:, 1])), ref)
    assert np.abs(un[:, 0] - K["x"]).max() > 1.0      # the distortion does move points


def test_bow_transform_restatements_agree(src, ref_out):
    """Frame::ComputeBoW of the reference on the DBoW2 stand-in (TemplatedVocabulary::transform restated from DBoW2's
    published algorithm; DBoW2 itself is not shipped with the reference) against an independent numpy restatement: same
    words, bit-equal L1-normalised weights, same FeatureVector (node ids 4 levels above the leaves)."""
    for (k, L, seed) in [(10, 5, 3), (6, 6, 4), (10, 4, 5), (4, 3, 6)]:
        parent, nd, w = src.synth_vocabulary(seed, k, L)
        rng = np.random.default_rng(seed)
        leaves = np.nonzero(w > 0)[0]
        desc = nd[rng.choice(leaves, 700)].copy()
        desc[:, :2] ^= rng.integers(0, 256, size=(700, 2), dtype=np.uint8)
        a = src.bow_transform_py(k, L, parent, nd, w, desc)
        ref_out.same((k, L), a, lambda: src.src_bow_transform(k, L, parent, nd, w, desc))
        assert len(a[0]) > 50 and abs(sum(a[0].values()) - 1.0) < 1e-9
        assert len(a[1]) >= (1 if L <= 4 else 6)
