"""GPU parity of the ORBmatcher members beyond the tracking searches.
(1) C-ABI entries (orbm_search_best / _for_initialization / _for_triangulation) against the flat CPU oracles, which
    tests/test_refsrc_cpu.py pins to the reference's own sources.
(2) THE DROP-IN CHECK: oracle/_ref/libshimsrc.so is the reference's own src/Frame.cc, KeyFrame.cc, MapPoint.cc, Map.cc
    compiled unmodified against shim/ORBextractor.h and shim/ORBmatcher.h; every public ORBmatcher member is run on the
    same real Frame / KeyFrame / MapPoint graphs through the shim (-> libb200orb.so -> GPU) and through the reference's
    own ORBmatcher.cc (oracle/_ref/librefsrc.so), and must leave the identical pointer state."""
import os

import numpy as np
import pytest

from orb_slam2_ssd_semantic_b200 import synth
from orb_slam2_ssd_semantic_b200._abi import BowView, FrameView, LastView, TrackPointsView
from tests import members_gen as G

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def matcher():
    from orb_slam2_ssd_semantic_b200 import ORBmatcher
    return ORBmatcher


def _rframe(rng, n, with_obs=False):
    x = rng.uniform(5, 635, n).astype(np.float32)
    y = rng.uniform(5, 475, n).astype(np.float32)
    octv = rng.integers(0, 8, n).astype(np.int32)
    desc = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    z = rng.uniform(0.5, 4.0, n).astype(np.float32)
    ur = np.where(rng.random(n) < 0.7, x - synth.BF / z, -1).astype(np.float32)
    F = FrameView(x, y, octv, rng.uniform(0, 360, n).astype(np.float32), ur, desc, np.eye(4, dtype=np.float32), synth.FX, synth.FY,
                  synth.CX, synth.CY, synth.BF, 0, 640, 0, 480, G.SF)
    if with_obs:
        F.mp_obs = rng.integers(-1, 2, n).astype(np.int32)
    return F, z


def test_search_best_matches_oracle(matcher, oracle):
    rng = np.random.default_rng(171)
    m = matcher(0.6, True)
    hits = 0
    for case in range(8):
        F, _ = _rframe(rng, int(rng.integers(150, 2200)))
        q = G.best_queries(rng, F, 400)
        inv_s2 = (1.0 / (G.SF * G.SF)).astype(np.float32)
        for gate in (0, 1):
            a = m.SearchBest(F, q, gate, inv_s2)
            b = oracle.search_best(F, q, gate, inv_s2)
            assert (a[0] == b[0]).all() and (a[1] == b[1]).all(), (case, gate)
            hits += int((a[0] >= 0).sum())
    assert hits > 2000
    # a crowded window: far more than 64 candidates per query
    n = 3000
    F, _ = _rframe(rng, n)
    F.x[:] = rng.uniform(300, 340, n)
    F.y[:] = rng.uniform(220, 260, n)
    q = G.best_queries(rng, F, 100)
    q.radius[:] = 40.0
    a, b = m.SearchBest(F, q, 0), oracle.search_best(F, q, 0)
    assert (a[0] == b[0]).all() and (a[1] == b[1]).all()


def test_search_for_initialization_matches_oracle(matcher, oracle):
    rng = np.random.default_rng(141)
    tot = 0
    for case in range(8):
        n = int(rng.integers(150, 900))
        x = rng.uniform(5, 635, n).astype(np.float32)
        y = rng.uniform(5, 475, n).astype(np.float32)
        octv = rng.integers(0, 3, n).astype(np.int32)
        desc = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
        ang = rng.uniform(0, 360, n).astype(np.float32)
        mk = lambda xx, yy, dd, aa: FrameView(xx, yy, octv, aa, np.full(n, -1, np.float32), dd, np.eye(4, dtype=np.float32),
                                              synth.FX, synth.FY, synth.CX, synth.CY, synth.BF, 0, 640, 0, 480, G.SF)
        F1 = mk(x, y, desc, ang)
        d2 = desc.copy()
        d2[:, :2] ^= rng.integers(0, 256, size=(n, 2), dtype=np.uint8)
        dup = rng.integers(0, n, n // 6)
        d2[dup] = d2[(dup + 1) % n]
        F2 = mk((x + rng.normal(0, 6, n)).astype(np.float32), (y + rng.normal(0, 6, n)).astype(np.float32), d2,
                (ang + rng.normal(0, 4, n)).astype(np.float32) % np.float32(360))
        prev = np.stack([x, y], 1)
        for window, ori in ((100, True), (30, False)):
            a = matcher(0.9, ori).SearchForInitialization(F1, F2, prev, window)
            b = oracle.search_for_initialization(F1, F2, prev, window, 0.9, ori)
            assert a[0] == b[0] and (a[1] == b[1]).all() and a[2].tobytes() == b[2].tobytes(), (case, window, ori)
            tot += a[0]
    assert tot > 300


def test_search_for_triangulation_matches_oracle(matcher, oracle):
    rng = np.random.default_rng(173)
    tot = 0
    for case in range(8):
        k1, k2, T1, T2, cam, F12 = G.tri_pair(rng, n=int(rng.integers(200, 1500)), mono_frac=[0.6, 0.0, 1.0, 0.3][case % 4])
        only_stereo, ori = case % 4 == 1, case % 3 != 2
        ep = (float(rng.uniform(-200, 800)), float(rng.uniform(-200, 700)))
        a = matcher(0.6, ori).SearchForTriangulation(k1, k2, F12, ep, G.SF, G.SF * G.SF, only_stereo)
        b = oracle.search_for_triangulation(k1, k2, F12, ep, G.SF, G.SF * G.SF, only_stereo, ori)
        assert a[0] == b[0] and (a[1] == b[1]).all(), case
        tot += a[0]
    assert tot > 300


# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def both(oracle):
    if not (oracle.refsrc_available() and os.path.exists(oracle._SHIMSO)):
        pytest.skip("no oracle/_ref libraries: they are built from the reference's own sources")
    return oracle.SrcMembers("refsrc"), oracle.SrcMembers("shimsrc")


def test_reference_callers_through_shims_tracking_searches(both):
    """SearchByProjection(cur, last) / (F, MapPoints), SearchByBoW x2, SearchForInitialization: the shim class on the
    reference's own Frame / KeyFrame / MapPoint objects == the reference's ORBmatcher.cc on the same objects."""
    R, S = both
    rng = np.random.default_rng(205)
    tot = 0
    for case in range(6):
        n = int(rng.integers(100, 1200))
        cur, z = _rframe(rng, n, case % 2 == 0)
        T = np.eye(4, dtype=np.float32)
        T[:3, 3] = rng.normal(0, 0.02, 3)
        T[2, 3] = [0.0, 0.3, -0.3][case % 3]
        cur.Tcw = T.reshape(16)
        m = int(rng.integers(100, 1200))
        sel = rng.integers(0, n, m)
        zz = z[sel] * rng.uniform(0.98, 1.02, m).astype(np.float32)
        xw = np.stack([(cur.x[sel] + rng.normal(0, 3, m) - synth.CX) * zz / synth.FX,
                       (cur.y[sel] + rng.normal(0, 3, m) - synth.CY) * zz / synth.FY, zz], 1).astype(np.float32)
        d2 = cur.desc[sel].copy()
        d2[:, :4] ^= rng.integers(0, 256, size=(m, 4), dtype=np.uint8)
        last = LastView(xw, (rng.random(m) < 0.9).astype(np.uint8), np.clip(cur.octave[sel] + rng.integers(-1, 2, m), 0, 7),
                        rng.uniform(0, 360, m).astype(np.float32), d2, np.eye(4, dtype=np.float32),
                        mp_obs=rng.integers(0, 2, m).astype(np.int32))
        a, b = R.search_by_projection_last(cur, last, 15.0, case == 5, 0.9, case != 4), S.search_by_projection_last(cur, last, 15.0, case == 5, 0.9, case != 4)
        assert a[0] == b[0] and (a[1] == b[1]).all(), ("last", case)
        tot += a[0]
        px = (cur.x[sel] + rng.normal(0, 4, m)).astype(np.float32)
        py = (cur.y[sel] + rng.normal(0, 4, m)).astype(np.float32)
        pts = TrackPointsView((rng.random(m) < 0.9).astype(np.uint8), px, py, (px - synth.BF / z[sel]).astype(np.float32),
                              np.clip(cur.octave[sel] + rng.integers(0, 2, m), 0, 7), rng.uniform(0.99, 1.0, m).astype(np.float32), d2,
                              mp_obs=rng.integers(0, 2, m).astype(np.int32))
        a, b = R.search_by_projection_points(cur, pts, 3.0, 0.8), S.search_by_projection_points(cur, pts, 3.0, 0.8)
        assert a[0] == b[0] and (a[1] == b[1]).all(), ("points", case)
        nw = int(rng.integers(4, 40))
        fv1, fv2 = {}, {}
        for i, w in enumerate(rng.integers(0, nw, n)):
            fv1.setdefault(int(w) * 3, []).append(i)
        for i, w in enumerate(rng.integers(0, nw, m)):
            fv2.setdefault(int(w) * 3 + (0 if rng.random() < 0.8 else 1), []).append(i)
        ang2 = rng.uniform(0, 360, m).astype(np.float32)
        K = BowView(cur.desc, cur.angle, fv1, valid=(rng.random(n) < 0.85).astype(np.uint8))
        Fr = BowView(d2, ang2, fv2)
        K2 = BowView(d2, ang2, fv2, valid=(rng.random(m) < 0.85).astype(np.uint8))
        a, b = R.search_by_bow(K, Fr, 0.7, True), S.search_by_bow(K, Fr, 0.7, True)
        assert a[0] == b[0] and (a[1] == b[1]).all(), ("bow", case)
        a, b = R.search_by_bow(K, K2, 0.75, True, kfkf=True), S.search_by_bow(K, K2, 0.75, True, kfkf=True)
        assert a[0] == b[0] and (a[1] == b[1]).all(), ("bow_kf", case)
        octv = rng.integers(0, 3, n).astype(np.int32)
        mk = lambda xx, yy, dd, aa: FrameView(xx, yy, octv, aa, np.full(n, -1, np.float32), dd, np.eye(4, dtype=np.float32),
                                              synth.FX, synth.FY, synth.CX, synth.CY, synth.BF, 0, 640, 0, 480, G.SF)
        F1 = mk(cur.x, cur.y, cur.desc, cur.angle)
        d3 = cur.desc.copy()
        d3[:, :2] ^= rng.integers(0, 256, size=(n, 2), dtype=np.uint8)
        F2 = mk((cur.x + rng.normal(0, 6, n)).astype(np.float32), (cur.y + rng.normal(0, 6, n)).astype(np.float32), d3,
                (cur.angle + rng.normal(0, 4, n)).astype(np.float32) % np.float32(360))
        prev = np.stack([cur.x, cur.y], 1)
        a, b = R.search_for_initialization(F1, F2, prev, 100, 0.9, True), S.search_for_initialization(F1, F2, prev, 100, 0.9, True)
        assert a[0] == b[0] and (a[1] == b[1]).all() and a[2].tobytes() == b[2].tobytes(), ("init", case)
    assert tot > 500


def test_reference_callers_through_shims_graph_members(both, oracle):
    """Relocalisation and loop-closing projections, Fuse x2, SearchBySim3, SearchForTriangulation on real KeyFrame /
    MapPoint graphs: shim == reference, including the Replace / AddObservation mutations Fuse performs."""
    R, S = both
    rng = np.random.default_rng(279)
    tot = np.zeros(6, int)
    for case in range(5):
        sc = G.scene(rng, oracle, n=int(rng.integers(300, 1500)))
        a, b = R.fuse(sc["KF"], sc["kf_mps"], sc["pts"], sc["in_kf"], 3.0), S.fuse(sc["KF"], sc["kf_mps"], sc["pts"], sc["in_kf"], 3.0)
        assert a[0] == b[0] and all((x == y).all() for x, y in zip(a[1:], b[1:])), ("fuse", case)
        tot[0] += a[0]
        a, b = R.fuse_sim3(sc["KF"], sc["kf_mps"], sc["S"], sc["pts"], 4.0), S.fuse_sim3(sc["KF"], sc["kf_mps"], sc["S"], sc["pts"], 4.0)
        assert a[0] == b[0] and (a[1] == b[1]).all() and (a[2] == b[2]).all(), ("fuse_sim3", case)
        tot[1] += a[0]
        a, b = R.projection_sim3(sc["KF"], sc["S"], sc["pts"], sc["matched"], 10), S.projection_sim3(sc["KF"], sc["S"], sc["pts"], sc["matched"], 10)
        assert a[0] == b[0] and (a[1] == b[1]).all(), ("projection_sim3", case)
        tot[2] += a[0]
        a = R.projection_kf(sc["cur"], sc["KF"], sc["kf_mps"], sc["found"], 15.0, 100, 0.9, case != 3)
        b = S.projection_kf(sc["cur"], sc["KF"], sc["kf_mps"], sc["found"], 15.0, 100, 0.9, case != 3)
        assert a[0] == b[0] and (a[1] == b[1]).all(), ("projection_kf", case)
        tot[3] += a[0]
        m0 = np.full(sc["KF"].n, -1, np.int32)
        a = R.search_by_sim3(sc["KF"], sc["KF2"], sc["kf_mps"], sc["mp2"], m0, 1.0, sc["R12"], sc["t12"], 7.5)
        b = S.search_by_sim3(sc["KF"], sc["KF2"], sc["kf_mps"], sc["mp2"], m0, 1.0, sc["R12"], sc["t12"], 7.5)
        assert a[0] == b[0] and (a[1] == b[1]).all(), ("sim3", case)
        tot[4] += a[0]
        k1, k2, T1, T2, cam, F12 = G.tri_pair(rng, n=int(rng.integers(200, 1200)), mono_frac=[0.6, 0.0, 1.0, 0.3, 0.5][case])
        a = R.triangulation(k1, k2, T1, T2, cam, F12, case == 1, 0.6, case != 2)
        b = S.triangulation(k1, k2, T1, T2, cam, F12, case == 1, 0.6, case != 2)
        assert a[0] == b[0] and (a[1] == b[1]).all(), ("triangulation", case)
        tot[5] += a[0]
    assert (tot > 50).all(), tot


def test_reference_frame_constructor_and_pipeline_through_shims(both):
    """The reference's RGB-D Frame constructor (src/Frame.cc:176-240, unmodified) running on the shim ORBextractor, and
    the whole per-frame tracking path (Frame ctor + MapPoints + SearchByProjection) on shim extractor + shim matcher,
    give what the reference's own ORBextractor.cc / ORBmatcher.cc give."""
    R, S = both
    rs = synth.RoomStream(seed=5, n=40)
    fr = [rs.frame(3 * t) for t in range(5)]
    gray, depth, T = np.stack([f[0] for f in fr]), np.stack([f[1] for f in fr]), np.stack([f[3] for f in fr])
    a = R.frame_rgbd(gray[0], depth[0], T[0], synth.FX, synth.FY, synth.CX, synth.CY, synth.BF, 1000)
    b = S.frame_rgbd(gray[0], depth[0], T[0], synth.FX, synth.FY, synth.CX, synth.CY, synth.BF, 1000)
    assert len(a[0]) == len(b[0]) > 900
    for x, y in zip(a, b):
        assert x.tobytes() == y.tobytes()
    pa = R.pipeline_run(gray, depth, T, 2, 1000, synth.FX, synth.FY, synth.CX, synth.CY, synth.BF)
    pb = S.pipeline_run(gray, depth, T, 2, 1000, synth.FX, synth.FY, synth.CX, synth.CY, synth.BF)
    assert (pa[1] == pb[1]).all() and (pa[2] == pb[2]).all() and pa[2][1:].min() > 100


def test_frame_glue_is_in_frustum_and_undistort_match_oracle(matcher, oracle):
    """orbm_is_in_frustum (Frame::isInFrustum + PredictScale) and orbm_undistort_keypoints (Frame::UndistortKeyPoints)
    against the flat oracles (pinned to the reference's Frame.cc / MapPoint.cc in tests/test_refsrc_cpu.py)."""
    rng = np.random.default_rng(191)
    m = matcher(0.8, True)
    for case in range(4):
        n = 20000
        X = G.world_points(rng, n)
        X[: n // 10, 2] *= -1
        T = G.pose(rng, 0.3, 8.0)
        F, _ = _rframe(rng, 50)
        F.Tcw = T.reshape(16)
        PO = X - G.camera_centre(T)
        dist = np.linalg.norm(PO, axis=1)
        normal = PO / dist[:, None] + rng.normal(0, 0.5, (n, 3))
        normal /= np.linalg.norm(normal, axis=1)[:, None]
        lvl = rng.integers(0, 9, n)
        maxd = (dist * 1.2 ** lvl * rng.uniform(0.999, 1.001, n)).astype(np.float32)   # ratios AT the level boundaries
        mind = (maxd / 1.2 ** 7 * rng.uniform(0.5, 1.4, n)).astype(np.float32)
        lsf = float(np.log(np.float32(1.2)))
        a = m.IsInFrustum(F, X, normal, mind, maxd, 0.5, lsf)
        b = oracle.is_in_frustum(F, X, normal, mind, maxd, 0.5, lsf, "oracle")
        assert 0.15 * n < b[0].sum() < 0.9 * n
        for x, y in zip(a, b):
            assert np.asarray(x).tobytes() == np.asarray(y).tobytes(), case
    Kmat = np.array([synth.FX, 0, synth.CX, 0, synth.FY, synth.CY, 0, 0, 1], np.float32)
    xy = np.stack([rng.uniform(0, 640, 5000), rng.uniform(0, 480, 5000)], 1).astype(np.float32)
    for dist in ([-0.28, 0.07, 0.0002, 0.0001], [0.26, -0.95, -0.005, 0.003, 1.16], [0.0, 0.1, 0, 0]):
        a = m.UndistortKeyPoints(xy, Kmat, np.array(dist, np.float32))
        b = oracle.undistort(xy, Kmat, np.array(dist, np.float32))
        assert a.tobytes() == b.tobytes(), dist


def test_bow_transform_matches_reference_sources(oracle):
    """orbv_transform + the map assembly of the Python mirror, and the shim ORBVocabulary under the reference's own
    Frame::ComputeBoW, against Frame::ComputeBoW on the CPU (DBoW2 stand-in): identical BowVector (bit-equal doubles)
    and FeatureVector.  The reference's output is recorded (tests/reference_outputs.py) and also computed live where
    oracle/_ref holds its library; the shim leg needs oracle/_ref/libshimsrc.so."""
    from orb_slam2_ssd_semantic_b200 import ORBVocabulary
    from tests.reference_outputs import Reference
    R = Reference("test_bow_transform_matches_reference_sources", oracle.refsrc_available())
    for (k, L, seed) in [(10, 5, 3), (6, 6, 4), (10, 4, 5), (4, 3, 6)]:
        parent, nd, w = oracle.synth_vocabulary(seed, k, L)
        rng = np.random.default_rng(seed)
        leaves = np.nonzero(w > 0)[0]
        desc = nd[rng.choice(leaves, 2000)].copy()
        desc[:, :2] ^= rng.integers(0, 256, size=(2000, 2), dtype=np.uint8)
        voc = ORBVocabulary(k, L, parent, nd, w)
        bow, fv = voc.transform(desc, 4)
        R.same((k, L), (bow, fv), lambda: oracle.src_bow_transform(k, L, parent, nd, w, desc, "refsrc"))
        if os.path.exists(oracle._SHIMSO):
            R.same((k, L), oracle.src_bow_transform(k, L, parent, nd, w, desc, "shimsrc"))
