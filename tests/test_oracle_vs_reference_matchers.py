"""The oracle's matchers (oracle/match_oracle.cpp, oracle/proj_oracle.cpp) against the REFERENCE'S OWN cslam/src/ORBmatcher.cpp, compiled
where it lies into oracle/_ref/libmatch_ref.so (oracle/Makefile `ref`).  Frame / KeyFrame / MapPoint are plain stand-ins exposing the
members the matcher source names (oracle/ref_stub/cslam/Frame.h); every search method — candidate walks, best / second-best bookkeeping,
thresholds, ratio tests, rotation histograms, mutual checks and the geometric gates in front of them — is the reference's object code.
Index-exact.  The reference's outputs are stored under tests/golden/reference (tests/reference_outputs.py)."""
import numpy as np
import pytest

from ccm_slam_b200 import synth_match as sm
from tests.reference_outputs import ALL, Recorded, same

f32 = np.float32


@pytest.fixture(scope="module")
def ref(oracle):
    return Recorded(oracle, __file__, oracle.ref_match, keep=ALL)


def _two_frames(seed, n=800):
    """descriptor sets with true matches (a few flipped bits), vocabulary-node labels and angles, as SearchByBoW sees them"""
    rng = np.random.default_rng(seed)
    d1 = rng.integers(0, 256, size=(n, 32), dtype=np.uint8); d2 = rng.integers(0, 256, size=(n + 40, 32), dtype=np.uint8)
    perm = rng.permutation(n + 40)[: (2 * n) // 3]
    d2[perm] = sm.flip_bits(d1[: len(perm)], rng.integers(0, 60, len(perm)), rng)
    node1 = rng.integers(0, 40, n); node2 = rng.integers(0, 40, n + 40); node2[perm] = node1[: len(perm)]
    a1 = rng.uniform(0, 360, n).astype(f32); a2 = rng.uniform(0, 360, n + 40).astype(f32)
    a2[perm] = (a1[: len(perm)] + rng.normal(0, 3, len(perm)) + np.where(rng.random(len(perm)) < 0.1, 90, 0)).astype(f32) % f32(360)
    has1 = (rng.random(n) < 0.75).astype(np.uint8); has2 = (rng.random(n + 40) < 0.75).astype(np.uint8)
    return d1, d2, node1, node2, a1, a2, has1, has2


@pytest.mark.parametrize("seed,nnratio,ori", [(0, 0.7, True), (1, 0.9, False), (2, 0.6, True)])
def test_search_by_bow(ref, seed, nnratio, ori):
    d1, d2, node1, node2, a1, a2, has1, has2 = _two_frames(seed)
    fv1, fv2 = ref.FeatureVector(node1), ref.FeatureVector(node2)
    got, n = ref.match_bow_kf_frame(d1, has1, a1, fv1, d2, a2, fv2, nnratio, ori)
    want, wn = ref.ref_match_bow_kf_frame(d1, has1, a1, fv1, d2, a2, fv2, nnratio, ori)
    assert n == wn and same(got, want) and n > 100
    got, n = ref.match_bow_kf_kf(d1, has1, a1, fv1, d2, has2, a2, fv2, nnratio, ori)
    want, wn = ref.ref_match_bow_kf_kf(d1, has1, a1, fv1, d2, has2, a2, fv2, nnratio, ori)
    assert n == wn and same(got, want) and n > 60
    assert ref.ref_descriptor_distance(d1[0], d2[0]) == ref.descriptor_distance(d1[0], d2[0])


@pytest.mark.parametrize("seed,ori", [(3, False), (4, True)])
def test_search_for_triangulation(ref, seed, ori):
    rng = np.random.default_rng(seed)
    n = 700
    d1 = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    d2 = sm.flip_bits(d1, rng.integers(0, 70, n), rng)                      # keypoint i of view 2 is keypoint i of view 1, noisily
    d2[500:] = rng.integers(0, 256, size=(n - 500, 32), dtype=np.uint8)     # ... except the last 200
    node1 = rng.integers(0, 30, n); node2 = node1.copy(); node2[650:] = rng.integers(0, 30, n - 650)
    a1 = rng.uniform(0, 360, n).astype(f32); a2 = ((a1 + rng.normal(0, 3, n) + np.where(rng.random(n) < 0.1, 90, 0)) % 360).astype(f32)
    has1 = (rng.random(n) < 0.3).astype(np.uint8); has2 = (rng.random(n) < 0.3).astype(np.uint8)   # only untracked keypoints are triangulated
    # pure x-translation between the views: F12 = K^-T [t]_x K^-1, matches lie on (nearly) the same image row
    fx, fy, cx, cy = f32(512.0), f32(512.0), f32(376.0), f32(240.0)
    xy1 = np.round(rng.uniform([20, 20], [730, 460], size=(n, 2)) * 4) / 4
    xy2 = xy1 + np.stack([rng.uniform(-40, 40, n), rng.normal(0, 1.2, n)], 1); xy2 = np.round(xy2 * 4) / 4
    oct1 = rng.integers(0, 8, n).astype(np.int32); oct2 = rng.integers(0, 8, n).astype(np.int32)
    Kinv = np.linalg.inv(np.array([[fx, 0, cx], [0, fy, cy], [0, 0, 1]], np.float64))
    F12 = (Kinv.T @ np.array([[0, 0, 0], [0, 0, -1.0], [0, 1.0, 0]]) @ Kinv).astype(f32)
    fv1, fv2 = ref.FeatureVector(node1), ref.FeatureVector(node2)
    v = lambda d, has, xy, oc, an, fv: dict(desc=d, has_mp=has, kp_xy=xy.astype(f32), octave=oc, angle=an, fv=fv, intr=(fx, fy, cx, cy))
    v1, v2 = v(d1, has1, xy1, oct1, a1, fv1), v(d2, has2, xy2, oct2, a2, fv2)
    # camera 1 sits at Cw in camera 2's frame; its image there is the epipole — float32, in the reference's evaluation order (:704-712)
    Cw = np.array([-8.0, 0.5, 2.0], f32)
    invz = f32(1.0) / Cw[2]
    ex = f32(f32(f32(fx * Cw[0]) * invz) + cx); ey = f32(f32(f32(fy * Cw[1]) * invz) + cy)
    sf = np.empty(8, f32); sf[0] = 1
    for i in range(1, 8):
        sf[i] = f32(sf[i - 1] * f32(1.2))
    got = ref.match_triangulation(v1, v2, F12, float(ex), float(ey), (sf * sf).astype(f32), sf, ori)
    want = ref.ref_match_triangulation(v1, v2, F12, Cw, ori)
    assert same(got, want) and len(want) > 30


@pytest.mark.parametrize("seed,nnratio,ori", [(5, 0.9, True), (6, 0.7, False)])
def test_search_for_initialization(ref, seed, nnratio, ori):
    g2, q = sm.make_init_pair(n=900, seed=seed)
    g1 = dict(desc=q["desc"], kp_xy=q["uv"], octave=q["level"], angle=q["angle"], bounds=g2["bounds"], cols=g2["cols"], rows=g2["rows"])
    got, n = ref.search_for_initialization(g2, q, nnratio, ori)
    want, wn, prev = ref.ref_search_for_initialization(g1, g2, q["uv"], 100, nnratio, ori)
    assert n == wn and same(got, want) and n > 100
    hit = want >= 0
    assert same(prev[hit], g2["kp_xy"][want[hit]]) and same(prev[~hit], q["uv"][~hit])   # vbPrevMatched refreshed (:557-560)


@pytest.mark.parametrize("seed,th,nnratio", [(7, 1.0, 0.8), (8, 3.0, 0.8), (9, 5.0, 0.6)])
def test_search_by_projection_track(ref, seed, th, nnratio):
    g = sm.make_grid(n=1200, seed=seed); q = sm.make_queries(g, m=1500, seed=seed + 50)
    rng = np.random.default_rng(seed + 100)
    m = 1500
    view_cos = np.where(rng.random(m) < 0.5, f32(0.9995), f32(0.9)).astype(f32)
    n_obs = np.where(rng.random(m) < 0.85, 3, 0).astype(np.int32); bad = (rng.random(m) < 0.05).astype(np.uint8)
    blocked = (rng.random(1200) < 0.2).astype(np.uint8)
    points = dict(desc=q["desc"], bad=bad, n_obs=n_obs, track_in_view=q["valid"], track_xy=q["uv"], track_level=q["level"], track_view_cos=view_cos)
    # the oracle takes the window the reference derives: RadiusByViewingCos [* th] * mvScaleFactors[level], in float32 (:86-93)
    sf = np.empty(8, f32); sf[0] = 1
    for i in range(1, 8):
        sf[i] = f32(sf[i - 1] * f32(1.2))
    r = np.where(view_cos > f32(0.998), f32(2.5), f32(4.0)).astype(f32)
    if th != 1.0:
        r = (r * f32(th)).astype(f32)
    oq = dict(q, valid=(q["valid"].astype(bool) & ~bad.astype(bool)).astype(np.uint8), radius=(r * sf[q["level"]]).astype(f32))
    got, n = ref.search_by_projection_track(g, oq, (n_obs > 0).astype(np.uint8), blocked, nnratio)
    want, wn = ref.ref_search_by_projection_track(g, points, blocked, th, nnratio)
    assert n == wn and same(got, want) and n > 200


# ---- the overloads with a geometric prelude ------------------------------------------------------------------------------------
# The reference runs its own prelude (cv::Mat pose algebra, projection, image bounds, distance / angle gates, PredictScale) in front of
# the window search; the oracle starts at the window.  To compare them the scene is built so that the prelude's arithmetic is EXACT in
# float32 (identity rotations, dyadic translations and depths, power-of-two focal length): whatever rounding a matrix product uses, the
# projected pixel is the intended quarter-pixel position, and the gate quantities sit far from their thresholds.
INTR = (f32(512.0), f32(512.0), f32(376.0), f32(240.0))
BOUNDS = (0.0, 0.0, 752.0, 480.0)
SF = np.empty(8, f32); SF[0] = 1
for _i in range(1, 8):
    SF[_i] = f32(SF[_i - 1] * f32(1.2))
CATS = ("good", "behind", "outside", "too_far", "too_near", "bad_angle", "bad")


TIES = False   # set by the tie-storm tests below: every descriptor becomes one of six nearby patterns (sm.tie_storm)


def _scene(seed, n=900, m=1300, th=3.0, t=(0.25, -0.5, 1.0), scale=1.0, th_is_int=False):
    """keypoints of one image + map points whose projection through Tcw = [I | t] (or Scw = scale * [I | t]) lands on intended pixels"""
    rng = np.random.default_rng(seed)
    g = sm.make_grid(n=n, seed=seed, bounds=BOUNDS)
    fx, fy, cx, cy = [float(v) for v in INTR]
    src = rng.integers(0, n, m)
    dup = rng.random(m) < 0.12
    for i in range(1, m):
        if dup[i]:
            src[i] = src[rng.integers(0, i)]
    uv = np.round((g["kp_xy"][src].astype(np.float64) + rng.normal(0, 1.5, (m, 2))) * 4) / 4
    cat = rng.choice(len(CATS), size=m, p=[0.64, 0.06, 0.06, 0.06, 0.06, 0.06, 0.06])
    uv[cat == CATS.index("outside")] += np.array([900.0, 0.0])
    zc = rng.choice([2.0, 4.0, 8.0], m)
    zc[cat == CATS.index("behind")] *= -1
    cam = np.stack([(uv[:, 0] - cx) * zc / fx, (uv[:, 1] - cy) * zc / fy, zc], 1)        # exact dyadic numbers
    world = cam - np.asarray(t, np.float64)                                             # R = I: Xc = Xw + t
    assert same(world.astype(f32).astype(np.float64), world) and same(cam.astype(f32).astype(np.float64), cam)
    dist = np.sqrt((cam * cam).sum(1))
    level = np.clip(g["octave"][src] + rng.choice([0, 0, 0, 1, 1, -1], m), 0, 7).astype(np.int32)
    max_d = dist * 1.2 ** (level - 0.5)                                                  # PredictScale lands mid-interval on `level`
    min_d = dist / 3.0
    max_d[cat == CATS.index("too_far")] = dist[cat == CATS.index("too_far")] / 2.0
    level[cat == CATS.index("too_far")] = 0
    min_d[cat == CATS.index("too_near")] = dist[cat == CATS.index("too_near")] * 2.0
    normal = cam / dist[:, None]
    normal[cat == CATS.index("bad_angle")] *= -1
    desc = sm.flip_bits(g["desc"][src], rng.integers(0, 70, m), rng)
    if TIES:
        g, qd = sm.tie_storm(g, dict(desc=desc), pool=6, seed=seed + 1000)
        desc = qd["desc"]
    n_obs = rng.integers(1, 6, m).astype(np.int32)
    points = dict(pos=world.astype(f32), normal=normal.astype(f32), min_dist=min_d.astype(f32), max_dist=max_d.astype(f32), desc=desc,
                  bad=(cat == CATS.index("bad")).astype(np.uint8), n_obs=n_obs)
    thf = f32(int(th)) if th_is_int else f32(th)
    # a few keypoints of make_grid lie outside the image on purpose; a point projected next to one of them fails the bounds test:
    # KeyFrame::IsInImage is half-open (KeyFrame.cpp:1203), the Frame overloads compare against [mnMin, mnMax] inclusively
    in_kf_image = (uv[:, 0] >= 0) & (uv[:, 0] < 752) & (uv[:, 1] >= 0) & (uv[:, 1] < 480)
    in_frame_image = (uv[:, 0] >= 0) & (uv[:, 0] <= 752) & (uv[:, 1] >= 0) & (uv[:, 1] <= 480)
    q = dict(valid=((cat == 0) & in_kf_image).astype(np.uint8), uv=uv.astype(f32), radius=(thf * SF[level]).astype(f32), level=level, desc=desc,
             angle=np.zeros(m, f32))
    Scw = np.eye(4, dtype=f32) * f32(scale); Scw[:3, 3] = np.asarray(t, f32) * f32(scale); Scw[3, 3] = 1
    return dict(g=g, points=points, q=q, cat=cat, t=np.asarray(t, f32), Scw=Scw, rng=rng, src=src, in_frame_image=in_frame_image)


def _holders(rng, n, frac=0.3):
    return np.where(rng.random(n) < frac, rng.integers(1, 6, n), -1).astype(np.int32)


@pytest.mark.parametrize("seed,th", [(20, 3.0), (21, 5.0)])
def test_fuse(ref, seed, th):
    S = _scene(seed, th=th)
    rng = S["rng"]; m = len(S["cat"])
    held = _holders(rng, 900)
    in_kf = np.where(rng.random(m) < 0.08, rng.integers(0, 900, m), -1).astype(np.int32)      # IsInKeyFrame -> skipped
    dnr = (rng.random(m) < 0.05).astype(np.uint8)                                             # mbDoNotReplace -> skipped
    pts = dict(S["points"], index_in_kf=in_kf, do_not_replace=dnr)
    q = dict(S["q"], valid=(S["q"]["valid"].astype(bool) & (in_kf < 0) & (dnr == 0)).astype(np.uint8))
    got, n = ref.fuse_search(S["g"], q, sm.INV_LEVEL_SIGMA2)
    want, wn = ref.ref_fuse(S["g"], INTR, S["t"], held, pts, th)
    assert n == wn and n > 150                                   # nFused
    seen = want >= 0                                             # (a second point fused onto a replaced placeholder leaves no trace: not compared)
    assert same(got[seen], want[seen]) and seen.sum() >= 0.9 * n


@pytest.mark.parametrize("seed,th,scale", [(22, 4.0, 2.0), (23, 3.0, 0.5)])
def test_fuse_sim3(ref, seed, th, scale):
    S = _scene(seed, th=th, scale=scale)
    held = _holders(S["rng"], 900)
    got, n = ref.fuse_search(S["g"], S["q"], None)
    want, wn = ref.ref_fuse(S["g"], INTR, None, held, S["points"], th, Scw=S["Scw"])
    assert n == wn and same(got, want) and n > 150


@pytest.mark.parametrize("seed,scale", [(24, 2.0), (25, 1.0)])
def test_search_by_projection_sim3(ref, seed, scale):
    S = _scene(seed, th=10, scale=scale, th_is_int=True)
    rng = S["rng"]; m = len(S["cat"])
    matched = (rng.random(900) < 0.2).astype(np.uint8)
    existing = np.where(rng.random(m) < 0.12, rng.integers(0, 900, m), -1).astype(np.int32)
    existing[np.unique(existing[existing >= 0], return_index=True)[1]] = existing[np.unique(existing[existing >= 0], return_index=True)[1]]
    pts = dict(S["points"], index_in_kf=existing)
    best, mof, n = ref.search_by_projection_sim3(S["g"], S["q"], matched, existing)
    wmof, remap, wn = ref.ref_search_by_projection_sim3(S["g"], INTR, S["Scw"], pts, matched, 10)
    assert n == wn and same(mof, wmof) and n > 100
    # RemapMapPointMatch calls: (point, where it sat, where it goes) for every observed point that found a keypoint
    exp = [(i, int(existing[i]), int(best[i])) for i in range(m) if best[i] >= 0 and existing[i] >= 0]
    assert [tuple(r) for r in remap.tolist()] == exp and len(exp) > 10


def test_search_by_sim3(ref):
    rng = np.random.default_rng(26)
    fx, fy, cx, cy = [float(v) for v in INTR]
    g1 = sm.make_grid(n=700, seed=27, bounds=BOUNDS); g2 = sm.make_grid(n=720, seed=28, bounds=BOUNDS)
    share = rng.permutation(700)[:350]                           # keypoint share[k] of KF1 and keypoint k of KF2 see the same thing
    g2["desc"][:350] = sm.flip_bits(g1["desc"][share], rng.integers(0, 30, 350), rng); g2["octave"][:350] = g1["octave"][share]
    t1, t2, t12, s12 = np.array([0.5, 0.25, -1.0]), np.array([-0.25, 1.0, 0.5]), np.array([1.0, -0.5, 0.25]), 2.0

    def side(src_g, dst_g, src_idx, dst_idx, to_dst, t_src):
        """one map point per keypoint of the source keyframe; those in src_idx project next to dst_idx's keypoints in the other keyframe"""
        n = src_g["desc"].shape[0]
        uv = np.round(rng.uniform([30, 30], [720, 450], (n, 2)) * 4) / 4
        uv[src_idx] = np.round((dst_g["kp_xy"][dst_idx].astype(np.float64) + rng.normal(0, 1.0, (len(src_idx), 2))) * 4) / 4
        zc = rng.choice([2.0, 4.0, 8.0], n)
        c_dst = np.stack([(uv[:, 0] - cx) * zc / fx, (uv[:, 1] - cy) * zc / fy, zc], 1)   # in the destination camera
        world = to_dst(c_dst) - t_src                                                    # source camera frame -> world (R = I)
        assert same(world.astype(f32).astype(np.float64), world)
        dist = np.sqrt((c_dst * c_dst).sum(1)); level = src_g["octave"].astype(np.int32)
        valid = rng.random(n) < 0.85
        pts = dict(pos=world.astype(f32), min_dist=(dist / 3).astype(f32), max_dist=(dist * 1.2 ** (level - 0.5)).astype(f32), desc=src_g["desc"],
                   bad=(~valid).astype(np.uint8))
        q = dict(valid=valid.astype(np.uint8), uv=uv.astype(f32), radius=(f32(7.5) * SF[level]).astype(f32), level=level, desc=src_g["desc"])
        return pts, q
    # c2 = (1/s12) (c1 - t12)  <=>  c1 = s12 c2 + t12   (R12 = I), S/ORBmatcher.cpp:1139-1142
    p1, q12 = side(g1, g2, share, np.arange(350), lambda c2: s12 * c2 + t12, t1)
    p2, q21 = side(g2, g1, np.arange(350), share, lambda c1: (c1 - t12) / s12, t2)
    got, n = ref.search_by_sim3(g1, g2, q12, q21)
    want, wn = ref.ref_search_by_sim3(g1, g2, INTR, t1.astype(f32), t2.astype(f32), p1, np.arange(700), p2, np.arange(720), s12, np.eye(3, dtype=f32),
                                      t12.astype(f32), 7.5)
    assert n == wn and same(got, want) and n > 80


@pytest.mark.parametrize("seed,th,ori", [(30, 7.0, True), (31, 15.0, False)])
def test_search_by_projection_last_frame(ref, seed, th, ori):
    S = _scene(seed, n=900, m=800, th=th)                        # one map point per keypoint of the last frame
    rng = S["rng"]; m = 800
    g_last = sm.make_grid(n=m, seed=seed + 5, bounds=BOUNDS)
    g_last["octave"] = S["q"]["level"].copy()                    # nLastOctave drives the window and the level range
    g_last["angle"] = ((S["g"]["angle"][S["src"]] + rng.normal(0, 4, m) + np.where(rng.random(m) < 0.1, 120, 0)) % 360).astype(f32)
    has_point = rng.random(m) < 0.9; outlier = (rng.random(m) < 0.08).astype(np.uint8)
    last_point = np.where(has_point, np.arange(m), -1).astype(np.int32)
    blocked = (rng.random(900) < 0.2).astype(np.uint8)
    # what the reference lets through here (:1376-1396): a point, not an outlier, 1/z >= 0, inside [mnMin, mnMax] (inclusive)
    cat = S["cat"]
    ok = has_point & (outlier == 0) & (cat != CATS.index("behind")) & S["in_frame_image"]
    q = dict(S["q"], valid=ok.astype(np.uint8), angle=g_last["angle"])
    has_obs = (S["points"]["n_obs"] > 0).astype(np.uint8)
    got, n = ref.search_by_projection_frame(S["g"], q, has_obs, blocked, False, 100, ori)
    want, wn = ref.ref_search_by_projection_last(S["g"], g_last, INTR, S["t"], S["points"], last_point, outlier, blocked, th, ori)
    assert n == wn and same(np.where(got == -2, -1, got), want) and n > 150


@pytest.mark.parametrize("seed,th,orb_dist,ori", [(32, 10.0, 100, True), (33, 3.0, 64, False)])
def test_search_by_projection_relocalisation(ref, seed, th, orb_dist, ori):
    S = _scene(seed, n=900, m=800, th=th)
    rng = S["rng"]; m = 800
    g_kf = sm.make_grid(n=m, seed=seed + 5, bounds=BOUNDS)
    g_kf["angle"] = ((S["g"]["angle"][S["src"]] + rng.normal(0, 4, m) + np.where(rng.random(m) < 0.1, 120, 0)) % 360).astype(f32)
    has_point = rng.random(m) < 0.9; found = (rng.random(m) < 0.08).astype(np.uint8)
    kf_point = np.where(has_point, np.arange(m), -1).astype(np.int32)
    blocked = (rng.random(900) < 0.2).astype(np.uint8)
    # (:1500-1530): a good point not already found, inside the image, inside its distance range — this overload has neither a depth nor a
    # viewing-angle gate, so a point BEHIND the camera that projects into the image is searched like any other (1/z < 0 flips x and y back)
    cat = S["cat"]
    ok = has_point & (found == 0) & np.isin(cat, [CATS.index("good"), CATS.index("bad_angle"), CATS.index("behind")]) & S["in_frame_image"]
    q = dict(S["q"], valid=ok.astype(np.uint8), angle=g_kf["angle"])
    got, n = ref.search_by_projection_frame(S["g"], q, np.ones(m, np.uint8), blocked, True, orb_dist, ori)
    want, wn = ref.ref_search_by_projection_reloc(S["g"], g_kf, INTR, S["t"], S["points"], kf_point, found, blocked, th, orb_dist, ori)
    assert n == wn and same(np.where(got == -2, -1, got), want) and n > 150


# ---- the same scenes with ties everywhere ----------------------------------------------------------------------------------------
# Six descriptor patterns 8..30 bits apart: every search window holds several candidates at exactly the same distance, under the
# acceptance thresholds.  The outcome then rests on the visiting order alone — first minimum, second best on the same level, which query
# keeps a contested keypoint — and must still be the reference's, index for index.
@pytest.fixture
def ties():
    global TIES
    TIES = True
    yield
    TIES = False


def test_ties_projection_overloads(ref, ties):
    test_fuse(ref, 40, 4.0)
    test_fuse_sim3(ref, 41, 4.0, 2.0)
    test_search_by_projection_sim3(ref, 42, 2.0)
    test_search_by_projection_last_frame(ref, 43, 7.0, True)
    test_search_by_projection_relocalisation(ref, 44, 10.0, 100, False)


def test_ties_track_and_initialization(ref):
    # these two build their inputs with sm.make_grid / make_queries directly
    g = sm.make_grid(n=1200, seed=45); q = sm.make_queries(g, m=1500, seed=46)
    g, q = sm.tie_storm(g, q, pool=6, seed=47)
    rng = np.random.default_rng(48)
    m = 1500
    view_cos = np.where(rng.random(m) < 0.5, f32(0.9995), f32(0.9)).astype(f32)
    n_obs = np.where(rng.random(m) < 0.85, 3, 0).astype(np.int32); bad = (rng.random(m) < 0.05).astype(np.uint8)
    blocked = (rng.random(1200) < 0.2).astype(np.uint8)
    points = dict(desc=q["desc"], bad=bad, n_obs=n_obs, track_in_view=q["valid"], track_xy=q["uv"], track_level=q["level"], track_view_cos=view_cos)
    r = (np.where(view_cos > f32(0.998), f32(2.5), f32(4.0)).astype(f32) * f32(3.0)).astype(f32)
    oq = dict(q, valid=(q["valid"].astype(bool) & ~bad.astype(bool)).astype(np.uint8), radius=(r * SF[q["level"]]).astype(f32))
    for nnratio in (0.8, 1.0):                      # at 1.0 a tie between best and second best on one level still passes (d > ratio * d2 is false)
        got, n = ref.search_by_projection_track(g, oq, (n_obs > 0).astype(np.uint8), blocked, nnratio)
        want, wn = ref.ref_search_by_projection_track(g, points, blocked, 3.0, nnratio)
        assert n == wn and same(got, want)
    assert n > 100
    g2, qi = sm.make_init_pair(n=900, seed=49)
    g2, qi = sm.tie_storm(g2, qi, pool=6, seed=50)
    g1 = dict(desc=qi["desc"], kp_xy=qi["uv"], octave=qi["level"], angle=qi["angle"], bounds=g2["bounds"], cols=g2["cols"], rows=g2["rows"])
    for nnratio in (0.9, 1.01):
        got, n = ref.search_for_initialization(g2, qi, nnratio, True)
        want, wn, prev = ref.ref_search_for_initialization(g1, g2, qi["uv"], 100, nnratio, True)
        assert n == wn and same(got, want)
