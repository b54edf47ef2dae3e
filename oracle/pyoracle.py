"""ctypes binding of the CPU oracle (oracle/liboracle.so).  TEST INFRASTRUCTURE, NOT PRODUCT.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs import this module.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None
TRACE_COLS = 6


def build(force: bool = False) -> str:
    so = os.path.join(_HERE, "liboracle.so")
    srcs = [os.path.join(_HERE, f) for f in os.listdir(_HERE) if f.endswith((".cpp", ".hpp", ".h"))]
    if force or not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.check_call(["make", "-C", _HERE, "-s", "liboracle.so"])
    return so


class _BAProblem(C.Structure):
    _fields_ = [("K", C.c_int32), ("P", C.c_int32), ("E", C.c_int32),
                ("poses", C.c_void_p), ("intr", C.c_void_p), ("fixed", C.c_void_p), ("points", C.c_void_p),
                ("obs_kf", C.c_void_p), ("obs_mp", C.c_void_p), ("obs_uv", C.c_void_p), ("obs_w", C.c_void_p),
                ("edge_flags", C.c_void_p)]


class _BAOptions(C.Structure):
    _fields_ = [("iterations", C.c_int32), ("robust", C.c_int32), ("huber_delta", C.c_double),
                ("lambda_init", C.c_double), ("max_trials", C.c_int32), ("stop", C.c_void_p)]


class _BAResult(C.Structure):
    _fields_ = [("poses", C.c_void_p), ("points", C.c_void_p), ("chi2", C.c_void_p), ("depth_pos", C.c_void_p),
                ("trace", C.c_void_p), ("trace_cap", C.c_int32), ("trace_len", C.c_int32),
                ("iters_done", C.c_int32), ("trials_total", C.c_int32),
                ("chi2_initial", C.c_double), ("chi2_final", C.c_double), ("lambda_final", C.c_double),
                ("t_build_s", C.c_double), ("t_schur_s", C.c_double), ("t_solve_s", C.c_double),
                ("t_resid_s", C.c_double), ("t_total_s", C.c_double), ("t_structure_s", C.c_double)]


class _PGOProblem(C.Structure):
    _fields_ = [("K", C.c_int32), ("E", C.c_int32), ("sim3", C.c_void_p), ("fixed", C.c_void_p),
                ("edge_i", C.c_void_p), ("edge_j", C.c_void_p), ("meas", C.c_void_p), ("fix_scale", C.c_int32)]


class _PGOResult(C.Structure):
    _fields_ = [("sim3", C.c_void_p), ("trace", C.c_void_p), ("trace_cap", C.c_int32), ("trace_len", C.c_int32),
                ("iters_done", C.c_int32), ("chi2_initial", C.c_double), ("chi2_final", C.c_double),
                ("lambda_final", C.c_double), ("t_total_s", C.c_double)]


def lib():
    global _LIB
    if _LIB is None:
        _LIB = C.CDLL(build())
        _LIB.orc_ba_linearize.restype = C.c_double
    return _LIB


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _ba_struct(p, keep):
    arrs = dict(poses=np.ascontiguousarray(p.poses, np.float64), intr=np.ascontiguousarray(p.intr, np.float64),
                fixed=np.ascontiguousarray(p.fixed, np.uint8), points=np.ascontiguousarray(p.points, np.float64),
                obs_kf=np.ascontiguousarray(p.obs_kf, np.int32), obs_mp=np.ascontiguousarray(p.obs_mp, np.int32),
                obs_uv=np.ascontiguousarray(p.obs_uv, np.float32), obs_w=np.ascontiguousarray(p.obs_w, np.float32),
                edge_flags=None if p.edge_flags is None else np.ascontiguousarray(p.edge_flags, np.uint8))
    keep.append(arrs)
    return _BAProblem(p.K, p.P, p.E, *[_p(arrs[k]) for k in
                                      ("poses", "intr", "fixed", "points", "obs_kf", "obs_mp", "obs_uv", "obs_w", "edge_flags")])


def ba_solve(p, iterations=20, robust=True, huber_delta=np.sqrt(5.99), lambda_init=-1.0, max_trials=10,
             chi2_in=None, stop=None, fn=None):
    keep = []
    prob = _ba_struct(p, keep)
    poses = np.empty((p.K, 7)); points = np.empty((p.P, 3))
    chi2 = np.zeros(p.E) if chi2_in is None else np.array(chi2_in, np.float64)
    depth = np.zeros(p.E, np.uint8)
    trace = np.zeros((max(iterations, 1), TRACE_COLS))
    opt = _BAOptions(iterations, int(robust), float(huber_delta), float(lambda_init), max_trials, _p(stop))
    res = _BAResult(_p(poses), _p(points), _p(chi2), _p(depth), _p(trace), trace.shape[0])
    rc = (fn or lib().orc_ba_solve)(C.byref(prob), C.byref(opt), C.byref(res))
    assert rc == 0
    return dict(poses=poses, points=points, chi2=chi2, depth_pos=depth, trace=trace[:res.trace_len],
                iters_done=res.iters_done, trials_total=res.trials_total, chi2_initial=res.chi2_initial,
                chi2_final=res.chi2_final, lambda_final=res.lambda_final,
                timing=dict(build=res.t_build_s, schur=res.t_schur_s, solve=res.t_solve_s, resid=res.t_resid_s,
                            structure=res.t_structure_s, total=res.t_total_s))


def ba_linearize(p, robust=True, huber_delta=np.sqrt(5.99), fn=None):
    keep = []
    prob = _ba_struct(p, keep)
    err = np.empty((p.E, 2)); Jp = np.empty((p.E, 2, 6)); Jl = np.empty((p.E, 2, 3))
    rho1 = np.empty(p.E); chi2 = np.empty(p.E)
    fn = fn or lib().orc_ba_linearize
    fn.restype = C.c_double
    tot = fn(C.byref(prob), int(robust), C.c_double(huber_delta), _p(err), _p(Jp), _p(Jl), _p(rho1), _p(chi2))
    return dict(err=err, Jpose=Jp, Jpoint=Jl, rho1=rho1, chi2=chi2, chi2_robust_sum=tot)


def ba_build(p, robust=True, huber_delta=np.sqrt(5.99), fn=None):
    keep = []
    prob = _ba_struct(p, keep)
    Hpp = np.empty((p.K, 6, 6)); bp = np.empty((p.K, 6)); Hll = np.empty((p.P, 3, 3)); bl = np.empty((p.P, 3))
    W = np.empty((p.E, 6, 3))
    (fn or lib().orc_ba_build)(C.byref(prob), int(robust), C.c_double(huber_delta), _p(Hpp), _p(bp), _p(Hll), _p(bl), _p(W))
    return dict(Hpp=Hpp, bp=bp, Hll=Hll, bl=bl, W=W)


def ba_schur_solve(p, lam, robust=True, huber_delta=np.sqrt(5.99), dense=False):
    keep = []
    prob = _ba_struct(p, keep)
    dxp = np.empty((p.K, 6)); dxl = np.empty((p.P, 3))
    S = np.empty((6 * p.K, 6 * p.K)) if dense else None
    bs = np.empty(6 * p.K) if dense else None
    rc = lib().orc_ba_schur_solve(C.byref(prob), int(robust), C.c_double(huber_delta), C.c_double(lam), _p(dxp), _p(dxl), _p(S), _p(bs))
    return dict(rc=rc, dx_pose=dxp, dx_point=dxl, S=S, bschur=bs)


def _vec(fn, inp, nout):
    a = np.ascontiguousarray(inp, np.float64)
    o = np.empty(nout)
    fn(_p(a), _p(o))
    return o


def se3_exp(u): return _vec(lib().orc_se3_exp, u, 7)
def sim3_exp(u): return _vec(lib().orc_sim3_exp, u, 8)
def sim3_log(s): return _vec(lib().orc_sim3_log, s, 7)
def sim3_inv(s): return _vec(lib().orc_sim3_inv, s, 8)


def se3_mul(a, b):
    a = np.ascontiguousarray(a, np.float64); b = np.ascontiguousarray(b, np.float64); o = np.empty(7)
    lib().orc_se3_mul(_p(a), _p(b), _p(o)); return o


def sim3_mul(a, b):
    a = np.ascontiguousarray(a, np.float64); b = np.ascontiguousarray(b, np.float64); o = np.empty(8)
    lib().orc_sim3_mul(_p(a), _p(b), _p(o)); return o


def se3_map(qt, x):
    qt = np.ascontiguousarray(qt, np.float64); x = np.ascontiguousarray(x, np.float64); o = np.empty(3)
    lib().orc_se3_map(_p(qt), _p(x), _p(o)); return o


def pose_from_Tcw_f32(T):
    T = np.ascontiguousarray(T, np.float32); o = np.empty(7)
    lib().orc_pose_from_Tcw_f32(_p(T), _p(o)); return o


def pose_to_Tcw_f32(qt):
    qt = np.ascontiguousarray(qt, np.float64); o = np.empty((4, 4), np.float32)
    lib().orc_pose_to_Tcw_f32(_p(qt), _p(o)); return o


def huber(e, delta):
    o = np.empty(3)
    lib().orc_huber(C.c_double(e), C.c_double(delta), _p(o)); return o


def pgo_edge_error(meas, si, sj):
    m = np.ascontiguousarray(meas, np.float64); a = np.ascontiguousarray(si, np.float64); b = np.ascontiguousarray(sj, np.float64)
    o = np.empty(7)
    lib().orc_pgo_edge_error(_p(m), _p(a), _p(b), _p(o)); return o


def pgo_solve(p, iterations=20, lambda_init=1e-16, analytic_jac=False, stop=None, fn=None):
    arrs = dict(sim3=np.ascontiguousarray(p.sim3, np.float64), fixed=np.ascontiguousarray(p.fixed, np.uint8),
                ei=np.ascontiguousarray(p.edge_i, np.int32), ej=np.ascontiguousarray(p.edge_j, np.int32),
                meas=np.ascontiguousarray(p.meas, np.float64))
    K, E = arrs["sim3"].shape[0], arrs["ei"].shape[0]
    prob = _PGOProblem(K, E, _p(arrs["sim3"]), _p(arrs["fixed"]), _p(arrs["ei"]), _p(arrs["ej"]), _p(arrs["meas"]), int(p.fix_scale))
    out = np.empty((K, 8)); trace = np.zeros((max(iterations, 1), TRACE_COLS))
    res = _PGOResult(_p(out), _p(trace), trace.shape[0])
    rc = (fn or lib().orc_pgo_solve)(C.byref(prob), iterations, C.c_double(lambda_init), int(analytic_jac), _p(stop), C.byref(res))
    assert rc == 0
    return dict(sim3=out, trace=trace[:res.trace_len], iters_done=res.iters_done, chi2_initial=res.chi2_initial,
                chi2_final=res.chi2_final, lambda_final=res.lambda_final, t_total=res.t_total_s)


# ---- ORB extractor / matching ------------------------------------------------------------------------------------
class _OrbCfg(C.Structure):
    _fields_ = [("nfeatures", C.c_int32), ("scale_factor", C.c_float), ("nlevels", C.c_int32),
                ("ini_th_fast", C.c_int32), ("min_th_fast", C.c_int32), ("blur_2413", C.c_int32)]


class _KP(C.Structure):
    _fields_ = [("x", C.c_float), ("y", C.c_float), ("size", C.c_float), ("angle", C.c_float),
                ("response", C.c_float), ("octave", C.c_int32)]


KP_DTYPE = np.dtype([("x", "f4"), ("y", "f4"), ("size", "f4"), ("angle", "f4"), ("response", "f4"), ("octave", "i4")])


def orb_cfg(nfeatures=1000, scale_factor=1.2, nlevels=8, ini_th=20, min_th=7, blur_2413=0):
    return _OrbCfg(nfeatures, scale_factor, nlevels, ini_th, min_th, blur_2413)


def orb_extract(img, cfg=None, max_kp=8192):
    cfg = cfg or orb_cfg()
    img = np.ascontiguousarray(img, np.uint8)
    h, w = img.shape
    kps = np.zeros(max_kp, KP_DTYPE); desc = np.zeros((max_kp, 32), np.uint8); n = C.c_int()
    lib().orc_orb_extract(_p(img), w, h, w, C.byref(cfg), _p(kps), max_kp, C.byref(n), _p(desc))
    return kps[:n.value].copy(), desc[:n.value].copy()


def orb_tables(cfg, w, h):
    npl = np.zeros(cfg.nlevels, np.int32); umax = np.zeros(16, np.int32); wh = np.zeros((cfg.nlevels, 2), np.int32)
    lib().orc_orb_tables(C.byref(cfg), w, h, _p(npl), _p(umax), _p(wh))
    return npl, umax, wh


def resize_linear_u8(src, dw, dh):
    src = np.ascontiguousarray(src, np.uint8); dst = np.empty((dh, dw), np.uint8)
    lib().orc_resize_linear_u8(_p(src), src.shape[1], src.shape[0], _p(dst), dw, dh)
    return dst


def gaussian_blur7(src, taps2413=False):
    src = np.ascontiguousarray(src, np.uint8); dst = np.empty_like(src)
    lib().orc_gaussian_blur7(_p(src), src.shape[1], src.shape[0], _p(dst), int(taps2413))
    return dst


def fast(img, threshold, max_out=100000):
    img = np.ascontiguousarray(img, np.uint8)
    xy = np.zeros((max_out, 2), np.int32); sc = np.zeros(max_out, np.int32)
    n = lib().orc_fast(_p(img), img.shape[1], img.shape[0], threshold, _p(xy), _p(sc), max_out)
    return xy[:n], sc[:n]


def fast_atan2(y, x):
    f = lib().orc_fast_atan2
    f.restype = C.c_float
    return f(C.c_float(y), C.c_float(x))


def orb_level_candidates(img, cfg, level, max_out=200000):
    img = np.ascontiguousarray(img, np.uint8)
    out = np.zeros((max_out, 3), np.float32)
    n = lib().orc_orb_level_candidates(_p(img), img.shape[1], img.shape[0], C.byref(cfg), level, _p(out), max_out)
    return out[:n]


def orb_descriptor(img, x, y, angle):
    img = np.ascontiguousarray(img, np.uint8); d = np.zeros(32, np.uint8)
    lib().orc_orb_descriptor(_p(img), img.shape[1], img.shape[0], C.c_float(x), C.c_float(y), C.c_float(angle), _p(d))
    return d


def ic_angle(img, x, y):
    img = np.ascontiguousarray(img, np.uint8)
    f = lib().orc_ic_angle
    f.restype = C.c_float
    m01 = C.c_int(); m10 = C.c_int()
    a = f(_p(img), img.shape[1], img.shape[0], C.c_float(x), C.c_float(y), C.byref(m01), C.byref(m10))
    return a, m01.value, m10.value


class _FV(C.Structure):
    _fields_ = [("n_nodes", C.c_int32), ("node_id", C.c_void_p), ("node_ptr", C.c_void_p), ("feat", C.c_void_p)]


class FeatureVector:
    """Flattened DBoW2::FeatureVector: nodes ascending, features per node in insertion order."""

    def __init__(self, node_of_feature):
        node_of_feature = np.asarray(node_of_feature)
        order = np.argsort(node_of_feature, kind="stable")
        nodes, counts = np.unique(node_of_feature, return_counts=True)
        self.node_id = nodes.astype(np.uint32)
        self.node_ptr = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
        self.feat = order.astype(np.uint32)

    def c(self, cls=_FV):
        return cls(len(self.node_id), _p(self.node_id), _p(self.node_ptr), _p(self.feat))


def descriptor_distance(a, b):
    a = np.ascontiguousarray(a, np.uint8); b = np.ascontiguousarray(b, np.uint8)
    return lib().orc_descriptor_distance(_p(a), _p(b))


def match_bow_kf_frame(desc_kf, has_mp, ang_kf, fv_kf, desc_f, ang_f, fv_f, nnratio=0.7, check_ori=True):
    desc_kf = np.ascontiguousarray(desc_kf, np.uint8); desc_f = np.ascontiguousarray(desc_f, np.uint8)
    has_mp = np.ascontiguousarray(has_mp, np.uint8); ang_kf = np.ascontiguousarray(ang_kf, np.float32); ang_f = np.ascontiguousarray(ang_f, np.float32)
    out = np.empty(desc_f.shape[0], np.int32)
    fk, ff = fv_kf.c(), fv_f.c()
    n = lib().orc_match_bow_kf_frame(_p(desc_kf), desc_kf.shape[0], _p(has_mp), _p(ang_kf), C.byref(fk), _p(desc_f), desc_f.shape[0],
                                     _p(ang_f), C.byref(ff), C.c_float(nnratio), int(check_ori), _p(out))
    return out, n


def match_bow_kf_kf(d1, has1, a1, fv1, d2, has2, a2, fv2, nnratio=0.8, check_ori=True):
    d1 = np.ascontiguousarray(d1, np.uint8); d2 = np.ascontiguousarray(d2, np.uint8)
    has1 = np.ascontiguousarray(has1, np.uint8); has2 = np.ascontiguousarray(has2, np.uint8)
    a1 = np.ascontiguousarray(a1, np.float32); a2 = np.ascontiguousarray(a2, np.float32)
    out = np.empty(d1.shape[0], np.int32)
    f1, f2 = fv1.c(), fv2.c()
    n = lib().orc_match_bow_kf_kf(_p(d1), d1.shape[0], _p(has1), _p(a1), C.byref(f1), _p(d2), d2.shape[0], _p(has2), _p(a2), C.byref(f2),
                                  C.c_float(nnratio), int(check_ori), _p(out))
    return out, n


class _TriView(C.Structure):
    _fields_ = [("desc", C.c_void_p), ("n", C.c_int32), ("has_mp", C.c_void_p), ("kp_xy", C.c_void_p), ("octave", C.c_void_p),
                ("angle", C.c_void_p), ("fv", C.POINTER(_FV)), ("fx", C.c_float), ("fy", C.c_float), ("cx", C.c_float), ("cy", C.c_float)]


def match_triangulation(v1, v2, F12, ex, ey, level_sigma2, scale_factors, check_ori=False):
    """v = dict(desc, has_mp, kp_xy, octave, angle, fv, intr)"""
    keep = []

    def view(v):
        arrs = dict(desc=np.ascontiguousarray(v["desc"], np.uint8), has=np.ascontiguousarray(v["has_mp"], np.uint8),
                    xy=np.ascontiguousarray(v["kp_xy"], np.float32), oc=np.ascontiguousarray(v["octave"], np.int32),
                    an=np.ascontiguousarray(v["angle"], np.float32))
        fv = v["fv"].c(); keep.extend([arrs, fv])
        fx, fy, cx, cy = v["intr"]
        return _TriView(_p(arrs["desc"]), arrs["desc"].shape[0], _p(arrs["has"]), _p(arrs["xy"]), _p(arrs["oc"]), _p(arrs["an"]),
                        C.pointer(fv), fx, fy, cx, cy)
    a, b = view(v1), view(v2)
    F = np.ascontiguousarray(F12, np.float32); ls = np.ascontiguousarray(level_sigma2, np.float32); sf = np.ascontiguousarray(scale_factors, np.float32)
    pairs = np.empty((min(a.n, b.n) + 1, 2), np.int32)
    n = lib().orc_match_triangulation(C.byref(a), C.byref(b), _p(F), C.c_float(ex), C.c_float(ey), _p(ls), _p(sf), int(check_ori), _p(pairs))
    return pairs[:n].copy()


# ---- projection-guided matchers (proj_oracle.cpp) and the DBoW2 transform (bow_oracle.cpp) -----------------------------
class _Grid(C.Structure):
    _fields_ = [("n", C.c_int32), ("desc", C.c_void_p), ("kp_xy", C.c_void_p), ("octave", C.c_void_p), ("angle", C.c_void_p),
                ("min_x", C.c_float), ("min_y", C.c_float), ("max_x", C.c_float), ("max_y", C.c_float),
                ("grid_w_inv", C.c_float), ("grid_h_inv", C.c_float), ("grid_cols", C.c_int32), ("grid_rows", C.c_int32)]


class _Queries(C.Structure):
    _fields_ = [("m", C.c_int32), ("valid", C.c_void_p), ("uv", C.c_void_p), ("radius", C.c_void_p), ("level", C.c_void_p),
                ("desc", C.c_void_p), ("angle", C.c_void_p)]


def grid_struct(g, keep, cls=_Grid):
    """g = dict(desc, kp_xy, octave, angle, bounds=(min_x, min_y, max_x, max_y), cols, rows)"""
    a = dict(desc=np.ascontiguousarray(g["desc"], np.uint8), xy=np.ascontiguousarray(g["kp_xy"], np.float32),
             oc=np.ascontiguousarray(g["octave"], np.int32), an=np.ascontiguousarray(g["angle"], np.float32))
    keep.append(a)
    x0, y0, x1, y1 = [np.float32(v) for v in g["bounds"]]
    wi = np.float32(g["cols"]) / np.float32(x1 - x0); hi = np.float32(g["rows"]) / np.float32(y1 - y0)   # S/Frame.cpp:86-87
    return cls(a["desc"].shape[0], _p(a["desc"]), _p(a["xy"]), _p(a["oc"]), _p(a["an"]), x0, y0, x1, y1, wi, hi, int(g["cols"]), int(g["rows"]))


def queries_struct(q, keep, cls=_Queries):
    """q = dict(valid, uv, radius, level, desc, angle)"""
    a = dict(valid=np.ascontiguousarray(q["valid"], np.uint8), uv=np.ascontiguousarray(q["uv"], np.float32),
             r=np.ascontiguousarray(q["radius"], np.float32), lv=np.ascontiguousarray(q["level"], np.int32),
             desc=np.ascontiguousarray(q["desc"], np.uint8), an=np.ascontiguousarray(q.get("angle", np.zeros(len(q["valid"]))), np.float32))
    keep.append(a)
    return cls(a["valid"].shape[0], _p(a["valid"]), _p(a["uv"]), _p(a["r"]), _p(a["lv"]), _p(a["desc"]), _p(a["an"]))


def features_in_area(g, x, y, r, min_level=-1, max_level=-1):
    keep = []; G = grid_struct(g, keep)
    out = np.empty(G.n + 1, np.int32)
    n = lib().orc_features_in_area(C.byref(G), C.c_float(x), C.c_float(y), C.c_float(r), int(min_level), int(max_level), _p(out), G.n)
    return out[:n].copy()


def search_by_projection_track(g, q, query_has_obs, feat_blocked, nnratio=0.8):
    keep = []; G = grid_struct(g, keep); Q = queries_struct(q, keep)
    ho = np.ascontiguousarray(query_has_obs, np.uint8); fb = np.ascontiguousarray(feat_blocked, np.uint8)
    out = np.empty(G.n, np.int32)
    n = lib().orc_search_by_projection_track(C.byref(G), C.byref(Q), _p(ho), _p(fb), C.c_float(nnratio), _p(out))
    return out, n


def search_by_projection_frame(g, q, query_has_obs, feat_blocked, reloc=False, orb_dist=100, check_ori=True):
    keep = []; G = grid_struct(g, keep); Q = queries_struct(q, keep)
    ho = np.ascontiguousarray(query_has_obs, np.uint8); fb = np.ascontiguousarray(feat_blocked, np.uint8)
    out = np.empty(G.n, np.int32)
    n = lib().orc_search_by_projection_frame(C.byref(G), C.byref(Q), _p(ho), _p(fb), int(reloc), int(orb_dist), int(check_ori), _p(out))
    return out, n


def search_by_projection_sim3(g, q, feat_matched, existing_idx):
    keep = []; G = grid_struct(g, keep); Q = queries_struct(q, keep)
    fm = np.ascontiguousarray(feat_matched, np.uint8); ex = np.ascontiguousarray(existing_idx, np.int32)
    best = np.empty(Q.m, np.int32); out = np.empty(G.n, np.int32)
    n = lib().orc_search_by_projection_sim3(C.byref(G), C.byref(Q), _p(fm), _p(ex), _p(best), _p(out))
    return best, out, n


def fuse_search(g, q, inv_level_sigma2=None):
    keep = []; G = grid_struct(g, keep); Q = queries_struct(q, keep)
    w = None if inv_level_sigma2 is None else np.ascontiguousarray(inv_level_sigma2, np.float32)
    best = np.empty(Q.m, np.int32)
    n = lib().orc_fuse_search(C.byref(G), C.byref(Q), _p(w), _p(best))
    return best, n


def search_by_sim3(g1, g2, q12, q21):
    keep = []; G1 = grid_struct(g1, keep); G2 = grid_struct(g2, keep); Q12 = queries_struct(q12, keep); Q21 = queries_struct(q21, keep)
    out = np.empty(Q12.m, np.int32)
    n = lib().orc_search_by_sim3(C.byref(G1), C.byref(G2), C.byref(Q12), C.byref(Q21), _p(out))
    return out, n


def search_for_initialization(g2, q, nnratio=0.9, check_ori=True):
    keep = []; G = grid_struct(g2, keep); Q = queries_struct(q, keep)
    out = np.empty(Q.m, np.int32)
    n = lib().orc_search_for_initialization(C.byref(G), C.byref(Q), C.c_float(nnratio), int(check_ori), _p(out))
    return out, n


class Vocabulary:
    """v = dict(k, L, scoring, weighting, parent, is_leaf, desc, weight) with row 0 = root (ccm_slam_b200.synth.make_vocabulary)."""

    def __init__(self, v):
        self.parent = np.ascontiguousarray(v["parent"], np.int32); self.is_leaf = np.ascontiguousarray(v["is_leaf"], np.uint8)
        self.desc = np.ascontiguousarray(v["desc"], np.uint8); self.weight = np.ascontiguousarray(v["weight"], np.float64)
        f = lib().orc_voc_create; f.restype = C.c_void_p
        self.h = f(int(v["k"]), int(v["L"]), int(v["scoring"]), int(v["weighting"]), len(self.parent), _p(self.parent), _p(self.is_leaf),
                   _p(self.desc), _p(self.weight))
        assert self.h, "malformed vocabulary"

    def transform(self, feat, levelsup=4):
        feat = np.ascontiguousarray(feat, np.uint8); n = feat.shape[0]
        word = np.empty(n, np.uint32); node = np.empty(n, np.uint32); w = np.empty(n, np.float64)
        bid = np.empty(n, np.uint32); bval = np.empty(n, np.float64); bn = C.c_int32()
        fid = np.empty(n, np.uint32); fptr = np.empty(n + 1, np.int32); ff = np.empty(n, np.uint32); fn = C.c_int32()
        lib().orc_voc_transform(C.c_void_p(self.h), _p(feat), n, int(levelsup), _p(word), _p(node), _p(w), _p(bid), _p(bval), C.byref(bn),
                                _p(fid), _p(fptr), _p(ff), C.byref(fn))
        return dict(word=word, node=node, weight=w, bow_id=bid[:bn.value].copy(), bow_val=bval[:bn.value].copy(),
                    fv_node_id=fid[:fn.value].copy(), fv_node_ptr=fptr[:fn.value + 1].copy(), fv_feat=ff[:fptr[fn.value] if fn.value else 0].copy())

    def close(self):
        if self.h:
            lib().orc_voc_destroy(C.c_void_p(self.h)); self.h = None


# ---- the reference's own DBoW2, compiled in place by `make -C oracle ref` (only where /root/reference exists) ---------------
_REF_DBOW2 = None


def build_ref() -> str | None:
    """oracle/_ref/libdbow2_ref.so from the reference's DBoW2 sources (nothing copied); None where the reference tree is absent
    and no prebuilt library travelled with the repository."""
    so = os.path.join(_HERE, "_ref", "libdbow2_ref.so")
    if os.path.isdir("/root/reference/cslam/thirdparty/DBoW2"):
        subprocess.check_call(["make", "-C", _HERE, "-s", "-j", str(min(8, os.cpu_count() or 1)), "ref"])
    return so if os.path.exists(so) else None


def ref_dbow2():
    global _REF_DBOW2
    if _REF_DBOW2 is None:
        so = build_ref()
        if so is None:
            return None
        _REF_DBOW2 = C.CDLL(so)
        _REF_DBOW2.ref_voc_load.restype = C.c_void_p
    return _REF_DBOW2


def ref_orb_cli():
    """oracle/_ref/orb_ref_cli: the reference's own ORBextractor.cpp on the oracle's OpenCV-primitive restatements; None if absent"""
    if build_ref() is None:
        return None
    exe = os.path.join(_HERE, "_ref", "orb_ref_cli")
    return exe if os.path.exists(exe) else None


def ref_orb_extract(img, cfg=None, allocator="bump"):
    """ORBextractor::operator() of the reference itself (cslam/src/ORBextractor.cpp) -> (keypoints, descriptors) like orb_extract.
    allocator: "bump" = monotone addresses (pointer ties of DistributeOctTree follow creation order), "malloc" = glibc."""
    import tempfile
    cfg = cfg or orb_cfg()
    img = np.ascontiguousarray(img, np.uint8)
    with tempfile.TemporaryDirectory() as d:
        fin, fout = os.path.join(d, "in.raw"), os.path.join(d, "out.bin")
        img.tofile(fin)
        subprocess.check_call([ref_orb_cli(), fin, str(img.shape[1]), str(img.shape[0]), str(cfg.nfeatures), repr(float(cfg.scale_factor)),
                               str(cfg.nlevels), str(cfg.ini_th_fast), str(cfg.min_th_fast), str(cfg.blur_2413), allocator, fout])
        raw = open(fout, "rb").read()
    n = int(np.frombuffer(raw[:4], np.int32)[0])
    kps = np.frombuffer(raw[4:4 + n * KP_DTYPE.itemsize], KP_DTYPE).copy()
    desc = np.frombuffer(raw[4 + n * KP_DTYPE.itemsize:], np.uint8).reshape(n, 32).copy()
    return kps, desc


# ---- the reference's own Levenberg-Marquardt driver on the oracle's linear algebra (oracle/_ref/liblm_ref.so) -------------------------
_REF_LM = None


def ref_lm():
    global _REF_LM
    if _REF_LM is None:
        if build_ref() is None:
            return None
        so = os.path.join(_HERE, "_ref", "liblm_ref.so")
        if not os.path.exists(so):
            return None
        _REF_LM = C.CDLL(so)
    return _REF_LM


_REF_BA_FULL = None


def ref_ba_full():
    global _REF_BA_FULL
    if _REF_BA_FULL is None:
        if build_ref() is None:
            return None
        so = os.path.join(_HERE, "_ref", "libba_full_ref.so")
        if not os.path.exists(so):
            return None
        _REF_BA_FULL = C.CDLL(so)
    return _REF_BA_FULL


def ref_ba_full_solve(p, **kw):
    """ba_solve() where the reference's LM driver runs over the reference's own vertices, edges and kernels (oracle/ref_ba_full_wrap.cpp);
    only the Schur complement + LDL^T under Solver::solve() are the oracle's."""
    return ba_solve(p, fn=ref_ba_full().ref_ba_full_solve, **kw)


_REF_BA_BLOCK = None


def ref_ba_block():
    global _REF_BA_BLOCK
    if _REF_BA_BLOCK is None:
        if build_ref() is None:
            return None
        so = os.path.join(_HERE, "_ref", "libba_block_ref.so")
        if not os.path.exists(so):
            return None
        _REF_BA_BLOCK = C.CDLL(so)
    return _REF_BA_BLOCK


def ref_ba_block_solve(p, **kw):
    """ba_solve() with the reference's LM driver, vertices / edges / kernels AND its BlockSolver_6_3 (structure, Schur complement,
    back-substitution); the oracle supplies only the sparse LDL^T under LinearSolver::solve (oracle/ref_ba_block_wrap.cpp).
    Trace columns 1 and 3 are NaN."""
    return ba_solve(p, fn=ref_ba_block().ref_ba_block_solve, **kw)


def ref_ba_solve(p, **kw):
    """ba_solve() with g2o's own OptimizationAlgorithmLevenberg::solve (compiled from the reference tree, oracle/ref_lm_wrap.cpp)
    deciding lambda, trials and termination; trace column 3 (rho) is NaN — it is a local of the reference's function."""
    return ba_solve(p, fn=ref_lm().ref_lm_solve, **kw)


# ---- g2o's own vertex / edge types, Lie groups and Huber kernel (oracle/_ref/libg2o_types_ref.so, oracle/ref_g2o_wrap.cpp) ---------------
_REF_G2O = None


def ref_g2o():
    global _REF_G2O
    if _REF_G2O is None:
        if build_ref() is None:
            return None
        so = os.path.join(_HERE, "_ref", "libg2o_types_ref.so")
        if not os.path.exists(so):
            return None
        _REF_G2O = C.CDLL(so)
    return _REF_G2O


class Pieces:
    """The same piece-level entry points on either side: which='oracle' (liboracle.so, orc_*) or 'ref' (the reference's compiled
    g2o types, ref_*).  Arrays in, arrays out; layouts as in oracle.h."""

    def __init__(self, which):
        self.l = lib() if which == "oracle" else ref_g2o()
        self.pre = "orc_" if which == "oracle" else "ref_"

    def _f(self, name):
        return getattr(self.l, self.pre + name)

    def vec(self, name, nout, *ins):
        arrs = [np.ascontiguousarray(a, np.float64) for a in ins]
        o = np.empty(nout)
        self._f(name)(*[_p(a) for a in arrs], _p(o))
        return o

    def huber(self, e, delta):
        o = np.empty(3)
        self._f("huber")(C.c_double(e), C.c_double(delta), _p(o))
        return o

    def ba_linearize(self, p, **kw):
        return ba_linearize(p, fn=self._f("ba_linearize"), **kw)

    def ba_build(self, p, **kw):
        return ba_build(p, fn=self._f("ba_build"), **kw)

    def pose_opt_build(self, Tcw, Xw, uv, inv_sigma2, intr, robust, delta):
        a = dict(Tcw=np.ascontiguousarray(Tcw, np.float64), Xw=np.ascontiguousarray(Xw, np.float32).reshape(-1, 3),
                 uv=np.ascontiguousarray(uv, np.float32).reshape(-1, 2), w=np.ascontiguousarray(inv_sigma2, np.float32))
        n = a["Xw"].shape[0]
        prob = _PoseOpt(n, _p(a["Tcw"]), _p(a["Xw"]), _p(a["uv"]), _p(a["w"]), *[float(v) for v in intr])
        H = np.empty((6, 6)); b = np.empty(6); err = np.empty((n, 2))
        self._f("pose_opt_build")(C.byref(prob), _p(a["Tcw"]), int(robust), C.c_double(delta), _p(H), _p(b), _p(err))
        return H, b, err

    def sim3_opt_build(self, S12, P1c, P2c, uv1, uv2, w1, w2, K1, K2, fix_scale, robust, delta):
        f32 = lambda x, c: np.ascontiguousarray(x, np.float32).reshape(-1, c) if c else np.ascontiguousarray(x, np.float32)
        a = dict(S=np.ascontiguousarray(S12, np.float64), P1=f32(P1c, 3), P2=f32(P2c, 3), u1=f32(uv1, 2), u2=f32(uv2, 2), w1=f32(w1, 0), w2=f32(w2, 0))
        n = a["P1"].shape[0]
        prob = _Sim3Opt(n, _p(a["S"]), _p(a["P1"]), _p(a["P2"]), _p(a["u1"]), _p(a["u2"]), _p(a["w1"]), _p(a["w2"]),
                        (C.c_float * 4)(*[float(v) for v in K1]), (C.c_float * 4)(*[float(v) for v in K2]), 0.0, int(bool(fix_scale)))
        H = np.empty((7, 7)); b = np.empty(7); err = np.empty((2 * n, 2))
        self._f("sim3_opt_build")(C.byref(prob), _p(a["S"]), int(robust), C.c_double(delta), _p(H), _p(b), _p(err))
        return H, b, err

    def pgo_edge_jacobian(self, meas, si, sj, fix_scale):
        m, a, b = [np.ascontiguousarray(v, np.float64) for v in (meas, si, sj)]
        Ji = np.empty((7, 7)); Jj = np.empty((7, 7))
        self._f("pgo_edge_jacobian")(_p(m), _p(a), _p(b), int(bool(fix_scale)), _p(Ji), _p(Jj))
        return Ji, Jj


def ref_vertex_oplus(kind, est, upd, flag=0):
    """the reference's VertexSE3Expmap (kind 0) / VertexSim3Expmap (1, flag = _fix_scale) / VertexSBAPointXYZ (2) ::oplus"""
    e = np.ascontiguousarray(est, np.float64); u = np.ascontiguousarray(upd, np.float64); o = np.empty(len(e))
    ref_g2o().ref_vertex_oplus(int(kind), _p(e), _p(u), int(flag), _p(o))
    return o


# ---- the reference's own ORBmatcher.cpp on stand-in Frame / KeyFrame / MapPoint (oracle/_ref/libmatch_ref.so) -----------------------
_REF_MATCH = None
_SHIM_MATCH = {}
_MATCH_SIDE = "ref"


def ref_match():
    """the matcher library the ref_* wrappers below talk to: the reference's own ORBmatcher.cpp (default) or, inside
    `with matcher_side("shim")`, this repository's shim/ORBmatcher*_shim.cpp built over the same stand-in classes"""
    global _REF_MATCH, _SHIM_MATCH
    if _MATCH_SIDE in ("shim", "shim_gpu"):     # "shim": device half doubled on the CPU; "shim_gpu": the real device entry points
        if _SHIM_MATCH.get(_MATCH_SIDE) is None:
            so = os.path.join(_HERE, "_ref", "libmatch_shim.so" if _MATCH_SIDE == "shim" else "libmatch_shim_gpu.so")
            if build_ref() is None or not os.path.exists(so):
                return None
            _SHIM_MATCH[_MATCH_SIDE] = C.CDLL(so)
        return _SHIM_MATCH[_MATCH_SIDE]
    if _REF_MATCH is None:
        if build_ref() is None:
            return None
        so = os.path.join(_HERE, "_ref", "libmatch_ref.so")
        if not os.path.exists(so):
            return None
        _REF_MATCH = C.CDLL(so)
    return _REF_MATCH


class matcher_side:
    def __init__(self, side):
        self.side = side

    def __enter__(self):
        global _MATCH_SIDE
        self.prev, _MATCH_SIDE = _MATCH_SIDE, self.side

    def __exit__(self, *a):
        global _MATCH_SIDE
        _MATCH_SIDE = self.prev


class _RefImage(C.Structure):
    _fields_ = [("n", C.c_int32), ("desc", C.c_void_p), ("kp_xy", C.c_void_p), ("octave", C.c_void_p), ("angle", C.c_void_p),
                ("min_x", C.c_float), ("min_y", C.c_float), ("max_x", C.c_float), ("max_y", C.c_float), ("grid_w_inv", C.c_float),
                ("grid_h_inv", C.c_float), ("grid_cols", C.c_int32), ("grid_rows", C.c_int32),
                ("fx", C.c_float), ("fy", C.c_float), ("cx", C.c_float), ("cy", C.c_float), ("R", C.c_void_p), ("t", C.c_void_p),
                ("nlevels", C.c_int32), ("scale_factors", C.c_void_p), ("level_sigma2", C.c_void_p), ("inv_level_sigma2", C.c_void_p),
                ("log_scale_factor", C.c_float), ("fv", C.POINTER(_FV))]


class _RefPoints(C.Structure):
    _fields_ = [("m", C.c_int32), ("pos", C.c_void_p), ("normal", C.c_void_p), ("min_dist", C.c_void_p), ("max_dist", C.c_void_p),
                ("desc", C.c_void_p), ("bad", C.c_void_p), ("do_not_replace", C.c_void_p), ("n_obs", C.c_void_p), ("index_in_kf", C.c_void_p),
                ("track_in_view", C.c_void_p), ("track_xy", C.c_void_p), ("track_level", C.c_void_p), ("track_view_cos", C.c_void_p)]


def ref_image_struct(g, keep, intr=(0, 0, 0, 0), R=None, t=None, fv=None, nlevels=8, scale_factor=1.2):
    """g: grid dict (desc, kp_xy, octave, angle, bounds, cols, rows); cols = 0 -> no lookup grid.  Level tables as ORBextractor builds them."""
    a = dict(desc=np.ascontiguousarray(g["desc"], np.uint8), xy=np.ascontiguousarray(g["kp_xy"], np.float32),
             oc=np.ascontiguousarray(g["octave"], np.int32), an=np.ascontiguousarray(g["angle"], np.float32))
    sf = np.empty(nlevels, np.float32); sf[0] = 1.0
    for i in range(1, nlevels):
        sf[i] = np.float32(sf[i - 1] * np.float32(scale_factor))
    a["sf"] = sf; a["ls2"] = (sf * sf).astype(np.float32); a["ils2"] = (np.float32(1.0) / a["ls2"]).astype(np.float32)
    a["R"] = None if R is None else np.ascontiguousarray(R, np.float32); a["t"] = None if t is None else np.ascontiguousarray(t, np.float32)
    cfv = None
    if fv is not None:
        cfv = fv.c(); a["fv"] = (fv, cfv)
    keep.append(a)
    x0, y0, x1, y1 = [np.float32(v) for v in g.get("bounds", (0, 0, 1, 1))]
    cols, rows = int(g.get("cols", 0)), int(g.get("rows", 0))
    wi = np.float32(cols) / np.float32(x1 - x0) if cols else np.float32(0); hi = np.float32(rows) / np.float32(y1 - y0) if rows else np.float32(0)
    fx, fy, cx, cy = [np.float32(v) for v in intr]
    return _RefImage(a["desc"].shape[0], _p(a["desc"]), _p(a["xy"]), _p(a["oc"]), _p(a["an"]), x0, y0, x1, y1, wi, hi, cols, rows, fx, fy, cx, cy,
                     _p(a["R"]), _p(a["t"]), nlevels, _p(a["sf"]), _p(a["ls2"]), _p(a["ils2"]), np.float32(np.log(np.float32(scale_factor))),
                     C.pointer(cfv) if cfv is not None else None)


def ref_points_struct(p, keep):
    """p: dict with any of pos, normal, min_dist, max_dist, desc, bad, do_not_replace, n_obs, index_in_kf, track_in_view, track_xy, track_level, track_view_cos"""
    m = len(p["desc"])
    spec = dict(pos=np.float32, normal=np.float32, min_dist=np.float32, max_dist=np.float32, desc=np.uint8, bad=np.uint8, do_not_replace=np.uint8,
                n_obs=np.int32, index_in_kf=np.int32, track_in_view=np.uint8, track_xy=np.float32, track_level=np.int32, track_view_cos=np.float32)
    a = {k: (np.ascontiguousarray(p[k], dt) if k in p and p[k] is not None else None) for k, dt in spec.items()}
    keep.append(a)
    return _RefPoints(m, *[_p(a[k]) for k in ("pos", "normal", "min_dist", "max_dist", "desc", "bad", "do_not_replace", "n_obs", "index_in_kf",
                                               "track_in_view", "track_xy", "track_level", "track_view_cos")])


def _plain(desc, angle, octave=None, xy=None):
    n = len(desc)
    return dict(desc=desc, kp_xy=np.zeros((n, 2), np.float32) if xy is None else xy, octave=np.zeros(n, np.int32) if octave is None else octave,
                angle=angle)


def ref_descriptor_distance(a, b):
    """ORBmatcher::DescriptorDistance of the matcher library"""
    a = np.ascontiguousarray(a, np.uint8); b = np.ascontiguousarray(b, np.uint8)
    return ref_match().ref_descriptor_distance(_p(a), _p(b))


def ref_match_bow_kf_frame(desc_kf, has_mp, ang_kf, fv_kf, desc_f, ang_f, fv_f, nnratio=0.7, check_ori=True):
    keep = []; K = ref_image_struct(_plain(desc_kf, ang_kf), keep, fv=fv_kf); F = ref_image_struct(_plain(desc_f, ang_f), keep, fv=fv_f)
    has = np.ascontiguousarray(has_mp, np.uint8); out = np.empty(len(desc_f), np.int32)
    n = ref_match().ref_match_bow_kf_frame(C.byref(K), _p(has), C.byref(F), C.c_float(nnratio), int(check_ori), _p(out))
    return out, n


def ref_match_bow_kf_kf(d1, has1, a1, fv1, d2, has2, a2, fv2, nnratio=0.8, check_ori=True):
    keep = []; K1 = ref_image_struct(_plain(d1, a1), keep, fv=fv1); K2 = ref_image_struct(_plain(d2, a2), keep, fv=fv2)
    h1 = np.ascontiguousarray(has1, np.uint8); h2 = np.ascontiguousarray(has2, np.uint8); out = np.empty(len(d1), np.int32)
    n = ref_match().ref_match_bow_kf_kf(C.byref(K1), _p(h1), C.byref(K2), _p(h2), C.c_float(nnratio), int(check_ori), _p(out))
    return out, n


def ref_match_triangulation(v1, v2, F12, Cw, check_ori=False):
    """v = dict(desc, has_mp, kp_xy, octave, angle, fv, intr); Cw = camera centre of keyframe 1 in world = in camera 2 (its pose is identity)"""
    keep = []
    Cw = np.asarray(Cw, np.float32)
    K1 = ref_image_struct(_plain(v1["desc"], v1["angle"], v1["octave"], v1["kp_xy"]), keep, intr=v1["intr"], t=-Cw, fv=v1["fv"])
    K2 = ref_image_struct(_plain(v2["desc"], v2["angle"], v2["octave"], v2["kp_xy"]), keep, intr=v2["intr"], fv=v2["fv"])
    h1 = np.ascontiguousarray(v1["has_mp"], np.uint8); h2 = np.ascontiguousarray(v2["has_mp"], np.uint8)
    F = np.ascontiguousarray(F12, np.float32); pairs = np.empty((min(K1.n, K2.n) + 1, 2), np.int32)
    n = ref_match().ref_match_triangulation(C.byref(K1), _p(h1), C.byref(K2), _p(h2), _p(F), int(check_ori), _p(pairs))
    return pairs[:n].copy()


def ref_search_for_initialization(g1, g2, prev_matched, window, nnratio=0.9, check_ori=True):
    keep = []; F1 = ref_image_struct(g1, keep); F2 = ref_image_struct(g2, keep)
    prev = np.ascontiguousarray(prev_matched, np.float32).copy(); out = np.empty(F1.n, np.int32)
    n = ref_match().ref_search_for_initialization(C.byref(F1), C.byref(F2), _p(prev), int(window), C.c_float(nnratio), int(check_ori), _p(out))
    return out, n, prev


def ref_search_by_projection_track(g, points, feat_blocked, th, nnratio=0.8):
    keep = []; F = ref_image_struct(g, keep); P = ref_points_struct(points, keep)
    fb = np.ascontiguousarray(feat_blocked, np.uint8); out = np.empty(F.n, np.int32)
    n = ref_match().ref_search_by_projection_track(C.byref(F), C.byref(P), _p(fb), C.c_float(th), C.c_float(nnratio), _p(out))
    return out, n


def ref_fuse(g, intr, t, kf_mp_obs, points, th, Scw=None):
    """Fuse(pKF, vpMapPoints, th) (Scw None) or Fuse(pKF, Scw, vpPoints, th, vpReplacePoint) -> (best_idx per point, nFused)"""
    keep = []; K = ref_image_struct(g, keep, intr=intr, t=t); P = ref_points_struct(points, keep)
    obs = np.ascontiguousarray(kf_mp_obs, np.int32); best = np.empty(P.m, np.int32)
    if Scw is None:
        n = ref_match().ref_fuse(C.byref(K), _p(obs), C.byref(P), C.c_float(th), _p(best))
    else:
        S = np.ascontiguousarray(Scw, np.float32)
        n = ref_match().ref_fuse_sim3(C.byref(K), _p(obs), _p(S), C.byref(P), C.c_float(th), _p(best))
    return best, n


def ref_search_by_projection_sim3(g, intr, Scw, points, feat_matched, th):
    keep = []; K = ref_image_struct(g, keep, intr=intr); P = ref_points_struct(points, keep)
    S = np.ascontiguousarray(Scw, np.float32); fm = np.ascontiguousarray(feat_matched, np.uint8)
    mof = np.empty(K.n, np.int32); remap = np.empty((P.m + 1, 3), np.int32); nr = C.c_int32()
    n = ref_match().ref_search_by_projection_sim3(C.byref(K), _p(S), C.byref(P), _p(fm), int(th), _p(mof), _p(remap), C.byref(nr))
    return mof, remap[:nr.value].copy(), n


def ref_search_by_sim3(g1, g2, intr, t1, t2, pts1, p1_of_feat, pts2, p2_of_feat, s12, R12, t12, th):
    keep = []; K1 = ref_image_struct(g1, keep, intr=intr, t=t1); K2 = ref_image_struct(g2, keep, intr=intr, t=t2)
    P1 = ref_points_struct(pts1, keep); P2 = ref_points_struct(pts2, keep)
    a = np.ascontiguousarray(p1_of_feat, np.int32); b = np.ascontiguousarray(p2_of_feat, np.int32)
    R = np.ascontiguousarray(R12, np.float32); t = np.ascontiguousarray(t12, np.float32); out = np.empty(K1.n, np.int32)
    n = ref_match().ref_search_by_sim3(C.byref(K1), C.byref(K2), C.byref(P1), _p(a), C.byref(P2), _p(b), C.c_float(s12), _p(R), _p(t), C.c_float(th), _p(out))
    return out, n


def ref_search_by_projection_last(g_cur, g_last, intr, t_cur, points, last_point, last_outlier, feat_blocked, th, check_ori=True):
    keep = []; Cur = ref_image_struct(g_cur, keep, intr=intr, t=t_cur); Last = ref_image_struct(g_last, keep, intr=intr)
    P = ref_points_struct(points, keep)
    lp = np.ascontiguousarray(last_point, np.int32); lo = np.ascontiguousarray(last_outlier, np.uint8); fb = np.ascontiguousarray(feat_blocked, np.uint8)
    out = np.empty(Cur.n, np.int32)
    n = ref_match().ref_search_by_projection_last(C.byref(Cur), C.byref(Last), C.byref(P), _p(lp), _p(lo), _p(fb), C.c_float(th), int(check_ori), _p(out))
    return out, n


def ref_search_by_projection_reloc(g_cur, g_kf, intr, t_cur, points, kf_point, already_found, feat_blocked, th, orb_dist, check_ori=True):
    keep = []; Cur = ref_image_struct(g_cur, keep, intr=intr, t=t_cur); KF = ref_image_struct(g_kf, keep, intr=intr)
    P = ref_points_struct(points, keep)
    kp = np.ascontiguousarray(kf_point, np.int32); af = np.ascontiguousarray(already_found, np.uint8); fb = np.ascontiguousarray(feat_blocked, np.uint8)
    out = np.empty(Cur.n, np.int32)
    n = ref_match().ref_search_by_projection_reloc(C.byref(Cur), C.byref(KF), C.byref(P), _p(kp), _p(af), _p(fb), C.c_float(th), int(orb_dist),
                                                   int(check_ori), _p(out))
    return out, n


def write_vocabulary_text(v, path):
    """the rows of make_vocabulary() in the format TemplatedVocabulary::saveToTextFile writes and loadFromTextFile reads
    (D/TemplatedVocabulary.h:1428-1448, :1338-1422); no trailing newline (the loader turns an empty last line into a node)"""
    lines = ["%d %d  %d %d" % (v["k"], v["L"], v["scoring"], v["weighting"])]
    for i in range(1, len(v["parent"])):
        lines.append("%d %d %s %r" % (v["parent"][i], 1 if v["is_leaf"][i] else 0, " ".join(str(int(b)) for b in v["desc"][i]), float(v["weight"][i])))
    with open(path, "w") as f:
        f.write("\n".join(lines))


class RefVocabulary:
    """DBoW2::TemplatedVocabulary<FORB> of the reference itself, loaded from a text file"""

    def __init__(self, path):
        self.lib = ref_dbow2()
        assert self.lib is not None, "oracle/_ref/libdbow2_ref.so is not available"
        self.h = self.lib.ref_voc_load(path.encode())
        assert self.h, "loadFromTextFile failed"

    def words(self):
        return self.lib.ref_voc_words(C.c_void_p(self.h))

    def transform(self, feat, levelsup=4):
        feat = np.ascontiguousarray(feat, np.uint8); n = feat.shape[0]
        word = np.empty(n, np.uint32); node = np.empty(n, np.uint32); w = np.empty(n, np.float64)
        bid = np.empty(n, np.uint32); bval = np.empty(n, np.float64); bn = C.c_int32()
        fid = np.empty(n, np.uint32); fptr = np.empty(n + 1, np.int32); ff = np.empty(n, np.uint32); fn = C.c_int32()
        self.lib.ref_voc_transform(C.c_void_p(self.h), _p(feat), n, int(levelsup), _p(word), _p(node), _p(w), _p(bid), _p(bval), C.byref(bn),
                                   _p(fid), _p(fptr), _p(ff), C.byref(fn))
        return dict(word=word, node=node, weight=w, bow_id=bid[:bn.value].copy(), bow_val=bval[:bn.value].copy(),
                    fv_node_id=fid[:fn.value].copy(), fv_node_ptr=fptr[:fn.value + 1].copy(), fv_feat=ff[:fptr[fn.value] if fn.value else 0].copy())

    def close(self):
        if self.h:
            self.lib.ref_voc_free(C.c_void_p(self.h)); self.h = None


def ref_forb_distance(a, b):
    a = np.ascontiguousarray(a, np.uint8); b = np.ascontiguousarray(b, np.uint8)
    return ref_dbow2().ref_forb_distance(_p(a), _p(b))


# ---- single-vertex optimisations (PoseOptimizationClient, OptimizeSim3) ---------------------------------------------
class _PoseOpt(C.Structure):
    _fields_ = [("n", C.c_int32), ("Tcw", C.c_void_p), ("Xw", C.c_void_p), ("uv", C.c_void_p), ("inv_sigma2", C.c_void_p),
                ("fx", C.c_float), ("fy", C.c_float), ("cx", C.c_float), ("cy", C.c_float)]


class _Sim3Opt(C.Structure):
    _fields_ = [("n", C.c_int32), ("S12", C.c_void_p), ("P1c", C.c_void_p), ("P2c", C.c_void_p), ("uv1", C.c_void_p),
                ("uv2", C.c_void_p), ("inv_sigma2_1", C.c_void_p), ("inv_sigma2_2", C.c_void_p), ("K1", C.c_float * 4),
                ("K2", C.c_float * 4), ("th2", C.c_float), ("fix_scale", C.c_int32)]


def pose_optimize(Tcw, Xw, uv, inv_sigma2, intr, fn=None):
    """Optimizer::PoseOptimizationClient on flat arrays -> (Tcw (7,), outlier (n,) u8, n_inliers)."""
    a = dict(Tcw=np.ascontiguousarray(Tcw, np.float64), Xw=np.ascontiguousarray(Xw, np.float32).reshape(-1, 3),
             uv=np.ascontiguousarray(uv, np.float32).reshape(-1, 2), w=np.ascontiguousarray(inv_sigma2, np.float32))
    n = a["Xw"].shape[0]
    prob = _PoseOpt(n, _p(a["Tcw"]), _p(a["Xw"]), _p(a["uv"]), _p(a["w"]), *[float(v) for v in intr])
    out = np.empty(7); outlier = np.zeros(max(n, 1), np.uint8)
    nin = (fn or lib().orc_pose_optimize)(C.byref(prob), _p(out), _p(outlier))
    return out, outlier[:n], nin


def sim3_optimize(S12, P1c, P2c, uv1, uv2, w1, w2, K1, K2, th2, fix_scale, fn=None):
    """Optimizer::OptimizeSim3 on flat arrays -> (S12 (8,), inlier (n,) u8, n_inliers)."""
    f32 = lambda x, c: np.ascontiguousarray(x, np.float32).reshape(-1, c) if c else np.ascontiguousarray(x, np.float32)
    a = dict(S=np.ascontiguousarray(S12, np.float64), P1=f32(P1c, 3), P2=f32(P2c, 3), u1=f32(uv1, 2), u2=f32(uv2, 2),
             w1=f32(w1, 0), w2=f32(w2, 0))
    n = a["P1"].shape[0]
    prob = _Sim3Opt(n, _p(a["S"]), _p(a["P1"]), _p(a["P2"]), _p(a["u1"]), _p(a["u2"]), _p(a["w1"]), _p(a["w2"]),
                    (C.c_float * 4)(*[float(v) for v in K1]), (C.c_float * 4)(*[float(v) for v in K2]), float(th2), int(bool(fix_scale)))
    out = np.empty(8); inl = np.zeros(max(n, 1), np.uint8)
    nin = (fn or lib().orc_sim3_optimize)(C.byref(prob), _p(out), _p(inl))
    return out, inl[:n], nin


# ---- the two single-vertex optimisations run by the reference's LM driver over the reference's vertices / edges (oracle/ref_single_full_wrap.cpp)
_REF_SINGLE = None


def ref_single_full():
    global _REF_SINGLE
    if _REF_SINGLE is None:
        if build_ref() is None:
            return None
        so = os.path.join(_HERE, "_ref", "libsingle_full_ref.so")
        if not os.path.exists(so):
            return None
        _REF_SINGLE = C.CDLL(so)
    return _REF_SINGLE


def ref_pose_optimize(*a):
    return pose_optimize(*a, fn=ref_single_full().ref_pose_optimize)


def ref_sim3_optimize(*a):
    return sim3_optimize(*a, fn=ref_single_full().ref_sim3_optimize)


# ---- the essential graph run by the reference's LM driver over the reference's VertexSim3Expmap / EdgeSim3 (oracle/ref_pgo_full_wrap.cpp)
_REF_PGO = None


def ref_pgo_full():
    global _REF_PGO
    if _REF_PGO is None:
        if build_ref() is None:
            return None
        so = os.path.join(_HERE, "_ref", "libpgo_full_ref.so")
        if not os.path.exists(so):
            return None
        _REF_PGO = C.CDLL(so)
    return _REF_PGO


def ref_pgo_solve(p, **kw):
    return pgo_solve(p, fn=ref_pgo_full().ref_pgo_solve, **kw)


_REF_PGO_BLOCK = None


def ref_pgo_block():
    global _REF_PGO_BLOCK
    if _REF_PGO_BLOCK is None:
        if build_ref() is None:
            return None
        so = os.path.join(_HERE, "_ref", "libpgo_block_ref.so")
        if not os.path.exists(so):
            return None
        _REF_PGO_BLOCK = C.CDLL(so)
    return _REF_PGO_BLOCK


def ref_pgo_block_solve(p, **kw):
    """as ref_pgo_solve, with g2o's own BlockSolver_7_3 between the LM driver and the oracle's sparse LDL^T (oracle/ref_pgo_block_wrap.cpp)"""
    return pgo_solve(p, fn=ref_pgo_block().ref_pgo_block_solve, **kw)


def gba_map_update(sc, fn=None):
    """Map::RunGBA's update loop (S/Map.cpp:1441-1570) on the flat map view of ccm_slam_b200.synth.make_map_update; same result layout
    as ccm_slam_b200.api.gba_map_update.  fn: another entry point of the same signature (tests/host build of the product's header)."""
    from ccm_slam_b200.api import _map_update_args, _map_update_result
    a, argv, K, P = _map_update_args(sc)
    rc = (fn or lib().orc_gba_map_update)(*argv)
    if rc != 0:
        raise ValueError("gba_map_update: a map origin has no BA result")
    return _map_update_result(a, K, P)
