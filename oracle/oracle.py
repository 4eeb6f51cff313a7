"""ctypes binding of the CPU oracle (oracle/libdsac_oracle.so).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference leg.  Never imported by the product package dsac_b200.
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libdsac_oracle.so")
GRID = 40
N = GRID * GRID


def build(force=False):
    """Compile the oracle with the recipe in oracle/Makefile (g++ only, no dependencies)."""
    src = [os.path.join(_HERE, f) for f in ("dsac_oracle.cpp", "dsac_oracle_pipeline.inc", "dsac_oracle.h")]
    if (not force) and os.path.exists(_LIB_PATH) and all(os.path.getmtime(_LIB_PATH) >= os.path.getmtime(s) for s in src):
        return _LIB_PATH
    subprocess.check_call(["make", "-C", _HERE, "-s"])
    return _LIB_PATH


class Config(C.Structure):
    _fields_ = [
        ("f", C.c_double), ("cx", C.c_double), ("cy", C.c_double),
        ("n_hyps", C.c_int32), ("thr2d", C.c_int32), ("inlier_count", C.c_int32), ("ref_steps", C.c_int32),
        ("sub_sample", C.c_double), ("alpha", C.c_double), ("beta", C.c_double),
        ("seed", C.c_uint32), ("n_streams", C.c_int32), ("stream_skip", C.c_uint32), ("max_candidates", C.c_int32),
        ("fix_q4", C.c_int32), ("grad_clamp", C.c_double),
    ]


class ForwardOut(C.Structure):
    _fields_ = [
        ("hyp_rvec", C.c_void_p), ("hyp_tvec", C.c_void_p), ("img_idx", C.c_void_p), ("cand_idx", C.c_void_p),
        ("diffmaps", C.c_void_p), ("scores", C.c_void_p), ("sf", C.c_void_p),
        ("entropy", C.c_double), ("avg", C.c_double * 6), ("ref", C.c_double * 6),
        ("inlier_map", C.c_void_p), ("pixel_idxs", C.c_void_p),
        ("ref_steps_done", C.c_int32), ("n_perm_steps", C.c_int32),
        ("loss", C.c_double), ("rot_err", C.c_double), ("t_err", C.c_double),
        ("correct", C.c_int32), ("n_candidates", C.c_int64), ("n_fragile", C.c_int64),
    ]


class DsacOut(C.Structure):
    _fields_ = [
        ("hyp_rvec", C.c_void_p), ("hyp_tvec", C.c_void_p), ("img_idx", C.c_void_p), ("sf", C.c_void_p),
        ("ref_pose", C.c_void_p), ("losses", C.c_void_p), ("inlier_maps", C.c_void_p), ("steps_done", C.c_void_p),
        ("entropy", C.c_double), ("expected_loss", C.c_double), ("rot_err", C.c_double), ("t_err", C.c_double),
        ("hyp_idx", C.c_int32), ("correct", C.c_int32), ("stream0_endpos", C.c_uint64),
    ]


class BackwardDsacOut(C.Structure):
    _fields_ = [
        ("dloss_dobj", C.c_void_p), ("path1", C.c_void_p), ("path2", C.c_void_p), ("score_grads", C.c_void_p),
        ("n_selected", C.c_int32), ("n_refine_jobs", C.c_int32),
    ]


class BackwardOut(C.Structure):
    _fields_ = [
        ("dloss_dobj", C.c_void_p), ("dloss_dref", C.c_double * 6), ("dref_dobj", C.c_void_p),
        ("dref_dhyp", C.c_double * 36), ("score_grads", C.c_void_p), ("dpnp", C.c_void_p),
    ]


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_LIB_PATH)
        _lib.orc_soft_inlier_score.restype = C.c_double
        _lib.orc_entropy.restype = C.c_double
        _lib.orc_max_loss.restype = C.c_double
        _lib.orc_bench_forward.restype = C.c_double
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def default_config(**kw):
    c = Config()
    lib().orc_default_config(C.byref(c))
    for k, v in kw.items():
        setattr(c, k, v)
    return c


def _d(x):
    return C.c_double(float(x))


def rodrigues(r, jac=False):
    r = np.ascontiguousarray(r, np.float64).reshape(3)
    R = np.empty(9)
    J = np.empty(27) if jac else None
    lib().orc_rodrigues(_p(r), _p(R), _p(J))
    return (R.reshape(3, 3), J.reshape(3, 9)) if jac else R.reshape(3, 3)


def rodrigues_inv(R):
    R = np.ascontiguousarray(R, np.float64).reshape(9)
    r = np.empty(3)
    lib().orc_rodrigues_inv(_p(R), _p(r))
    return r


def project_points(X, rvec, tvec, f=525.0, cx=320.0, cy=240.0, jac=False):
    X = np.ascontiguousarray(X, np.float64).reshape(-1, 3)
    n = X.shape[0]
    rvec = np.ascontiguousarray(rvec, np.float64).reshape(3)
    tvec = np.ascontiguousarray(tvec, np.float64).reshape(3)
    uv = np.empty((n, 2))
    dr = np.empty((2 * n, 3)) if jac else None
    dt = np.empty((2 * n, 3)) if jac else None
    lib().orc_project_points(n, _p(X), _p(rvec), _p(tvec), _d(f), _d(cx), _d(cy), _p(uv), _p(dr), _p(dt))
    return (uv, dr, dt) if jac else uv


def solve_p3p(obj, img, f=525.0, cx=320.0, cy=240.0):
    obj = np.ascontiguousarray(obj, np.float32).reshape(12)
    img = np.ascontiguousarray(img, np.float32).reshape(8)
    r, t = np.empty(3), np.empty(3)
    ok = lib().orc_solve_p3p(_p(obj), _p(img), _d(f), _d(cx), _d(cy), _p(r), _p(t))
    return bool(ok), r, t


def solve_pnp_iterative(obj, img, rvec, tvec, f=525.0, cx=320.0, cy=240.0):
    obj = np.ascontiguousarray(obj, np.float32).reshape(-1, 3)
    img = np.ascontiguousarray(img, np.float32).reshape(-1, 2)
    r = np.array(rvec, np.float64).reshape(3).copy()
    t = np.array(tvec, np.float64).reshape(3).copy()
    it = C.c_int(0)
    lib().orc_solve_pnp_iterative(obj.shape[0], _p(obj), _p(img), _d(f), _d(cx), _d(cy), _p(r), _p(t), C.byref(it))
    return r, t, it.value


def svd3(A):
    A = np.ascontiguousarray(A, np.float64).reshape(9)
    U, w, Vt = np.empty(9), np.empty(3), np.empty(9)
    lib().orc_svd3(_p(A), _p(U), _p(w), _p(Vt))
    return U.reshape(3, 3), w, Vt.reshape(3, 3)


def kabsch(a, b):
    a = np.ascontiguousarray(a, np.float64).reshape(-1, 3)
    b = np.ascontiguousarray(b, np.float64).reshape(-1, 3)
    R, t = np.empty(9), np.empty(3)
    lib().orc_kabsch(a.shape[0], _p(a), _p(b), _p(R), _p(t))
    return R.reshape(3, 3), t


def stochastic_subsample(seed=1305, width=640, height=480):
    pix = np.empty((N, 2), np.int32)
    lib().orc_stochastic_subsample(C.c_uint32(seed), width, height, _p(pix))
    return pix


def candidates(seed, skip, n_cand):
    cells = np.empty((n_cand, 4, 2), np.int32)
    draws = np.empty(n_cand, np.uint32)
    lib().orc_candidates(C.c_uint32(seed), C.c_uint32(skip), n_cand, _p(cells), _p(draws))
    return cells, draws


def refine_permutations(steps=8):
    perm = np.empty((steps, N), np.int32)
    lib().orc_refine_permutations(steps, _p(perm))
    return perm


def mt19937_raw(seed, n):
    out = np.empty(n, np.uint32)
    lib().orc_mt19937_raw(C.c_uint32(seed), n, _p(out))
    return out


def diff_map(coords, pix, rvec, tvec, f=525.0, cx=320.0, cy=240.0):
    coords = np.ascontiguousarray(coords, np.int16).reshape(N, 3)
    pix = np.ascontiguousarray(pix, np.int32).reshape(N, 2)
    rvec = np.ascontiguousarray(rvec, np.float64).reshape(3)
    tvec = np.ascontiguousarray(tvec, np.float64).reshape(3)
    d = np.empty(N, np.float32)
    lib().orc_diff_map(_p(coords), _p(pix), _p(rvec), _p(tvec), _d(f), _d(cx), _d(cy), _p(d))
    return d


def soft_inlier_score(diff, tau=10.0, alpha=0.1, beta=0.5):
    diff = np.ascontiguousarray(diff, np.float32).reshape(-1)
    return lib().orc_soft_inlier_score(_p(diff), diff.size, _d(tau), _d(alpha), _d(beta))


def softmax(s):
    s = np.ascontiguousarray(s, np.float64).reshape(-1)
    p = np.empty_like(s)
    lib().orc_softmax(_p(s), s.size, _p(p))
    return p


def entropy(p):
    p = np.ascontiguousarray(p, np.float64).reshape(-1)
    return lib().orc_entropy(_p(p), p.size)


def cv2our(rvec, tvec):
    rvec = np.ascontiguousarray(rvec, np.float64).reshape(3)
    tvec = np.ascontiguousarray(tvec, np.float64).reshape(3)
    R, t = np.empty(9), np.empty(3)
    lib().orc_cv2our(_p(rvec), _p(tvec), _p(R), _p(t))
    return R.reshape(3, 3), t


def our2cv(R, t):
    R = np.ascontiguousarray(R, np.float64).reshape(9)
    t = np.ascontiguousarray(t, np.float64).reshape(3)
    r, tv = np.empty(3), np.empty(3)
    lib().orc_our2cv(_p(R), _p(t), _p(r), _p(tv))
    return r, tv


def jp6(rvec, tvec):
    rvec = np.ascontiguousarray(rvec, np.float64).reshape(3)
    tvec = np.ascontiguousarray(tvec, np.float64).reshape(3)
    o = np.empty(6)
    lib().orc_jp6(_p(rvec), _p(tvec), _p(o))
    return o


def max_loss(R1, t1, R2, t2):
    a = [np.ascontiguousarray(x, np.float64).reshape(-1) for x in (R1, t1, R2, t2)]
    re, te = C.c_double(0), C.c_double(0)
    loss = lib().orc_max_loss(_p(a[0]), _p(a[1]), _p(a[2]), _p(a[3]), C.byref(re), C.byref(te))
    return loss, re.value, te.value


def dloss_max(est6, gt6):
    est6 = np.ascontiguousarray(est6, np.float64).reshape(6)
    gt6 = np.ascontiguousarray(gt6, np.float64).reshape(6)
    j = np.empty(6)
    lib().orc_dloss_max(_p(est6), _p(gt6), _p(j))
    return j


def dpnp(obj, img, f=525.0, cx=320.0, cy=240.0):
    obj = np.ascontiguousarray(obj, np.float32).reshape(12)
    img = np.ascontiguousarray(img, np.float32).reshape(8)
    j = np.empty((6, 12))
    lib().orc_dpnp(_p(obj), _p(img), _d(f), _d(cx), _d(cy), _p(j))
    return j


def dproject_dobj(pt, obj, R, t, f=525.0, cx=320.0, cy=240.0):
    pt = np.ascontiguousarray(pt, np.float32).reshape(2)
    obj = np.ascontiguousarray(obj, np.float32).reshape(3)
    R = np.ascontiguousarray(R, np.float64).reshape(9)
    t = np.ascontiguousarray(t, np.float64).reshape(3)
    o = np.empty(3)
    lib().orc_dproject_dobj(_p(pt), _p(obj), _p(R), _p(t), _d(f), _d(cx), _d(cy), _p(o))
    return o


def dproject_dhyp(pt, obj, R, t, f=525.0, cx=320.0, cy=240.0):
    pt = np.ascontiguousarray(pt, np.float32).reshape(2)
    obj = np.ascontiguousarray(obj, np.float32).reshape(3)
    R = np.ascontiguousarray(R, np.float64).reshape(9)
    t = np.ascontiguousarray(t, np.float64).reshape(3)
    o = np.empty(6)
    lib().orc_dproject_dhyp(_p(pt), _p(obj), _p(R), _p(t), _d(f), _d(cx), _d(cy), _p(o))
    return o


class Forward:
    """Result of orc_forward for one frame (numpy arrays own the memory)."""

    def __init__(self, cfg, want_diffmaps=True):
        H = cfg.n_hyps
        self.hyp_rvec = np.zeros((H, 3))
        self.hyp_tvec = np.zeros((H, 3))
        self.img_idx = np.zeros((H, 4), np.int32)
        self.cand_idx = np.zeros(H, np.int32)
        self.diffmaps = np.zeros((H, N), np.float32) if want_diffmaps else None
        self.scores = np.zeros(H)
        self.sf = np.zeros(H)
        self.inlier_map = np.zeros(N, np.int32)
        self.pixel_idxs = np.zeros((max(cfg.ref_steps, 1), N), np.int32)
        self.raw = ForwardOut()
        for k in ("hyp_rvec", "hyp_tvec", "img_idx", "cand_idx", "diffmaps", "scores", "sf", "inlier_map", "pixel_idxs"):
            setattr(self.raw, k, _p(getattr(self, k)))

    def __getattr__(self, k):
        raw = self.__dict__.get("raw")
        if raw is not None and k in ("entropy", "ref_steps_done", "n_perm_steps", "loss", "rot_err", "t_err", "correct",
                                     "n_candidates", "n_fragile"):
            return getattr(raw, k)
        if raw is not None and k in ("avg", "ref"):
            return np.array(list(getattr(raw, k)))
        raise AttributeError(k)


def forward(cfg, coords, pix, gt_R=None, gt_t=None, want_diffmaps=True):
    coords = np.ascontiguousarray(coords, np.int16).reshape(N, 3)
    pix = np.ascontiguousarray(pix, np.int32).reshape(N, 2)
    out = Forward(cfg, want_diffmaps)
    gR = np.ascontiguousarray(gt_R, np.float64).reshape(9) if gt_R is not None else None
    gt = np.ascontiguousarray(gt_t, np.float64).reshape(3) if gt_t is not None else None
    out.status = lib().orc_forward(C.byref(cfg), _p(coords), _p(pix), _p(gR), _p(gt), C.byref(out.raw))
    out._keep = (coords, pix)
    return out


class ForwardDsac:
    def __init__(self, cfg):
        H = cfg.n_hyps
        self.hyp_rvec = np.zeros((H, 3)); self.hyp_tvec = np.zeros((H, 3)); self.img_idx = np.zeros((H, 4), np.int32)
        self.sf = np.zeros(H); self.ref_pose = np.zeros((H, 6)); self.losses = np.zeros(H)
        self.inlier_maps = np.zeros((H, N), np.int32); self.steps_done = np.zeros(H, np.int32)
        self.raw = DsacOut()
        for k in ("hyp_rvec", "hyp_tvec", "img_idx", "sf", "ref_pose", "losses", "inlier_maps", "steps_done"):
            setattr(self.raw, k, _p(getattr(self, k)))

    def __getattr__(self, k):
        raw = self.__dict__.get("raw")
        if raw is not None and k in ("entropy", "expected_loss", "rot_err", "t_err", "hyp_idx", "correct", "stream0_endpos"):
            return getattr(raw, k)
        raise AttributeError(k)


def forward_dsac(cfg, coords, pix, gt_R, gt_t, random_draw=True):
    """DSAC / RANSAC variant (cnn.h processImage): draw + refine all hypotheses + expected loss."""
    coords = np.ascontiguousarray(coords, np.int16).reshape(N, 3)
    pix = np.ascontiguousarray(pix, np.int32).reshape(N, 2)
    gR = np.ascontiguousarray(gt_R, np.float64).reshape(9)
    gt = np.ascontiguousarray(gt_t, np.float64).reshape(3)
    out = ForwardDsac(cfg)
    out.status = lib().orc_forward_dsac(C.byref(cfg), int(random_draw), _p(coords), _p(pix), _p(gR), _p(gt), C.byref(out.raw))
    return out


def refine(cfg, pixel_idxs, n_perm_steps, coords, pix, init6):
    coords = np.ascontiguousarray(coords, np.int16).reshape(N, 3)
    pix = np.ascontiguousarray(pix, np.int32).reshape(N, 2)
    pixel_idxs = np.ascontiguousarray(pixel_idxs, np.int32)
    init6 = np.ascontiguousarray(init6, np.float64).reshape(6)
    o = np.empty(6)
    lib().orc_refine(C.byref(cfg), _p(pixel_idxs), int(n_perm_steps), _p(coords), _p(pix), _p(init6), _p(o))
    return o


class Backward:
    def __init__(self, cfg):
        H = cfg.n_hyps
        self.dloss_dobj = np.zeros((N, 3))
        self.dref_dobj = np.zeros((6, N * 3))
        self.score_grads = np.zeros(H)
        self.dpnp = np.zeros((H, 6, 12))
        self.raw = BackwardOut()
        for k in ("dloss_dobj", "dref_dobj", "score_grads", "dpnp"):
            setattr(self.raw, k, _p(getattr(self, k)))

    @property
    def dloss_dref(self):
        return np.array(list(self.raw.dloss_dref))

    @property
    def dref_dhyp(self):
        return np.array(list(self.raw.dref_dhyp)).reshape(6, 6)


def backward(cfg, coords, pix, gt_R, gt_t, fwd):
    coords = np.ascontiguousarray(coords, np.int16).reshape(N, 3)
    pix = np.ascontiguousarray(pix, np.int32).reshape(N, 2)
    gR = np.ascontiguousarray(gt_R, np.float64).reshape(9)
    gt = np.ascontiguousarray(gt_t, np.float64).reshape(3)
    out = Backward(cfg)
    lib().orc_backward(C.byref(cfg), _p(coords), _p(pix), _p(gR), _p(gt), C.byref(fwd.raw), C.byref(out.raw))
    return out


class BackwardDsac:
    def __init__(self, cfg):
        self.dloss_dobj = np.zeros((N, 3)); self.path1 = np.zeros((N, 3)); self.path2 = np.zeros((N, 3))
        self.score_grads = np.zeros(cfg.n_hyps)
        self.raw = BackwardDsacOut()
        for k in ("dloss_dobj", "path1", "path2", "score_grads"):
            setattr(self.raw, k, _p(getattr(self, k)))

    def __getattr__(self, k):
        raw = self.__dict__.get("raw")
        if raw is not None and k in ("n_selected", "n_refine_jobs"):
            return getattr(raw, k)
        raise AttributeError(k)


def backward_dsac(cfg, coords, pix, gt_R, gt_t, fwd):
    """Backward of the DSAC / RANSAC variant (train_ransac.cpp:304-381) from a forward_dsac result."""
    coords = np.ascontiguousarray(coords, np.int16).reshape(N, 3)
    pix = np.ascontiguousarray(pix, np.int32).reshape(N, 2)
    gR = np.ascontiguousarray(gt_R, np.float64).reshape(9)
    gt = np.ascontiguousarray(gt_t, np.float64).reshape(3)
    out = BackwardDsac(cfg)
    lib().orc_backward_dsac.restype = C.c_int
    lib().orc_backward_dsac(C.byref(cfg), _p(coords), _p(pix), _p(gR), _p(gt), C.byref(fwd.raw), C.byref(out.raw))
    return out


_variants = {}


def variant_lib(variant):
    """A differently COMPILED build of the same oracle sources, for the CPU timing arm only (bench.py): "parity" = the -O2
    -ffp-contract=off library the tests use; "perf" = -O3 -march=x86-64-v3 -fopenmp; "native" / "ofast" = -O3 / -Ofast
    -march=native, built on the calling machine into a temporary directory (BASELINE.md section 3).  Returns (CDLL, flags
    description) or (None, why)."""
    if variant == "parity":
        return lib(), "-O2 -ffp-contract=off (parity build)"
    if variant in _variants:
        return _variants[variant]
    target = {"perf": "libdsac_oracle_perf.so", "native": "libdsac_oracle_native.so", "ofast": "libdsac_oracle_ofast.so"}[variant]
    flags = {"perf": "-O3 -march=x86-64-v3 -fopenmp", "native": "-O3 -march=native -fopenmp", "ofast": "-Ofast -march=native -fopenmp"}[variant]
    try:
        if variant == "perf":
            path = os.path.join(_HERE, target)
            if not os.path.exists(path):
                subprocess.check_call(["make", "-C", _HERE, "-s", target], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            l = C.CDLL(path)
        else:
            with tempfile.TemporaryDirectory() as d:   # the library stays mapped once the directory is gone
                path = os.path.join(d, target)
                subprocess.check_call(["make", "-C", _HERE, "-s", "VARIANT_DIR=" + d, path], stdout=subprocess.DEVNULL,
                                      stderr=subprocess.DEVNULL)
                l = C.CDLL(path)
        l.orc_bench_forward.restype = C.c_double
        _variants[variant] = (l, flags)
    except Exception as e:   # no compiler on this box, or an instruction set this CPU lacks
        _variants[variant] = (None, "unavailable: %s" % e)
    return _variants[variant]


def bench_forward(cfg, coords, pix, n_threads=1, with_refine=False, want_avg=False, variant="parity", stages=None):
    """Wall-clock seconds of orc_forward over the frames with n_threads host threads (frames in parallel).
    stages: a list that receives the per-stage seconds summed over threads [sampling, scoring, averaging, refinement]."""
    coords = np.ascontiguousarray(coords, np.int16).reshape(-1, N, 3)
    pix = np.ascontiguousarray(pix, np.int32).reshape(-1, N, 2)
    nf = coords.shape[0]
    avg = np.zeros((nf, 6)) if want_avg else None
    l, _ = variant_lib(variant)
    if l is None:
        raise RuntimeError("oracle build %r is not available" % variant)
    four = (C.c_double * 4)()
    l.orc_stage_seconds(four, 1)
    secs = l.orc_bench_forward(C.byref(cfg), nf, _p(coords), _p(pix), int(n_threads), int(with_refine), _p(avg))
    l.orc_stage_seconds(four, 1)
    if stages is not None:
        stages[:] = list(four)
    return (secs, avg) if want_avg else secs


# ---- upstream step (SURVEY.md section 8f row N3), numpy restatement
def gather_patches(frame_bgr, pix, mean=127.0, patch=42):
    """getCoordImg's patch assembly (cnn_softam.h:221-256) + forward()'s normalisation (lua/train_obj.lua:117-124) in
    pushMaps' channel-major order (lua_calls.h:65-82).  frame_bgr: [H][W][3] uint8; pix: [N][2] (origX, origY).
    Returns float32 [N][3][42][42]; border cells (which the reference skips) come back as zero patches."""
    frame_bgr = np.asarray(frame_bgr, np.uint8)
    pix = np.asarray(pix).reshape(-1, 2)
    Hh, W = frame_bgr.shape[:2]
    half = patch // 2
    out = np.zeros((pix.shape[0], 3, patch, patch), np.float32)
    for i, (ox, oy) in enumerate(pix):
        if ox < half or oy < half or ox > W - half or oy > Hh - half:
            continue
        p = frame_bgr[oy - half:oy + half, ox - half:ox + half, :].astype(np.float32)   # patch(curY-minY, curX-minX) = colorData(curY, curX)
        out[i] = np.transpose(p, (2, 0, 1)) - np.float32(mean)
    return out


def coords_from_prediction(pred):
    """modeImg(y, x) = prediction[i] * 1000 (cnn_softam.h:262-268): Vec3f * 1000 in float, then cv::saturate_cast<short>
    (cvRound = round half to even via cvtss2si: NaN / out-of-int-range -> INT_MIN -> -32768)."""
    v = np.asarray(pred, np.float32) * np.float32(1000.0)
    bad = ~(np.abs(v) < np.float32(2147483648.0))
    r = np.where(bad, -2147483648.0, np.rint(np.where(bad, 0, v).astype(np.float64)))
    return np.clip(r, -32768, 32767).astype(np.int16)
