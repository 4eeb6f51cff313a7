"""ctypes binding of oracle/_ref: the reference's OWN pipeline sources compiled unmodified (oracle/Makefile, oracle/shim,
oracle/ref_harness).  TEST INFRASTRUCTURE ONLY, and only where the reference's sources are present:
tests/golden/make_ref_golden.py and make_ref_cases_golden.py freeze its outputs as the fixtures that
tests/test_oracle_vs_ref.py compares the oracle against (write_dataset() alone needs no reference).
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
REF_TREE = os.environ.get("DSAC_REFERENCE", "/root/reference/core")
GRID, N = 40, 1600


def available():
    return os.path.exists(os.path.join(REF_TREE, "cnn_softam.h"))


def build():
    subprocess.check_call(["make", "-C", _HERE, "-s", "ref", "REF=" + REF_TREE])


class Config(C.Structure):
    _fields_ = [("alpha", C.c_double), ("beta", C.c_double), ("grad_clamp", C.c_double),
                ("n_hyps", C.c_int32), ("thr2d", C.c_int32), ("inlier_count", C.c_int32), ("ref_steps", C.c_int32),
                ("sub_sample", C.c_float), ("seed", C.c_uint32), ("n_threads", C.c_int32), ("frame", C.c_int64)]


def config(**kw):
    c = Config(alpha=0.1, beta=0.5, grad_clamp=0.1, n_hyps=256, thr2d=10, inlier_count=100, ref_steps=8, sub_sample=0.01,
               seed=1305, n_threads=1, frame=0)
    for k, v in kw.items():
        setattr(c, k, v)
    return c


class ForwardOut(C.Structure):
    _fields_ = [("pix", C.c_void_p), ("est_obj", C.c_void_p), ("hyp_rvec", C.c_void_p), ("hyp_tvec", C.c_void_p),
                ("img_idx", C.c_void_p), ("diffmaps", C.c_void_p), ("scores", C.c_void_p), ("sf", C.c_void_p),
                ("entropy", C.c_double), ("avg", C.c_double * 6), ("ref", C.c_double * 6),
                ("inlier_map", C.c_void_p), ("pixel_idxs", C.c_void_p), ("n_perm_steps", C.c_int32),
                ("loss", C.c_double), ("rot_err", C.c_double), ("t_err", C.c_double), ("correct", C.c_int32)]


_libs = {}


def _lib(name):
    if name not in _libs:
        build()
        _libs[name] = C.CDLL(os.path.join(_HERE, "_ref", name))
    return _libs[name]


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


class Forward:
    def __init__(self, cfg):
        H = cfg.n_hyps
        self.pix = np.zeros((N, 2), np.int32); self.est_obj = np.zeros((N, 3), np.int16)
        self.hyp_rvec = np.zeros((H, 3)); self.hyp_tvec = np.zeros((H, 3)); self.img_idx = np.zeros((H, 4), np.int32)
        self.diffmaps = np.zeros((H, N), np.float32); self.scores = np.zeros(H); self.sf = np.zeros(H)
        self.inlier_map = np.zeros(N, np.int32); self.pixel_idxs = np.zeros((max(cfg.ref_steps, 1), N), np.int32)
        self.raw = ForwardOut()
        for k in ("pix", "est_obj", "hyp_rvec", "hyp_tvec", "img_idx", "diffmaps", "scores", "sf", "inlier_map", "pixel_idxs"):
            setattr(self.raw, k, _p(getattr(self, k)))

    def __getattr__(self, k):
        raw = self.__dict__.get("raw")
        if raw is not None and k in ("entropy", "n_perm_steps", "loss", "rot_err", "t_err", "correct"):
            return getattr(raw, k)
        if raw is not None and k in ("avg", "ref"):
            return np.array(list(getattr(raw, k)))
        raise AttributeError(k)


def forward(cfg, coords, gt_R, gt_t):
    """processImage (cnn_softam.h:960-1180) of the reference on one synthetic frame."""
    coords = np.ascontiguousarray(coords, np.int16).reshape(N, 3)
    gR = np.ascontiguousarray(gt_R, np.float64).reshape(9)
    gt = np.ascontiguousarray(gt_t, np.float64).reshape(3)
    out = Forward(cfg)
    rc = _lib("libref_softam.so").ref_softam_forward(C.byref(cfg), _p(coords), _p(gR), _p(gt), C.byref(out.raw))
    assert rc == 0
    out._keep = coords
    return out


def factors(cfg, score_out_grads=None, want_dref_dobj=True):
    """Backward factors by the reference's own functions, on the outputs of the last forward()."""
    H = cfg.n_hyps
    dloss_dref = np.zeros(6); dref_dobj = np.zeros((6, N * 3)) if want_dref_dobj else None; dref_dhyp = np.zeros((6, 6))
    dpnp = np.zeros((H, 6, 12))
    sog = np.ascontiguousarray(score_out_grads, np.float64) if score_out_grads is not None else None
    dscore = np.zeros(N * 3) if sog is not None else None
    rc = _lib("libref_softam.so").ref_softam_factors(C.byref(cfg), _p(dloss_dref), _p(dref_dobj), _p(dref_dhyp), _p(dpnp), _p(sog), _p(dscore))
    assert rc == 0
    return dict(dloss_dref=dloss_dref, dref_dobj=dref_dobj, dref_dhyp=dref_dhyp, dpnp=dpnp, dscore_sum=dscore)


def stochastic_subsample(seed=1305, skip_draws=0):
    pix = np.zeros((N, 2), np.int32)
    _lib("libref_softam.so").ref_stochastic_subsample(C.c_uint32(seed), int(skip_draws), _p(pix))
    return pix


def read_pose(directory, pose_file):
    R = np.zeros(9); t = np.zeros(3)
    rc = _lib("libref_softam.so").ref_read_pose(directory.encode(), pose_file.encode(), _p(R), _p(t))
    assert rc == 0, rc
    return R.reshape(3, 3), t


def _argv(args):
    arr = (C.c_char_p * len(args))(*[a.encode() for a in args])
    return arr


def write_dataset(root, split, gt_jp, translation=None, scene="synth"):
    """A 7-Scenes-shaped directory tree for the reference's drivers: <root>/<split>/<scene>/{rgb_noseg,depth_noseg,poses}.
    gt_jp [n][12]: the jp poses (R row-major, t in mm) the frames shall have; the pose files hold the 4x4 camera-to-world
    matrices in metres that read_data.cpp:69-133 turns back into them (through float)."""
    base = os.path.join(root, split, scene)
    for d in ("rgb_noseg", "depth_noseg", "poses"):
        os.makedirs(os.path.join(base, d), exist_ok=True)
    tr = np.zeros(3) if translation is None else np.asarray(translation, float)
    if translation is not None:
        with open(os.path.join(root, "translation.txt"), "w") as f:
            f.write("%.17g %.17g %.17g\n" % tuple(tr))
    corr = np.diag([1.0, -1.0, -1.0, 1.0])
    for i, g in enumerate(np.asarray(gt_jp).reshape(-1, 12)):
        M = np.eye(4)
        M[:3, :3] = g[:9].reshape(3, 3)
        M[:3, 3] = g[9:] / 1000.0
        P = np.linalg.inv(M) @ corr          # read_data: inv(P * correction) = M
        P[:3, 3] += tr
        open(os.path.join(base, "rgb_noseg", "frame-%06d.color.png" % i), "w").close()
        open(os.path.join(base, "depth_noseg", "frame-%06d.depth.png" % i), "w").close()
        with open(os.path.join(base, "poses", "frame-%06d.pose.txt" % i), "w") as f:
            for r in range(4):
                f.write("\t".join("%.17g" % v for v in P[r]) + "\n")
    return base


def run_test_main(cfg, root, coords, args=()):
    """main() of the reference's test_ransac_softam.cpp in `root` (needs ./test/<scene>/...); returns its two log files' text."""
    coords = np.ascontiguousarray(coords, np.int16).reshape(-1, N, 3)
    a = _argv(list(args))
    rc = _lib("libref_softam.so").ref_run_test_main(C.byref(cfg), root.encode(), _p(coords), coords.shape[0], len(args), a)
    assert rc == 0, rc
    logs = {}
    for fn in os.listdir(root):
        if fn.startswith("ransac_test_"):
            logs[fn] = open(os.path.join(root, fn)).read()
    return logs


def train_round(cfg, root, coords, args=()):
    """One round of main() of the reference's train_ransac_softam.cpp on the one-frame dataset in `root`
    (./training/<scene>/...): returns (dLoss_dObj [N,3], loss, scoreOutputGradients [H])."""
    coords = np.ascontiguousarray(coords, np.int16).reshape(1, N, 3)
    dloss = np.zeros((N, 3)); loss = C.c_double(0); sog = np.zeros(cfg.n_hyps)
    a = _argv(list(args))
    rc = _lib("libref_train_softam.so").ref_train_softam_round(C.byref(cfg), root.encode(), _p(coords), len(args), a, _p(dloss), C.byref(loss), _p(sog))
    assert rc == 0, rc
    return dloss, loss.value, sog


# ---------------------------------------------------------------- DSAC / RANSAC variant (core/cnn.h, test_ransac.cpp, train_ransac.cpp)
class DsacOut(C.Structure):
    _fields_ = [("hyp_rvec", C.c_void_p), ("hyp_tvec", C.c_void_p), ("img_idx", C.c_void_p), ("sf", C.c_void_p),
                ("ref_pose", C.c_void_p), ("losses", C.c_void_p), ("inlier_maps", C.c_void_p),
                ("entropy", C.c_double), ("expected_loss", C.c_double), ("rot_err", C.c_double), ("t_err", C.c_double),
                ("hyp_idx", C.c_int32), ("correct", C.c_int32)]


class ForwardDsac:
    def __init__(self, cfg):
        H = cfg.n_hyps
        self.hyp_rvec = np.zeros((H, 3)); self.hyp_tvec = np.zeros((H, 3)); self.img_idx = np.zeros((H, 4), np.int32)
        self.sf = np.zeros(H); self.ref_pose = np.zeros((H, 6)); self.losses = np.zeros(H); self.inlier_maps = np.zeros((H, N), np.int32)
        self.raw = DsacOut()
        for k in ("hyp_rvec", "hyp_tvec", "img_idx", "sf", "ref_pose", "losses", "inlier_maps"):
            setattr(self.raw, k, _p(getattr(self, k)))

    def __getattr__(self, k):
        raw = self.__dict__.get("raw")
        if raw is not None and k in ("entropy", "expected_loss", "rot_err", "t_err", "hyp_idx", "correct"):
            return getattr(raw, k)
        raise AttributeError(k)


def forward_dsac(cfg, coords, gt_R, gt_t, random_draw=True):
    """processImage of the DSAC variant (cnn.h:1028-1257) of the reference on one synthetic frame."""
    coords = np.ascontiguousarray(coords, np.int16).reshape(N, 3)
    gR = np.ascontiguousarray(gt_R, np.float64).reshape(9)
    gt = np.ascontiguousarray(gt_t, np.float64).reshape(3)
    out = ForwardDsac(cfg)
    rc = _lib("libref_dsac.so").ref_dsac_forward(C.byref(cfg), int(random_draw), _p(coords), _p(gR), _p(gt), C.byref(out.raw))
    assert rc == 0
    return out


def train_round_dsac(cfg, root, coords, args=()):
    """One round of main() of the reference's train_ransac.cpp on the one-frame dataset in `root`: (dLoss_dObj [N,3], expected loss)."""
    coords = np.ascontiguousarray(coords, np.int16).reshape(1, N, 3)
    dloss = np.zeros((N, 3)); loss = C.c_double(0)
    a = _argv(list(args))
    rc = _lib("libref_train_dsac.so").ref_train_dsac_round(C.byref(cfg), root.encode(), _p(coords), len(args), a, _p(dloss), C.byref(loss))
    assert rc == 0, rc
    return dloss, loss.value
