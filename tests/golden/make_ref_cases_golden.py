"""Freeze what tests/test_oracle_vs_ref.py compares the oracle against: the outputs of the reference's own code
(oracle/_ref, compiled by oracle/Makefile from the reference's sources against oracle/shim) for exactly the parameter
sets of those tests, so that the comparisons run on any machine.

    python tests/golden/make_ref_cases_golden.py  ->  tests/golden/ref_cases_golden.npz

Needs oracle/_ref (built by __graft_entry__.build() where the reference's sources are present).  Keys are
"<case>/<field>".  Integer arrays that the tests compare bit for bit and that would make the file large are stored as the
SHA-256 of their bytes (field "<name>_sha256", see digest()); real-valued arrays compared with a tolerance are stored as
they are, except the gradients and the largest factors: of those a fixed, seeded sample of entries is kept together
with the largest magnitude of the whole array (see SAMPLES).
"""
import hashlib
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

RNG_SEEDS = (1305, 1306, 99)
FORWARD = [(1, 64, (0, 1, 2)), (1, 256, (4,)), (8, 256, (2,)), (3, 64, (6,)), (8, 64, (9, 10))]
FACTORS = [(1, 64, 1), (8, 256, 3)]
TRAIN = [(1, 64, 0), (1, 256, 2), (8, 256, 5)]
DRIVER_FRAMES, DRIVER_H, DRIVER_TRANSLATION = 12, 64, (0.25, -0.5, 1.0)
POSE_FRAMES, POSE_TRANSLATION = 5, (0.5, -1.25, 2.0)
DSAC_FORWARD = [(1, 64, 0, True), (1, 64, 3, False), (4, 32, 2, True)]
DSAC_TRAIN = [(1, 32, 1), (4, 48, 6)]
# entries kept of the gradients (N x 3) and of the two largest factors (6 x 3N and H x 6 x 12)
SAMPLES = {"dloss_dobj": 1024, "dref_dobj": 1024, "dpnp": 1024}


def digest(a):
    """SHA-256 of an array's dtype, shape and bytes (C order)."""
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(("%s %s " % (a.dtype.str, a.shape)).encode())
    h.update(a.tobytes())
    return h.hexdigest()


def sample_index(name, size):
    """The fixed positions (into the flattened array) kept of array `name`."""
    rng = np.random.default_rng(20170721)
    return np.sort(rng.choice(size, size=min(size, SAMPLES[name]), replace=False))


def sampled(name, a):
    """{name_sample, name_absmax}: the kept entries of `a` and its largest magnitude."""
    a = np.asarray(a).reshape(-1)
    return {name + "_sample": a[sample_index(name, a.size)], name + "_absmax": np.abs(a).max()}


def forward_key(T, H, g):
    return "fwd_t%d_h%d_f%d" % (T, H, g)


def factors_key(T, H, g):
    return "fac_t%d_h%d_f%d" % (T, H, g)


def train_key(T, H, g):
    return "train_t%d_h%d_f%d" % (T, H, g)


def dsac_forward_key(T, H, g, random_draw):
    return "dsacfwd_t%d_h%d_f%d_r%d" % (T, H, g, int(random_draw))


def dsac_train_key(T, H, g):
    return "dsactrain_t%d_h%d_f%d" % (T, H, g)


def main():
    import dsac_b200.engine as E
    from oracle import ref as R
    assert R.available(), "the reference's sources are needed to build oracle/_ref"
    out = {}

    def put(key, **fields):
        for k, v in fields.items():
            out[key + "/" + k] = np.asarray(v)

    for seed in RNG_SEEDS:
        put("rng_%d" % seed, pix=R.stochastic_subsample(seed))

    for T, H, frames in FORWARD:
        for g in frames:
            coords, pix, gt_cv, gt_jp = E.synth_frames(1, frame0=g, n_streams=T)
            r = R.forward(R.config(n_hyps=H, n_threads=T, frame=g), coords[0], gt_jp[0, :9], gt_jp[0, 9:])
            put(forward_key(T, H, g), pix_sha256=digest(r.pix), est_obj_sha256=digest(r.est_obj), img_idx=r.img_idx,
                hyp_rvec=r.hyp_rvec, hyp_tvec=r.hyp_tvec, scores=r.scores, sf=r.sf, entropy=r.entropy, avg=r.avg, ref=r.ref,
                inlier_map=r.inlier_map, n_perm_steps=r.n_perm_steps, loss=r.loss, rot_err=r.rot_err, t_err=r.t_err,
                correct=r.correct, diffmaps_sha256=digest(r.diffmaps), pixel_idxs_sha256=digest(r.pixel_idxs))

    for T, H, g in FACTORS:
        coords, pix, gt_cv, gt_jp = E.synth_frames(1, frame0=g, n_streams=T)
        cfg = R.config(n_hyps=H, n_threads=T, frame=g)
        R.forward(cfg, coords[0], gt_jp[0, :9], gt_jp[0, 9:])
        fa = R.factors(cfg)
        put(factors_key(T, H, g), dloss_dref=fa["dloss_dref"], dref_dhyp=fa["dref_dhyp"], **sampled("dref_dobj", fa["dref_dobj"]),
            **sampled("dpnp", fa["dpnp"]))

    for T, H, g in TRAIN:
        coords, pix, gt_cv, gt_jp = E.synth_frames(1, frame0=g, n_streams=T)
        with tempfile.TemporaryDirectory() as d:
            R.write_dataset(d, "training", gt_jp)
            Rg, tg = R.read_pose(d, os.path.join("training", "synth", "poses", "frame-000000.pose.txt"))
            dl, loss, sog = R.train_round(R.config(n_hyps=H, n_threads=T, frame=g), d, coords[0], args=("-rI", str(H)))
        put(train_key(T, H, g), gt_R=Rg, gt_t=tg, loss=loss, score_out_grads=sog, **sampled("dloss_dobj", dl))

    coords, pix, gt_cv, gt_jp = E.synth_frames(DRIVER_FRAMES, traj=True)
    with tempfile.TemporaryDirectory() as d:
        R.write_dataset(d, "test", gt_jp, translation=DRIVER_TRANSLATION)
        gts = [R.read_pose(d, os.path.join("test", "synth", "poses", "frame-%06d.pose.txt" % i)) for i in range(DRIVER_FRAMES)]
        logs = R.run_test_main(R.config(n_hyps=DRIVER_H), d, coords, args=("-rI", str(DRIVER_H)))
    per_frame = [[float(v) for v in ln.split()] for ln in logs["ransac_test_errors_obj_model_init.net_rdraw1_softam.txt"].strip().splitlines()]
    put("driver", gt_R=np.array([R_ for R_, t_ in gts]), gt_t=np.array([t_ for R_, t_ in gts]), per_frame=np.array(per_frame),
        summary=np.array([float(v) for v in logs["ransac_test_loss_obj_model_init.net_rdraw1_softam.txt"].split()]))

    coords, pix, gt_cv, gt_jp = E.synth_frames(POSE_FRAMES, traj=True)
    with tempfile.TemporaryDirectory() as d:
        R.write_dataset(d, "test", gt_jp, translation=POSE_TRANSLATION)
        gts = [R.read_pose(d, os.path.join("test", "synth", "poses", "frame-%06d.pose.txt" % i)) for i in range(POSE_FRAMES)]
    put("pose", gt_R=np.array([R_ for R_, t_ in gts]), gt_t=np.array([t_ for R_, t_ in gts]))

    for T, H, g, random_draw in DSAC_FORWARD:
        coords, pix, gt_cv, gt_jp = E.synth_frames(1, frame0=g, n_streams=T)
        r = R.forward_dsac(R.config(n_hyps=H, n_threads=T, frame=g), coords[0], gt_jp[0, :9], gt_jp[0, 9:], random_draw)
        put(dsac_forward_key(T, H, g, random_draw), img_idx=r.img_idx, hyp_idx=r.hyp_idx, correct=r.correct,
            inlier_maps_sha256=digest(r.inlier_maps), hyp_rvec=r.hyp_rvec, hyp_tvec=r.hyp_tvec, sf=r.sf, ref_pose=r.ref_pose,
            losses=r.losses, expected_loss=r.expected_loss, rot_err=r.rot_err, t_err=r.t_err)

    for T, H, g in DSAC_TRAIN:
        coords, pix, gt_cv, gt_jp = E.synth_frames(1, frame0=g, n_streams=T)
        with tempfile.TemporaryDirectory() as d:
            R.write_dataset(d, "training", gt_jp)
            Rg, tg = R.read_pose(d, os.path.join("training", "synth", "poses", "frame-000000.pose.txt"))
            dl, loss = R.train_round_dsac(R.config(n_hyps=H, n_threads=T, frame=g), d, coords[0], args=("-rI", str(H)))
        put(dsac_train_key(T, H, g), gt_R=Rg, gt_t=tg, loss=loss, **sampled("dloss_dobj", dl))

    path = os.path.join(ROOT, "tests", "golden", "ref_cases_golden.npz")
    np.savez_compressed(path, **out)
    print(path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
