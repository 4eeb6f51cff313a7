"""Pins the oracle (oracle/dsac_oracle.cpp, the CPU restatement every GPU parity test is checked against) to the
REFERENCE'S OWN CODE.

oracle/_ref is the reference's core/{cnn_softam.h, maxloss.h, Hypothesis.cpp, types.h, thread_rand.cpp, properties.cpp,
read_data.cpp, dataset.h, lua_calls.h, test_ransac_softam.cpp, train_ransac_softam.cpp} compiled UNMODIFIED against API
shims (oracle/shim: OpenCV containers with the calib3d numerics forwarded to the oracle's restated primitives, a Lua
C-API stand-in whose "score CNN" is the closed-form soft-inlier score, png++) -- see oracle/Makefile.  What is pinned
is therefore everything above the OpenCV boundary: the sampling loop and its RNG use, reprojection-error maps, softmax /
soft-argmax, the refinement loop and its stop rules, evaluation, every finite-difference factor of the backward pass
and the gradient assembly inside the reference's own main(), including the quirks Q1, Q2, Q4, Q6, Q7, Q8, Q10
(SURVEY.md section 7).  The OpenCV boundary itself is pinned to cv2 4.13 in tests/test_oracle_golden.py.

The reference's outputs are frozen from oracle/_ref as fixtures: tests/golden/ref_golden.npz (make_ref_golden.py) and,
for the parameter sets of the tests below, tests/golden/ref_cases_golden.npz (make_ref_cases_golden.py, which also says
how large arrays are stored: digests of bit-exact integer arrays, seeded samples of the gradients).

Tolerances: integer work (sampled indices, inlier maps, permutations, step counts) bit-exact; poses, scores, softmax,
losses and all gradient factors 1e-12 relative (measured: 0 .. 3e-14).
"""
import importlib.util
import os

import numpy as np
import pytest

from oracle import ref as R

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
GOLD = os.path.join(GOLDEN, "ref_golden.npz")
_spec = importlib.util.spec_from_file_location("make_ref_cases_golden", os.path.join(GOLDEN, "make_ref_cases_golden.py"))
G = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(G)


@pytest.fixture(scope="module")
def ref_cases():
    """tests/golden/ref_cases_golden.npz as {case: {field: array}}."""
    z = np.load(os.path.join(GOLDEN, "ref_cases_golden.npz"))
    out = {}
    for k in z.files:
        case, field = k.split("/")
        out.setdefault(case, {})[field] = z[k]
    return out


def rel(a, b):
    a, b = np.asarray(a, float), np.asarray(b, float)
    return np.abs(a - b).max() / max(1e-300, np.abs(b).max())


def sampled_rel(a, g, name):
    """rel() of `a` against a reference array stored as a sample (G.sampled): over the sampled entries, normalised by the
    whole reference array's largest magnitude, which is compared with a's as well."""
    a = np.asarray(a, float).reshape(-1)
    m = float(g[name + "_absmax"])
    d = np.abs(a[G.sample_index(name, a.size)] - g[name + "_sample"]).max()
    return max(d, abs(np.abs(a).max() - m)) / max(1e-300, m)


def check_forward(o, r, H):
    assert np.array_equal(o.img_idx, r["img_idx"])
    assert rel(o.hyp_rvec, r["hyp_rvec"]) <= 1e-12 and rel(o.hyp_tvec, r["hyp_tvec"]) <= 1e-12
    assert rel(o.scores, r["scores"]) <= 1e-12 and np.abs(o.sf - r["sf"]).max() <= 1e-12
    assert abs(o.entropy - float(r["entropy"])) <= 1e-12
    assert rel(o.avg, r["avg"]) <= 1e-12 and rel(o.ref, r["ref"]) <= 1e-12
    assert np.array_equal(o.inlier_map, r["inlier_map"]) and o.n_perm_steps == int(r["n_perm_steps"])
    assert abs(o.loss - float(r["loss"])) <= 1e-10 and abs(o.rot_err - float(r["rot_err"])) <= 1e-10
    assert abs(o.t_err - float(r["t_err"])) <= 1e-9 and o.correct == int(r["correct"])


# ------------------------------------------------------------------------------------------------ reference cases
def test_rng_contract_is_the_references(oracle, engine_mod, ref_cases):
    """stochasticSubSample through the reference's ThreadRand (thread_rand.cpp:59-81, cnn_softam.h:283-309)."""
    for seed in G.RNG_SEEDS:
        ref_pix = ref_cases["rng_%d" % seed]["pix"]
        assert np.array_equal(ref_pix, oracle.stochastic_subsample(seed))
        assert np.array_equal(ref_pix, engine_mod.stochastic_subsample(seed))


@pytest.mark.parametrize("T,H,frames", [(1, 64, (0, 1, 2)), (1, 256, (4,)), (8, 256, (2,)), (3, 64, (6,)), (8, 64, (9, 10))])
def test_forward_equals_reference_process_image(oracle, engine_mod, ref_cases, T, H, frames):
    """processImage (cnn_softam.h:960-1180) with OMP_NUM_THREADS = T  <->  orc_forward with n_streams = T (configs 1, 2)."""
    O, E = oracle, engine_mod
    for g in frames:
        coords, pix, gt_cv, gt_jp = E.synth_frames(1, frame0=g, n_streams=T)
        r = ref_cases[G.forward_key(T, H, g)]
        assert r["pix_sha256"] == G.digest(pix[0]) and r["est_obj_sha256"] == G.digest(coords[0])
        o = O.forward(O.default_config(seed=1305 + g * T, n_hyps=H, n_streams=T), coords[0], pix[0], gt_jp[0, :9], gt_jp[0, 9:])
        assert o.n_fragile == 0
        check_forward(o, r, H)
        assert G.digest(o.diffmaps) == r["diffmaps_sha256"]              # getDiffMap, cnn_softam.h:319-362
        assert G.digest(o.pixel_idxs) == r["pixel_idxs_sha256"]          # std::shuffle permutations, quirk Q2


@pytest.mark.parametrize("T,H,g", [(1, 64, 1), (8, 256, 3)])
def test_backward_factors_equal_the_references(oracle, engine_mod, ref_cases, T, H, g):
    """dLossMax, dRefineObj (x skip, Q8), dRefineHyp (unit mix, Q7), dPNP by the reference's own functions (config 3)."""
    O, E = oracle, engine_mod
    coords, pix, gt_cv, gt_jp = E.synth_frames(1, frame0=g, n_streams=T)
    oc = O.default_config(seed=1305 + g * T, n_hyps=H, n_streams=T)
    o = O.forward(oc, coords[0], pix[0], gt_jp[0, :9], gt_jp[0, 9:])
    ob = O.backward(oc, coords[0], pix[0], gt_jp[0, :9], gt_jp[0, 9:], o)
    fa = ref_cases[G.factors_key(T, H, g)]
    assert rel(ob.dloss_dref, fa["dloss_dref"]) <= 1e-12
    assert rel(ob.dref_dhyp, fa["dref_dhyp"]) <= 1e-12
    assert sampled_rel(ob.dref_dobj, fa, "dref_dobj") <= 1e-12 and float(fa["dref_dobj_absmax"]) > 0
    assert sampled_rel(ob.dpnp, fa, "dpnp") <= 1e-12


@pytest.mark.parametrize("T,H,g", [(1, 64, 0), (1, 256, 2), (8, 256, 5)])
def test_training_round_gradient_equals_the_references_main(oracle, engine_mod, ref_cases, T, H, g):
    """One round of main() of train_ransac_softam.cpp (forward, paths I and II, the x-major dScore columns of quirk Q4, the
    assembly of lines 288-394) on a one-frame dataset on disk; dLoss_dObj is captured where the driver hands it to the
    coordinate CNN (:412).  The ground truth goes through the reference's 7-Scenes pose reader (read_data.cpp:69-133)."""
    O, E = oracle, engine_mod
    coords, pix, gt_cv, gt_jp = E.synth_frames(1, frame0=g, n_streams=T)
    r = ref_cases[G.train_key(T, H, g)]
    Rg, tg = r["gt_R"], r["gt_t"]
    assert np.abs(Rg.reshape(-1) - gt_jp[0, :9]).max() < 1e-6 and np.abs(tg - gt_jp[0, 9:]).max() < 1e-3   # float round trip
    oc = O.default_config(seed=1305 + g * T, n_hyps=H, n_streams=T)
    o = O.forward(oc, coords[0], pix[0], Rg, tg)
    ob = O.backward(oc, coords[0], pix[0], Rg, tg, o)
    assert abs(o.loss - float(r["loss"])) <= 1e-10
    assert rel(ob.score_grads, r["score_out_grads"]) <= 1e-10
    assert sampled_rel(ob.dloss_dobj, r, "dloss_dobj") <= 1e-12 and float(r["dloss_dobj_absmax"]) > 0


def test_test_driver_logs_equal_the_references_main(oracle, engine_mod, ref_cases):
    """main() of test_ransac_softam.cpp over a 12-frame trajectory (config 5 in small): its per-frame log (loss, entropy,
    errors, pose converted back to the 7-Scenes convention, :161-223) and its summary line (:251-263) against the same
    quantities from the oracle, compared at the 6 significant digits the reference prints."""
    O, E = oracle, engine_mod
    n, H = G.DRIVER_FRAMES, G.DRIVER_H
    coords, pix, gt_cv, gt_jp = E.synth_frames(n, traj=True)
    tr = np.array(G.DRIVER_TRANSLATION)
    r = ref_cases["driver"]
    gts = list(zip(r["gt_R"], r["gt_t"]))
    per_frame, summary = r["per_frame"], r["summary"]
    assert per_frame.shape == (n, 10)
    losses, ents, rots, ts, corr = [], [], [], [], []
    for i in range(n):
        o = O.forward(O.default_config(seed=1305 + i, n_hyps=H), coords[i], pix[i], gts[i][0], gts[i][1])
        Rj, tj = O.cv2our(o.ref[:3], o.ref[3:])
        M = np.eye(4); M[:3, :3] = Rj; M[:3, 3] = tj
        P = np.linalg.inv(M) @ np.diag([1.0, -1.0, -1.0, 1.0])
        want = [o.loss, o.entropy, o.t_err, o.rot_err] + list(O.rodrigues_inv(P[:3, :3])) + list(P[:3, 3] / 1000.0 + tr)
        got = [float(v) for v in per_frame[i]]
        for w, gv in zip(want, got):
            assert abs(w - gv) <= 1e-5 * max(1.0, abs(w)), (i, want, got)
        losses.append(o.loss); ents.append(o.entropy); rots.append(o.rot_err); ts.append(o.t_err); corr.append(o.correct)
    want = [np.mean(corr), np.mean(losses), np.std(losses), np.mean(ents), np.std(ents), sorted(rots)[n // 2], sorted(ts)[n // 2]]
    assert len(summary) == len(want)
    for w, gv in zip(want, [float(v) for v in summary]):
        assert abs(w - gv) <= 1e-5 * max(1.0, abs(w))


# ------------------------------------------------------------------------------------------------ frozen fixtures
def _cases():
    z = np.load(GOLD)
    names = sorted({k.split("/")[0] for k in z.files})
    return z, names


def test_oracle_matches_the_reference_fixtures(oracle):
    """The same comparison against outputs of oracle/_ref frozen in tests/golden/ref_golden.npz (runs on any box)."""
    O = oracle
    z, names = _cases()
    assert len(names) >= 7
    for name in names:
        g = {k.split("/")[1]: z[k] for k in z.files if k.startswith(name + "/")}
        H, T, f = int(g["H"]), int(g["T"]), int(g["frame"])
        oc = O.default_config(seed=1305 + f * T, n_hyps=H, n_streams=T)
        o = O.forward(oc, g["coords"], g["pix"], g["gt_R"], g["gt_t"])
        check_forward(o, g, H)
        assert np.abs(o.diffmaps[:: max(1, H // 8)] - g["diffmap_rows"]).max() == 0.0
        if "dloss_dobj" in g:
            ob = O.backward(oc, g["coords"], g["pix"], g["gt_R"], g["gt_t"], o)
            assert rel(ob.dloss_dobj, g["dloss_dobj"]) <= 1e-12
            assert rel(ob.score_grads, g["score_out_grads"]) <= 1e-10
            assert rel(ob.dloss_dref, g["dloss_dref"]) <= 1e-12 and rel(ob.dref_dhyp, g["dref_dhyp"]) <= 1e-12


def test_pose_file_reader_equals_the_references(engine_mod, ref_cases, tmp_path):
    """SURVEY.md section 8(f) N3: the host mirror's 7-Scenes pose reader (dsac_b200/host/read_data.cpp) against the
    reference's own readData + Hypothesis(info) (core/read_data.cpp:69-133) on pose files with a scene offset."""
    import subprocess
    E = engine_mod
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    subprocess.check_call(["make", "-C", os.path.join(root, "apps"), "-s", "host_selftest"])
    coords, pix, gt_cv, gt_jp = E.synth_frames(G.POSE_FRAMES, traj=True)
    d = str(tmp_path)
    R.write_dataset(d, "test", gt_jp, translation=G.POSE_TRANSLATION)
    r = ref_cases["pose"]
    for i in range(G.POSE_FRAMES):
        rel_path = os.path.join("test", "synth", "poses", "frame-%06d.pose.txt" % i)
        Rg, tg = r["gt_R"][i], r["gt_t"][i]
        out = subprocess.run([os.path.join(root, "apps", "host_selftest"), "pose", rel_path], cwd=d, capture_output=True, text=True, timeout=60)
        assert out.returncode == 0, out.stdout + out.stderr
        v = np.array([float(x) for x in out.stdout.split()])
        assert np.abs(v[:9] - Rg.reshape(-1)).max() <= 2e-7 and np.abs(v[9:] - tg).max() <= 1e-3   # float arithmetic on both sides
        assert np.abs(v[:9] - gt_jp[i, :9]).max() <= 1e-6 and np.abs(v[9:] - gt_jp[i, 9:]).max() <= 5e-3


# ------------------------------------------------------------------------------------------------ DSAC / RANSAC variant (SURVEY.md 8f, N1)
@pytest.mark.parametrize("T,H,g,random_draw", [(1, 64, 0, True), (1, 64, 3, False), (4, 32, 2, True)])
def test_dsac_variant_forward_equals_reference_process_image(oracle, engine_mod, ref_cases, T, H, g, random_draw):
    """processImage of core/cnn.h:1028-1257 (draw :102-126, refinement of every hypothesis :1155-1228, expectedMaxLoss
    :137-151) by the reference's own code  <->  orc_forward_dsac."""
    O, E = oracle, engine_mod
    coords, pix, gt_cv, gt_jp = E.synth_frames(1, frame0=g, n_streams=T)
    r = ref_cases[G.dsac_forward_key(T, H, g, random_draw)]
    o = O.forward_dsac(O.default_config(seed=1305 + g * T, n_hyps=H, n_streams=T), coords[0], pix[0], gt_jp[0, :9], gt_jp[0, 9:], random_draw)
    assert np.array_equal(o.img_idx, r["img_idx"]) and o.hyp_idx == int(r["hyp_idx"]) and o.correct == int(r["correct"])
    assert G.digest(o.inlier_maps) == r["inlier_maps_sha256"]
    assert rel(o.hyp_rvec, r["hyp_rvec"]) <= 1e-12 and rel(o.hyp_tvec, r["hyp_tvec"]) <= 1e-12
    assert np.abs(o.sf - r["sf"]).max() <= 1e-12 and rel(o.ref_pose, r["ref_pose"]) <= 1e-12
    assert np.abs(o.losses - r["losses"]).max() <= 1e-9 and abs(o.expected_loss - float(r["expected_loss"])) <= 1e-10
    assert abs(o.rot_err - float(r["rot_err"])) <= 1e-9 and abs(o.t_err - float(r["t_err"])) <= 1e-9


@pytest.mark.parametrize("T,H,g", [(1, 32, 1), (4, 48, 6)])
def test_dsac_variant_gradient_equals_the_references_main(oracle, engine_mod, ref_cases, T, H, g):
    """One round of main() of core/train_ransac.cpp (expectation of the loss: sum_h sf_h dLossMax dRefine_h + dSMScore,
    lines 304-381) on a one-frame dataset  <->  orc_backward_dsac."""
    O, E = oracle, engine_mod
    coords, pix, gt_cv, gt_jp = E.synth_frames(1, frame0=g, n_streams=T)
    r = ref_cases[G.dsac_train_key(T, H, g)]
    Rg, tg = r["gt_R"], r["gt_t"]
    oc = O.default_config(seed=1305 + g * T, n_hyps=H, n_streams=T)
    o = O.forward_dsac(oc, coords[0], pix[0], Rg, tg, True)
    ob = O.backward_dsac(oc, coords[0], pix[0], Rg, tg, o)
    assert abs(o.expected_loss - float(r["loss"])) <= 1e-10
    assert sampled_rel(ob.dloss_dobj, r, "dloss_dobj") <= 1e-10 and float(r["dloss_dobj_absmax"]) > 0
