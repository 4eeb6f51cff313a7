"""GPU parity at BASELINE.json's FULL configs (VERDICT r1, "parity tests undersample BASELINE's configs"), through the C ABI:

  config 4  all 1024 frames x 256 hypotheses against the oracle, frame by frame (the oracle runs on the box's host threads);
  config 3  the backward pass at H = 256 on 4 frames, both dScore column layouts (quirk Q4);
  config 5  the 1000-frame trajectory through apps/test_ransac_softam, its per-frame log against oracle-derived lines;
  and the CUDA engine directly against the fixtures frozen from the REFERENCE'S OWN CODE (tests/golden/ref_golden.npz,
  written by tests/golden/make_ref_golden.py from oracle/_ref).

Measured maxima are printed (pytest -s) and recorded in BASELINE.md section 6.
"""
import os
import subprocess
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _threads():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return os.cpu_count() or 1


def _oracle_frames(O, coords, pix, gt_jp, H, T=1, frame0=0, want_diffmaps=False):
    """orc_forward for every frame on the host threads (ctypes releases the GIL)."""
    def one(f):
        cfg = O.default_config(seed=1305 + (frame0 + f) * T, n_hyps=H, n_streams=T)
        return O.forward(cfg, coords[f], pix[f], gt_jp[f, :9], gt_jp[f, 9:], want_diffmaps=want_diffmaps)
    with ThreadPoolExecutor(max_workers=_threads()) as ex:
        return list(ex.map(one, range(coords.shape[0])))


def test_config4_all_1024_frames_match_the_oracle(engine_mod, oracle):
    E, O = engine_mod, oracle
    nf, H = 1024, 256
    coords, pix, gt_cv, gt_jp = E.synth_frames(nf)
    eng = E.Engine(max_frames=nf)
    res = eng.forward(coords, pix, gt_jp)
    eng.close()
    ora = _oracle_frames(O, coords, pix, gt_jp, H)
    mx = dict(rvec=0.0, tvec=0.0, score_rel=0.0, sf=0.0, avg_r=0.0, avg_t=0.0, ref_r=0.0, ref_t=0.0, loss=0.0)
    for f, o in enumerate(ora):
        assert o.n_fragile == 0
        assert np.array_equal(o.img_idx, res.img_idx[f]), f                 # sampled point indices: bit-exact
        assert np.array_equal(o.cand_idx, res.cand_idx[f]), f
        assert o.n_candidates == res.n_candidates[f], f
        assert np.array_equal(o.inlier_map, res.inlier_map[f]), f
        assert o.ref_steps_done == res.ref_steps_done[f] and o.n_perm_steps == res.n_perm_steps[f] and res.status[f] == 0
        assert o.correct == res.correct[f]
        mx["rvec"] = max(mx["rvec"], np.abs(o.hyp_rvec - res.hyp_pose[f][:, :3]).max())
        mx["tvec"] = max(mx["tvec"], np.abs(o.hyp_tvec - res.hyp_pose[f][:, 3:]).max())
        mx["score_rel"] = max(mx["score_rel"], np.abs(o.scores - res.scores[f]).max() / np.abs(o.scores).max())
        mx["sf"] = max(mx["sf"], np.abs(o.sf - res.sf[f]).max())
        mx["avg_r"] = max(mx["avg_r"], np.abs(o.avg[:3] - res.avg_pose[f][:3]).max())
        mx["avg_t"] = max(mx["avg_t"], np.abs(o.avg[3:] - res.avg_pose[f][3:]).max())
        mx["ref_r"] = max(mx["ref_r"], np.abs(o.ref[:3] - res.ref_pose[f][:3]).max())
        mx["ref_t"] = max(mx["ref_t"], np.abs(o.ref[3:] - res.ref_pose[f][3:]).max())
        mx["loss"] = max(mx["loss"], abs(o.loss - res.loss[f]))
    print("config 4, measured maxima over 1024 frames x 256 hypotheses:", {k: float("%.3g" % v) for k, v in mx.items()})
    # asserted at ~5x the measured maxima (BASELINE.md section 6: rvec 2.7e-10, tvec 3.9e-7, scores 1.05e-5, sf 4.1e-6,
    # soft-argmax pose 6.4e-8 rad / 1.6e-4 mm, refined pose 1.3e-10 rad / 4.5e-7 mm, loss 3.0e-8)
    assert mx["rvec"] <= 1e-9 and mx["tvec"] <= 2e-6
    assert mx["score_rel"] <= 2e-5 and mx["sf"] <= 2e-5
    assert mx["avg_r"] <= 1e-6 and mx["avg_t"] <= 2e-3         # soft-argmax pose: rad / mm (propagated fp32 score error)
    assert mx["ref_r"] <= 1e-8 and mx["ref_t"] <= 1e-5          # refined pose: far inside the 0.01 deg / 0.1 mm contract
    assert mx["loss"] <= 1e-6


@pytest.mark.parametrize("fix_q4", [0, 1])
def test_config3_backward_at_256_hypotheses(engine_mod, oracle, fix_q4):
    E, O = engine_mod, oracle
    nf, H = 4, 256
    coords, pix, gt_cv, gt_jp = E.synth_frames(nf, frame0=40)
    eng = E.Engine(max_frames=nf, n_hyps=H, fix_q4=fix_q4)
    fwd = eng.forward(coords, pix, gt_jp, frame0=40)
    bw = eng.backward(coords, pix, gt_jp)
    eng.close()

    def one(f):
        cfg = O.default_config(seed=1305 + 40 + f, n_hyps=H, fix_q4=fix_q4)
        ofw = O.forward(cfg, coords[f], pix[f], gt_jp[f, :9], gt_jp[f, 9:], want_diffmaps=False)
        return ofw, O.backward(cfg, coords[f], pix[f], gt_jp[f, :9], gt_jp[f, 9:], ofw)
    with ThreadPoolExecutor(max_workers=min(nf, _threads())) as ex:
        ora = list(ex.map(one, range(nf)))
    rel = lambda a, b, floor=1e-300: np.abs(a - b).max() / max(floor, np.abs(b).max())   # noqa: E731
    worst = 0.0
    for f, (ofw, obw) in enumerate(ora):
        assert np.array_equal(ofw.img_idx, fwd.img_idx[f]) and np.array_equal(ofw.inlier_map, fwd.inlier_map[f])
        assert rel(bw.dloss_dref[f], obw.dloss_dref) <= 1e-9
        assert rel(bw.dref_dhyp[f], obw.dref_dhyp, 1e-3) <= 1e-7
        assert rel(bw.dref_dobj[f], obw.dref_dobj, 1e-3) <= 1e-7
        assert rel(bw.dpnp[f], obw.dpnp) <= 1e-7
        assert rel(bw.score_grads[f], obw.score_grads, 1e-6) <= 1e-4
        worst = max(worst, rel(bw.dloss_dobj[f], obw.dloss_dobj, 1e-6))
    print("config 3 (H=256, fix_q4=%d): final gradient, max relative-to-max difference %.3g" % (fix_q4, worst))
    assert worst <= 1e-4     # measured 9.3e-6: BASELINE.md's 1e-4-of-max contract holds at config 3's full size


def test_config5_thousand_frame_sequence_logs(engine_mod, oracle, tmp_path):
    """apps/test_ransac_softam (the C++ driver on the C ABI) over the 1000-frame 7Scenes-shaped trajectory: every line of its
    per-frame log against the same line derived from the oracle, compared as text at the 6 significant digits the
    reference's ofstream prints -- fields may differ in the last printed digit where the fp32 score error moves them."""
    E, O = engine_mod, oracle
    apps = os.path.join(ROOT, "apps")
    subprocess.check_call(["make", "-C", apps, "-s"])
    nf, H = 1000, 256
    out = subprocess.run([os.path.join(apps, "test_ransac_softam"), "-frames", str(nf), "-batch", "250"], cwd=tmp_path,
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout + out.stderr
    errs = np.loadtxt(tmp_path / "ransac_test_errors_obj_model_init.net_rdraw1_softam.txt")
    summ = np.loadtxt(tmp_path / "ransac_test_loss_obj_model_init.net_rdraw1_softam.txt")
    assert errs.shape == (nf, 10) and summ.shape == (7,)
    coords, pix, gt_cv, gt_jp = E.synth_frames(nf, traj=True)
    ora = _oracle_frames(O, coords, pix, gt_jp, H)
    want = np.zeros((nf, 10))
    for f, o in enumerate(ora):
        Rj, tj = O.cv2our(o.ref[:3], o.ref[3:])
        M = np.eye(4); M[:3, :3] = Rj; M[:3, 3] = tj
        P = np.linalg.inv(M) @ np.diag([1.0, -1.0, -1.0, 1.0])     # back to the 7-Scenes convention, test_ransac_softam.cpp:161-185
        want[f] = [o.loss, o.entropy, o.t_err, o.rot_err] + list(O.rodrigues_inv(P[:3, :3])) + list(P[:3, 3] / 1000.0)
    tol = 2e-5 * np.maximum(1.0, np.abs(want)) + np.array([1e-4, 1e-3, 1e-3, 1e-4, 1e-5, 1e-5, 1e-5, 1e-5, 1e-5, 1e-5])
    bad = np.abs(errs - want) > tol
    print("config 5: max |log - oracle| per column", np.abs(errs - want).max(0))
    assert not bad.any(), (np.argwhere(bad)[:5], errs[bad][:5], want[bad][:5])
    acc = np.mean([o.correct for o in ora])
    assert abs(summ[0] - acc) < 1e-9 and abs(summ[5] - np.sort([o.rot_err for o in ora])[nf // 2]) < 1e-4
    assert abs(summ[6] - np.sort([o.t_err for o in ora])[nf // 2]) < 1e-2


def test_engine_matches_the_reference_fixtures(engine_mod):
    """The CUDA engine against outputs of the reference's own code (oracle/_ref frozen in tests/golden/ref_golden.npz):
    sampled indices, inlier maps, step counts bit-exact; poses, scores, softmax, refined pose, loss and the gradient of one
    training round within the fp32-score tolerances."""
    E = engine_mod
    z = np.load(os.path.join(ROOT, "tests", "golden", "ref_golden.npz"))
    names = sorted({k.split("/")[0] for k in z.files})
    assert len(names) >= 7
    for name in names:
        g = {k.split("/")[1]: z[k] for k in z.files if k.startswith(name + "/")}
        H, T, f = int(g["H"]), int(g["T"]), int(g["frame"])
        gt = np.concatenate([g["gt_R"].reshape(9), g["gt_t"].reshape(3)])[None]
        eng = E.Engine(max_frames=1, n_hyps=H, n_streams=T)
        r = eng.forward(g["coords"][None], g["pix"][None], gt, frame0=f, want_diffmaps=True)
        assert np.array_equal(r.img_idx[0], g["img_idx"]), name
        assert np.array_equal(r.inlier_map[0], g["inlier_map"]) and r.n_perm_steps[0] == int(g["n_perm_steps"])
        assert np.abs(r.hyp_pose[0][:, :3] - g["hyp_rvec"]).max() <= 1e-9 and np.abs(r.hyp_pose[0][:, 3:] - g["hyp_tvec"]).max() <= 1e-6
        assert np.abs(r.diffmaps[0][:: max(1, H // 8)] - g["diffmap_rows"]).max() <= 2e-3
        assert np.abs(r.scores[0] - g["scores"]).max() <= 1e-5 * np.abs(g["scores"]).max()
        assert np.abs(r.sf[0] - g["sf"]).max() <= 1e-4 and abs(r.entropy[0] - float(g["entropy"])) <= 1e-3
        assert np.abs(r.ref_pose[0][:3] - g["ref"][:3]).max() <= 1e-6 and np.abs(r.ref_pose[0][3:] - g["ref"][3:]).max() <= 1e-3
        assert abs(r.loss[0] - float(g["loss"])) <= 1e-4 and r.correct[0] == int(g["correct"])
        if "dloss_dobj" in g:
            bw = eng.backward(g["coords"][None], g["pix"][None], gt)
            d = np.abs(bw.dloss_dobj[0] - g["dloss_dobj"]).max() / np.abs(g["dloss_dobj"]).max()
            assert d <= 5e-3, (name, d)   # measured up to 1.0e-3 at H = 64 (few hypotheses carry the soft-argmax; 9e-6 at H = 256)
            # dLossMax at the GPU's refined pose vs at the reference's: the poses differ by <= 1e-6 rad (fp32 scores ->
            # soft-argmax -> refinement) and d(angle)/d(pose) carries a 1 / sin(angle) factor at sub-degree errors
            assert np.abs(bw.dloss_dref[0] - g["dloss_dref"]).max() <= 1e-3 * max(1.0, np.abs(g["dloss_dref"]).max())
        eng.close()


def test_score_seam_adjoint_hook(engine_mod):
    """dsac_set_score_backward_hook (lua_calls.h:312-341).  The forward hook leaves the scores alone (k_score has already
    written the closed-form soft-inlier scores, so softmax and soft-argmax are those of the plain engine); the backward
    hook differentiates the same score with torch autograd on the DEVICE diffmaps.
      (a) autograd hook == analytic torch hook (-alpha beta s (1 - s) * clamped output gradient) to 1e-9: the plumbing;
      (b) hook gradient == the engine's closed-form gradient to 5e-3 of max: the only difference is that the hook sees the
          materialised fp32 error matrix (<= 2e-3 px from the exact errors, times beta = 0.5), while the closed-form kernel
          re-evaluates the errors with the reference's exact roundings;
      (c) one hook without the other is an error, not a silently different gradient."""
    import torch
    E = engine_mod
    nf, H = 2, 64
    coords, pix, gt_cv, gt_jp = E.synth_frames(nf)
    plain = E.Engine(max_frames=nf, n_hyps=H)
    plain.forward(coords, pix, gt_jp)
    want = plain.backward(coords, pix, gt_jp, full=False)
    plain.close()

    class _W:
        def __init__(self, ptr, shape, typestr):
            self.__cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (ptr, False), "version": 2}

    seen = {}

    def fwd_hook(dm, n, Hh, sc, stream):
        return 0

    def bwd_autograd(dm, sg, n, Hh, out, stream):
        with torch.cuda.stream(torch.cuda.ExternalStream(stream)):   # the engine's backward stream
            d = torch.as_tensor(_W(dm, (n, Hh, 1600), "<f4"), device="cuda").double().requires_grad_(True)
            g = torch.as_tensor(_W(sg, (n, Hh), "<f8"), device="cuda")
            seen["max_out_grad"] = float(g.abs().max())
            o = torch.as_tensor(_W(out, (n, Hh, 1600), "<f8"), device="cuda")
            score = 0.1 * torch.sigmoid(0.5 * (10.0 - d)).sum(2)
            score.backward(g.clone())
            o.copy_(d.grad)
        return 0

    def bwd_analytic(dm, sg, n, Hh, out, stream):
        with torch.cuda.stream(torch.cuda.ExternalStream(stream)):
            d = torch.as_tensor(_W(dm, (n, Hh, 1600), "<f4"), device="cuda").double()
            g = torch.as_tensor(_W(sg, (n, Hh), "<f8"), device="cuda")
            o = torch.as_tensor(_W(out, (n, Hh, 1600), "<f8"), device="cuda")
            s = torch.sigmoid(0.5 * (10.0 - d))
            o.copy_(g[:, :, None] * (-0.1 * 0.5) * s * (1 - s))
        return 0

    eng = E.Engine(max_frames=nf, n_hyps=H)
    eng.set_score_hook(fwd_hook)
    eng.forward(coords, pix, gt_jp)
    with pytest.raises(RuntimeError, match="both hooks"):
        eng.backward(coords, pix, gt_jp, full=False)          # (c) forward hook only
    eng.set_score_backward_hook(bwd_autograd)
    eng.forward(coords, pix, gt_jp)
    got = eng.backward(coords, pix, gt_jp, full=False)
    assert seen["max_out_grad"] <= 0.1 + 1e-15                # the hook receives the clamped output gradients
    eng.set_score_backward_hook(bwd_analytic)
    eng.forward(coords, pix, gt_jp)
    got2 = eng.backward(coords, pix, gt_jp, full=False)
    eng.set_score_hook(None)
    with pytest.raises(RuntimeError, match="both hooks"):
        eng.backward(coords, pix, gt_jp, full=False)          # (c) backward hook only
    eng.close()
    for f in range(nf):
        scale = np.abs(want.dloss_dobj[f]).max()
        assert np.array_equal(got.score_grads[f], want.score_grads[f])                       # same scores, same softmax
        assert np.abs(got.dloss_dobj[f] - got2.dloss_dobj[f]).max() <= 1e-9 * scale          # (a)
        assert np.abs(got.dloss_dobj[f] - want.dloss_dobj[f]).max() <= 5e-3 * scale          # (b)
        assert np.abs(got.dloss_dobj[f] - want.dloss_dobj[f]).max() > 0                      # ... and it really took the hook's path


def test_two_lanes_are_scheduling_only(engine_mod):
    """A batch of >= 768 frames runs as two concurrent half-batches with their own queues, counters and side streams
    (engine.cu: forward_split, lane 1); dsac_set_tail_split(0) keeps it in one pass.  Frames are independent and sampler
    streams keyed by the global frame index: the results must be those of the single pass, bit for bit."""
    E = engine_mod
    nf = 800
    coords, pix, gt_cv, gt_jp = E.synth_frames(nf)
    out = {}
    for lanes in ("1", "0"):
        eng = E.Engine(max_frames=nf)
        eng.set_tail_split(int(lanes))
        out[lanes] = eng.forward(coords, pix, gt_jp)
        out[lanes + "b"] = eng.forward(coords, pix, gt_jp)      # a second call: the lanes' own acceptance-rate priors are in use
        eng.close()
    for name in ("img_idx", "cand_idx", "n_candidates", "hyp_pose", "scores", "sf", "avg_pose", "ref_pose", "inlier_map", "loss", "status"):
        assert np.array_equal(getattr(out["1"], name), getattr(out["0"], name)), name
        assert np.array_equal(getattr(out["1b"], name), getattr(out["0"], name)), name
    assert int(out["1"].status.sum()) == 0

