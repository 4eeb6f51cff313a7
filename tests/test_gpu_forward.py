"""GPU parity tests proper: the CUDA engine, called through the C ABI, against the oracle on the
same seeded inputs (SURVEY.md section 8c(3)); plus size-independent properties at BASELINE.json's sizes.

Tolerances (stated here, mirrored in DESIGN.md):
  sampled indices / candidate indices / candidate counts ... bit-exact
  hypothesis poses (fp64 P3P) ............................. 1e-9 rad, 1e-6 mm
  diffmap entries (fp32 projection) ....................... 2e-3 px abs
  scores .................................................. 1e-5 relative to max score
  softmax of identical scores ............................. 1e-12 abs;  end-to-end sf: 1e-4 abs
  soft-argmax pose ........................................ 1e-3 rad-or-mm abs (propagated fp32 score error)
  refined pose ............................................ 1e-6 rad, 1e-3 mm  (0.01 deg / 0.1 mm is the contract)
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _oracle_frame(O, cfg_kw, coords, pix, gt_jp, f, T):
    cfg = O.default_config(seed=1305 + f * T, n_streams=T, **cfg_kw)
    return O.forward(cfg, coords, pix, gt_jp[:9], gt_jp[9:])


@pytest.mark.parametrize("T,H", [(1, 256), (8, 256), (3, 64), (64, 64)])
def test_forward_matches_oracle(engine_mod, oracle, T, H):
    E, O = engine_mod, oracle
    nf = 3
    coords, pix, gt_cv, gt_jp = E.synth_frames(nf, n_streams=T)
    eng = E.Engine(max_frames=nf, n_streams=T, n_hyps=H)
    res = eng.forward(coords, pix, gt_jp, want_diffmaps=True)
    for f in range(nf):
        fw = _oracle_frame(O, dict(n_hyps=H), coords[f], pix[f], gt_jp[f], f, T)
        assert fw.n_fragile == 0
        # --- bit-exact integer work
        assert np.array_equal(fw.img_idx, res.img_idx[f])
        assert np.array_equal(fw.cand_idx, res.cand_idx[f])
        assert fw.n_candidates == res.n_candidates[f]
        assert res.status[f] == 0
        # --- hypothesis poses
        assert np.abs(fw.hyp_rvec - res.hyp_pose[f][:, :3]).max() <= 1e-9
        assert np.abs(fw.hyp_tvec - res.hyp_pose[f][:, 3:]).max() <= 1e-6
        # --- H x N reprojection-error matrix
        assert np.abs(fw.diffmaps - res.diffmaps[f]).max() <= 2e-3
        assert res.diffmaps[f].max() <= 100.0 and res.diffmaps[f].min() >= 0.0
        # --- scores / softmax / soft-argmax
        assert np.abs(fw.scores - res.scores[f]).max() <= 1e-5 * np.abs(fw.scores).max()
        assert np.abs(O.softmax(res.scores[f]) - res.sf[f]).max() <= 1e-12
        assert abs(O.entropy(res.sf[f]) - res.entropy[f]) <= 1e-9
        assert np.abs(fw.sf - res.sf[f]).max() <= 1e-4
        avg_from_gpu_sf = (res.sf[f][:, None] * res.hyp_pose[f]).sum(0)
        assert np.abs(avg_from_gpu_sf - res.avg_pose[f]).max() <= 1e-9 * max(1.0, np.abs(avg_from_gpu_sf).max())
        assert np.abs(fw.avg - res.avg_pose[f]).max() <= 1e-3
        # --- refinement + evaluation
        assert fw.ref_steps_done == res.ref_steps_done[f] and fw.n_perm_steps == res.n_perm_steps[f]
        assert np.array_equal(fw.inlier_map, res.inlier_map[f])
        assert np.abs(fw.ref[:3] - res.ref_pose[f][:3]).max() <= 1e-6
        assert np.abs(fw.ref[3:] - res.ref_pose[f][3:]).max() <= 1e-3
        assert abs(fw.loss - res.loss[f]) <= 1e-4 and abs(fw.rot_err - res.rot_err[f]) <= 1e-4
        assert abs(fw.t_err - res.t_err[f]) <= 1e-2 and fw.correct == res.correct[f]
    eng.close()


@pytest.mark.parametrize("T,nf", [(1, 1), (1, 3), (2, 2), (3, 1), (1, 8)])
def test_speculative_first_round_is_scheduling_only(engine_mod, oracle, T, nf, monkeypatch):
    """k1_spec / k1_stitch / k1_gather (a few streams: the first round generated window by window on many SMs, four alignments
    per window, stitched afterwards) must give exactly the candidates of the one-CTA-per-stream generator -- and the oracle's."""
    E, O = engine_mod, oracle
    H = 256
    coords, pix, gt_cv, gt_jp = E.synth_frames(nf, n_streams=T)
    out = {}
    for spec in ("1", "0"):
        monkeypatch.setenv("DSAC_K1_SPEC", spec)
        eng = E.Engine(max_frames=nf, n_streams=T, n_hyps=H)
        l0 = eng.launches
        res = eng.forward(coords, pix, gt_jp)
        out[spec] = (res, eng.launches - l0)
        eng.close()
    a, b = out["1"][0], out["0"][0]
    assert out["1"][1] > out["0"][1]                     # the speculative path really ran (three more launches in round 0)
    for name in ("img_idx", "cand_idx", "n_candidates", "hyp_pose", "scores", "ref_pose", "inlier_map", "status"):
        assert np.array_equal(getattr(a, name), getattr(b, name)), name
    for f in range(nf):
        fw = _oracle_frame(O, dict(n_hyps=H), coords[f], pix[f], gt_jp[f], f, T)
        assert np.array_equal(fw.img_idx, a.img_idx[f]) and np.array_equal(fw.cand_idx, a.cand_idx[f])
        assert fw.n_candidates == a.n_candidates[f]


@pytest.mark.parametrize("T,nf", [(1, 12), (2, 20), (1, 150)])
def test_chained_generator_is_scheduling_only(engine_mod, oracle, T, nf, monkeypatch):
    """k1_pipe (DSAC_K1_PIPE=1: K CTAs per stream, window w on CTA w mod K, the first candidate's position handed from window to
    window through a spin on a global flag) must give exactly the candidates of the one-CTA-per-stream generator and the oracle's."""
    E, O = engine_mod, oracle
    H = 256
    coords, pix, gt_cv, gt_jp = E.synth_frames(nf, n_streams=T)
    out = {}
    for pipe in ("1", "0"):
        monkeypatch.setenv("DSAC_K1_PIPE", pipe)
        eng = E.Engine(max_frames=nf, n_streams=T, n_hyps=H)
        out[pipe] = eng.forward(coords, pix, gt_jp)
        eng.close()
    a, b = out["1"], out["0"]
    for name in ("img_idx", "cand_idx", "n_candidates", "hyp_pose", "scores", "ref_pose", "inlier_map", "status"):
        assert np.array_equal(getattr(a, name), getattr(b, name)), name
    for f in (0, nf - 1):
        fw = _oracle_frame(O, dict(n_hyps=H), coords[f], pix[f], gt_jp[f], f, T)
        assert np.array_equal(fw.img_idx, a.img_idx[f]) and np.array_equal(fw.cand_idx, a.cand_idx[f])
        assert fw.n_candidates == a.n_candidates[f]


@pytest.mark.parametrize("threads", [256, 512, 1024])
def test_generator_thread_counts_sample_the_same_sets(engine_mod, oracle, threads, monkeypatch):
    """k1_slot is instantiated for 256 / 512 / 1024 threads per (frame, stream) and chosen by the number of streams
    (engine.cu); every instantiation must give the oracle's minimal sets, candidate for candidate."""
    E, O = engine_mod, oracle
    nf, T, H = 5, 3, 64
    monkeypatch.setenv("DSAC_K1_SLOT_THREADS", str(threads))
    coords, pix, gt_cv, gt_jp = E.synth_frames(nf, n_streams=T)
    eng = E.Engine(max_frames=nf, n_streams=T, n_hyps=H)
    res = eng.forward(coords, pix, gt_jp)
    eng.close()
    for f in range(nf):
        fw = _oracle_frame(O, dict(n_hyps=H), coords[f], pix[f], gt_jp[f], f, T)
        assert np.array_equal(fw.img_idx, res.img_idx[f]) and np.array_equal(fw.cand_idx, res.cand_idx[f])
        assert fw.n_candidates == res.n_candidates[f] and res.status[f] == 0


def test_refine_is_exact_given_the_same_start(engine_mod, oracle):
    """K4 alone (fp64): start the oracle's refine() from the GPU's own average pose."""
    E, O = engine_mod, oracle
    coords, pix, gt_cv, gt_jp = E.synth_frames(2)
    eng = E.Engine(max_frames=2)
    res = eng.forward(coords, pix, gt_jp)
    for f in range(2):
        cfg = O.default_config(seed=1305 + f)
        fw = O.forward(cfg, coords[f], pix[f])
        rep = O.refine(cfg, fw.pixel_idxs, 8, coords[f], pix[f], res.avg_pose[f])
        got = O.jp6(res.ref_pose[f][:3], res.ref_pose[f][3:])
        assert np.abs(rep[:3] - got[:3]).max() <= 1e-10 and np.abs(rep[3:] - got[3:]).max() <= 1e-7


def test_shared_grid_and_no_diffmap_mode(engine_mod):
    E = engine_mod
    coords, pix, gt_cv, gt_jp = E.synth_frames(4)
    shared = np.ascontiguousarray(pix[0])
    a = E.Engine(max_frames=4, write_diffmaps=1).forward(coords, shared, gt_jp)
    b = E.Engine(max_frames=4, write_diffmaps=0).forward(coords, shared, gt_jp)
    c = E.Engine(max_frames=4).forward(coords, np.broadcast_to(shared, (4, 1600, 2)).copy(), gt_jp)
    for x in (b, c):
        assert np.array_equal(a.img_idx, x.img_idx) and np.array_equal(a.scores, x.scores)
        assert np.array_equal(a.ref_pose, x.ref_pose)


def test_edge_cases_exhausted_sampler_and_aborted_refinement(engine_mod, oracle):
    """All-outlier frame: the reference would loop forever; the engine bounds the loop and value-encodes."""
    E, O = engine_mod, oracle
    coords, pix, gt_cv, gt_jp = E.synth_frames(1, rho=0.0)
    eng = E.Engine(max_frames=1, max_candidates=2048, n_hyps=8)
    res = eng.forward(coords, pix, gt_jp)
    cfg = O.default_config(n_hyps=8, max_candidates=2048)
    fw = O.forward(cfg, coords[0], pix[0], gt_jp[0, :9], gt_jp[0, 9:])
    assert np.array_equal(fw.img_idx, res.img_idx[0])
    if fw.status != 0:
        assert res.status[0] & E.ST_SAMPLER_EXHAUSTED
    assert fw.ref_steps_done == res.ref_steps_done[0]
    if res.ref_steps_done[0] < 8:
        assert res.status[0] & E.ST_REFINE_ABORTED
    assert np.isfinite(res.ref_pose).all()
    # saturated / extreme coordinates must not produce NaNs in the scores
    coords2 = coords.copy()
    coords2[0, ::7] = 32767
    coords2[0, 1::7] = -32768
    res2 = eng.forward(coords2, pix, gt_jp, want_diffmaps=True)
    assert np.isfinite(res2.scores).all() and np.isfinite(res2.diffmaps).all()
    assert abs(res2.sf.sum() - 1) < 1e-9


def test_capacity_and_argument_errors(engine_mod):
    E = engine_mod
    eng = E.Engine(max_frames=2)
    coords, pix, _, gt = E.synth_frames(3)
    with pytest.raises(RuntimeError) as ei:
        eng.forward(coords, pix, gt)
    assert "capacity" in str(ei.value)
    with pytest.raises(RuntimeError):
        E.Engine(n_hyps=0)
    with pytest.raises(RuntimeError):
        E.Engine(inlier_count=1000)


def test_full_size_properties(engine_mod):
    """BASELINE.json config 4 sizes on one GPU: 1024 frames x 256 hypotheses (size-independent properties)."""
    E = engine_mod
    n = 1024
    coords, pix, gt_cv, gt_jp = E.synth_frames(n)
    eng = E.Engine(max_frames=n)
    a = eng.forward(coords, pix, gt_jp)
    # determinism: a second pass is bit-identical
    b = eng.forward(coords, pix, gt_jp)
    for k in ("img_idx", "cand_idx", "hyp_pose", "scores", "sf", "avg_pose", "ref_pose", "inlier_map", "loss"):
        assert np.array_equal(getattr(a, k), getattr(b, k)), k
    # sharding invariance: frames [512, 1024) processed alone with frame0 = 512 give the same results
    c = eng.forward(coords[512:], pix[512:], gt_jp[512:], frame0=512)
    assert np.array_equal(a.img_idx[512:], c.img_idx) and np.array_equal(a.ref_pose[512:], c.ref_pose)
    # softmax properties
    assert np.abs(a.sf.sum(1) - 1).max() < 1e-12 and (a.sf >= 0).all()
    assert (a.entropy >= 0).all() and (a.entropy <= 8.0 + 1e-9).all()
    # every minimal set: 4 distinct cells in range, candidates strictly increasing within a stream
    assert a.img_idx.min() >= 0 and a.img_idx.max() < 1600
    s = np.sort(a.img_idx, axis=2)
    assert (np.diff(s, axis=2) > 0).all()
    assert (np.diff(a.cand_idx, axis=1) > 0).all()
    assert (a.n_candidates == a.cand_idx[:, -1] + 1).all()
    # scores bounded by alpha * N, inlier maps bounded by steps, accuracy on the synthetic data
    assert a.scores.min() >= 0 and a.scores.max() <= 0.1 * 1600
    assert a.inlier_map.max() <= 8 and (a.inlier_map.sum(1) <= 800).all()
    assert (a.status == 0).all()
    assert a.correct.mean() > 0.95 and np.median(a.rot_err) < 1.0 and np.median(a.t_err) < 30.0


def test_score_hook_seam(engine_mod, oracle):
    """The score seam (lua_calls.h:284-300): an external scorer sees the device diffmaps and its
    scores drive softmax / soft-argmax.  Here the hook re-implements the soft-inlier score with torch."""
    import torch
    E, O = engine_mod, oracle
    coords, pix, gt_cv, gt_jp = E.synth_frames(2)
    ref = E.Engine(max_frames=2).forward(coords, pix, gt_jp)
    eng = E.Engine(max_frames=2)
    seen = {}

    def hook(dm, n, H, sc, stream):
        seen["n"] = (n, H)
        import ctypes
        # wrap raw device pointers as torch tensors via __cuda_array_interface__
        class _W:
            def __init__(self, ptr, shape, typestr):
                self.__cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (ptr, False), "version": 2}
        with torch.cuda.stream(torch.cuda.ExternalStream(stream)):   # the engine's stream: ordered after k_score, before the soft-argmax tail
            d = torch.as_tensor(_W(dm, (n, H, 1600), "<f4"), device="cuda")
            s = torch.as_tensor(_W(sc, (n, H), "<f8"), device="cuda")
            s.copy_(0.1 * torch.sigmoid(0.5 * (10.0 - d.double())).sum(2))
        return 0

    eng.set_score_hook(hook)
    res = eng.forward(coords, pix, gt_jp)
    assert seen["n"] == (2, 256)
    assert np.abs(res.scores - ref.scores).max() <= 1e-5 * ref.scores.max()
    assert np.abs(res.avg_pose - ref.avg_pose).max() <= 1e-3
    assert np.array_equal(res.img_idx, ref.img_idx)


@pytest.mark.parametrize("random_draw,T", [(True, 1), (False, 4)])
def test_dsac_variant_forward_matches_oracle(engine_mod, oracle, random_draw, T):
    """SURVEY.md section 8(f) N1: the DSAC / RANSAC variant's forward (core/cnn.h:1028-1257) -- draw, refinement of ALL hypotheses,
    per-hypothesis losses, expected loss."""
    E, O = engine_mod, oracle
    nf, H = 2, 32
    coords, pix, gt_cv, gt_jp = E.synth_frames(nf, n_streams=T)
    eng = E.Engine(max_frames=nf, n_hyps=H, n_streams=T)
    res = eng.forward_dsac(coords, pix, gt_jp, random_draw=random_draw, want_inlier_maps=True)
    for f in range(nf):
        cfg = O.default_config(seed=1305 + f * T, n_hyps=H, n_streams=T)
        o = O.forward_dsac(cfg, coords[f], pix[f], gt_jp[f, :9], gt_jp[f, 9:], random_draw)
        assert np.array_equal(o.img_idx, res.img_idx[f])
        assert o.hyp_idx == res.hyp_idx[f]                       # same draw (same stream position, same libstdc++ calls)
        assert np.array_equal(o.steps_done, res.steps_done[f])
        assert np.array_equal(o.inlier_maps, res.inlier_maps[f])
        assert np.abs(o.ref_pose[:, :3] - res.ref_pose[f][:, :3]).max() <= 1e-8
        assert np.abs(o.ref_pose[:, 3:] - res.ref_pose[f][:, 3:]).max() <= 1e-5
        assert np.abs(o.losses - res.losses[f]).max() <= 1e-6 * max(1.0, np.abs(o.losses).max())
        assert np.abs(o.sf - res.sf[f]).max() <= 1e-4
        assert abs(o.expected_loss - res.expected_loss[f]) <= 1e-3 * max(1.0, abs(o.expected_loss))
        assert abs(o.rot_err - res.rot_err[f]) <= 1e-6 and abs(o.t_err - res.t_err[f]) <= 1e-4 and o.correct == res.correct[f]


def test_score_cnn_plugin_behind_the_seam(engine_mod, oracle):
    """SURVEY.md section 8(f) N2: the reference's Score-CNN architecture as a zero-copy plug-in behind dsac_set_score_hook."""
    import torch
    from dsac_b200.score_cnn import ScoreCNN, MEAN
    E, O = engine_mod, oracle
    coords, pix, gt_cv, gt_jp = E.synth_frames(2)
    H = 64
    cnn = ScoreCNN(seed=3)
    eng = E.Engine(max_frames=2, n_hyps=H)
    eng.set_score_hook(cnn)
    res = eng.forward(coords, pix, gt_jp, want_diffmaps=True)
    plain = E.Engine(max_frames=2, n_hyps=H).forward(coords, pix, gt_jp)
    assert np.array_equal(res.img_idx, plain.img_idx)            # sampling does not depend on the scorer
    # scores = the same network evaluated on the fetched diffmaps
    with torch.no_grad():
        x = torch.from_numpy(res.diffmaps.reshape(-1, 1, 40, 40)).cuda() - MEAN
        want = cnn.model(x).reshape(2, H).double().cpu().numpy()
    assert np.abs(res.scores - want).max() <= 1e-4 * max(1.0, np.abs(want).max())
    for f in range(2):
        assert np.abs(O.softmax(res.scores[f]) - res.sf[f]).max() <= 1e-12
        assert np.abs((res.sf[f][:, None] * res.hyp_pose[f]).sum(0) - res.avg_pose[f]).max() <= 1e-9 * 3000
    assert np.isfinite(res.ref_pose).all()


def test_submit_wait_equals_blocking_forward(engine_mod):
    """dsac_forward_submit / dsac_forward_wait (two engines in flight) give what the blocking dsac_forward gives."""
    E = engine_mod
    coords, pix, gt_cv, gt_jp = E.synth_frames(6)
    a, b = E.Engine(max_frames=3, n_hyps=32), E.Engine(max_frames=3, n_hyps=32)
    ra = a.forward_submit(coords[:3], pix[:3], gt_jp[:3], frame0=0)
    rb = b.forward_submit(coords[3:], pix[3:], gt_jp[3:], frame0=3)
    with pytest.raises(RuntimeError):
        a.forward_submit(coords[:3], pix[:3], gt_jp[:3], frame0=0)      # one pending pass per engine
    a.forward_wait(); b.forward_wait()
    a.forward_wait()                                                    # idempotent
    ref = E.Engine(max_frames=6, n_hyps=32).forward(coords, pix, gt_jp)
    for k in ("img_idx", "cand_idx", "ref_pose", "avg_pose", "sf", "loss", "n_candidates"):
        assert np.array_equal(np.concatenate([getattr(ra, k), getattr(rb, k)]), getattr(ref, k)), k


@pytest.mark.parametrize("T,H,n", [(8, 32, 40), (1, 16, 300)])
def test_tail_split_is_scheduling_only(engine_mod, T, H, n):
    """dsac_set_tail_split decides which calls may run a large batch as two lanes: every output must be bit-identical
    with the split off, on (blocking call, device-resident call) and on for submitted passes."""
    import torch
    E = engine_mod
    coords, pix, gt_cv, gt_jp = E.synth_frames(n, n_streams=T)
    keys = ("img_idx", "cand_idx", "hyp_pose", "scores", "sf", "avg_pose", "ref_pose", "inlier_map", "loss", "n_candidates", "status")
    eng = E.Engine(max_frames=n, n_streams=T, n_hyps=H)
    eng.set_tail_split(0)
    ref = eng.forward(coords, pix, gt_jp, want_diffmaps=True)
    eng.set_tail_split(1)
    got = eng.forward(coords, pix, gt_jp, want_diffmaps=True)
    for k in keys + ("diffmaps",):
        assert np.array_equal(getattr(ref, k), getattr(got, k)), k
    eng.set_tail_split(2)
    sub = eng.forward_submit(coords, pix, gt_jp)
    eng.forward_wait()
    for k in keys:
        assert np.array_equal(getattr(ref, k), getattr(sub, k)), k
    # device-resident inputs on the caller's stream
    eng.set_tail_split(1)
    d_c, d_p, d_g = torch.from_numpy(coords).cuda(), torch.from_numpy(pix).cuda(), torch.from_numpy(gt_jp).cuda()
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        eng.forward_device(n, d_c.data_ptr(), d_p.data_ptr(), 0, d_g.data_ptr(), 0, st.cuda_stream)
        dev = eng.fetch(n, stream=st.cuda_stream)
    for k in keys:
        assert np.array_equal(getattr(ref, k), getattr(dev, k)), k
    with pytest.raises(RuntimeError):
        eng.set_tail_split(7)
    eng.close()


def test_points_in_the_camera_plane_and_on_their_pixel(engine_mod, oracle):
    """k_score's unguarded error formula hands a warp to the guarded form when A z^2 leaves the normal range: z = 0
    exactly (cv::projectPoints then uses 1/z := 1) or a point exactly on its pixel.  All-outlier frame with a bounded
    sampler -> zero poses (R = I, t = 0), scene coordinates (0, 0, 0) and (x, y, 0) -> z = 0 for those cells."""
    E, O = engine_mod, oracle
    coords, pix, gt_cv, gt_jp = E.synth_frames(1, rho=0.0)
    coords = coords.copy()
    coords[0, ::3] = 0                       # projects to the principal point: error = |pixel - (cx, cy)|, < 100 near the centre
    coords[0, 1::11, 2] = 0                  # z = 0 with non-zero x, y
    eng = E.Engine(max_frames=1, max_candidates=1024, n_hyps=8)
    res = eng.forward(coords, pix, gt_jp, want_diffmaps=True)
    cfg = O.default_config(n_hyps=8, max_candidates=1024)
    fw = O.forward(cfg, coords[0], pix[0], gt_jp[0, :9], gt_jp[0, 9:])
    assert np.array_equal(fw.img_idx, res.img_idx[0])
    zero = np.flatnonzero((res.img_idx[0] < 0).all(1))
    assert len(zero) > 0, "the test needs at least one value-encoded (zero) pose"
    d = np.hypot(pix[0][::3, 0] - 320.0, pix[0][::3, 1] - 240.0)
    want = np.minimum(d, 100.0).astype(np.float32)
    for h in zero:
        assert np.abs(res.diffmaps[0][h].reshape(-1)[::3] - want).max() <= 1e-4
    assert (res.diffmaps[0][zero].reshape(len(zero), -1)[:, ::3].min(1) < 100.0).all()
    assert np.abs(fw.diffmaps - res.diffmaps[0]).max() <= 2e-3
    # scores of an all-outlier frame are tiny (~0.025): k_score rounds a sigmoid below 2^-25 up to 2^-25 (it shares one
    # reciprocal between five sigmoids), i.e. at most alpha * N * 2^-25 = 4.8e-6 absolute on a score
    assert np.abs(fw.scores - res.scores[0]).max() <= 5e-6 + 1e-5 * np.abs(fw.scores).max()
    eng.close()
