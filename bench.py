#!/usr/bin/env python
"""bench.py -- hypotheses scored / second on synthetic 640x480 scene-coordinate maps.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
    (N > 1: launched by torchrun, one rank per GPU; frames shard with no data-path collective)

A step = one pass of the hot path (sample -> HxN reprojection errors -> soft-inlier score ->
softmax / soft-argmax -> refinement -> evaluation) over one batch of frames per GPU.
Workload (config.workload): BASELINE.json config 4's batch on every GPU -- 1024 frames x 256
hypotheses x 40x40 points per GPU (weak scaling); the single-frame config 2 latency is reported
beside it under "single_frame".  Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the tree may be read-only: nothing is cached in it

import numpy as np  # noqa: E402

H = 256
NPTS = 1600
FRAMES_PER_GPU = 1024
BYTES_F = NPTS * (6 + 8) + H * (48 + 8) + 56           # fused, scores only   (BASELINE.md section 5)
BYTES_M = BYTES_F + H * NPTS * 4                       # diffmap materialised (reference behaviour)
FLOPS_PER_PAIR = 38                                    # BASELINE.md section 5
# fp64 flop model of the sampler's conservative filter (one thread per candidate; DESIGN.md section 5, counted from
# p3p_quick_core / quartic_roots_banded in pose_math.cuh with FMA = 2 flops, a Newton-refined reciprocal = 8, rsqrt = 11):
#   set-up (triangle, quadrics, quartic coefficients, Ferrari + cubic Newton, world frame) ... 388 fp64 flops
#   one root slot: Newton step on the two quadrics + positivity ............................... 91 fp64 flops
#                  4th point by congruence + pixel test (fp32 since round 2) ................. 78 fp32 flops
# ALGORITHMIC work = set-up + the REAL roots of the quartic: 96.9 % of the candidates have two, 0.7 % four, 2.4 % none
# (tools/filter_stats.py over 2 * 10^6 candidates of the benchmark frames) -> 1.97 root slots = 567 fp64 (+ 154 fp32)
# flops per candidate.  The kernel evaluates slots 0 and 1 in every lane and slots 2, 3 only in warps that hold a
# four-root candidate (one in five): ~2.4 slots = 606 executed fp64 flops per candidate.
FILTER_FLOPS_SETUP, FILTER_FLOPS_ROOT, FILTER_FP32_ROOT, FILTER_MEAN_ROOTS, FILTER_EXEC_SLOTS = 388, 91, 78, 1.97, 2.4
FP64_PEAK_TFLOPS = 148 * 64 * 2 * 1.965e9 / 1e12       # 148 SMs x 64 FMA/clk x 2 x 1.965 GHz = 37.2 (B200 non-tensor fp64)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames", type=int, default=FRAMES_PER_GPU, help="frames per GPU per step")
    ap.add_argument("--cpu-frames", type=int, default=0, help="frames in the cpu_baseline sample (0 = auto)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (rank 0's frames) as DIR/<name>.npy, float32 / float64, < 64 MB")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_BYTES = 60 << 20         # array bytes of a dump: with the .npy headers below 64 MB in either unit
DUMP_DIFFMAP_ROWS = 2048     # (frame, hypothesis) rows of the H x N diffmaps kept: 13 MB of the 1.7 GB a step writes
DUMP_SEED = 20170721


def dump_outputs(d, res):
    """The arrays dsac_fetch returns for the step, as d/<name>.npy: real arrays in their own precision, integer arrays as
    float64 (exact).  Of the diffmaps a fixed, seeded sample of rows is kept (diffmaps_rows, with their (frame, hypothesis)
    in diffmaps_rows_index); if the per-frame arrays still exceed the budget, a fixed, seeded sample of frames is kept
    (frame_index)."""
    os.makedirs(d, exist_ok=True)
    rng = np.random.default_rng(DUMP_SEED)
    nf, H = res.scores.shape
    rows = np.sort(rng.choice(nf * H, size=min(nf * H, DUMP_DIFFMAP_ROWS), replace=False))
    out = {"diffmaps_rows": res.diffmaps.reshape(nf * H, -1)[rows],
           "diffmaps_rows_index": np.stack([rows // H, rows % H], 1).astype(np.float64)}
    per_frame = {k: (a if a.dtype.kind == "f" else a.astype(np.float64)) for k, a in vars(res).items()
                 if isinstance(a, np.ndarray) and k != "diffmaps"}
    room = DUMP_BYTES - sum(a.nbytes for a in out.values())
    keep = min(nf, room // sum(a.nbytes // nf for a in per_frame.values()))
    if keep < nf:
        frames = np.sort(rng.choice(nf, size=keep, replace=False))
        per_frame = {k: a[frames] for k, a in per_frame.items()}
        out["frame_index"] = frames.astype(np.float64)
    out.update(per_frame)
    for k, a in out.items():
        np.save(os.path.join(d, k + ".npy"), np.ascontiguousarray(a))


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json, burst copy)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                       "-lms", "100"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name).read().splitlines() if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))
        return out


def cpu_threads():
    """Host threads the CPU arm uses: the affinity mask, capped by the cgroup CPU quota if there is one."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(round(int(txt[0]) / int(txt[1])))))
            else:
                q = int(txt[0])
                per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                if q > 0:
                    n = min(n, max(1, int(round(q / per))))
            break
        except Exception:
            continue
    return n


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def run_cpu_sample(n_frames, threads, frame0=0, variant="perf", stages=None):
    """The oracle (CPU restatement of the reference path) on `n_frames` frames of the SAME workload.  Inputs come from the
    host-only generator library (dsac_b200/libdsac_synth.so: no CUDA library is mapped by this leg)."""
    from dsac_b200 import synth
    from oracle import oracle as O
    coords, pix, _, _ = synth.synth_frames(n_frames, frame0=frame0)
    cfg = O.default_config(seed=1305 + frame0)
    secs = O.bench_forward(cfg, coords, pix, n_threads=threads, with_refine=True, variant=variant, stages=stages)
    return n_frames * H / secs, secs


def pick_cpu_variant():
    """-O3 -march=native build made on THIS box if a compiler is here, else the shipped -O3 -march=x86-64-v3 build."""
    from oracle import oracle as O
    for v in ("native", "perf", "parity"):
        lib, flags = O.variant_lib(v)
        if lib is not None:
            return v, flags
    raise SystemExit("no oracle library available")


def cpu_report(threads, n_frames, frame0=0):
    """CPU baseline per BASELINE.md section 3: perf build, 1 thread and all threads, per-stage split at the reference's
    print points (cnn_softam.h:1062, 1074, 1096, 1156), plus the reference's own -Ofast for information."""
    from oracle import oracle as O
    variant, flags = pick_cpu_variant()
    run_cpu_sample(min(n_frames, threads), threads, variant=variant)             # page in, spin the cores up
    st = []
    v_all, secs = run_cpu_sample(n_frames, threads, frame0=frame0, variant=variant, stages=st)
    tot = sum(st) or 1.0
    n1 = max(8, n_frames // max(1, threads))
    v_one, secs1 = run_cpu_sample(n1, 1, frame0=frame0, variant=variant)
    out = {"value": v_all, "unit": "hyp/s", "cores": threads, "kind": "port", "build": flags,
           "sample": "%d frames x %d hyp x 1600 pts of the same batch, full pipeline (sample+score+softargmax+refine), %.2f s wall" % (n_frames, H, secs),
           "one_thread": {"value": v_one, "frames": n1, "seconds": secs1},
           "stage_share": {"sampling": st[0] / tot, "scoring": st[1] / tot, "averaging": st[2] / tot, "refinement": st[3] / tot},
           "cpu": cpu_model(),
           "note": "oracle = CPU restatement of the reference path with the closed-form score, pinned to the reference's own code "
                   "(tests/test_oracle_vs_ref.py); it omits the reference's Lua/cuDNN round trip, i.e. a lower bound on the reference's CPU time"}
    lib, oflags = O.variant_lib("ofast")
    if lib is not None:
        run_cpu_sample(min(n_frames, threads), threads, variant="ofast")
        v_fast, _ = run_cpu_sample(n_frames, threads, frame0=frame0, variant="ofast")
        out["ofast"] = {"value": v_fast, "build": oflags + " (the reference's own flag, core/CMakeLists.txt:7; informational)"}
    return out


def reference_arm(args, rank):
    """--impl reference: the reference's own CPU implementation of the path.  The reference cannot be linked against its
    real dependencies here (OpenCV C++/Lua/Torch7/png++ missing; oracle/_ref compiles it against shims for PINNING only),
    so this arm times the oracle port -- built for speed -- on all host threads.  It maps no CUDA library."""
    if rank != 0:
        return
    threads = cpu_threads()
    variant, flags = pick_cpu_variant()
    per_step = max(threads * 4, 64)
    for _ in range(max(1, args.warmup)):
        run_cpu_sample(max(threads, 16), threads, variant=variant)
    t = 0.0
    for s in range(args.steps):
        _, secs = run_cpu_sample(per_step, threads, frame0=s * per_step, variant=variant)
        t += secs
    value = per_step * H * args.steps / t
    sample = "%d frames/step x %d hyp x 1600 pts (same generator, seeds and config as the GPU arm, whose step is %d frames: " \
             "throughput-normalised), %d threads, build %s" % (per_step, H, FRAMES_PER_GPU, threads, flags)
    line = {
        "impl": "reference", "metric": "hypotheses scored/sec (256 hyp x 1600 pts/img)", "value": value, "unit": "hyp/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "config4-shaped batch, CPU sample: " + sample, "n_hyps": H, "points": NPTS, "frames_per_step": per_step,
                   "stages": "sample+score+softargmax+refine+eval"},
        "cpu_baseline": {"value": value, "unit": "hyp/s", "cores": threads, "kind": "port", "sample": sample, "cpu": cpu_model(), "build": flags},
        "e2e": {"value": value, "unit": "hyp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        reference_arm(args, rank)
        return

    import torch
    import torch.distributed as dist
    import dsac_b200.engine as E
    from dsac_b200.sharding import shard_range

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU path (use --impl reference for the CPU arm)")
    E.load(build_if_missing=False)      # the library as built; the benchmark never compiles into the tree
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # NCCL's debug lines must not mix with the ONE JSON line on stdout
        # ... and its "NCCL version" banner is printed to stdout regardless (seen on the 2-GPU box): file descriptor 1 points
        # at stderr while the communicator is set up (init + the first collective)
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    nf = args.frames
    n_total = nf * world
    lo, hi = shard_range(n_total, rank, world)          # weak scaling: every rank owns `nf` frames
    frame0 = lo
    coords, pix, gt_cv, gt_jp = E.synth_frames(nf, frame0=frame0)
    eng = E.Engine(max_frames=nf, device=local_rank)
    stream = torch.cuda.current_stream().cuda_stream

    # inputs resident in HBM for `value`
    d_coords = torch.from_numpy(coords).cuda()
    d_pix = torch.from_numpy(pix).cuda()
    d_gt = torch.from_numpy(gt_jp).cuda()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")   # 2x the 126 MB L2

    def step_device():
        eng.forward_device(nf, d_coords.data_ptr(), d_pix.data_ptr(), 0, d_gt.data_ptr(), frame0, stream)

    def timed_steps(fn, k):
        """k steps, each bracketed by its own CUDA events on the launching stream, L2 flushed between."""
        tot = 0.0
        for _ in range(k):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            tot += e0.elapsed_time(e1)
        return tot

    eng.set_stages(E.STAGE_ALL)
    for _ in range(max(args.warmup, 3)):
        step_device()
    barrier()
    clocks = ClockSampler(local_rank) if rank == 0 else None
    launches0 = eng.launches
    ms_total = timed_steps(step_device, args.steps)
    gpu_launches = eng.launches - launches0
    barrier()
    t = torch.tensor([ms_total], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    value = n_total * H * args.steps / (ms_total * 1e-3)

    # quality of the result (pose error vs the generating pose)
    dump = bool(args.dump_outputs) and rank == 0
    res = eng.fetch(nf, want_diffmaps=dump)
    if dump:
        dump_outputs(args.dump_outputs, res)
        res.diffmaps = None
    quality = {"accuracy_5cm5deg": float(res.correct.mean()), "median_rot_deg": float(np.median(res.rot_err)),
               "median_t_mm": float(np.median(res.t_err)), "candidates_per_frame": float(res.n_candidates.mean()),
               "frames_with_status": int((res.status != 0).sum())}

    # ---- e2e: HOST (pinned) buffers through dsac_forward, H2D + kernels + D2H every step
    def pinned(a):
        t_ = torch.from_numpy(a).pin_memory()
        return t_, t_.numpy()
    k1, h_coords = pinned(coords); k2, h_pix = pinned(pix); k3, h_gt = pinned(gt_jp)
    h2d = h_coords.nbytes + h_pix.nbytes + h_gt.nbytes
    keep = []

    def host_result():
        out = E.ForwardResult(nf, H, False)
        nbytes = 0
        for name in ("ref_pose", "avg_pose", "sf", "scores", "entropy", "loss", "rot_err", "t_err", "correct", "status", "n_candidates"):
            tt, arr = pinned(getattr(out, name))
            keep.append(tt)
            setattr(out, name, arr)
            setattr(out.raw, name, arr.ctypes.data)
            nbytes += arr.nbytes
        for name in ("hyp_pose", "img_idx", "cand_idx", "diffmaps", "inlier_map", "ref_steps_done", "n_perm_steps"):
            setattr(out.raw, name, None)
        return out, nbytes

    # (a) one synchronous dsac_forward per step: H2D, kernels and D2H strictly one after the other
    out, d2h = host_result()

    def step_host():
        eng.forward(h_coords, h_pix, h_gt, frame0=frame0, out=out)

    for _ in range(max(args.warmup, 3)):
        step_host()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_host()
    torch.cuda.synchronize()
    sync_s = time.perf_counter() - t0
    # (b) the driver loop with DEPTH engines in flight (dsac_forward_submit / dsac_forward_wait): every step still copies its
    # inputs from pinned host memory and reads its results back, but the copies of one step overlap the kernels of the others
    # (measured, tools/e2e_depth_probe.py: 1 / 2 / 3 / 4 engines in flight 4.21 / 2.74 / 2.60 / 2.59 ms per step)
    DEPTH = 3
    engs = [eng] + [E.Engine(max_frames=nf, device=local_rank) for _ in range(DEPTH - 1)]
    outs = [out] + [host_result()[0] for _ in range(DEPTH - 1)]

    def run_pipelined(steps):
        for i in range(steps):
            engs[i % DEPTH].forward_wait()
            engs[i % DEPTH].forward_submit(h_coords, h_pix, h_gt, frame0=frame0, out=outs[i % DEPTH])
        for e_ in engs:
            e_.forward_wait()

    run_pipelined(max(args.warmup, 3) + DEPTH)
    barrier()
    t0 = time.perf_counter()
    run_pipelined(args.steps)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    barrier()
    for o_ in outs[1:]:
        assert np.array_equal(outs[0].correct, o_.correct) and np.array_equal(outs[0].ref_pose, o_.ref_pose)
    # (c) for information: the same DEPTH engines on DEVICE-resident inputs, consecutive steps in flight on DEPTH streams (no
    # host copies, no L2 flush: every step streams 1.7 GB of diffmaps, far more than the 126 MB L2) -- the steady-state
    # throughput of the kernels alone, between the step-isolated `value` and `e2e`
    pstreams = [torch.cuda.Stream(device=local_rank) for _ in range(DEPTH)]

    def run_device_pipelined(steps):
        for i in range(steps):
            engs[i % DEPTH].forward_device(nf, d_coords.data_ptr(), d_pix.data_ptr(), 0, d_gt.data_ptr(), frame0, pstreams[i % DEPTH].cuda_stream)

    run_device_pipelined(2 * DEPTH)
    barrier()
    pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    pe0.record()
    for st_ in pstreams:
        st_.wait_event(pe0)
    run_device_pipelined(args.steps)
    for st_ in pstreams:
        torch.cuda.current_stream().wait_stream(st_)
    pe1.record()
    pe1.synchronize()
    dev_pipe_ms = pe0.elapsed_time(pe1) / args.steps
    barrier()
    for e_ in engs[1:]:
        e_.close()
    t = torch.tensor([e2e_s, sync_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = n_total * H * args.steps / float(t[0].item())
    e2e_sync_value = n_total * H * args.steps / float(t[1].item())
    clk = clocks.stop() if clocks else None

    # ---- per-stage durations (stage-isolated launches, CUDA events), the sampler's per-kernel split and the rooflines
    stage_ms = {}
    reps_s = max(3, min(args.steps, 10))
    for name, mask in (("sampler", E.STAGE_SAMPLE), ("k_score", E.STAGE_SCORE), ("k_refine", E.STAGE_REFINE | E.STAGE_EVAL)):
        eng.set_stages(E.STAGE_ALL)
        step_device()
        eng.set_stages(mask)
        step_device()
        torch.cuda.synchronize()
        stage_ms[name] = timed_steps(step_device, reps_s) / reps_s
    # the sampler's kernels, from CUDA events the engine records between its launches (dsac_sampler_profile)
    eng.set_stages(E.STAGE_SAMPLE)
    eng.sampler_profile(True)
    k1_ms, k1_cnt = [0.0] * 4, [0] * 4
    for _ in range(reps_s):
        flush.zero_()
        step_device()
        ms_k, cnt_k = eng.sampler_profile_read()
        k1_ms = [a + b / reps_s for a, b in zip(k1_ms, ms_k)]
        k1_cnt = cnt_k
    eng.sampler_profile(False)
    eng.set_stages(E.STAGE_ALL)
    peak, peak_src = peaks()
    k2_s = stage_ms["k_score"] * 1e-3
    achieved = BYTES_M * nf / k2_s / 1e9
    traffic = None
    tp = os.path.join(ROOT, "profiles", "k_score_traffic.json")
    if os.path.exists(tp):
        try:
            traffic = json.load(open(tp)).get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    filt_traffic = None
    try:
        filt_traffic = json.load(open(os.path.join(ROOT, "profiles", "k1_filter_traffic.json"))).get("dram_bytes_per_launch")
    except Exception:
        filt_traffic = None
    ssum = sum(stage_ms.values())
    kernels_ms = {"k1_cells+k1_slot (MT19937 streams, candidate boundaries, ordered selection)": k1_ms[0],
                  "k1_filter (conservative fp64 P3P filter, 1 thread per candidate)": k1_ms[1],
                  "k1_solve (full fp64 P3P + reprojection check on the flagged)": k1_ms[2],
                  "k_sample resume tail (streams the rounds left unfinished; normally empty)": k1_ms[3],
                  "k_score": stage_ms["k_score"], "k_refine": stage_ms["k_refine"]}
    # dominant kernel: the sampler's filter.  Point-wise fp64 arithmetic on shared-memory-resident data: neither HBM nor
    # tensor cores bound it, the fp64 pipe does -- reported against the chip's non-tensor fp64 peak.
    filt_s = max(k1_ms[1], 1e-9) * 1e-3
    flops_alg = (FILTER_FLOPS_SETUP + FILTER_MEAN_ROOTS * FILTER_FLOPS_ROOT) * k1_cnt[0]
    flops_exec = (FILTER_FLOPS_SETUP + FILTER_EXEC_SLOTS * FILTER_FLOPS_ROOT) * k1_cnt[0]
    roofline = {"kernel": "k1_filter (dominant: %.0f %% of the stage-isolated step) -- conservative fp64 P3P filter over every sampled minimal set" % (100 * k1_ms[1] / ssum),
                "bound": "fp64",
                "bound_note": "fp64 pipe, not hbm / tensor: point-wise fp64 arithmetic on data staged in shared memory (DRAM throughput 4 % of peak under ncu); see roofline_hbm for the HBM-bound kernel of the path",
                "achieved": flops_alg / filt_s / 1e12, "peak": FP64_PEAK_TFLOPS, "unit": "TFLOP/s", "frac": flops_alg / filt_s / 1e12 / FP64_PEAK_TFLOPS,
                "traffic": filt_traffic, "traffic_note": "DRAM bytes of ONE k1_filter launch (launch set 0: 4 194 304 candidates) from the committed ncu --set full capture, profiles/k1_filter_traffic.json",
                "peak_source": "148 SMs x 64 fp64 FMA/clk x 2 x 1.965 GHz (no measured fp64 peak in MEASURED_PEAKS.json)",
                "algorithmic_flops_per_candidate": FILTER_FLOPS_SETUP + FILTER_MEAN_ROOTS * FILTER_FLOPS_ROOT,
                "fp32_flops_per_candidate_beside": FILTER_MEAN_ROOTS * FILTER_FP32_ROOT,
                "executed_flops_per_candidate": FILTER_FLOPS_SETUP + FILTER_EXEC_SLOTS * FILTER_FLOPS_ROOT, "executed_frac": flops_exec / filt_s / 1e12 / FP64_PEAK_TFLOPS,
                "candidates_per_launch_set": k1_cnt[0], "ms_per_step": k1_ms[1], "share_of_step": k1_ms[1] / ssum}
    roofline_hbm = {"kernel": "k_score<write_diffmaps=1> (HxN reprojection-error matrix + soft-inlier score + soft-argmax tail)",
                    "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": traffic, "peak_source": peak_src, "algorithmic_bytes_per_launch": BYTES_M * nf,
                    "ms_per_launch": stage_ms["k_score"], "share_of_step": stage_ms["k_score"] / ssum,
                    "fp32_gflops": FLOPS_PER_PAIR * H * NPTS * nf / k2_s / 1e9,
                    "step_level": {"achieved": BYTES_M * nf / (ms_total / args.steps * 1e-3) / 1e9, "frac": BYTES_M * nf / (ms_total / args.steps * 1e-3) / 1e9 / peak,
                                   "note": "algorithmic bytes of the whole step (mode M) over the whole step's time"}}

    # ---- BASELINE config 4 verbatim (strong scaling): the SAME 1024 frames split over the ranks, 1024 / N per GPU
    strong = None
    nf_s = FRAMES_PER_GPU // world
    if world > 1 and nf_s >= 1:
        lo_s = rank * nf_s

        def step_strong():
            eng.forward_device(nf_s, d_coords.data_ptr(), d_pix.data_ptr(), 0, d_gt.data_ptr(), lo_s, stream)
        for _ in range(3):
            step_strong()
        barrier()
        ms_s = timed_steps(step_strong, args.steps)
        barrier()
        ts = torch.tensor([ms_s], dtype=torch.float64, device="cuda")
        dist.all_reduce(ts, op=dist.ReduceOp.MAX)
        ms_s = float(ts.item())
        strong = {"workload": "BASELINE config 4 as written: %d frames in total, %d per GPU" % (nf_s * world, nf_s), "frames_total": nf_s * world,
                  "frames_per_gpu": nf_s, "ms_per_step": ms_s / args.steps, "value": nf_s * world * H * args.steps / (ms_s * 1e-3), "unit": "hyp/s",
                  "note": "strong scaling: per-GPU work shrinks with N, so launch latency and the sampler's round structure (a fixed "
                          "number of dependent kernel launches per pass) weigh more than in the weak-scaling `value`"}
    elif world == 1:
        strong = {"workload": "BASELINE config 4 as written: 1024 frames on one GPU (identical to `value`)", "frames_total": nf, "frames_per_gpu": nf,
                  "ms_per_step": ms_total / args.steps, "value": value, "unit": "hyp/s"}

    # ---- config 2: single frame latency (1 frame, 256 hyp, forward scoring + soft-argmax)
    single = None
    config1 = None
    if rank == 0:
        def frame_latency(H1, T, stages, reps=1000, warm=100):
            """One frame per call; every call bracketed by its own pair of CUDA events on the launching stream; median."""
            d1 = E.synth_frames(1, frame0=frame0, n_streams=T)
            c1 = torch.from_numpy(d1[0]).cuda(); p1 = torch.from_numpy(d1[1]).cuda(); g1 = torch.from_numpy(d1[3]).cuda()
            eng1 = E.Engine(max_frames=1, device=local_rank, n_streams=T, n_hyps=H1)
            eng1.set_stages(stages)
            for _ in range(warm):
                eng1.forward_device(1, c1.data_ptr(), p1.data_ptr(), 0, g1.data_ptr(), frame0, stream)
            torch.cuda.synchronize()
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
            for a, b in ev:
                a.record()
                eng1.forward_device(1, c1.data_ptr(), p1.data_ptr(), 0, g1.data_ptr(), frame0, stream)
                b.record()
            torch.cuda.synchronize()
            us = sorted(a.elapsed_time(b) * 1e3 for a, b in ev)
            eng1.close()
            return us[len(us) // 2], us[len(us) // 10], us[(9 * len(us)) // 10]

        single = {"workload": "config 2: 1 frame x 256 hyp x 1600 pts, sample+score+soft-argmax (a CUDA-event pair per call, median of 1000 after 100 warm-ups)"}
        # n_streams is part of the sampler contract (= OpenMP threads of the reference loop): 1 reproduces
        # OMP_NUM_THREADS=1, 8 an 8-thread run; more streams = more CTAs sampling the one frame in parallel
        for T in (1, 8):
            med, p10, p90 = frame_latency(H, T, E.STAGE_SAMPLE | E.STAGE_SCORE)
            single["streams_%d" % T] = {"latency_us": med, "p10_us": p10, "p90_us": p90, "hyp_per_s": H / (med * 1e-6)}
        single["bound"] = "latency: one stream's first round is generated window by window on many SMs (k1_spec: twist-ahead, four alignments per window, stitched afterwards); what remains serial is the MT19937 twist chain to the last window, then stitch, filter, solve (DESIGN.md section 5)"
        # config 1: the reference's own CPU-runnable case (1 frame, 64 hypotheses, full test pipeline)
        med1, p10_1, p90_1 = frame_latency(64, 1, E.STAGE_ALL)
        config1 = {"workload": "config 1: 1 frame x 64 hyp x 1600 pts, full test pipeline (sample+score+softargmax+refine+eval)",
                   "gpu_latency_us": med1, "gpu_hyp_per_s": 64 / (med1 * 1e-6)}
        if world == 1:
            try:
                from dsac_b200 import synth
                from oracle import oracle as O
                variant, flags = pick_cpu_variant()
                cs, ps, _, _ = synth.synth_frames(16, frame0=frame0)
                cfg1 = O.default_config(seed=1305 + frame0, n_hyps=64)
                O.bench_forward(cfg1, cs[:2], ps[:2], n_threads=1, with_refine=True, variant=variant)
                secs = O.bench_forward(cfg1, cs, ps, n_threads=1, with_refine=True, variant=variant)
                config1["cpu_ms_per_frame_1thread"] = secs * 1e3 / 16
                config1["cpu_hyp_per_s_1thread"] = 16 * 64 / secs
                config1["cpu_build"] = flags
            except Exception as ex:   # the CPU leg is informational
                config1["cpu_error"] = str(ex)[:200]

    # ---- config 3: 256 hyp, 8 refinement iterations + soft-argmax backward (one training round per frame)
    train = None
    if rank == 0:
        nb3 = 64
        eng3 = E.Engine(max_frames=nb3, device=local_rank)
        eng3.forward(coords[:nb3], pix[:nb3], gt_jp[:nb3])
        eng3.backward(coords[:nb3], pix[:nb3], gt_jp[:nb3], full=False)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        reps3 = 3
        for _ in range(reps3):
            eng3.forward(coords[:nb3], pix[:nb3], gt_jp[:nb3])
            eng3.backward(coords[:nb3], pix[:nb3], gt_jp[:nb3], full=False)
        torch.cuda.synchronize()
        ms_round = (time.perf_counter() - t0) * 1e3 / (reps3 * nb3)
        train = {"workload": "config 3: forward + backward (train_ransac_softam round), %d frames per call, host buffers" % nb3,
                 "gpu_ms_per_round": ms_round, "rounds_per_s": 1e3 / ms_round}
        if world == 1:
            from oracle import oracle as O
            cfg3 = O.default_config(seed=1305 + frame0)
            t0 = time.perf_counter()
            ofw = O.forward(cfg3, coords[0], pix[0], gt_jp[0, :9], gt_jp[0, 9:])
            O.backward(cfg3, coords[0], pix[0], gt_jp[0, :9], gt_jp[0, 9:], ofw)
            train["cpu_ms_per_round_1thread"] = (time.perf_counter() - t0) * 1e3
        eng3.close()
        # the DSAC / RANSAC variant's round (SURVEY.md 8f N1): refine all 256 hypotheses, expected loss, dRefine of every
        # hypothesis with sf > 1e-4 (~45 hypotheses x ~40 finite-differenced refinements each) + dSMScore
        nb5 = 16
        eng5 = E.Engine(max_frames=nb5, device=local_rank)
        eng5.forward_dsac(coords[:nb5], pix[:nb5], gt_jp[:nb5], random_draw=True)
        bwd = eng5.backward_dsac(nb5)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps3):
            eng5.forward_dsac(coords[:nb5], pix[:nb5], gt_jp[:nb5], random_draw=True)
            eng5.backward_dsac(nb5)
        torch.cuda.synchronize()
        ms5 = (time.perf_counter() - t0) * 1e3 / (reps3 * nb5)
        train["dsac_variant"] = {"workload": "train_ransac round (forward_dsac + backward_dsac), %d frames per call, host buffers" % nb5,
                                 "gpu_ms_per_round": ms5, "rounds_per_s": 1e3 / ms5,
                                 "refine_jobs_per_round": float(bwd.n_refine_jobs.mean()), "selected_hyps_per_round": float(bwd.n_selected.mean())}
        if world == 1:
            t0 = time.perf_counter()
            ofw = O.forward_dsac(cfg3, coords[0], pix[0], gt_jp[0, :9], gt_jp[0, 9:], True)
            O.backward_dsac(cfg3, coords[0], pix[0], gt_jp[0, :9], gt_jp[0, 9:], ofw)
            train["dsac_variant"]["cpu_ms_per_round_1thread"] = (time.perf_counter() - t0) * 1e3
        eng5.close()

    # ---- upstream step (SURVEY.md 8f N3): BGR frame -> normalised CNN patches, a pure streaming kernel
    upstream = None
    if rank == 0:
        nbu = 64
        rng = np.random.default_rng(7)
        fr = torch.from_numpy(rng.integers(0, 256, size=(nbu, 480, 640, 3), dtype=np.uint8)).cuda()
        pxu = torch.from_numpy(pix[:nbu]).cuda()
        patches = torch.empty((nbu, E.N, 3, 42, 42), dtype=torch.float32, device="cuda")
        engu = E.Engine(max_frames=1, n_hyps=8, device=local_rank)

        def gather():
            engu.gather_patches_device(nbu, fr.data_ptr(), 640, 480, pxu.data_ptr(), 0, patches.data_ptr(), stream=stream)
        for _ in range(3):
            gather()
        torch.cuda.synchronize()
        reps_u = 10
        tot = 0.0
        for _ in range(reps_u):
            flush.zero_()
            a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a_.record(); gather(); b_.record(); b_.synchronize()
            tot += a_.elapsed_time(b_)
        ms_u = tot / reps_u
        bytes_u = nbu * (E.N * 3 * 42 * 42 * 4 + 480 * 640 * 3 + E.N * 8)
        peak_u, _src = peaks()
        upstream = {"kernel": "k_gather_patches (getCoordImg patch assembly + normalisation, %d frames x 1600 patches of 3x42x42 f32)" % nbu,
                    "ms_per_launch": ms_u, "algorithmic_bytes_per_launch": bytes_u, "achieved_gbs": bytes_u / (ms_u * 1e-3) / 1e9,
                    "peak_gbs": peak_u, "frac": bytes_u / (ms_u * 1e-3) / 1e9 / peak_u, "patches_per_s": nbu * E.N / (ms_u * 1e-3)}
        engu.close()
        del patches, fr

    # ---- BASELINE config 5: the 1000-frame 7Scenes-shaped sequence through the C++ test driver (its own engines, one host
    #      thread per GPU; the other ranks idle meanwhile)
    sequence = None
    barrier()
    if rank == 0:
        try:
            with tempfile.TemporaryDirectory() as d:
                cmd = [os.path.join(ROOT, "apps", "test_ransac_softam"), "-frames", "1000", "-batch", "250", "-gpus", str(world)]
                subprocess.run(cmd, cwd=d, capture_output=True, text=True, timeout=300)   # first run: engine creation, page-in
                o = subprocess.run(cmd, cwd=d, capture_output=True, text=True, timeout=300)
                summ = [float(x) for x in open(os.path.join(d, "ransac_test_loss_obj_model_init.net_rdraw1_softam.txt")).read().split()]
                tail = o.stdout.strip().splitlines()[-1]
                fps = float(tail.split(" s: ")[1].split(" frames/s")[0])
                sequence = {"workload": "config 5: 1000-frame synthetic chess-shaped trajectory, apps/test_ransac_softam -gpus %d (host buffers, "
                                        "log files written), scores only (no diffmap materialisation)" % world,
                            "frames_per_s": fps, "hyp_per_s": fps * H, "accuracy_5cm5deg": summ[0], "median_rot_deg": summ[5], "median_t_mm": summ[6]}
        except Exception as ex:   # the driver is an extra: never lose the bench line over it
            sequence = {"error": str(ex)[:200]}
    barrier()

    # ---- CPU baseline (rank 0, N = 1 only): bounded sample of the same workload on the host cores
    cpu = None
    if rank == 0 and world == 1:
        threads = cpu_threads()
        cpu = cpu_report(threads, args.cpu_frames or max(256, 4 * threads), frame0=frame0)

    if rank == 0:
        line = {
            "metric": "hypotheses scored/sec (256 hyp x 1600 pts/img)", "value": value, "unit": "hyp/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64 (P3P, softmax, LM) + f32 (HxN matrix, scores)",
            "data": "synthetic",
            "config": {"workload": "BASELINE config 4 batch per GPU: %d frames x %d hyp x 40x40 pts (640x480, f=525), full test pipeline "
                                   "sample+score+softargmax+refine+eval, diffmaps materialised" % (nf, H),
                       "frames_per_gpu": nf, "n_hyps": H, "points": NPTS, "streams_per_frame": 1, "inlier_ratio": 0.5,
                       "noise_mm": 25.0, "data_seed": 20170721, "sampler_seed": 1305, "alpha": 0.1, "beta": 0.5,
                       "parallelism": "frames sharded over %d GPU(s), no collective" % world,
                       "sampler": "round-based pipeline of flat kernels (sampler_split.cuh), %d launches per pass" % (gpu_launches // max(1, args.steps)),
                       "l2": "256 MB buffer written between timed steps (flush); each step also streams %.2f GB of diffmaps" % (BYTES_M * nf / 1e9),
                       "schedule": "one step = one dsac_forward_device call; inside it a batch of >= 768 frames runs as two concurrent half-batches (lanes: own queues, counters, side streams; bit-identical results), DESIGN.md section 9"},
            "e2e": {"value": e2e_value, "unit": "hyp/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": 1e3 * float(t[0].item()) / args.steps,
                    "api": "dsac_forward_submit / dsac_forward_wait, three engines in flight on the GPU (the driver's frame loop): every step "
                           "copies its inputs from pinned host buffers (H2D) and reads poses/scores/errors back (D2H); the copies of one "
                           "step overlap the kernels of the other",
                    "pipeline_depth": 3,
                    "device_resident_pipelined": {"ms_per_step": dev_pipe_ms, "value": nf * H / (dev_pipe_ms * 1e-3) * world, "unit": "hyp/s",
                                                  "note": "for information: the same three engines on device-resident inputs, consecutive steps in flight on three streams (no host copies); rank 0's time"},
                    "note": "can exceed `value`: consecutive steps overlap on the GPU (the last, partial wave of one step's sampler is "
                            "filled by the other engine's kernels), which the per-step-isolated, L2-flushed `value` measurement forbids",
                    "sync_call": {"value": e2e_sync_value, "ms_per_step": 1e3 * float(t[1].item()) / args.steps,
                                  "api": "one blocking dsac_forward per step (H2D, kernels, D2H strictly serial)"}},
            "gpu_launches": gpu_launches,
            "roofline": roofline,
            "roofline_hbm": roofline_hbm,
            "stages_ms": stage_ms,
            "kernels_ms": kernels_ms,
            "sampler": {"ms_per_step": stage_ms["sampler"], "share_of_step": stage_ms["sampler"] / ssum,
                        "candidates_per_s": k1_cnt[0] / (stage_ms["sampler"] * 1e-3),
                        "candidates_per_accepted_hypothesis": quality["candidates_per_frame"] / H,
                        "generated_over_consumed": k1_cnt[0] / max(1.0, quality["candidates_per_frame"] * nf),
                        "flagged_by_filter": k1_cnt[1], "accepted": k1_cnt[2], "rounds_with_work": k1_cnt[3]},
            "strong_scaling": strong,
            "sequence": sequence,
            "cpu_baseline": cpu,
            "single_frame": single,
            "config1": config1,
            "train_round": train,
            "upstream": upstream,
            "quality": quality,
            "clocks": clk,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
