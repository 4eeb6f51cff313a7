// engine.cu -- C ABI of the B200 hypothesis engine (include/dsac_b200.h): device memory,
// launches and host<->device copies.  No CPU fallback: every compute entry point needs a
// CUDA device and fails loudly otherwise.
#include <cuda_runtime.h>

#include <chrono>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <random>
#include <string>
#include <vector>

#include "../../include/dsac_b200.h"
#include "backward.cuh"
#include "device_block.h"
#include "kernels.cuh"
#include "refine.cuh"
#include "sampler_split.cuh"
#include "upstream.cuh"

using namespace dsac;

static std::string g_create_error;

// One lane of the split sampler (sampler_split.cuh): the streams, events, queue counters and acceptance statistics of one
// pass.  Lane 0 runs its generator on the caller's stream; lane 1, the second half of a large batch (forward_split), on `main`.
struct K1Lane {
    cudaStream_t main = nullptr;                  // lane 1 only
    cudaStream_t side = nullptr;                  // k1_filter (and k1_solve), next to the generator on the lane's stream
    cudaStream_t side2 = nullptr;                 // k1_solve, when it runs next to the following set's filter
    cudaEvent_t ev_filt[K1S_MAX_SETS] = {};       // filter of launch set i done
    cudaEvent_t ev_solve[K1S_MAX_SETS] = {};      // solve of launch set i done
    cudaEvent_t ev_gen[K1S_MAX_SETS] = {};        // generation of launch set i done
    cudaEvent_t ev_round = nullptr;               // last solve of a round done
    int* counters = nullptr;                      // wq_n[K1S_MAX_SETS], fq_n[K1S_MAX_SETS]
    unsigned long long* stats = nullptr;          // [2][2]: candidates / hypotheses of finished streams, by call parity
    unsigned long long calls = 0;
};

struct dsac_engine {
    dsac_config cfg;
    std::string err;
    int64_t launches = 0;
    uint32_t stages = DSAC_STAGE_ALL;
    dsac_score_hook hook = nullptr;
    void* hook_user = nullptr;
    dsac_score_backward_hook bw_hook = nullptr;
    void* bw_hook_user = nullptr;
    cudaEvent_t ev_fwd = nullptr;   // recorded after the last forward launch: the backward waits on it
    int sm_count = 148;
    // device memory for the engine's lifetime (dev_alloc): freed by dsac_engine_destroy
    std::vector<void*> owned;
    // grow-only device memory, (re)allocated on use
    DeviceBlock ext_g;              // [n][H][N] dScore/dDiffMap from the backward hook, then [n][H] clamped output gradients
    DeviceBlock kabsch;             // dsac_kabsch: inputs and outputs in one block
    BackwardScratch bw;             // dsac_backward (bw.block)
    DeviceBlock ra;                 // refine-all (DSAC variant): d_ra_* below are carved from it for ra_jobs jobs
    DeviceBlock ra_imap;            // refine-all inlier maps
    std::vector<DeviceBlock> bw_pool;   // device buffers of dsac_backward_dsac, kept across calls
    // inputs (device copies for the host-buffer entry point)
    int16_t* d_coords = nullptr;
    int32_t* d_pix = nullptr;
    double* d_gt = nullptr;
    // last-call input views (device), used by fetch / backward
    const int16_t* cur_coords = nullptr;
    const int32_t* cur_pix = nullptr;
    int cur_pix_shared = 0;
    const double* cur_gt = nullptr;
    int cur_n = 0;
    int dsac_n = 0;                 // frames of the last dsac_forward_dsac (0: none), for dsac_backward_dsac
    long long cur_frame0 = 0;
    // state
    uint16_t* d_perm = nullptr;
    double* d_hyp_pose = nullptr;
    float* d_hyp_P = nullptr;
    int32_t* d_img_idx = nullptr;
    int32_t* d_cand_idx = nullptr;
    long long* d_stream_ncand = nullptr;
    unsigned long long* d_stream_endpos = nullptr;
    int32_t* d_ra_frame = nullptr; double* d_ra_pose = nullptr; double* d_ra_loss = nullptr; double* d_ra_rot = nullptr;
    double* d_ra_t = nullptr; int32_t* d_ra_correct = nullptr; int32_t* d_ra_steps = nullptr;
    size_t ra_jobs = 0;
    uint32_t* d_status = nullptr;
    unsigned long long* d_fragile = nullptr;
    unsigned long long* d_phase = nullptr;   // K1 per-phase cycle counters (DSAC_K1_TIMERS=1), else null
    float* d_diffmaps = nullptr;
    double* d_scores = nullptr;
    double* d_sf = nullptr;
    double* d_entropy = nullptr;
    double* d_avg = nullptr;
    double* d_ref = nullptr;
    int32_t* d_inlier_map = nullptr;
    int32_t* d_steps_done = nullptr;
    int32_t* d_n_perm = nullptr;
    double* d_loss = nullptr;
    double* d_rot_err = nullptr;
    double* d_t_err = nullptr;
    int32_t* d_correct = nullptr;
    unsigned int* d_frame_counter = nullptr;
    long long* h_stream_ncand = nullptr;   // [max_frames][n_streams], pinned (so that a submitted pass stays asynchronous)
    dsac_forward_out* pending_out = nullptr;   // results of a submitted, not yet awaited pass
    int pending_n = 0;
    bool pending = false;
    cudaStream_t stream = nullptr;          // the engine's stream: host-buffer passes and the backward passes
    cudaStream_t kabsch_stream = nullptr;   // dsac_kabsch
    // two lanes (forward_split): fork / join of lane 1 with the caller's stream
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    int tail_split = 1;             // dsac_set_tail_split
    // split sampler (sampler_split.cuh): per-stream state and round buffers, sized at creation
    int k1_cap = 0;
    int k1_filter_grid = 0, k1_solve_grid = 0;
    K1Lane lane[2];
    K1SlotState* d_k1_state = nullptr;
    CellRec* d_k1_celltab = nullptr;
    uint2* d_k1_cells = nullptr;
    uint32_t* d_k1_endw = nullptr;
    uint32_t* d_k1_accbits = nullptr;
    double* d_k1_pose = nullptr;
    uint2* d_k1_wq = nullptr;
    uint32_t* d_k1_fq = nullptr;
    unsigned long long* d_k1_dbg = nullptr;       // [K1S_MAX_ROUNDS][4] (DSAC_K1_DEBUG=1 or dsac_sampler_profile), else null
    // dsac_sampler_profile: CUDA events between the sampler's launches of the last forward pass
    int k1_profile = 0;
    std::vector<cudaEvent_t> k1_ev;               // event i is recorded after launch i (event 0 before the first)
    std::vector<int> k1_ev_kind;                  // 0 cells/slot (integer generation + selection), 1 filter, 2 solve, 3 resume tail
    int k1_ev_n = 0;
    K1SlotState* d_k1_vstate = nullptr;           // k1_spec: virtual slots of the speculative first round (few streams)
    uint2* d_k1_vcells = nullptr;
    uint32_t* d_k1_vendw = nullptr;
    int* d_k1_spec_result = nullptr;
    int* d_k1_spec_table = nullptr;
    uint32_t* d_k1_chain = nullptr;               // k1_pipe: hand-over records of the window chain, [slots][K1Q_MAX_WIN + 1][4]
    unsigned long long k1_epoch = 0;              // k1_pipe: one value per launch, engine-wide (a stale hand-over record never matches)
    int k1_pipe = 0;                              // DSAC_K1_PIPE=1: chained generator for 9 .. ~190 streams (experimental, off by default)
    int k1_slot_capacity = 0;                     // CTAs of k1_pipe / k1_slot (256 threads) the GPU holds at once
    int k1_spec_slots = 0;                        // streams the scratch above was sized for (0: speculative round off)
    int k1_slot_threads = 0;                      // DSAC_K1_SLOT_THREADS: 256 / 512 / 1024 (0: by the number of streams)
    int k1_wq_stride = 0;
};

// Rounds of the split sampler per pass: rounds 0..2 finish every stream of the benchmark batches; a straggler continues in
// k_sample (resume).  5 rounds = 6 empty launches per pass (measured +0.02 ms).
constexpr int K1_ROUNDS = 3;

// Engine-lifetime device memory: recorded in e->owned and freed by dsac_engine_destroy.
template <typename T>
static cudaError_t dev_alloc(dsac_engine* e, T** p, size_t bytes) {
    const cudaError_t st = cudaMalloc(p, bytes);
    if (st != cudaSuccess) {
        *p = nullptr;
        return st;
    }
    e->owned.push_back(*p);
    return cudaSuccess;
}

static int fail(dsac_engine* e, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (e) e->err = buf;
    else g_create_error = buf;
    return code;
}

#define CU(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t _st = (call);                                                                        \
        if (_st != cudaSuccess)                                                                          \
            return fail(e, DSAC_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_st), __FILE__, __LINE__); \
    } while (0)

extern "C" {

const char* dsac_version(void) { return "dsac_b200 0.1 (sm_100a)"; }

int dsac_default_config(dsac_config* c) {
    if (!c) return DSAC_ERR_ARG;
    memset(c, 0, sizeof(*c));
    c->focal = 525.0;                  // properties.cpp:55
    c->cx = 320.0; c->cy = 240.0;      // properties.cpp:310-311 (iw 640, ih 480, xs = ys = 0)
    c->n_hyps = 256;                   // properties.cpp:45
    c->thr2d = 10;                     // properties.cpp:50, int-truncated at test_ransac_softam.cpp:51
    c->inlier_count = 100;             // properties.cpp:47
    c->ref_steps = 8;                  // properties.cpp:46
    c->sub_sample = 0.01;              // properties.cpp:48
    c->alpha = 0.1; c->beta = 0.5;     // engine defaults (BASELINE.md section 2); not reference values
    c->seed = 1305;                    // thread_rand.h:100
    c->n_streams = 1;
    c->stream_skip = 6400;
    c->max_candidates = 1 << 20;
    c->fix_q4 = 0;
    c->grad_clamp = 0.1;               // train_score_softam.lua:13
    c->write_diffmaps = 1;
    c->device = 0;
    c->max_frames = 1;
    c->hyps_per_cta = 0;
    return DSAC_OK;
}

const char* dsac_last_error(const dsac_engine* e) { return e ? e->err.c_str() : g_create_error.c_str(); }

int dsac_engine_config(const dsac_engine* e, dsac_config* out) {
    if (!e || !out) return DSAC_ERR_ARG;
    *out = e->cfg;
    return DSAC_OK;
}

void dsac_engine_destroy(dsac_engine* e) {
    if (!e) return;
    cudaSetDevice(e->cfg.device);
    const cudaStream_t streams[] = {e->stream, e->kabsch_stream, e->lane[0].side, e->lane[0].side2,
                                    e->lane[1].main, e->lane[1].side, e->lane[1].side2};
    for (cudaStream_t st : streams)
        if (st) cudaStreamSynchronize(st);
    if (e->d_phase) {
        unsigned long long h[16];
        if (cudaMemcpy(h, e->d_phase, sizeof(h), cudaMemcpyDeviceToHost) == cudaSuccess)
            fprintf(stderr, "[dsac K1 thread-0 cycles] A1 gen %llu  A2 bounds %llu  B filter %llu  C queue %llu  D full %llu  E advance %llu\n"
                            "[dsac k1_slot thread-0 cycles] regenerate+decode %llu  scan %llu  walk %llu  starts %llu  write %llu  leftover %llu\n",
                    h[0], h[1], h[2], h[3], h[4], h[5], h[8], h[9], h[10], h[11], h[12], h[13]);
    }
    if (e->d_k1_dbg && e->d_k1_spec_result && e->k1_spec_slots > 0) {
        int h[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        if (cudaMemcpy(h, e->d_k1_spec_result, std::min(8, e->k1_spec_slots) * sizeof(int), cudaMemcpyDeviceToHost) == cudaSuccess)
            fprintf(stderr, "[dsac k1_spec, last call] windows stitched per stream (0 = speculation abandoned or not used): %d %d %d %d %d %d %d %d\n",
                    h[0], h[1], h[2], h[3], h[4], h[5], h[6], h[7]);
    }
    if (e->d_k1_dbg) {
        unsigned long long h[K1S_MAX_ROUNDS * 4];
        if (cudaMemcpy(h, e->d_k1_dbg, sizeof(h), cudaMemcpyDeviceToHost) == cudaSuccess)
            for (int r = 0; r < K1S_MAX_ROUNDS && (h[r * 4] || r == 0); r++)
                fprintf(stderr, "[dsac K1 split, last call] round %d: %llu active streams, %llu candidates, %llu flagged, %llu accepted\n", r,
                        h[r * 4], h[r * 4 + 1], h[r * 4 + 2], h[r * 4 + 3]);
    }
    for (cudaStream_t st : streams)
        if (st) cudaStreamDestroy(st);
    for (K1Lane& L : e->lane) {
        for (int i = 0; i < K1S_MAX_SETS; i++)
            for (cudaEvent_t ev : {L.ev_filt[i], L.ev_solve[i], L.ev_gen[i]})
                if (ev) cudaEventDestroy(ev);
        if (L.ev_round) cudaEventDestroy(L.ev_round);
    }
    for (cudaEvent_t ev : {e->ev_fork, e->ev_join, e->ev_fwd})
        if (ev) cudaEventDestroy(ev);
    for (cudaEvent_t ev : e->k1_ev) cudaEventDestroy(ev);
    for (void* p : e->owned) cudaFree(p);
    for (DeviceBlock* b : {&e->ext_g, &e->kabsch, &e->bw.block, &e->ra, &e->ra_imap}) b->release();
    for (DeviceBlock& b : e->bw_pool) b.release();
    if (e->h_stream_ncand) cudaFreeHost(e->h_stream_ncand);
    delete e;
}

int dsac_engine_create(const dsac_config* cfg, dsac_engine** out) {
    dsac_engine* e = nullptr;
    if (!cfg || !out) return fail(e, DSAC_ERR_ARG, "null argument");
    *out = nullptr;
    if (cfg->n_hyps < 1 || cfg->n_hyps > DSAC_MAX_HYPS) return fail(e, DSAC_ERR_ARG, "n_hyps out of range [1,%d]", DSAC_MAX_HYPS);
    if (cfg->n_streams < 1 || cfg->n_streams > cfg->n_hyps) return fail(e, DSAC_ERR_ARG, "n_streams out of range [1,n_hyps]");
    if (cfg->inlier_count < 1 || cfg->inlier_count > K4_MAX_INLIERS) return fail(e, DSAC_ERR_ARG, "inlier_count out of range [1,%d]", K4_MAX_INLIERS);
    if (cfg->ref_steps < 0 || cfg->ref_steps > DSAC_MAX_REF_STEPS) return fail(e, DSAC_ERR_ARG, "ref_steps out of range [0,%d]", DSAC_MAX_REF_STEPS);
    if (cfg->max_frames < 1) return fail(e, DSAC_ERR_ARG, "max_frames must be >= 1");
    int ndev = 0;
    cudaError_t st = cudaGetDeviceCount(&ndev);
    if (st != cudaSuccess || ndev == 0)
        return fail(e, DSAC_ERR_NODEVICE, "no CUDA device available (%s); the engine has no CPU path",
                    st == cudaSuccess ? "device count 0" : cudaGetErrorString(st));
    if (cfg->device < 0 || cfg->device >= ndev) return fail(e, DSAC_ERR_ARG, "device %d out of range (have %d)", cfg->device, ndev);
    e = new dsac_engine();
    e->cfg = *cfg;
    if (e->cfg.max_candidates <= 0) e->cfg.max_candidates = 1 << 20;
    auto bail = [&](int code) {
        g_create_error = e->err;
        dsac_engine_destroy(e);
        return code;
    };
#define CUC(call)                                                                                   \
    do {                                                                                            \
        cudaError_t _s = (call);                                                                    \
        if (_s != cudaSuccess) {                                                                    \
            fail(e, DSAC_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(_s));                  \
            return bail(DSAC_ERR_CUDA);                                                             \
        }                                                                                           \
    } while (0)
    CUC(cudaSetDevice(cfg->device));
    cudaDeviceProp prop;
    CUC(cudaGetDeviceProperties(&prop, cfg->device));
    e->sm_count = prop.multiProcessorCount;
    const size_t n = (size_t)cfg->max_frames, H = (size_t)cfg->n_hyps, N = DSAC_N;
    CUC(dev_alloc(e, &e->d_coords, n * N * 3 * sizeof(int16_t)));
    CUC(dev_alloc(e, &e->d_pix, n * N * 2 * sizeof(int32_t)));
    CUC(dev_alloc(e, &e->d_gt, n * 12 * sizeof(double)));
    CUC(dev_alloc(e, &e->d_perm, (size_t)std::max(1, cfg->ref_steps) * N * sizeof(uint16_t)));
    CUC(dev_alloc(e, &e->d_hyp_pose, n * H * 6 * sizeof(double)));
    CUC(dev_alloc(e, &e->d_hyp_P, n * H * 12 * sizeof(float)));
    CUC(dev_alloc(e, &e->d_img_idx, n * H * 4 * sizeof(int32_t)));
    CUC(dev_alloc(e, &e->d_cand_idx, n * H * sizeof(int32_t)));
    CUC(dev_alloc(e, &e->d_stream_ncand, n * cfg->n_streams * sizeof(long long)));
    CUC(dev_alloc(e, &e->d_stream_endpos, n * cfg->n_streams * sizeof(unsigned long long)));
    CUC(dev_alloc(e, &e->d_status, n * sizeof(uint32_t)));
    CUC(dev_alloc(e, &e->d_fragile, sizeof(unsigned long long)));
    if (cfg->write_diffmaps) CUC(dev_alloc(e, &e->d_diffmaps, n * H * N * sizeof(float)));
    CUC(dev_alloc(e, &e->d_scores, n * H * sizeof(double)));
    CUC(dev_alloc(e, &e->d_sf, n * H * sizeof(double)));
    CUC(dev_alloc(e, &e->d_entropy, n * sizeof(double)));
    CUC(dev_alloc(e, &e->d_avg, n * 6 * sizeof(double)));
    CUC(dev_alloc(e, &e->d_ref, n * 6 * sizeof(double)));
    CUC(dev_alloc(e, &e->d_inlier_map, n * N * sizeof(int32_t)));
    CUC(dev_alloc(e, &e->d_steps_done, n * sizeof(int32_t)));
    CUC(dev_alloc(e, &e->d_n_perm, n * sizeof(int32_t)));
    CUC(dev_alloc(e, &e->d_loss, n * sizeof(double)));
    CUC(dev_alloc(e, &e->d_rot_err, n * sizeof(double)));
    CUC(dev_alloc(e, &e->d_t_err, n * sizeof(double)));
    CUC(dev_alloc(e, &e->d_correct, n * sizeof(int32_t)));
    CUC(dev_alloc(e, &e->d_frame_counter, n * sizeof(unsigned int)));
    CUC(cudaMemset(e->d_frame_counter, 0, n * sizeof(unsigned int)));
    CUC(cudaMemset(e->d_fragile, 0, sizeof(unsigned long long)));
    if (getenv("DSAC_K1_TIMERS")) {
        CUC(dev_alloc(e, &e->d_phase, 16 * sizeof(unsigned long long)));
        CUC(cudaMemset(e->d_phase, 0, 16 * sizeof(unsigned long long)));
    }
    CUC(cudaMemset(e->d_status, 0, n * sizeof(uint32_t)));
    CUC(cudaMemset(e->d_steps_done, 0, n * sizeof(int32_t)));
    CUC(cudaMemset(e->d_n_perm, 0, n * sizeof(int32_t)));
    CUC(cudaMemset(e->d_inlier_map, 0, n * N * sizeof(int32_t)));
    CUC(cudaMemset(e->d_ref, 0, n * 6 * sizeof(double)));
    CUC(cudaMemset(e->d_loss, 0, n * sizeof(double)));
    CUC(cudaMemset(e->d_rot_err, 0, n * sizeof(double)));
    CUC(cudaMemset(e->d_t_err, 0, n * sizeof(double)));
    CUC(cudaMemset(e->d_correct, 0, n * sizeof(int32_t)));
    // refinement permutations: std::mt19937 randG (default seed) once per frame, iota +
    // std::shuffle per step with the continuing generator (cnn_softam.h:1104,1112-1114) --
    // identical for every frame, so they are built once with the very same libstdc++ calls.
    {
        std::mt19937 randG;
        std::vector<uint16_t> perm((size_t)std::max(1, cfg->ref_steps) * N, 0);
        for (int s = 0; s < cfg->ref_steps; s++) {
            std::vector<int> idx(N);
            for (size_t i = 0; i < N; i++) idx[i] = (int)i;
            std::shuffle(idx.begin(), idx.end(), randG);
            for (size_t i = 0; i < N; i++) perm[(size_t)s * N + i] = (uint16_t)idx[i];
        }
        CUC(cudaMemcpy(e->d_perm, perm.data(), perm.size() * sizeof(uint16_t), cudaMemcpyHostToDevice));
    }
    CUC(cudaFuncSetAttribute(k_sample, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(K1Smem)));
    // k_refine wants 8 CTAs x 26 KB of shared memory per SM: ask for the carve-out explicitly (the default heuristic
    // need not pick the split the launch bounds were written for).  k_sample is left to the default: it spills to
    // local memory and measured 5 % slower with the largest carve-out (3.39 vs 3.24 ms), i.e. with the smallest L1.
    CUC(cudaFuncSetAttribute(k_refine, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
    CUC(cudaMallocHost(&e->h_stream_ncand, n * cfg->n_streams * sizeof(long long)));
    {
        const size_t T = (size_t)cfg->n_streams, slots = n * T;
        const int quota_max = (cfg->n_hyps + cfg->n_streams - 1) / cfg->n_streams;
        // few streams (single-frame latency): the first round takes 115 % of the expected need, so the capacity is larger
        const int cap_per_hyp = slots < 128 ? (K1S_CAP_PER_HYP * 3) / 2 : K1S_CAP_PER_HYP;
        int cap = std::min(K1S_MAX_CAP, std::max(1024, cap_per_hyp * quota_max));
        cap = (cap + 1023) & ~1023;     // a round is generated in portions of cap / 4, themselves multiples of 256
        e->k1_cap = cap;
        e->k1_wq_stride = (int)(slots * 128);
        CUC(dev_alloc(e, &e->d_k1_state, slots * sizeof(K1SlotState)));
        CUC(dev_alloc(e, &e->d_k1_celltab, n * N * sizeof(CellRec)));
        CUC(dev_alloc(e, &e->d_k1_cells, slots * cap * sizeof(uint2)));
        CUC(dev_alloc(e, &e->d_k1_endw, slots * cap * sizeof(uint32_t)));
        CUC(dev_alloc(e, &e->d_k1_accbits, slots * (cap / 32) * sizeof(uint32_t)));
        CUC(dev_alloc(e, &e->d_k1_pose, slots * cap * 6 * sizeof(double)));
        CUC(dev_alloc(e, &e->d_k1_wq, (size_t)K1S_MAX_SETS * slots * 128 * sizeof(uint2)));
        CUC(dev_alloc(e, &e->d_k1_fq, 2 * slots * cap * sizeof(uint32_t)));   // two regions: the filter of set k+1 writes one while the solve of set k reads the other
        CUC(dev_alloc(e, &e->d_k1_chain, slots * (K1Q_MAX_WIN + 1) * 4 * sizeof(uint32_t)));
        CUC(cudaMemset(e->d_k1_chain, 0, slots * (K1Q_MAX_WIN + 1) * 4 * sizeof(uint32_t)));
        {
            int per_sm = 0;
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k1_pipe, K1S_THREADS, 0);
            e->k1_slot_capacity = std::max(1, per_sm) * e->sm_count;
            if (const char* pv = getenv("DSAC_K1_PIPE")) e->k1_pipe = atoi(pv);
        }
        {   // speculative first round for a few streams (sampler_split.cuh: k1_spec / k1_stitch); DSAC_K1_SPEC=0 turns it off
            int want = 1;
            if (const char* sv = getenv("DSAC_K1_SPEC")) want = atoi(sv);
            if (want) {
                const size_t ss = std::min<size_t>(slots, 8);    // measured: 8 frames x 1 stream 0.546 -> 0.481 ms per step, 16 frames 0.565 -> 0.571 (1360 window CTAs: no longer one wave)
                CUC(dev_alloc(e, &e->d_k1_vstate, ss * K1P_VPER * sizeof(K1SlotState)));
                CUC(dev_alloc(e, &e->d_k1_vcells, ss * K1P_VPER * K1P_CAPW * sizeof(uint2)));
                CUC(dev_alloc(e, &e->d_k1_vendw, ss * K1P_VPER * K1P_CAPW * sizeof(uint32_t)));
                CUC(dev_alloc(e, &e->d_k1_spec_result, ss * sizeof(int)));
                CUC(cudaMemset(e->d_k1_spec_result, 0, ss * sizeof(int)));
                CUC(dev_alloc(e, &e->d_k1_spec_table, ss * K1P_TABLE * sizeof(int)));
                e->k1_spec_slots = (int)ss;
            }
        }
        // the lanes.  The fp64 kernels get the higher priority: when a generator launch and a filter launch become ready
        // together, the persistent filter CTAs are placed first and the generator's CTAs fill the registers they leave free
        int least = 0, greatest = 0;
        CUC(cudaDeviceGetStreamPriorityRange(&least, &greatest));
        for (int l = 0; l < 2; l++) {
            K1Lane& L = e->lane[l];
            if (l == 1) CUC(cudaStreamCreateWithFlags(&L.main, cudaStreamNonBlocking));
            CUC(cudaStreamCreateWithPriority(&L.side, cudaStreamNonBlocking, greatest));
            CUC(cudaStreamCreateWithPriority(&L.side2, cudaStreamNonBlocking, greatest));
            for (int i = 0; i < K1S_MAX_SETS; i++) {
                CUC(cudaEventCreateWithFlags(&L.ev_filt[i], cudaEventDisableTiming));
                CUC(cudaEventCreateWithFlags(&L.ev_solve[i], cudaEventDisableTiming));
                CUC(cudaEventCreateWithFlags(&L.ev_gen[i], cudaEventDisableTiming));
            }
            CUC(cudaEventCreateWithFlags(&L.ev_round, cudaEventDisableTiming));
            CUC(dev_alloc(e, &L.counters, 2 * K1S_MAX_SETS * sizeof(int)));
            CUC(dev_alloc(e, &L.stats, 4 * sizeof(unsigned long long)));
            CUC(cudaMemset(L.stats, 0, 4 * sizeof(unsigned long long)));
        }
        if (const char* stt = getenv("DSAC_K1_SLOT_THREADS")) e->k1_slot_threads = atoi(stt);
        if (getenv("DSAC_K1_DEBUG")) CUC(dev_alloc(e, &e->d_k1_dbg, K1S_MAX_ROUNDS * 4 * sizeof(unsigned long long)));
        CUC(cudaFuncSetAttribute(k1_filter, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(K1FSmem)));
        int per_sm = 0;
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k1_filter, K1F_THREADS, sizeof(K1FSmem));
        e->k1_filter_grid = std::max(1, per_sm) * e->sm_count;
        per_sm = 0;
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k1_solve, K1V_THREADS, 0);
        e->k1_solve_grid = std::max(1, per_sm) * e->sm_count;
    }
    CUC(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
    CUC(cudaStreamCreateWithFlags(&e->kabsch_stream, cudaStreamNonBlocking));
    CUC(cudaEventCreateWithFlags(&e->ev_fork, cudaEventDisableTiming));
    CUC(cudaEventCreateWithFlags(&e->ev_join, cudaEventDisableTiming));
    CUC(cudaEventCreateWithFlags(&e->ev_fwd, cudaEventDisableTiming));
#undef CUC
    *out = e;
    return DSAC_OK;
}

int dsac_set_stages(dsac_engine* e, uint32_t mask) {
    if (!e) return DSAC_ERR_ARG;
    e->stages = mask;
    return DSAC_OK;
}

int dsac_set_tail_split(dsac_engine* e, int32_t mode) {
    if (!e) return DSAC_ERR_ARG;
    if (mode < 0 || mode > 2) return fail(e, DSAC_ERR_ARG, "tail split mode %d out of range [0,2]", mode);
    e->tail_split = mode;
    return DSAC_OK;
}

int64_t dsac_launch_count(const dsac_engine* e) { return e ? e->launches : 0; }

int dsac_sampler_profile(dsac_engine* e, int32_t enable) {
    if (!e) return DSAC_ERR_ARG;
    CU(cudaSetDevice(e->cfg.device));
    if (enable && !e->d_k1_dbg) CU(dev_alloc(e, &e->d_k1_dbg, K1S_MAX_ROUNDS * 4 * sizeof(unsigned long long)));
    e->k1_profile = enable ? 1 : 0;
    return DSAC_OK;
}

int dsac_debug_spec_result(dsac_engine* e, int32_t out8[8]) {
    if (!e || !out8) return DSAC_ERR_ARG;
    for (int i = 0; i < 8; i++) out8[i] = 0;
    if (!e->d_k1_spec_result || e->k1_spec_slots <= 0) return DSAC_OK;
    CU(cudaSetDevice(e->cfg.device));
    CU(cudaDeviceSynchronize());
    CU(cudaMemcpy(out8, e->d_k1_spec_result, std::min(8, e->k1_spec_slots) * sizeof(int32_t), cudaMemcpyDeviceToHost));
    return DSAC_OK;
}

int dsac_sampler_profile_read(dsac_engine* e, double ms[4], uint64_t counts[4]) {
    if (!e || !ms || !counts) return DSAC_ERR_ARG;
    if (!e->k1_profile || e->k1_ev_n < 2) return fail(e, DSAC_ERR_ARG, "dsac_sampler_profile_read: no profiled forward pass");
    CU(cudaSetDevice(e->cfg.device));
    CU(cudaEventSynchronize(e->k1_ev[e->k1_ev_n - 1]));
    for (int k = 0; k < 4; k++) { ms[k] = 0; counts[k] = 0; }
    for (int i = 1; i < e->k1_ev_n; i++) {
        float t = 0;
        CU(cudaEventElapsedTime(&t, e->k1_ev[i - 1], e->k1_ev[i]));
        const int kind = e->k1_ev_kind[i];
        if (kind >= 0 && kind < 4) ms[kind] += t;
    }
    unsigned long long h[K1S_MAX_ROUNDS * 4];
    CU(cudaMemcpy(h, e->d_k1_dbg, sizeof(h), cudaMemcpyDeviceToHost));
    for (int r = 0; r < K1S_MAX_ROUNDS; r++) {
        counts[0] += h[r * 4 + 1]; counts[1] += h[r * 4 + 2]; counts[2] += h[r * 4 + 3];
        if (h[r * 4 + 0]) counts[3] = (uint64_t)(r + 1);
    }
    return DSAC_OK;
}

int dsac_set_score_hook(dsac_engine* e, dsac_score_hook fn, void* user) {
    if (!e) return DSAC_ERR_ARG;
    if (fn && !e->cfg.write_diffmaps) return fail(e, DSAC_ERR_ARG, "a score hook needs write_diffmaps=1");
    e->hook = fn;
    e->hook_user = user;
    return DSAC_OK;
}

int dsac_set_score_backward_hook(dsac_engine* e, dsac_score_backward_hook fn, void* user) {
    if (!e) return DSAC_ERR_ARG;
    e->bw_hook = fn;
    e->bw_hook_user = user;
    return DSAC_OK;
}

// Score seam in the backward pass: with hooks registered, dScore/dDiffMap comes from the backward hook (fills e->ext_g);
// returns the pointer k_dscore shall read (null: closed-form soft-inlier derivative).
static int seam_backward(dsac_engine* e, int n, const double* d_sog, cudaStream_t stream, const double** ext_g) {
    *ext_g = nullptr;
    if (!e->hook && !e->bw_hook) return DSAC_OK;
    if (!e->hook || !e->bw_hook)
        return fail(e, DSAC_ERR_ARG, "the score seam needs both hooks: %s is registered but %s is not (dsac_set_score_hook / dsac_set_score_backward_hook)",
                    e->hook ? "the forward hook" : "the backward hook", e->hook ? "the backward hook" : "the forward hook");
    if (!e->d_diffmaps) return fail(e, DSAC_ERR_ARG, "the score seam needs write_diffmaps=1");
    const size_t H = e->cfg.n_hyps, count = (size_t)n * H * DSAC_N;
    CU(e->ext_g.reserve((count + (size_t)n * H) * sizeof(double)));
    double* grad = (double*)e->ext_g.ptr;
    double* clamped = grad + count;   // [n][H] behind the gradient block
    k_clamp_copy<<<(unsigned)(((size_t)n * H + 255) / 256), 256, 0, stream>>>(d_sog, clamped, (size_t)n * H, e->cfg.grad_clamp);
    e->launches++;
    CU(cudaGetLastError());
    int rc = e->bw_hook(e->d_diffmaps, clamped, n, (int32_t)H, grad, (void*)stream, e->bw_hook_user);
    if (rc != 0) return fail(e, DSAC_ERR_ARG, "score backward hook returned %d", rc);
    *ext_g = grad;
    return DSAC_OK;
}

static int pick_tile(const dsac_engine* e, int n_frames) {
    int H = e->cfg.n_hyps, t = e->cfg.hyps_per_cta;
    if (t <= 0) {
        // enough CTAs to fill the chip a few times over, but no smaller than 8 hypotheses
        t = 64;
        while (t > 8 && (long long)n_frames * ((H + t - 1) / t) < 4ll * e->sm_count) t >>= 1;
    }
    t = std::max(8, std::min(t, K2_MAX_TILE));
    t = (t + 7) & ~7;
    return t;
}

// The split sampler (sampler_split.cuh) for the `n` frames at frame offset `off`, on lane L: the generator on `stream`, filter
// and solve on the lane's side streams.  One pass at a time per lane: the queues and per-slot arrays are the engine's,
// sliced by frame offset.
static int sample_split(dsac_engine* e, K1Lane& L, int32_t off, int32_t n, SampleParams sp, cudaStream_t stream) {
    const dsac_config& c = e->cfg;
    const size_t o = (size_t)off, Nn = DSAC_N, T = (size_t)c.n_streams, cap = (size_t)e->k1_cap;
    K1SplitParams q;
    q.sp = sp;
    q.state = e->d_k1_state + o * T; q.celltab = e->d_k1_celltab + o * Nn;
    q.cells = e->d_k1_cells + o * T * cap; q.endw = e->d_k1_endw + o * T * cap;
    q.accbits = e->d_k1_accbits + o * T * (cap / 32); q.pose_out = e->d_k1_pose + o * T * cap * 6;
    q.wq = e->d_k1_wq + o * T * 128; q.fq = e->d_k1_fq + o * T * cap;   // (work items / flagged candidates of this range's slots)
    q.wq_n = L.counters; q.fq_n = L.counters + K1S_MAX_SETS;
    q.wq_stride = e->k1_wq_stride;
    q.first_frac = (double)K1S_FIRST_ROUND_FRAC;
    q.spec = 0;
    const int par = (int)(L.calls & 1ull);
    L.calls++;
    q.stats_cur = L.stats + 2 * par; q.stats_prev = L.stats + 2 * (par ^ 1);
    q.dbg = e->d_k1_dbg;
    q.cap = e->k1_cap;
    const long long n_slots = (long long)n * c.n_streams;
    // a round is generated in up to 4 portions of cap / 4 candidates (round 0: 4, round 1: 2, later rounds: the whole
    // round at once); a filter work item is a chunk of a portion.  Measured at 128 frames: 2 / 4 / 8 / 16 portions
    // 0.885 / 0.896 / 0.951 / 1.207 ms per step (1024 frames: 2.94 / 2.89 / 2.97 / -)
    const int n_port = n_slots < 256 ? 2 : 4;   // portions of round 0 (round 1: half as many, twice as large)
    const int portion4 = e->k1_cap / n_port;
    const int want_chunk = n_slots >= 512 ? 2048 : (n_slots >= 64 ? 512 : 256);
    q.chunk = 256;
    for (int cc : {2048, 1024, 512, 256})
        if (cc <= want_chunk && cc <= K1F_MAX_CHUNK && portion4 % cc == 0) { q.chunk = cc; break; }
    q.n_slots = (int)n_slots;
    q.round = 0; q.select_only = 0; q.gen_only = 0;
    CU(cudaMemsetAsync(L.counters, 0, 2 * K1S_MAX_SETS * sizeof(int), stream));
    CU(cudaMemsetAsync(q.stats_cur, 0, 2 * sizeof(unsigned long long), stream));
    if (q.dbg) CU(cudaMemsetAsync(q.dbg, 0, K1S_MAX_ROUNDS * 4 * sizeof(unsigned long long), stream));
    e->k1_ev_n = 0;
    auto mark = [&](int kind) {   // dsac_sampler_profile: an event after every launch
        if (!e->k1_profile) return;
        if ((size_t)e->k1_ev_n >= e->k1_ev.size()) {
            cudaEvent_t ev;
            if (cudaEventCreate(&ev) != cudaSuccess) return;
            e->k1_ev.push_back(ev);
            e->k1_ev_kind.push_back(0);
        }
        e->k1_ev_kind[e->k1_ev_n] = kind;
        cudaEventRecord(e->k1_ev[e->k1_ev_n++], stream);
    };
    // threads per (frame, stream) of the generator.  A stream's generation is a serial chain of windows; with fewer
    // streams than the SMs hold at 256 threads, larger CTAs shorten the parallel phases of a window (measured, step in
    // ms at 256 / 512 / 1024 threads: 128 frames 0.931 / 0.922 / 0.934, 512 frames 1.794 / 1.811 / -; one frame
    // 295 / - / 272 us).  The MT19937 regeneration itself (half of a window) does not scale: 227 words are independent.
    int slot_threads = K1S_THREADS;
    if (n_slots <= 32) slot_threads = 1024;
    else if (n_slots <= 2 * e->sm_count) slot_threads = 512;
    if (e->k1_slot_threads > 0) slot_threads = e->k1_slot_threads;
    auto launch_slot = [&](const K1SplitParams& qq) {
        const dim3 g(c.n_streams, n);
        if (slot_threads == 1024) k1_slot_t<1024><<<g, 1024, 0, stream>>>(qq);
        else if (slot_threads == 512) k1_slot_t<512><<<g, 512, 0, stream>>>(qq);
        else k1_slot<<<g, K1S_THREADS, 0, stream>>>(qq);
    };
    // streams: generator on `stream`, filter (and solve) on a side stream; with a batch that does not fill the GPU several
    // times over the solve gets a stream of its own, so that the filter of set k+1 need not wait for the solve of set k
    // (measured, ms per step with the solve on the filter's stream / on its own: 128 frames 0.938 / 0.896, 256 frames
    // 1.21 / 1.18, 512 frames 1.78 / 1.69, 1024 frames 2.92 / 2.96).  With the profile on everything runs on one stream so
    // that the event intervals are the kernels' own durations.
    const bool overlap = !e->k1_profile;
    cudaStream_t side = overlap ? L.side : stream;
    cudaStream_t solve_side = (overlap && n_slots <= 768) ? L.side2 : side;
    const size_t n_slots_cap = (size_t)e->cfg.max_frames * c.n_streams * (size_t)e->k1_cap;
    mark(-1);
    {
        const int cell_blocks = (int)(((size_t)n * Nn + 255) / 256), seed_blocks = (int)((n_slots + 31) / 32);
        k1_cells<<<(unsigned)(cell_blocks + seed_blocks), 256, 0, stream>>>(q, n, seed_blocks);
    }
    mark(0);
    e->launches++;
    int set = 0;
    // few streams (single-frame latency): no previous call's shortfall to make up in later rounds -- the first round
    // takes 115 % of the expected need and one top-up round follows (every round is three dependent launches);
    // the rare straggler goes to the monolithic kernel
    const bool few = n_slots < 128;
    if (few) q.first_frac = 1.15;
    // speculative first round (k1_spec / k1_stitch): one stream generated window by window on many SMs; pays when a
    // stream's first round is several windows long (>= 64 hypotheses per stream) and the GPU is otherwise idle
    const int quota_max = (c.n_hyps + c.n_streams - 1) / c.n_streams;
    const bool use_spec = few && off == 0 && n_slots <= e->k1_spec_slots && quota_max >= 64 && c.max_candidates >= (1 << 16);   // (the candidate bound cannot fall inside the speculative round)
    // chained generator (k1_pipe): K CTAs per stream, all of them resident at once
    const int pipe_K = (int)std::min<long long>(8, e->k1_slot_capacity / std::max<long long>(1, n_slots));
    const bool use_pipe = e->k1_pipe && !use_spec && pipe_K >= 3 && n_slots >= 9 && quota_max >= 64 && c.max_candidates >= (1 << 16) &&
                          !e->k1_profile;
    const int n_rounds = few ? std::min(K1_ROUNDS, 2) : K1_ROUNDS;
    for (int r = 0; r < n_rounds; r++) {
        // portions only pay when the generator has the whole GPU to fill (many streams); a few streams (single-frame
        // latency, BASELINE config 2) take every round in one launch set: fewer dependent launches
        const bool portioned = n_slots >= 128 && r < 2 && !(use_pipe && r == 0);
        const int sets = portioned ? (r == 0 ? n_port : n_port / 2) : 1;
        q.round = r;
        q.portion = portioned ? (r == 0 ? portion4 : 2 * portion4) : e->k1_cap;   // round 1 may use the whole capacity too
        q.round_limit = q.portion * sets;
        const int fgrid = (int)std::min<long long>(e->k1_filter_grid, n_slots * ((q.portion + q.chunk - 1) / q.chunk));
        if (overlap && r > 0) CU(cudaStreamWaitEvent(stream, L.ev_round, 0));   // the selection needs the previous round's solves
        for (int k = 0; k < sets && set < K1S_MAX_SETS; k++, set++) {
            q.gen_only = (k > 0);
            q.qidx = set;
            q.fqidx = set;
            q.fq = e->d_k1_fq + o * T * cap + (size_t)(set & 1) * n_slots_cap;
            if (use_spec && r == 0 && k == 0) {
                K1SpecParams spp;
                spp.vstate = e->d_k1_vstate; spp.vcells = e->d_k1_vcells; spp.vendw = e->d_k1_vendw; spp.result = e->d_k1_spec_result; spp.table = e->d_k1_spec_table;
                k1_spec<<<dim3(K1P_VPER, (unsigned)n_slots), K1S_THREADS, 0, stream>>>(q, spp);
                k1_stitch<<<(unsigned)n_slots, K1T_THREADS, 0, stream>>>(q, spp);
                k1_gather<<<dim3((unsigned)((e->k1_cap + K1G_PER_CTA - 1) / K1G_PER_CTA), (unsigned)n_slots), K1G_THREADS, 0, stream>>>(q, spp);
                e->launches += 2;
            } else if (use_pipe && r == 0 && k == 0) {
                K1PipeParams ppm;
                ppm.chain = e->d_k1_chain + o * T * (K1Q_MAX_WIN + 1) * 4;
                ppm.epoch = (uint32_t)(++e->k1_epoch & 0x7fffffffull) + 1u;
                ppm.K = pipe_K;
                k1_pipe<<<dim3((unsigned)pipe_K, (unsigned)n_slots), K1S_THREADS, 0, stream>>>(q, ppm);
            } else {
                launch_slot(q);
            }
            mark(0);
            if (overlap) {
                CU(cudaEventRecord(L.ev_gen[set], stream));
                CU(cudaStreamWaitEvent(side, L.ev_gen[set], 0));
                if (solve_side != side && set >= 2) CU(cudaStreamWaitEvent(side, L.ev_solve[set - 2], 0));   // the flag-queue region is free again
            }
            k1_filter<<<fgrid, K1F_THREADS, sizeof(K1FSmem), side>>>(q);
            if (!overlap) mark(1);
            if (solve_side != side) {
                CU(cudaEventRecord(L.ev_filt[set], side));
                CU(cudaStreamWaitEvent(solve_side, L.ev_filt[set], 0));
            }
            if (few) k1_solve4<<<e->k1_solve_grid, K1V_THREADS, 0, solve_side>>>(q);
            else k1_solve<<<e->k1_solve_grid, K1V_THREADS, 0, solve_side>>>(q);
            if (solve_side != side) CU(cudaEventRecord(L.ev_solve[set], solve_side));
            if (!overlap) mark(2);
            e->launches += 3;
        }
        if (overlap) CU(cudaEventRecord(L.ev_round, solve_side));
    }
    if (overlap) CU(cudaStreamWaitEvent(stream, L.ev_round, 0));
    q.round = n_rounds; q.select_only = 1; q.gen_only = 0;
    launch_slot(q);
    mark(0);
    sp.resume = q.state;   // streams the rounds left unfinished (normally none) continue in the monolithic kernel
    k_sample<<<dim3(c.n_streams, n), K1_THREADS, sizeof(K1Smem), stream>>>(sp);
    mark(3);
    e->launches += 2;
    CU(cudaGetLastError());
    return DSAC_OK;
}

// Launches the forward stages for `n` frames whose per-frame engine buffers start at frame offset `off` (inputs are passed
// already offset), with the sampler on lane `lane`.  Used whole (off = 0) and per half-batch by forward_split.
static int forward_range(dsac_engine* e, int32_t off, int32_t n, int64_t frame0, const int16_t* d_coords, const int32_t* d_pix,
                         int32_t pix_shared, const double* d_gt_jp, cudaStream_t stream, int lane = 0) {
    const dsac_config& c = e->cfg;
    const size_t o = (size_t)off, Hh = (size_t)c.n_hyps, Nn = DSAC_N;

    if (e->stages & DSAC_STAGE_SAMPLE) {
        CU(cudaMemsetAsync(e->d_status + o, 0, (size_t)n * sizeof(uint32_t), stream));
        SampleParams sp;
        sp.coords = d_coords; sp.pix = d_pix; sp.pix_stride = pix_shared ? 0 : DSAC_N * 2;
        sp.f = c.focal; sp.cx = c.cx; sp.cy = c.cy;
        sp.H = c.n_hyps; sp.T = c.n_streams; sp.thr = c.thr2d;
        sp.seed = c.seed; sp.skip = c.stream_skip; sp.max_candidates = c.max_candidates;
        sp.frame0 = frame0;
        sp.hyp_pose = e->d_hyp_pose + o * Hh * 6; sp.hyp_P = e->d_hyp_P + o * Hh * 12; sp.img_idx = e->d_img_idx + o * Hh * 4; sp.cand_idx = e->d_cand_idx + o * Hh;
        sp.stream_ncand = e->d_stream_ncand + o * c.n_streams; sp.stream_endpos = e->d_stream_endpos + o * c.n_streams; sp.status = e->d_status + o; sp.n_fragile = e->d_fragile;
        sp.phase_cycles = e->d_phase;
        { const char* g = getenv("DSAC_K1_A2_GENERIC"); sp.a2_generic = (g && g[0] == '1') ? 1 : 0; }
        sp.resume = nullptr;
        const int rc = sample_split(e, e->lane[lane], off, n, sp, stream);
        if (rc != DSAC_OK) return rc;
    }
    if (e->stages & DSAC_STAGE_SCORE) {
        ScoreParams kp;
        kp.coords = d_coords; kp.pix = d_pix; kp.pix_stride = pix_shared ? 0 : DSAC_N * 2;
        kp.hyp_P = e->d_hyp_P + o * Hh * 12; kp.hyp_pose = e->d_hyp_pose + o * Hh * 6;
        kp.diffmaps = e->d_diffmaps ? e->d_diffmaps + o * Hh * Nn : nullptr; kp.scores = e->d_scores + o * Hh; kp.sf = e->d_sf + o * Hh; kp.entropy = e->d_entropy + o;
        kp.avg_pose = e->d_avg + o * 6; kp.frame_counter = e->d_frame_counter + o;
        kp.H = c.n_hyps;
        kp.tile = pick_tile(e, n);
        kp.tiles_per_frame = (c.n_hyps + kp.tile - 1) / kp.tile;
        kp.cxf = (float)c.cx; kp.cyf = (float)c.cy;
        kp.thr = (float)c.thr2d;
        kp.kbeta = (float)(c.beta * 1.4426950408889634);
        kp.alpha = c.alpha;
        kp.external_scores = 0;
        dim3 grid(kp.tiles_per_frame, n);
        if (e->d_diffmaps) k_score<true><<<grid, K2_THREADS, 0, stream>>>(kp);
        else k_score<false><<<grid, K2_THREADS, 0, stream>>>(kp);
        e->launches++;
        CU(cudaGetLastError());
        if (e->hook) {
            // score seam (lua_calls.h:284-300): external scorer on the materialised diffmaps,
            // then only the softmax / soft-argmax tail
            int rc = e->hook(kp.diffmaps, n, c.n_hyps, kp.scores, (void*)stream, e->hook_user);
            if (rc != 0) return fail(e, DSAC_ERR_ARG, "score hook returned %d", rc);
            kp.external_scores = 1;
            kp.tiles_per_frame = 1;
            k_score<false><<<dim3(1, n), K2_THREADS, 0, stream>>>(kp);
            e->launches++;
            CU(cudaGetLastError());
        }
    }
    if (e->stages & DSAC_STAGE_REFINE) {
        RefineParams rp;
        memset(&rp, 0, sizeof(rp));
        rp.coords = d_coords; rp.pix = d_pix; rp.pix_stride = pix_shared ? 0 : DSAC_N * 2;
        rp.perm = e->d_perm;
        rp.f = c.focal; rp.cx = c.cx; rp.cy = c.cy;
        rp.thr = c.thr2d; rp.inlier_count = c.inlier_count; rp.ref_steps = c.ref_steps;
        rp.n_jobs = n;
        rp.job_init = e->d_avg + o * 6;
        rp.out_pose = e->d_ref + o * 6;
        rp.inlier_map = e->d_inlier_map + o * Nn; rp.steps_done = e->d_steps_done + o; rp.n_perm_steps = e->d_n_perm + o;
        rp.status = e->d_status + o;
        if ((e->stages & DSAC_STAGE_EVAL) && d_gt_jp) {
            rp.gt_jp = d_gt_jp;
            rp.loss = e->d_loss + o; rp.rot_err = e->d_rot_err + o; rp.t_err = e->d_t_err + o; rp.correct = e->d_correct + o;
        }
        k_refine<<<n, K4_THREADS, 0, stream>>>(rp);
        e->launches++;
        CU(cudaGetLastError());
    }
    return DSAC_OK;
}

// forward_range over the whole batch.  With allow_split, a batch of at least 768 frames runs as two lanes: two concurrent
// half-batches, each a complete pass (sampler, H x N matrix, refinement) over its frames with its own queues, counters and
// side streams.  The passes de-phase on the GPU -- one half's generator and latency-bound refinement run beside the other
// half's register-filling filter -- which a single pass, whose kernels depend on each other in sequence, cannot: 2.90 ->
// 2.69 ms per 1024 frames; three or more lanes are slower (3.10 / 3.31 ms: tools/lane_probe.py).  Frames are independent
// (disjoint slices of every engine buffer) and sampler streams keyed by the global frame index, so results do not depend on
// the split.  Fork / join with events: for the caller everything still happens in stream order on `stream`.
static int forward_split(dsac_engine* e, int32_t n, int64_t frame0, const int16_t* d_coords, const int32_t* d_pix,
                         int32_t pix_shared, const double* d_gt_jp, cudaStream_t stream, bool allow_split) {
    if (!allow_split || n < 768 || e->k1_profile || e->d_k1_dbg || e->hook || !(e->stages & DSAC_STAGE_SAMPLE))
        return forward_range(e, 0, n, frame0, d_coords, d_pix, pix_shared, d_gt_jp, stream);
    const int32_t na = n / 2;
    const size_t N = DSAC_N, f = (size_t)na;
    cudaStream_t main1 = e->lane[1].main;
    CU(cudaEventRecord(e->ev_fork, stream));
    CU(cudaStreamWaitEvent(main1, e->ev_fork, 0));
    int rc = forward_range(e, na, n - na, frame0 + na, d_coords + f * N * 3, pix_shared ? d_pix : d_pix + f * N * 2, pix_shared,
                           d_gt_jp ? d_gt_jp + f * 12 : nullptr, main1, 1);
    cudaEventRecord(e->ev_join, main1);   // the caller's stream joins the lane again whatever happens below
    if (rc == DSAC_OK) rc = forward_range(e, 0, na, frame0, d_coords, d_pix, pix_shared, d_gt_jp, stream, 0);
    CU(cudaStreamWaitEvent(stream, e->ev_join, 0));
    return rc;
}

int dsac_forward_device(dsac_engine* e, int32_t n, int64_t frame0, const int16_t* d_coords, const int32_t* d_pix,
                        int32_t pix_shared, const double* d_gt_jp, void* stream_v) {
    if (!e) return DSAC_ERR_ARG;
    if (n < 1 || n > e->cfg.max_frames) return fail(e, DSAC_ERR_CAPACITY, "n_frames %d exceeds engine capacity %d", n, e->cfg.max_frames);
    if (!d_coords || !d_pix) return fail(e, DSAC_ERR_ARG, "null input");
    CU(cudaSetDevice(e->cfg.device));
    e->cur_coords = d_coords;
    e->cur_pix = d_pix;
    e->cur_pix_shared = pix_shared;
    e->cur_gt = d_gt_jp;
    e->cur_n = n;
    e->dsac_n = 0;
    e->cur_frame0 = frame0;
    if (e->pending) return fail(e, DSAC_ERR_ARG, "dsac_forward_device: a submitted pass has not been awaited (dsac_forward_wait)");
    int rc = forward_split(e, n, frame0, d_coords, d_pix, pix_shared, d_gt_jp, (cudaStream_t)stream_v, e->tail_split >= 1);
    if (rc != DSAC_OK) return rc;
    CU(cudaEventRecord(e->ev_fwd, (cudaStream_t)stream_v));   // dsac_backward (engine stream) waits on this
    return DSAC_OK;
}

// Queues the device->host copies of frames [off, off+n) into the caller's buffers (no synchronisation).
static int fetch_range(dsac_engine* e, int32_t off, int32_t n, dsac_forward_out* o, cudaStream_t stream) {
    const size_t H = e->cfg.n_hyps, N = DSAC_N, T = e->cfg.n_streams, nn = (size_t)n, f = (size_t)off;
#define D2H(dst, src, per)                                                                                          \
    do {                                                                                                            \
        if ((dst) && (src))                                                                                         \
            CU(cudaMemcpyAsync((dst) + f * (per), (src) + f * (per), nn * (per) * sizeof(*(dst)), cudaMemcpyDeviceToHost, stream)); \
    } while (0)
    D2H(o->hyp_pose, e->d_hyp_pose, H * 6);
    D2H(o->img_idx, e->d_img_idx, H * 4);
    D2H(o->cand_idx, e->d_cand_idx, H);
    D2H(o->scores, e->d_scores, H);
    D2H(o->sf, e->d_sf, H);
    if (o->diffmaps) {
        if (!e->d_diffmaps) return fail(e, DSAC_ERR_ARG, "diffmaps requested but the engine was created with write_diffmaps=0");
        D2H(o->diffmaps, e->d_diffmaps, H * N);
    }
    D2H(o->entropy, e->d_entropy, 1);
    D2H(o->avg_pose, e->d_avg, 6);
    D2H(o->ref_pose, e->d_ref, 6);
    D2H(o->inlier_map, e->d_inlier_map, N);
    D2H(o->ref_steps_done, e->d_steps_done, 1);
    D2H(o->n_perm_steps, e->d_n_perm, 1);
    D2H(o->loss, e->d_loss, 1);
    D2H(o->rot_err, e->d_rot_err, 1);
    D2H(o->t_err, e->d_t_err, 1);
    D2H(o->correct, e->d_correct, 1);
    D2H(o->status, e->d_status, 1);
    if (o->n_candidates) {
        long long* hdst = e->h_stream_ncand;
        D2H(hdst, e->d_stream_ncand, T);
    }
#undef D2H
    return DSAC_OK;
}

static void sum_candidates(dsac_engine* e, int32_t n, dsac_forward_out* o) {
    const size_t T = e->cfg.n_streams;
    if (!o->n_candidates) return;
    for (size_t f = 0; f < (size_t)n; f++) {
        long long s = 0;
        for (size_t t = 0; t < T; t++) s += e->h_stream_ncand[f * T + t];
        o->n_candidates[f] = s;
    }
}

int dsac_fetch(dsac_engine* e, int32_t n, dsac_forward_out* o, void* stream_v) {
    if (!e || !o) return DSAC_ERR_ARG;
    if (n < 1 || n > e->cfg.max_frames) return fail(e, DSAC_ERR_CAPACITY, "n_frames %d exceeds engine capacity %d", n, e->cfg.max_frames);
    cudaStream_t stream = (cudaStream_t)stream_v;
    CU(cudaSetDevice(e->cfg.device));
    int rc = fetch_range(e, 0, n, o, stream);
    if (rc != DSAC_OK) return rc;
    CU(cudaStreamSynchronize(stream));
    sum_candidates(e, n, o);
    return DSAC_OK;
}

int dsac_device_view_get(dsac_engine* e, dsac_device_view* v) {
    if (!e || !v) return DSAC_ERR_ARG;
    v->diffmaps = e->d_diffmaps;
    v->hyp_pose = e->d_hyp_pose;
    v->scores = e->d_scores;
    v->sf = e->d_sf;
    v->avg_pose = e->d_avg;
    v->ref_pose = e->d_ref;
    v->img_idx = e->d_img_idx;
    return DSAC_OK;
}

static int forward_submit_impl(dsac_engine* e, int32_t n, int64_t frame0, const int16_t* coords, const int32_t* pix,
                               int32_t pix_shared, const double* gt_jp, dsac_forward_out* out, bool blocking) {
    if (!e) return DSAC_ERR_ARG;
    if (e->pending) return fail(e, DSAC_ERR_ARG, "dsac_forward_submit: the previous submitted pass has not been awaited");
    if (n < 1 || n > e->cfg.max_frames) return fail(e, DSAC_ERR_CAPACITY, "n_frames %d exceeds engine capacity %d", n, e->cfg.max_frames);
    if (!coords || !pix) return fail(e, DSAC_ERR_ARG, "null input");
    CU(cudaSetDevice(e->cfg.device));
    const size_t N = DSAC_N;
    e->cur_coords = e->d_coords;
    e->cur_pix = e->d_pix;
    e->cur_pix_shared = pix_shared;
    e->cur_gt = gt_jp ? e->d_gt : nullptr;
    e->cur_n = n;
    e->dsac_n = 0;
    e->cur_frame0 = frame0;
    cudaStream_t st = e->stream;
    static const bool trace = getenv("DSAC_TRACE") != nullptr;
    cudaEvent_t tev[4];
    const auto t_host0 = std::chrono::steady_clock::now();
    if (trace) for (int k = 0; k < 4; k++) cudaEventCreate(&tev[k]);
    if (pix_shared) CU(cudaMemcpyAsync(e->d_pix, pix, N * 2 * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    if (trace) cudaEventRecord(tev[0], st);
    CU(cudaMemcpyAsync(e->d_coords, coords, (size_t)n * N * 3 * sizeof(int16_t), cudaMemcpyHostToDevice, st));
    if (!pix_shared) CU(cudaMemcpyAsync(e->d_pix, pix, (size_t)n * N * 2 * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    if (gt_jp) CU(cudaMemcpyAsync(e->d_gt, gt_jp, (size_t)n * 12 * sizeof(double), cudaMemcpyHostToDevice, st));
    if (trace) cudaEventRecord(tev[1], st);
    // two lanes (forward_split) for blocking calls in mode 1: with several submitted passes in flight the other pass already
    // fills the GPU; mode 2: always
    int rc = forward_split(e, n, frame0, e->d_coords, e->d_pix, pix_shared, gt_jp ? e->d_gt : nullptr, st,
                           blocking ? e->tail_split >= 1 : e->tail_split >= 2);
    if (trace) cudaEventRecord(tev[2], st);
    if (rc == DSAC_OK && out) rc = fetch_range(e, 0, n, out, st);
    if (rc != DSAC_OK) {   // copies from the caller's host buffers may already be queued: drain before reporting
        cudaStreamSynchronize(st);
        return rc;
    }
    if (trace) cudaEventRecord(tev[3], st);
    e->pending_out = out;
    e->pending_n = n;
    e->pending = true;
    CU(cudaEventRecord(e->ev_fwd, st));
    if (trace) {   // DSAC_TRACE=1: where one pass spends its time; forces the wait
        CU(cudaStreamSynchronize(st));
        float a = 0, b = 0, d = 0;
        cudaEventElapsedTime(&a, tev[0], tev[1]); cudaEventElapsedTime(&b, tev[1], tev[2]); cudaEventElapsedTime(&d, tev[2], tev[3]);
        const double host_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_host0).count();
        fprintf(stderr, "[dsac trace] H2D %.3f ms  kernels %.3f ms  D2H %.3f ms  | call %.3f ms (host wall)\n", a, b, d, host_ms);
        for (int k = 0; k < 4; k++) cudaEventDestroy(tev[k]);
    }
    return DSAC_OK;
}

int dsac_forward_wait(dsac_engine* e) {
    if (!e) return DSAC_ERR_ARG;
    if (!e->pending) return DSAC_OK;
    CU(cudaSetDevice(e->cfg.device));
    e->pending = false;
    CU(cudaStreamSynchronize(e->stream));
    if (e->pending_out) sum_candidates(e, e->pending_n, e->pending_out);
    e->pending_out = nullptr;
    return DSAC_OK;
}

int dsac_forward_submit(dsac_engine* e, int32_t n, int64_t frame0, const int16_t* coords, const int32_t* pix,
                        int32_t pix_shared, const double* gt_jp, dsac_forward_out* out) {
    return forward_submit_impl(e, n, frame0, coords, pix, pix_shared, gt_jp, out, false);
}

int dsac_forward(dsac_engine* e, int32_t n, int64_t frame0, const int16_t* coords, const int32_t* pix,
                 int32_t pix_shared, const double* gt_jp, dsac_forward_out* out) {
    int rc = forward_submit_impl(e, n, frame0, coords, pix, pix_shared, gt_jp, out, true);
    if (rc != DSAC_OK) return rc;
    return dsac_forward_wait(e);
}

int dsac_forward_dsac(dsac_engine* e, int32_t n, int64_t frame0, const int16_t* coords, const int32_t* pix,
                      int32_t pix_shared, const double* gt_jp, int32_t random_draw, dsac_dsac_out* out) {
    if (!e || !out) return DSAC_ERR_ARG;
    if (e->pending) return fail(e, DSAC_ERR_ARG, "dsac_forward_dsac: a submitted pass has not been awaited (dsac_forward_wait)");
    if (n < 1 || n > e->cfg.max_frames) return fail(e, DSAC_ERR_CAPACITY, "n_frames %d exceeds engine capacity %d", n, e->cfg.max_frames);
    if (!coords || !pix) return fail(e, DSAC_ERR_ARG, "null input");
    const dsac_config& c = e->cfg;
    CU(cudaSetDevice(c.device));
    cudaStream_t stream = e->stream;
    const size_t N = DSAC_N, nn = (size_t)n, H = c.n_hyps, jobs = nn * H, T = c.n_streams;
    // refine-all buffers: one block, carved for ra_jobs jobs; the job -> frame table is written when it grows
    if (jobs > e->ra_jobs) {
        e->ra_jobs = 0;
        auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
        const size_t b6 = al(jobs * 6 * sizeof(double)), bd = al(jobs * sizeof(double)), bi = al(jobs * sizeof(int32_t));
        CU(e->ra.reserve(b6 + 3 * bd + 3 * bi));
        char* p = (char*)e->ra.ptr;
        e->d_ra_pose = (double*)p; p += b6;
        e->d_ra_loss = (double*)p; p += bd;
        e->d_ra_rot = (double*)p; p += bd;
        e->d_ra_t = (double*)p; p += bd;
        e->d_ra_frame = (int32_t*)p; p += bi;
        e->d_ra_correct = (int32_t*)p; p += bi;
        e->d_ra_steps = (int32_t*)p;
        std::vector<int32_t> jf(jobs);
        for (size_t j = 0; j < jobs; j++) jf[j] = (int32_t)(j / H);
        CU(cudaMemcpy(e->d_ra_frame, jf.data(), jobs * sizeof(int32_t), cudaMemcpyHostToDevice));
        e->ra_jobs = jobs;
    }
    if (out->inlier_maps) CU(e->ra_imap.reserve(jobs * N * sizeof(int32_t)));
    int32_t* d_ra_imap = out->inlier_maps ? (int32_t*)e->ra_imap.ptr : nullptr;
    CU(cudaMemcpyAsync(e->d_coords, coords, nn * N * 3 * sizeof(int16_t), cudaMemcpyHostToDevice, stream));
    CU(cudaMemcpyAsync(e->d_pix, pix, (pix_shared ? 1 : nn) * N * 2 * sizeof(int32_t), cudaMemcpyHostToDevice, stream));
    if (gt_jp) CU(cudaMemcpyAsync(e->d_gt, gt_jp, nn * 12 * sizeof(double), cudaMemcpyHostToDevice, stream));
    e->cur_coords = e->d_coords; e->cur_pix = e->d_pix; e->cur_pix_shared = pix_shared; e->cur_gt = gt_jp ? e->d_gt : nullptr;
    e->cur_n = 0;   // the soft-argmax backward does not apply to this pass
    e->dsac_n = 0;
    e->cur_frame0 = frame0;
    const uint32_t saved = e->stages;
    e->stages = DSAC_STAGE_SAMPLE | DSAC_STAGE_SCORE;
    int rc = forward_range(e, 0, n, frame0, e->d_coords, e->d_pix, pix_shared, e->cur_gt, stream);
    e->stages = saved;
    if (rc != DSAC_OK) return rc;
    {   // every hypothesis is a refinement job starting from its own pose (cnn.h:1155-1218)
        RefineParams rp;
        memset(&rp, 0, sizeof(rp));
        rp.coords = e->d_coords; rp.pix = e->d_pix; rp.pix_stride = pix_shared ? 0 : DSAC_N * 2;
        rp.perm = e->d_perm;
        rp.f = c.focal; rp.cx = c.cx; rp.cy = c.cy;
        rp.thr = c.thr2d; rp.inlier_count = c.inlier_count; rp.ref_steps = c.ref_steps;
        rp.n_jobs = (int)jobs;
        rp.job_frame = e->d_ra_frame;
        rp.job_init = e->d_hyp_pose;
        rp.out_pose = e->d_ra_pose;
        rp.steps_done = e->d_ra_steps;
        rp.inlier_map = d_ra_imap;
        if (e->cur_gt) {
            rp.gt_jp = e->cur_gt;
            rp.loss = e->d_ra_loss; rp.rot_err = e->d_ra_rot; rp.t_err = e->d_ra_t; rp.correct = e->d_ra_correct;
        }
        k_refine<<<(unsigned)jobs, K4_THREADS, 0, stream>>>(rp);
        e->launches++;
        CU(cudaGetLastError());
    }
    std::vector<double> sf(nn * H), loss(jobs, 0.0), rot(jobs, 0.0), terr(jobs, 0.0);
    std::vector<int32_t> correct(jobs, 0), idx(nn * H * 4);
    std::vector<unsigned long long> endpos(nn * T);
    CU(cudaMemcpyAsync(sf.data(), e->d_sf, nn * H * sizeof(double), cudaMemcpyDeviceToHost, stream));
    CU(cudaMemcpyAsync(idx.data(), e->d_img_idx, nn * H * 4 * sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
    CU(cudaMemcpyAsync(endpos.data(), e->d_stream_endpos, nn * T * sizeof(unsigned long long), cudaMemcpyDeviceToHost, stream));
    if (e->cur_gt) {
        CU(cudaMemcpyAsync(loss.data(), e->d_ra_loss, jobs * sizeof(double), cudaMemcpyDeviceToHost, stream));
        CU(cudaMemcpyAsync(rot.data(), e->d_ra_rot, jobs * sizeof(double), cudaMemcpyDeviceToHost, stream));
        CU(cudaMemcpyAsync(terr.data(), e->d_ra_t, jobs * sizeof(double), cudaMemcpyDeviceToHost, stream));
        CU(cudaMemcpyAsync(correct.data(), e->d_ra_correct, jobs * sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
    }
#define D2H(dst, src, bytes)                                                                    \
    do {                                                                                        \
        if ((dst) && (src)) CU(cudaMemcpyAsync((dst), (src), (bytes), cudaMemcpyDeviceToHost, stream)); \
    } while (0)
    D2H(out->hyp_pose, e->d_hyp_pose, nn * H * 6 * sizeof(double));
    D2H(out->entropy, e->d_entropy, nn * sizeof(double));
    D2H(out->ref_pose, e->d_ra_pose, jobs * 6 * sizeof(double));
    D2H(out->steps_done, e->d_ra_steps, jobs * sizeof(int32_t));
    D2H(out->inlier_maps, d_ra_imap, jobs * N * sizeof(int32_t));
    D2H(out->status, e->d_status, nn * sizeof(uint32_t));
#undef D2H
    CU(cudaStreamSynchronize(stream));
    if (out->sf) memcpy(out->sf, sf.data(), nn * H * sizeof(double));
    if (out->img_idx) memcpy(out->img_idx, idx.data(), nn * H * 4 * sizeof(int32_t));
    if (out->losses) memcpy(out->losses, loss.data(), jobs * sizeof(double));
    for (size_t f = 0; f < nn; f++) {
        const double* p = &sf[f * H];
        // draw(), cnn.h:102-126
        double probSum = 0, maxProb = -1;
        int maxIdx = 0, pick = 0;
        for (size_t i = 0; i < H; i++) {
            if (p[i] < 1e-8) continue;
            probSum += p[i];
            if (maxProb < 0 || p[i] > maxProb) { maxProb = p[i]; maxIdx = (int)i; }
        }
        if (random_draw) {
            // thread 0's generator continues after the sampling loop: same libstdc++ calls as drand (thread_rand.cpp:71-81)
            std::mt19937 gen;
            gen.seed(c.seed + (uint32_t)((frame0 + (long long)f) * (long long)T));
            gen.discard(endpos[f * T]);
            std::uniform_real_distribution<double> dist(0, probSum);
            const double u = dist(gen);
            double cum = 0;
            bool found = false;
            for (size_t i = 0; i < H; i++) {
                if (p[i] < 1e-8) continue;
                cum += p[i];
                pick = (int)i;
                if (cum > u) { found = true; break; }   // std::map::upper_bound on the cumulative sums
            }
            (void)found;
        } else {
            pick = maxIdx;
        }
        double expected = 0;
        for (size_t h = 0; h < H; h++) expected += p[h] * loss[f * H + h];   // expectedMaxLoss, cnn.h:137-151
        if (out->expected_loss) out->expected_loss[f] = expected;
        if (out->hyp_idx) out->hyp_idx[f] = pick;
        if (out->rot_err) out->rot_err[f] = rot[f * H + pick];
        if (out->t_err) out->t_err[f] = terr[f * H + pick];
        if (out->correct) out->correct[f] = correct[f * H + pick];
        if (out->inlier_maps)   // the minimal set is excluded from its own inlier map (cnn.h:1221-1227)
            for (size_t h = 0; h < H; h++)
                for (int j = 0; j < 4; j++) {
                    int cidx = idx[(f * H + h) * 4 + j];
                    if (cidx >= 0) out->inlier_maps[(f * H + h) * N + cidx] = 0;
                }
    }
    e->dsac_n = n;
    return DSAC_OK;
}

int dsac_backward(dsac_engine* e, int32_t n, const int16_t* coords, const int32_t* pix, int32_t pix_shared,
                  const double* gt_jp, dsac_backward_out* out) {
    if (!e || !out) return DSAC_ERR_ARG;
    if (e->pending) return fail(e, DSAC_ERR_ARG, "dsac_backward: a submitted pass has not been awaited (dsac_forward_wait)");
    return backward_run(e, n, coords, pix, pix_shared, gt_jp, out);
}

int dsac_backward_dsac(dsac_engine* e, int32_t n, dsac_backward_dsac_out* out) {
    if (!e || !out) return DSAC_ERR_ARG;
    if (e->pending) return fail(e, DSAC_ERR_ARG, "dsac_backward_dsac: a submitted pass has not been awaited (dsac_forward_wait)");
    return backward_dsac_run(e, n, out);
}

int dsac_gather_patches_device(dsac_engine* e, int32_t n, const uint8_t* d_frames, int32_t width, int32_t height,
                               const int32_t* d_pix, int32_t pix_shared, float mean, float* d_patches, uint32_t* d_status,
                               void* stream_v) {
    if (!e) return DSAC_ERR_ARG;
    if (n < 1 || !d_frames || !d_pix || !d_patches) return fail(e, DSAC_ERR_ARG, "dsac_gather_patches_device: bad arguments");
    if (width < UP_PATCH || height < UP_PATCH) return fail(e, DSAC_ERR_ARG, "frame %dx%d smaller than a %d-pixel patch", width, height, UP_PATCH);
    CU(cudaSetDevice(e->cfg.device));
    cudaStream_t stream = (cudaStream_t)stream_v;
    GatherParams p;
    p.frames = d_frames; p.width = width; p.height = height;
    p.pix = d_pix; p.pix_stride = pix_shared ? 0 : DSAC_N * 2; p.n_cells = DSAC_N;
    p.mean = mean; p.patches = d_patches; p.status = d_status;
    if (d_status) CU(cudaMemsetAsync(d_status, 0, (size_t)n * sizeof(uint32_t), stream));
    k_gather_patches<<<dim3(DSAC_N, n), UP_THREADS, 0, stream>>>(p);
    e->launches++;
    CU(cudaGetLastError());
    return DSAC_OK;
}

int dsac_coords_from_prediction_device(dsac_engine* e, int32_t n, const float* d_prediction, int16_t* d_coords, void* stream_v) {
    if (!e) return DSAC_ERR_ARG;
    if (n < 1 || !d_prediction || !d_coords) return fail(e, DSAC_ERR_ARG, "dsac_coords_from_prediction_device: bad arguments");
    CU(cudaSetDevice(e->cfg.device));
    const size_t count = (size_t)n * DSAC_N * 3;
    k_coords_from_prediction<<<(unsigned)((count + 255) / 256), 256, 0, (cudaStream_t)stream_v>>>(d_prediction, d_coords, count);
    e->launches++;
    CU(cudaGetLastError());
    return DSAC_OK;
}

int dsac_kabsch(dsac_engine* e, int32_t n, int32_t m, const double* a, const double* b, double* R, double* t) {
    if (!e) return DSAC_ERR_ARG;
    return kabsch_run(e, n, m, a, b, R, t);
}

}  // extern "C"

#include "backward_host.inc"
#include "backward_dsac_host.inc"
