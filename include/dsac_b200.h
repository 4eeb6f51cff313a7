/*
 * dsac_b200.h -- C ABI of the B200-native DSAC soft-argmax hypothesis engine.
 *
 * This is the drop-in boundary for the ONE hot path of cvlab-dresden/DSAC
 * (/root/reference/core/cnn_softam.h processImage :960-1180 and the backward assembled in
 * train_ransac_softam.cpp:288-412).  Plain pointers and sizes only -- no CUDA, torch or
 * OpenCV types -- so the reference's C++ drivers (or any FFI) can bind it directly; see
 * INTEGRATION.md for the binding a DSAC maintainer would add.
 *
 * Each entry point cites the reference interface it replaces.
 *
 * Conventions (identical to the reference):
 *   - scene coordinates: int16 millimetres, [frame][y*40+x][3]     (types.h:43-51, cnn_softam.h:265)
 *   - sampling grid:     int32 pixel (x,y), [frame][y*40+x][2]      (cnn_softam.h:283-309)
 *   - "cv pose": 6 doubles (rvec[3], tvec[3] in mm), scene->camera, OpenCV axes (types.h:91)
 *   - "jp pose": 12 doubles (R row-major 3x3, t[3] in mm) after cv2our (types.h:186-214)
 *   - hypothesis h of a frame owns the 4 cells img_idx[h][0..3] = y*40+x (cnn_softam.h:1037)
 *
 * Error behaviour: every call returns 0 on success, <0 on failure (dsac_last_error gives
 * the text); numeric failures are value-encoded per frame exactly like the reference
 * (zero pose on PnP failure, cnn_softam.h:66-71; NaN translation -> 0, types.h:208-211).
 * The engine never falls back to a CPU path: without a CUDA device dsac_engine_create fails.
 */
#ifndef DSAC_B200_H
#define DSAC_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DSAC_GRID 40                      /* CNN_OBJ_PATCHSIZE, lua_calls.h:33 */
#define DSAC_N (DSAC_GRID * DSAC_GRID)    /* 1600 scene coordinates per frame */
#define DSAC_MAXINPUT 100.0f              /* CNN_OBJ_MAXINPUT, lua_calls.h:36 */
#define DSAC_MAX_HYPS 1024
#define DSAC_MAX_REF_STEPS 16

#define DSAC_OK 0
#define DSAC_ERR_ARG (-1)
#define DSAC_ERR_CUDA (-2)
#define DSAC_ERR_CAPACITY (-3)
#define DSAC_ERR_NODEVICE (-4)

/* per-frame status bits (dsac_forward_out.status) */
#define DSAC_ST_SAMPLER_EXHAUSTED 1u      /* max_candidates reached before n_hyps accepts */
#define DSAC_ST_BORDER_PATCH 4u           /* dsac_gather_patches_device met a border cell (the reference would skip it, cnn_softam.h:236-240) */
#define DSAC_ST_REFINE_ABORTED 2u         /* refinement stopped early (<50 inliers / NaN), cnn_softam.h:1136,1147 */

typedef struct dsac_engine dsac_engine;

/* Replaces GlobalProperties::pP / dP as consumed by the drivers
 * (properties.h:40-80, test_ransac_softam.cpp:44-57, train_ransac_softam.cpp:46-66). */
typedef struct dsac_config {
    double focal, cx, cy;     /* getCamMat(), properties.cpp:308-323 */
    int32_t n_hyps;           /* -rI  ransacIterations (256) */
    int32_t thr2d;            /* -rT2D ransacInlierThreshold2D truncated to int (10) */
    int32_t inlier_count;     /* -rB  ransacBatchSize (100) */
    int32_t ref_steps;        /* -rRI ransacRefinementIterations (8) */
    double sub_sample;        /* -rSS ransacSubSample (0.01) */
    double alpha, beta;       /* soft-inlier score s_h = alpha * sum_i sigmoid(beta*(thr2d - e_hi)) */
    uint32_t seed;            /* ThreadRand seed (1305), thread_rand.h:100 */
    int32_t n_streams;        /* sampler streams per frame (= OMP threads of the reference loop) */
    uint32_t stream_skip;     /* raw mt19937 words stream 0 skips first (6400 = stochasticSubSample's drand) */
    int32_t max_candidates;   /* bound on candidates per stream (the reference loops forever) */
    int32_t fix_q4;           /* 0 = bug-compatible dScore column layout (cnn_softam.h:628,641) */
    double grad_clamp;        /* clampE2E of the score backward (train_score_softam.lua:13,97) */
    int32_t write_diffmaps;   /* 1 = materialise the HxN reprojection-error matrix (reference behaviour) */
    int32_t device;           /* CUDA device ordinal */
    int32_t max_frames;       /* frames per call the engine is sized for */
    int32_t hyps_per_cta;     /* scoring tile (hypotheses per CTA); 0 = auto */
} dsac_config;

/* Caller-allocated host outputs of the forward pass; any pointer may be NULL.
 * These are the by-reference outputs of processImage (cnn_softam.h:971-988). */
typedef struct dsac_forward_out {
    double* hyp_pose;         /* [n][H][6]  hyps (cv)                  cnn_softam.h:974 */
    int32_t* img_idx;         /* [n][H][4]  imgIdx                     cnn_softam.h:979 */
    int32_t* cand_idx;        /* [n][H]     index of the accepted candidate in its stream */
    double* scores;           /* [n][H]     scores before softmax      cnn_softam.h:1072 */
    double* sf;               /* [n][H]     sfScores                   cnn_softam.h:981 */
    float* diffmaps;          /* [n][H][N]  diffMaps                   cnn_softam.h:1066 */
    double* entropy;          /* [n]        sfEntropy                  cnn_softam.h:972 */
    double* avg_pose;         /* [n][6]     avgHyp (cv)                cnn_softam.h:976 */
    double* ref_pose;         /* [n][6]     refAvgHyp (cv)             cnn_softam.h:975 */
    int32_t* inlier_map;      /* [n][N]     inlierMap                  cnn_softam.h:985 */
    int32_t* ref_steps_done;  /* [n] */
    int32_t* n_perm_steps;    /* [n]        permutations consumed (non-empty pixelIdxs entries) */
    double* loss;             /* [n]        loss   (needs gt)          cnn_softam.h:971 */
    double* rot_err;          /* [n]        rotErr                     cnn_softam.h:988 */
    double* t_err;            /* [n]        tErr                       cnn_softam.h:987 */
    int32_t* correct;         /* [n]        correct                    cnn_softam.h:973 */
    int64_t* n_candidates;    /* [n]        minimal sets drawn (all streams) */
    uint32_t* status;         /* [n]        DSAC_ST_* */
} dsac_forward_out;

/* Device-side views (valid until the next call on the engine); for zero-copy consumers
 * such as a CNN scorer behind the score seam (lua_calls.h:284-341). */
typedef struct dsac_device_view {
    const float* diffmaps;    /* [n][H][N] or NULL */
    const double* hyp_pose;   /* [n][H][6] */
    const double* scores;     /* [n][H] */
    const double* sf;         /* [n][H] */
    const double* avg_pose;   /* [n][6] */
    const double* ref_pose;   /* [n][6] */
    const int32_t* img_idx;   /* [n][H][4] */
} dsac_device_view;

/* Fills the defaults of GlobalProperties::GlobalProperties() (properties.cpp:39-83). */
int dsac_default_config(dsac_config* cfg);

/* Engine life-cycle.  Replaces the per-process state the drivers set up before the frame
 * loop (test_ransac_softam.cpp:66-82).  One engine per GPU; calls on one engine are not
 * re-entrant, different engines may be driven from different host threads. */
int dsac_engine_create(const dsac_config* cfg, dsac_engine** out);
void dsac_engine_destroy(dsac_engine* e);
const char* dsac_last_error(const dsac_engine* e);   /* e may be NULL: last create error */
int dsac_engine_config(const dsac_engine* e, dsac_config* out);

/* Forward of processImage (cnn_softam.h:960-1180) for n frames, HOST buffers:
 * copies inputs to the device, runs sampling -> HxN reprojection errors -> soft-inlier
 * score -> softmax / soft-argmax -> refinement -> evaluation, copies results back.
 * frame0: global index of the first frame (keys the sampler streams: stream s of frame g
 * is mt19937(seed + g*n_streams + s)), so results do not depend on how a batch is sharded.
 * pix_shared != 0: one sampling grid [N][2] shared by all frames.
 * gt_jp: [n][12] ground-truth jp poses or NULL. */
int dsac_forward(dsac_engine* e, int32_t n_frames, int64_t frame0, const int16_t* coords, const int32_t* pix,
                 int32_t pix_shared, const double* gt_jp, dsac_forward_out* out);

/* The same pass split in two, for drivers that overlap the copies of one batch with the kernels of another
 * (the frame loop of test_ransac_softam.cpp:107-160 with two engines in flight): dsac_forward_submit enqueues
 * H2D -> kernels -> D2H on the engine's streams and returns; dsac_forward_wait blocks until the results are in `out`.
 * coords / pix / gt_jp / out must stay valid (and should be page-locked for the copies to be asynchronous) until the
 * wait returns; one pass per engine may be pending.  dsac_forward == submit + wait. */
int dsac_forward_submit(dsac_engine* e, int32_t n_frames, int64_t frame0, const int16_t* coords, const int32_t* pix,
                        int32_t pix_shared, const double* gt_jp, dsac_forward_out* out);
int dsac_forward_wait(dsac_engine* e);

/* Same pass with inputs already resident in device memory; results stay on the device
 * (dsac_fetch copies them out).  stream: a cudaStream_t cast to void* (NULL = default). */
int dsac_forward_device(dsac_engine* e, int32_t n_frames, int64_t frame0, const int16_t* d_coords,
                        const int32_t* d_pix, int32_t pix_shared, const double* d_gt_jp, void* stream);
int dsac_fetch(dsac_engine* e, int32_t n_frames, dsac_forward_out* out, void* stream);
int dsac_device_view_get(dsac_engine* e, dsac_device_view* view);

/* Stage control for measurement: which stages dsac_forward_device runs. */
#define DSAC_STAGE_SAMPLE 1u
#define DSAC_STAGE_SCORE 2u
#define DSAC_STAGE_REFINE 4u
#define DSAC_STAGE_EVAL 8u
#define DSAC_STAGE_ALL 15u
int dsac_set_stages(dsac_engine* e, uint32_t mask);

/* Which calls may split a batch of at least 768 frames into two lanes (scheduling only, results are identical): two
 * concurrent half-batches, each a complete pass with its own internal streams, whose kernels fill the GPU in each other's
 * gaps.  mode 0: never; 1 (default): dsac_forward and dsac_forward_device; 2: dsac_forward_submit as well. */
int dsac_set_tail_split(dsac_engine* e, int32_t mode);

/* Number of kernels the engine launched since creation (bench.py's gpu_launches). */
int64_t dsac_launch_count(const dsac_engine* e);

/* Measurement aid for the sampler (the round-based pipeline of sampler_split.cuh): with the profile on, the engine records
 * a CUDA event after every sampler launch of a forward pass and counts the candidates per round.
 * dsac_sampler_profile_read waits for the last pass and returns
 *   ms[0..3]     device time in: generation + selection (k1_cells, k1_slot), conservative filter (k1_filter),
 *                full P3P solve (k1_solve), resume tail (k_sample; normally an empty launch);
 *   counts[0..3] candidates generated, candidates flagged by the filter, candidates accepted, rounds that had work. */
int dsac_sampler_profile(dsac_engine* e, int32_t enable);
int dsac_sampler_profile_read(dsac_engine* e, double ms[4], uint64_t counts[4]);
/* Development aid: per stream (first 8 of the last pass), the number of windows the speculative first round of a few streams
 * (k1_spec / k1_stitch, DESIGN.md section 5) stitched; 0 = speculation abandoned (the ordinary round generated the stream) or not used. */
int dsac_debug_spec_result(dsac_engine* e, int32_t out8[8]);

/* Score seam: replaces forward(diffMaps, stateObj) (lua_calls.h:284-300; call site
 * cnn_softam.h:1072).  If set, the engine materialises the diffmaps and calls the hook with
 * DEVICE pointers instead of evaluating the closed-form soft-inlier score.
 * diffmaps [n][H][N] float (row-major 40x40 images, lua_calls.h:98-104), scores [n][H] double. */
typedef int (*dsac_score_hook)(const float* d_diffmaps, int32_t n_frames, int32_t n_hyps, double* d_scores,
                               void* stream, void* user);
int dsac_set_score_hook(dsac_engine* e, dsac_score_hook fn, void* user);

/* The seam's adjoint: replaces backward(maps, stateObj, scoreOutputGradients, gradients) (lua_calls.h:312-341; call site
 * cnn_softam.h:607 in dScore, cnn.h:672 in dSMScore).  Called by dsac_backward / dsac_backward_dsac with DEVICE pointers:
 * the diffmaps of the preceding forward [n][H][N], the score output-gradients [n][H] already clamped to +-grad_clamp
 * (the clamp of train_score_softam.lua:97), and the buffer to fill: diffmap_grads [n][H][40][40] doubles, element (y, x) =
 * d score_h / d diffmap_h(y, x) -- what the reference holds in gradients[c](y, x) after lua_calls.h:326-338.
 * A forward hook and a backward hook must be registered together: with only one of them set the backward entry points
 * return DSAC_ERR_ARG (they would otherwise differentiate a score the forward did not compute). */
typedef int (*dsac_score_backward_hook)(const float* d_diffmaps, const double* d_score_grads, int32_t n_frames, int32_t n_hyps,
                                        double* d_diffmap_grads, void* stream, void* user);
int dsac_set_score_backward_hook(dsac_engine* e, dsac_score_backward_hook fn, void* user);

/* Backward of one training round (train_ransac_softam.cpp:288-394) for the n frames of the
 * preceding dsac_forward call: dLoss/dY, [n][N][3] doubles, row p = y*40+x
 * (what the driver hands to the coordinate-CNN backward, train_ransac_softam.cpp:412).
 * Optional diagnostics may be NULL. */
typedef struct dsac_backward_out {
    double* dloss_dobj;       /* [n][N][3] */
    double* dloss_dref;       /* [n][6]   dLossMax              maxloss.h:87 */
    double* dref_dhyp;        /* [n][36]  dRefineHyp            cnn_softam.h:738 */
    double* dref_dobj;        /* [n][6][N*3] dRefineObj         cnn_softam.h:853 */
    double* score_grads;      /* [n][H]   scoreOutputGradients  train_ransac_softam.cpp:361-376 */
    double* dpnp;             /* [n][H][6][12] dPNP             cnn_softam.h:101 */
} dsac_backward_out;
int dsac_backward(dsac_engine* e, int32_t n_frames, const int16_t* coords, const int32_t* pix, int32_t pix_shared,
                  const double* gt_jp, dsac_backward_out* out);

/* Forward of the DSAC / RANSAC variant (SURVEY.md section 8f row N1): processImage of core/cnn.h:1028-1257 -- same sampling and
 * scoring, then draw() of the winning hypothesis (cnn.h:102-126), refinement of ALL hypotheses, per-hypothesis
 * losses and the expectation of the loss (cnn.h:137-151).  random_draw != 0 draws with the stream-0 generator
 * continuing after the sampler (pP.randomDraw, -rdraw), else arg-max.  Any output may be NULL. */
typedef struct dsac_dsac_out {
    double* hyp_pose;         /* [n][H][6]  hyps                     cnn.h:1042 */
    int32_t* img_idx;         /* [n][H][4]  imgIdx                   cnn.h:1046 */
    double* sf;               /* [n][H]     sfScores                 cnn.h:1048 */
    double* entropy;          /* [n]        sfEntropy                cnn.h:1040 */
    double* ref_pose;         /* [n][H][6]  refHyps                  cnn.h:1043 */
    double* losses;           /* [n][H]     losses                   cnn.h:1052 */
    int32_t* inlier_maps;     /* [n][H][N]  inlierMaps (support cells zeroed, cnn.h:1221-1227) */
    int32_t* steps_done;      /* [n][H] */
    double* expected_loss;    /* [n]        expectedLoss             cnn.h:1039 */
    int32_t* hyp_idx;         /* [n]        hypIdx                   cnn.h:1057 */
    double* rot_err;          /* [n]        of the drawn hypothesis  cnn.h:1056 */
    double* t_err;            /* [n]                                 cnn.h:1055 */
    int32_t* correct;         /* [n]                                 cnn.h:1041 */
    uint32_t* status;         /* [n] */
} dsac_dsac_out;
int dsac_forward_dsac(dsac_engine* e, int32_t n_frames, int64_t frame0, const int16_t* coords, const int32_t* pix,
                      int32_t pix_shared, const double* gt_jp, int32_t random_draw, dsac_dsac_out* out);

/* Backward of the DSAC / RANSAC variant (replaces the gradient block of train_ransac.cpp:304-381; must follow a
 * dsac_forward_dsac over the same n_frames with ground truth):
 *   path I  : sum over the hypotheses with sf_h > 1e-4 of sf_h * dLossMax(refined_h, gt) (maxloss.h:87) * dRefine_h
 *             (cnn.h:866-990: central differences with eps = 2 through refine(), cnn.h:787-852 -- 18 evaluations on the
 *             perturbed minimal set plus 6 per sub-sampled inlier pixel, all of them jobs of the refinement kernel);
 *   path II : dSMScore (cnn.h:726-767) with scoreOutputGradients_i = sf_i * (loss_i - sum_j sf_j loss_j)
 *             (cnn.h:733-741) and the closed-form score backward at the score seam, rows in row-major order.
 * dloss_dobj = path I + path II is what train_ransac.cpp:399 hands to backward() of the coordinate CNN. */
typedef struct dsac_backward_dsac_out {
    double* dloss_dobj;       /* [n][N][3]  dLoss_dObj               train_ransac.cpp:353-377 */
    double* path1;            /* [n][N][3]  nullable */
    double* path2;            /* [n][N][3]  nullable */
    double* score_grads;      /* [n][H]     scoreOutputGradients, nullable  cnn.h:733-741 */
    int32_t* n_selected;      /* [n]        hypotheses with sf > 1e-4, nullable */
    int32_t* n_refine_jobs;   /* [n]        refine() evaluations of path I, nullable */
} dsac_backward_dsac_out;
int dsac_backward_dsac(dsac_engine* e, int32_t n_frames, dsac_backward_dsac_out* out);

/* Upstream step on the device (SURVEY.md section 8f row N3), so that frames never leave HBM between the image and the
 * hypothesis engine.  All pointers are DEVICE pointers; `stream` is a cudaStream_t (NULL: default stream).
 * dsac_gather_patches_device replaces the patch assembly of getCoordImg (cnn_softam.h:221-256) fused with forward()'s
 * normalisation (lua/train_obj.lua:117-124, mean = 127) and pushMaps' layout (lua_calls.h:65-82):
 *   patches[f][cell][c][y][x] = frames[f][oy-21+y][ox-21+x][c] - mean,   (ox, oy) = pix[f or 0][cell]
 * frames: [n][height][width][3] uint8 BGR (jp::img_bgr_t); patches: [n][N][3][42][42] float.  A border cell (which
 * stochasticSubSample never produces) yields a zero patch and DSAC_ST_BORDER_PATCH in status[f] (nullable).
 * dsac_coords_from_prediction_device replaces "modeImg(y,x) = prediction[i] * 1000" (cnn_softam.h:262-268):
 * prediction [n][N][3] float metres -> coords [n][N][3] int16 mm with cv::saturate_cast<short>. */
int dsac_gather_patches_device(dsac_engine* e, int32_t n_frames, const uint8_t* d_frames, int32_t width, int32_t height,
                               const int32_t* d_pix, int32_t pix_shared, float mean, float* d_patches, uint32_t* d_status,
                               void* stream);
int dsac_coords_from_prediction_device(dsac_engine* e, int32_t n_frames, const float* d_prediction, int16_t* d_coords,
                                       void* stream);

/* Batched Kabsch (Hypothesis::calcRigidBodyTransform, Hypothesis.cpp:145-200):
 * for each of n problems with m correspondences, b ~ R a + t.  a,b: [n][m][3] doubles. */
int dsac_kabsch(dsac_engine* e, int32_t n, int32_t m, const double* a, const double* b, double* R /* [n][9] */,
                double* t /* [n][3] */);

/* Host-side helpers that carry the reference's RNG contract (libstdc++ <random>). */
/* stochasticSubSample (cnn_softam.h:283-309) with ThreadRand thread-0 semantics
 * (thread_rand.cpp:40-81): mt19937(seed), 3200 uniform_real draws. */
int dsac_stochastic_subsample(uint32_t seed, int32_t width, int32_t height, int32_t* pix /* [N][2] */);
/* Synthetic frames of SURVEY.md section 8(d): GT pose, 40x40 int16 scene coordinates with inlier
 * ratio rho, inlier noise sigma (mm); sampling grid of frame g from mt19937(seed + g*n_streams).
 * traj != 0: smooth 7Scenes-like camera trajectory instead of i.i.d. poses. */
int dsac_synth_frames(uint32_t data_seed, uint32_t sampler_seed, int32_t n_streams, int64_t frame0, int32_t n_frames,
                      double rho, double sigma, int32_t traj, double focal, double cx, double cy, int16_t* coords,
                      int32_t* pix, double* gt_cv /* [n][6] */, double* gt_jp /* [n][12] */);

const char* dsac_version(void);

#ifdef __cplusplus
}
#endif
#endif
