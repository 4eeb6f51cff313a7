// backward.cuh -- K5/K6: backward of the soft-argmax pipeline, the chain rule assembled in
// train_ransac_softam.cpp:288-394 with the closed-form soft-inlier score in place of the Score CNN:
//
//   path I   dLoss/dY += dLossMax . dRefineObj                      (maxloss.h:87, cnn_softam.h:853)
//            dLoss/dY += dLossMax . dRefineHyp . sum_h sf_h dPNP_h   (cnn_softam.h:738, :101)
//   path II  dLoss/dY += sum_h dScore_h(scoreOutputGradients_h)      (train_ransac_softam.cpp:361-383,
//                                                                     cnn_softam.h:564-646)
//
// dRefineObj / dRefineHyp are central differences through the whole refinement: they are batched
// as jobs of the forward's k_refine kernel (refine.cuh).  dPNP is 24 full P3P solves per
// hypothesis.  dScore keeps a thread per scene coordinate, loops over the hypotheses in
// registers and reduces the per-hypothesis 1x6 with warp shuffles (all fp64, like the reference).
#pragma once
#include <cuda_runtime.h>

#include "device_block.h"
#include "pose_math.cuh"
#include "refine.cuh"

struct dsac_engine;
struct dsac_backward_out;

namespace dsac {

constexpr int BW_MAX_OBJ_PIX = 16;                       // ceil(1600 / skip) with skip = 1/rSS = 100
constexpr int BW_JOBS = 12 + BW_MAX_OBJ_PIX * 6;         // refine jobs per frame (dRefineHyp + dRefineObj)

struct BackwardScratch {
    DeviceBlock block;               // grow-only, owned by the engine
    int n_cap = 0;
    // carved from block
    int32_t* job_frame = nullptr;    // [n][BW_JOBS]
    double* job_init = nullptr;      // [n][BW_JOBS][6]
    int32_t* job_pert = nullptr;     // [n][BW_JOBS][2]
    double* job_pose = nullptr;      // [n][BW_JOBS][6]
    double* job_jp6 = nullptr;       // [n][BW_JOBS][6]
    int32_t* obj_cells = nullptr;    // [n][BW_MAX_OBJ_PIX]  cell of each processed pixel, -1 unused
    double* dl = nullptr;            // [n][6]   dLossMax
    double* dldavg = nullptr;        // [n][6]   dLossMax . dRefineHyp
    double* drefhyp = nullptr;       // [n][36]
    double* sog = nullptr;           // [n][H]   scoreOutputGradients
    double* dpnp = nullptr;          // [n][H][72]
    double* hypjp = nullptr;         // [n][H][39]  R(9) t(3) J(27) of every hypothesis in jp convention
    double* row = nullptr;           // [n][N*3]  dLoss_dObj_1row
    double* drefobj = nullptr;       // [n][6][N*3] (diagnostic, optional)
    double* part = nullptr;          // [n][groups][N*3] partial rows of k_dscore
    int groups = 1;
};

// Hypothesis(cv2our(pose)).getRodVecAndTrans()  (Hypothesis.cpp:274-290)
__device__ __forceinline__ void jp6_from_cv_dev(const double pose[6], double out[6]) {
    double R[9], t[3];
    cv2our_dev(pose, R, t);
    rodrigues_m2v(R, out);
    out[3] = t[0]; out[4] = t[1]; out[5] = t[2];
}

// dLossMax, maxloss.h:87-198
__device__ void dloss_max_dev(const double est[6], const double gt[6], double jac[6]) {
    for (int i = 0; i < 6; i++) jac[i] = 0;
    double rot1[9], rot2[9], dRod[27];
    rodrigues_jac(est, rot1, dRod);
    rodrigues_v2m(gt, rot2);
    double diag = 0;  // trace(rot1 * rot2^T)
    for (int i = 0; i < 3; i++)
        for (int k = 0; k < 3; k++) diag += rot1[i * 3 + k] * rot2[i * 3 + k];
    double trace = fmin(3.0, fmax(-1.0, diag));
    double rotErr = 180 * acos((trace - 1.0) / 2.0) / kPi;
    double a1[3] = {-est[3] / 10, -est[4] / 10, -est[5] / 10}, a2[3] = {-gt[3] / 10, -gt[4] / 10, -gt[5] / 10};
    double invT1[3], invT2[3];
    for (int r = 0; r < 3; r++) {  // invRot = rot^T
        invT1[r] = rot1[0 * 3 + r] * a1[0] + rot1[1 * 3 + r] * a1[1] + rot1[2 * 3 + r] * a1[2];
        invT2[r] = rot2[0 * 3 + r] * a2[0] + rot2[1 * 3 + r] * a2[1] + rot2[2 * 3 + r] * a2[2];
    }
    double d[3] = {invT1[0] - invT2[0], invT1[1] - invT2[1], invT1[2] - invT2[2]};
    double tErr = sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
    if (fmax(rotErr, tErr) > 10000000.0) return;
    if ((tErr + rotErr) < 1e-8) return;
    if (tErr > rotErr) {
        double dDist[3] = {d[0] / tErr, d[1] / tErr, d[2] / tErr};
        // cols 3..5 = dDist * (-invRot1), invRot1[i][j] = rot1[j][i]
        for (int j = 0; j < 3; j++) jac[3 + j] = -(dDist[0] * rot1[j * 3 + 0] + dDist[1] * rot1[j * 3 + 1] + dDist[2] * rot1[j * 3 + 2]);
        // dInvT1_dInvRot1 (3x9): row r has a1[0], a1[1], a1[2] at columns r, 3+r, 6+r   (maxloss.h:146-158)
        double v9[9];
        for (int k = 0; k < 9; k++) v9[k] = dDist[k % 3] * a1[k / 3];
        for (int j = 0; j < 3; j++) {
            double s = 0;
            for (int k = 0; k < 9; k++) s += v9[k] * dRod[j * 9 + k];
            jac[j] = s;
        }
    } else {
        // dTrace * dRotDiff: v9[k] = sum over the three diagonal blocks of invRot2 (maxloss.h:168-188)
        double v9[9];
        for (int blk = 0; blk < 3; blk++)
            for (int r = 0; r < 3; r++) v9[blk * 3 + r] = rot2[blk * 3 + r];  // invRot2[r][blk] = rot2[blk][r]
        double coef = 180 / kPi * -1 / sqrt(3 - trace * trace + 2 * trace);
        for (int j = 0; j < 3; j++) {
            double s = 0;
            for (int k = 0; k < 9; k++) s += v9[k] * dRod[j * 9 + k];
            jac[j] = coef * s;
        }
    }
    for (int i = 0; i < 6; i++)
        if (jac[i] != jac[i]) {
            for (int k = 0; k < 6; k++) jac[k] = 0;
            return;
        }
}

struct BwParams {
    const int16_t* coords;
    const int32_t* pix;
    int pix_stride;
    const double* gt_jp;        // [n][12]
    double f, cx, cy;
    int H, thr, skip, fix_q4;
    double alpha, beta, grad_clamp;
    // forward state
    const double* hyp_pose;     // [n][H][6]
    const int32_t* img_idx;     // [n][H][4]
    const double* sf;           // [n][H]
    const double* avg_pose;     // [n][6]
    const double* ref_pose;     // [n][6]
    const int32_t* inlier_map;  // [n][N]
    BackwardScratch s;
    // k_dscore splits the hypotheses of a frame over `groups` CTAs; group g accumulates into part[frame][g][N*3]
    // (zeroed by the caller) and k_dscore_reduce adds the groups to s.row in order
    double* part;
    int groups;
    // score seam, adjoint side (lua_calls.h:312-341): when set, dScore/dDiffMap of every hypothesis comes from the
    // registered backward hook -- [n][H][40][40] doubles, element (y, x) as the reference's gradients[c](y, x) -- instead
    // of the closed-form derivative of the soft-inlier score
    const double* ext_g;
};

// ------------------------------------------------------------------ DSAC / RANSAC variant (train_ransac.cpp:304-381)
// dRefine of hypothesis h (cnn.h:866-990) is a list of refine() evaluations (cnn.h:787-852); each is one k_refine job.
// The jobs that perturb a minimal-set point start from the P3P pose of the PERTURBED set: this kernel computes it.
struct DsacBwParams {
    const int16_t* coords;
    const int32_t* pix;
    int pix_stride;
    double f, cx, cy;
    int H;
    const int32_t* img_idx;     // [n][H][4]
    const double* ref_pose;     // [n*H][6] refined cv pose of every hypothesis (forward_dsac)
    const double* sf;           // [n*H]
    const double* gt_jp;        // [n][12]
    // jobs
    int n_jobs;
    const int32_t* job_frame;   // [n_jobs]
    const int32_t* job_p3p;     // [n_jobs][3] {global hypothesis index or -1, point*3+channel, delta}
    double* job_init;           // [n_jobs][6]
    const double* job_jp6;      // [n_jobs][6] results of k_refine
    // central-difference pairs (jobs 2p, 2p+1 = forward, backward step), sorted by frame, hypothesis
    int n_frames;
    const int32_t* frame_pair_begin;   // [n+1]
    const int32_t* pair_hyp;    // [n_pairs] global hypothesis index
    const int32_t* pair_col;    // [n_pairs] cell*3+channel
    const int32_t* pair_scale;  // [n_pairs] 1 or skip
    double* path1;              // [n][N*3]
};

__global__ void k_dsac_job_p3p(DsacBwParams p) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= p.n_jobs) return;
    const int hyp = p.job_p3p[j * 3];
    if (hyp < 0) return;
    const int frame = p.job_frame[j];
    const int16_t* coords = p.coords + (size_t)frame * DSAC_N_CONST * 3;
    const int32_t* pix = p.pix + (size_t)frame * p.pix_stride;
    const int32_t* idx = p.img_idx + (size_t)hyp * 4;
    float obj[12], img[8];
    for (int q = 0; q < 4; q++) {
        const int c = idx[q];
        img[q * 2] = (float)pix[c * 2];
        img[q * 2 + 1] = (float)pix[c * 2 + 1];
        for (int k = 0; k < 3; k++) obj[q * 3 + k] = (float)coords[c * 3 + k];
    }
    obj[p.job_p3p[j * 3 + 1]] += (float)p.job_p3p[j * 3 + 2];   // objPts[pt] +/- eps (integers in float: exact)
    double pose[6], R[9], t[3], e2;
    P3PProblem pr;
    make_problem(obj, img, p.f, p.cx, p.cy, pr);
    if (p3p_best(pr, p.f, p.cx, p.cy, R, t, &e2) > 0) {
        rodrigues_m2v(R, pose);
        pose[3] = t[0]; pose[4] = t[1]; pose[5] = t[2];
    } else {
        for (int k = 0; k < 6; k++) pose[k] = 0;   // safeSolvePnP leaves a zero pose (cnn.h:66-71)
    }
    for (int k = 0; k < 6; k++) p.job_init[(size_t)j * 6 + k] = pose[k];
}

// path I: dLoss_dObj(idx, c) += sf_h * (dLossMax(refined_h, gt) . dRefine_h)(idx*3+c), hypotheses and columns in the
// reference's order (one thread per frame: the sums are reproducible)
// path I of the DSAC variant: row[col] += sf_h * dLossMax_h . (refine(+eps) - refine(-eps)) / (2 eps) * scale over the
// central-difference pairs of a frame, in pair order (pairs are sorted by hypothesis; a hypothesis touches a column at
// most once, so within one hypothesis' run the additions are independent, and the runs are applied one after the other).
// One warp per frame: first the lanes evaluate dLossMax of the frame's selected hypotheses in parallel, then the runs
// are walked in order with the lanes spread over a run's pairs.
constexpr int DSAC_COMBINE_MAX_HYPS = 1024;   // = DSAC_MAX_HYPS
__global__ void __launch_bounds__(32) k_dsac_combine(DsacBwParams p) {
    __shared__ int s_run_begin[DSAC_COMBINE_MAX_HYPS + 1];
    __shared__ double s_dl[32][7];                       // dLossMax (1x6) and sf of 32 runs' hypotheses at a time
    const int frame = blockIdx.x, lane = threadIdx.x;
    if (frame >= p.n_frames) return;
    double* row = p.path1 + (size_t)frame * DSAC_N_CONST * 3;
    const int q_begin = p.frame_pair_begin[frame], q_end = p.frame_pair_begin[frame + 1];
    // runs of equal hypothesis
    int n_runs = 0;
    for (int q0 = q_begin; q0 < q_end; q0 += 32) {
        const int q = q0 + lane;
        const bool start = q < q_end && (q == q_begin || p.pair_hyp[q] != p.pair_hyp[q - 1]);
        const unsigned m = __ballot_sync(0xffffffffu, start);
        if (start) {
            const int r = n_runs + __popc(m & ((1u << lane) - 1u));
            if (r < DSAC_COMBINE_MAX_HYPS) s_run_begin[r] = q;
        }
        n_runs += __popc(m);
    }
    n_runs = min(n_runs, DSAC_COMBINE_MAX_HYPS);
    if (lane == 0) s_run_begin[n_runs] = q_end;
    __syncwarp();
    // dLossMax of every run's hypothesis
    const double* g = p.gt_jp + (size_t)frame * 12;
    double gt6[6];
    rodrigues_m2v(g, gt6);
    gt6[3] = g[9]; gt6[4] = g[10]; gt6[5] = g[11];
    for (int r0 = 0; r0 < n_runs; r0 += 32) {
        if (r0 + lane < n_runs) {
            const int hyp = p.pair_hyp[s_run_begin[r0 + lane]];
            double ref6[6], dl[6];
            jp6_from_cv_dev(p.ref_pose + (size_t)hyp * 6, ref6);
            dloss_max_dev(ref6, gt6, dl);
            for (int k = 0; k < 6; k++) s_dl[lane][k] = dl[k];
            s_dl[lane][6] = p.sf[hyp];
        }
        __syncwarp();
        for (int r = r0; r < min(n_runs, r0 + 32); r++) {
            const double sf = s_dl[r - r0][6];
            for (int q = s_run_begin[r] + lane; q < s_run_begin[r + 1]; q += 32) {
                const double* fS = p.job_jp6 + (size_t)(2 * q) * 6;
                const double* bS = fS + 6;
                const double scale = (double)p.pair_scale[q];
                double acc = 0;
                for (int k = 0; k < 6; k++) acc += s_dl[r - r0][k] * ((fS[k] - bS[k]) / 4.0 * scale);   // / (2 * eps), eps = 2; * skip
                row[p.pair_col[q]] += sf * acc;
            }
            __syncwarp();   // the next run may touch the same columns
        }
    }
}


// ---- per frame: dLossMax and the refine job list (one warp, lane 0 does the serial scan)
__global__ void k_bw_prep(BwParams p, int n) {
    const int frame = blockIdx.x * blockDim.x + threadIdx.x;
    if (frame >= n) return;
    // dLoss/dRefinedPose
    double ref6[6], gt6[6], dl[6];
    jp6_from_cv_dev(p.ref_pose + (size_t)frame * 6, ref6);
    const double* g = p.gt_jp + (size_t)frame * 12;
    rodrigues_m2v(g, gt6);  // poseGT.getRodVecAndTrans()
    gt6[3] = g[9]; gt6[4] = g[10]; gt6[5] = g[11];
    dloss_max_dev(ref6, gt6, dl);
    for (int k = 0; k < 6; k++) p.s.dl[(size_t)frame * 6 + k] = dl[k];
    // jobs 0..11: dRefineHyp (cnn_softam.h:756-833): +-eps on the cv rvec (eps = 0.001f) / cv tvec (eps*1000)
    int32_t* jf = p.s.job_frame + (size_t)frame * BW_JOBS;
    double* ji = p.s.job_init + (size_t)frame * BW_JOBS * 6;
    int32_t* jp = p.s.job_pert + (size_t)frame * BW_JOBS * 2;
    const double* avg = p.avg_pose + (size_t)frame * 6;
    const float eps = 0.001f;
    for (int i = 0; i < 6; i++) {
        double init[6];
        for (int k = 0; k < 6; k++) init[k] = avg[k];
        // the reference perturbs one shared copy in place: +eps, -2eps, +eps (the residue of earlier
        // parameters is below double rounding of these magnitudes only by luck, so replay it exactly)
        for (int q = 0; q < i; q++) {
            if (q < 3) { init[q] += eps; init[q] -= 2 * eps; init[q] += eps; }
            else { init[q] += eps * 1000; init[q] -= 2 * eps * 1000; init[q] += eps * 1000; }
        }
        double fwd = init[i], bwd;
        if (i < 3) { fwd += eps; bwd = fwd; bwd -= 2 * eps; }
        else { fwd += eps * 1000; bwd = fwd; bwd -= 2 * eps * 1000; }
        for (int sgn = 0; sgn < 2; sgn++) {
            int j = i * 2 + sgn;
            jf[j] = frame;
            for (int k = 0; k < 6; k++) ji[j * 6 + k] = init[k];
            ji[j * 6 + i] = sgn ? bwd : fwd;
            jp[j * 2] = -1; jp[j * 2 + 1] = 0;
        }
    }
    // jobs 12..: dRefineObj (cnn_softam.h:866-920): every skip-th ever-inlier pixel, x outer / y inner
    const int32_t* im = p.inlier_map + (size_t)frame * DSAC_N_CONST;
    int32_t* oc = p.s.obj_cells + (size_t)frame * BW_MAX_OBJ_PIX;
    int inCount = 0, npx = 0;
    for (int x = 0; x < DSAC_GRID_CONST; x++)
        for (int y = 0; y < DSAC_GRID_CONST; y++) {
            if (im[y * DSAC_GRID_CONST + x] == 0) continue;
            inCount++;
            if (inCount % p.skip != 0) continue;
            if (npx < BW_MAX_OBJ_PIX) oc[npx++] = y * DSAC_GRID_CONST + x;
        }
    for (int k = npx; k < BW_MAX_OBJ_PIX; k++) oc[k] = -1;
    for (int px = 0; px < BW_MAX_OBJ_PIX; px++)
        for (int c = 0; c < 3; c++)
            for (int sgn = 0; sgn < 2; sgn++) {
                int j = 12 + (px * 3 + c) * 2 + sgn;
                if (px < npx) {
                    jf[j] = frame;
                    for (int k = 0; k < 6; k++) ji[j * 6 + k] = avg[k];
                    jp[j * 2] = oc[px] * 3 + c;
                    jp[j * 2 + 1] = sgn ? -2 : 2;   // short += eps (2.f), then -= 2*eps  (cnn_softam.h:887,901)
                } else {
                    jf[j] = -1;
                    jp[j * 2] = -1; jp[j * 2 + 1] = 0;
                }
            }
}

// ---- per frame (one warp): dRefineHyp, dLossMax . dRefineObj into the row, scoreOutputGradients
__global__ void k_bw_combine(BwParams p, int n) {
    const int frame = blockIdx.x, lane = threadIdx.x;
    if (frame >= n) return;
    __shared__ double s_dref[36], s_dl[6], s_dldavg[6];
    const double* jp6 = p.s.job_jp6 + (size_t)frame * BW_JOBS * 6;
    const float eps = 0.001f;
    if (lane < 6) s_dl[lane] = p.s.dl[(size_t)frame * 6 + lane];
    if (lane < 6) {
        const int i = lane;
        const double* fS = jp6 + (i * 2) * 6;
        const double* bS = jp6 + (i * 2 + 1) * 6;
        for (int k = 0; k < 3; k++) s_dref[k * 6 + i] = (fS[k] - bS[k]) / (2 * eps);
        for (int k = 3; k < 6; k++) s_dref[k * 6 + i] = (fS[k] - bS[k]) / (2 * eps * 1000);
    }
    __syncwarp();
    if (lane < 6) {
        double s = 0;
        for (int k = 0; k < 6; k++) s += s_dl[k] * s_dref[k * 6 + lane];
        s_dldavg[lane] = s;
        p.s.dldavg[(size_t)frame * 6 + lane] = s;
    }
    for (int k = lane; k < 36; k += 32) p.s.drefhyp[(size_t)frame * 36 + k] = s_dref[k];
    __syncwarp();
    // dRefineObj columns -> row (and the optional 6 x 4800 diagnostic matrix)
    double* row = p.s.row + (size_t)frame * DSAC_N_CONST * 3;
    const int32_t* oc = p.s.obj_cells + (size_t)frame * BW_MAX_OBJ_PIX;
    for (int col = lane; col < BW_MAX_OBJ_PIX * 3; col += 32) {
        const int px = col / 3, c = col % 3;
        if (oc[px] < 0) continue;
        const double* fS = jp6 + (12 + col * 2) * 6;
        const double* bS = jp6 + (12 + col * 2 + 1) * 6;
        const float eps2 = 2.f;
        double s = 0;
        for (int k = 0; k < 6; k++) {
            double v = (fS[k] - bS[k]) / (2 * eps2) * p.skip;   // cnn_softam.h:918
            s += s_dl[k] * v;
            if (p.s.drefobj) p.s.drefobj[((size_t)frame * 6 + k) * DSAC_N_CONST * 3 + oc[px] * 3 + c] = v;
        }
        row[oc[px] * 3 + c] += s;   // distinct cells: no conflicts
    }
    __syncwarp();
    // scoreOutputGradients (train_ransac_softam.cpp:361-376): g_j = sf_j (hf_j - sum_h sf_h hf_h)
    const double* hp = p.hyp_pose + (size_t)frame * p.H * 6;
    const double* sf = p.sf + (size_t)frame * p.H;
    double part = 0;
    for (int h = lane; h < p.H; h += 32) {
        double hf = 0;
        for (int i = 0; i < 3; i++) hf += s_dldavg[i] * hp[h * 6 + i] + s_dldavg[3 + i] * (hp[h * 6 + 3 + i] / 1000);
        part += sf[h] * hf;
    }
    for (int off = 16; off; off >>= 1) part += __shfl_xor_sync(0xffffffffu, part, off);
    for (int h = lane; h < p.H; h += 32) {
        double hf = 0;
        for (int i = 0; i < 3; i++) hf += s_dldavg[i] * hp[h * 6 + i] + s_dldavg[3 + i] * (hp[h * 6 + 3 + i] / 1000);
        p.s.sog[(size_t)frame * p.H + h] = sf[h] * hf - sf[h] * part;
    }
}

// ---- dPNP (cnn_softam.h:101-146): thread = (hypothesis, column 0..11); 2 full P3P solves each.
// Also prepares the jp pose + Rodrigues Jacobian of every hypothesis for k_dscore.
__global__ void __launch_bounds__(192) k_dpnp(BwParams p) {
    const int frame = blockIdx.y;
    const int h = blockIdx.x * 16 + threadIdx.x / 12, col = threadIdx.x % 12;
    __shared__ int s_nan[16];
    if (threadIdx.x < 16) s_nan[threadIdx.x] = 0;
    __syncthreads();
    const bool active = h < p.H;
    double colv[6] = {0, 0, 0, 0, 0, 0};
    if (active) {
        const int16_t* coords = p.coords + (size_t)frame * DSAC_N_CONST * 3;
        const int32_t* pix = p.pix + (size_t)frame * p.pix_stride;
        const int32_t* idx = p.img_idx + ((size_t)frame * p.H + h) * 4;
        float obj[12], img[8];
        bool valid = true;
        for (int j = 0; j < 4; j++) {
            int c = idx[j];
            if (c < 0) { valid = false; c = 0; }
            img[j * 2] = (float)pix[c * 2];
            img[j * 2 + 1] = (float)pix[c * 2 + 1];
            for (int k = 0; k < 3; k++) obj[j * 3 + k] = (float)coords[c * 3 + k];
        }
        const float eps = 0.1f;
        // columns before `col` were perturbed and restored in float by the reference's serial loop
        for (int q = 0; q < col; q++) {
            obj[q] += eps;
            obj[q] -= 2 * eps;
            obj[q] += eps;
        }
        double fS[6], bS[6], pose[6], R[9], t[3], e2;
        P3PProblem pr;
        obj[col] += eps;
        make_problem(obj, img, p.f, p.cx, p.cy, pr);
        if (valid && p3p_best(pr, p.f, p.cx, p.cy, R, t, &e2) > 0) {
            rodrigues_m2v(R, pose);
            pose[3] = t[0]; pose[4] = t[1]; pose[5] = t[2];
        } else {
            for (int k = 0; k < 6; k++) pose[k] = 0;  // safeSolvePnP, cnn_softam.h:66-71
        }
        jp6_from_cv_dev(pose, fS);
        obj[col] -= 2 * eps;
        make_problem(obj, img, p.f, p.cx, p.cy, pr);
        if (valid && p3p_best(pr, p.f, p.cx, p.cy, R, t, &e2) > 0) {
            rodrigues_m2v(R, pose);
            pose[3] = t[0]; pose[4] = t[1]; pose[5] = t[2];
        } else {
            for (int k = 0; k < 6; k++) pose[k] = 0;
        }
        jp6_from_cv_dev(pose, bS);
        bool nan = false;
        for (int k = 0; k < 6; k++) {
            colv[k] = (fS[k] - bS[k]) / (2 * eps);
            if (colv[k] != colv[k]) nan = true;
        }
        if (nan) s_nan[threadIdx.x / 12] = 1;
    }
    __syncthreads();
    if (active) {
        // a NaN in column c makes the reference return zeros(6,12) at that point of its serial loop
        const bool zero = s_nan[threadIdx.x / 12] != 0;
        double* out = p.s.dpnp + ((size_t)frame * p.H + h) * 72;
        for (int k = 0; k < 6; k++) out[k * 12 + col] = zero ? 0.0 : colv[k];
        if (col == 0) {  // jp pose + Rodrigues Jacobian of this hypothesis (dScore re-solves the same P3P: cnn_softam.h:597-598)
            double* hj = p.s.hypjp + ((size_t)frame * p.H + h) * 39;
            double R[9], t[3], rod[3], Rt[9], J[27];
            cv2our_dev(p.hyp_pose + ((size_t)frame * p.H + h) * 6, R, t);
            rodrigues_m2v(R, rod);
            rodrigues_jac(rod, Rt, J);
            for (int k = 0; k < 9; k++) hj[k] = R[k];
            for (int k = 0; k < 3; k++) hj[9 + k] = t[k];
            for (int k = 0; k < 27; k++) hj[12 + k] = J[k];
        }
    }
}

// ---- per frame (one warp): row += dLdAvg . sum_h sf_h dPNP_h scattered to the support points
//      (train_ransac_softam.cpp:340-353); hypotheses in order, so the sums are reproducible
__global__ void k_bw_scatter_pnp(BwParams p, int n) {
    const int frame = blockIdx.x, lane = threadIdx.x;
    if (frame >= n || lane >= 12) return;
    double* row = p.s.row + (size_t)frame * DSAC_N_CONST * 3;
    const double* dld = p.s.dldavg + (size_t)frame * 6;
    double w[6];
    for (int k = 0; k < 6; k++) w[k] = dld[k];
    for (int h = 0; h < p.H; h++) {
        const int32_t* idx = p.img_idx + ((size_t)frame * p.H + h) * 4;
        const int c = idx[lane / 3];
        const double* J = p.s.dpnp + ((size_t)frame * p.H + h) * 72;
        double s = 0;
        for (int k = 0; k < 6; k++) s += w[k] * (p.sf[(size_t)frame * p.H + h] * J[k * 12 + lane]);
        if (c >= 0) row[c * 3 + lane % 3] += s;
        __syncwarp(0xfff);
    }
}

// ---- dScore (cnn_softam.h:564-646): thread = scene coordinate, loop over a group of the frame's hypotheses.
// grid (groups, frames): with one CTA per frame a training batch of 16..64 frames left most of the 148 SMs idle for the
// dominant kernel of the backward pass.  Every addition into a group's partial row is ordered (barriers of the h loop),
// and the groups are added in order, so the gradient is run-to-run reproducible.
constexpr int K5_THREADS = 320, K5_PTS = 5, K5_WARPS = K5_THREADS / 32;
constexpr int K5_MAX_GROUPS = 32;

// hypothesis groups for n frames: enough CTAs for ~4 per SM, at most K5_MAX_GROUPS, at least 8 hypotheses each
inline int dscore_groups(int n_frames, int n_hyps, int sm_count) {
    int g = (4 * sm_count + n_frames - 1) / std::max(1, n_frames);
    g = std::min(g, K5_MAX_GROUPS);
    g = std::min(g, std::max(1, n_hyps / 8));
    return std::max(1, g);
}

// scoreOutputGradients clamped to +-clamp, as the reference's score backward does before back-propagating
// (train_score_softam.lua:97) -- the copy a registered backward hook receives
__global__ void k_clamp_copy(const double* __restrict__ src, double* __restrict__ dst, size_t count, double clamp) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    double v = src[i];
    if (clamp > 0) v = fmax(-clamp, fmin(clamp, v));
    dst[i] = v;
}

__global__ void k_dscore_reduce(BwParams p) {
    const int frame = blockIdx.x;
    double* row = p.s.row + (size_t)frame * DSAC_N_CONST * 3;
    const double* part = p.part + (size_t)frame * p.groups * DSAC_N_CONST * 3;
    for (int c = threadIdx.x; c < DSAC_N_CONST * 3; c += blockDim.x) {
        double s = row[c];
        for (int g = 0; g < p.groups; g++) s += part[(size_t)g * DSAC_N_CONST * 3 + c];
        row[c] = s;
    }
}

__global__ void __launch_bounds__(K5_THREADS) k_dscore(BwParams p) {
    __shared__ double s_h[39];
    __shared__ double s_red[K5_WARPS][6];
    __shared__ double s_w[6];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int frame = blockIdx.y, group = blockIdx.x;
    const int per_group = (p.H + p.groups - 1) / p.groups, h_begin = group * per_group, h_end = min(p.H, h_begin + per_group);
    const int16_t* coords = p.coords + (size_t)frame * DSAC_N_CONST * 3;
    const int32_t* pix = p.pix + (size_t)frame * p.pix_stride;
    double* row = p.part + ((size_t)frame * p.groups + group) * DSAC_N_CONST * 3;
    double X[K5_PTS], Y[K5_PTS], Z[K5_PTS], pu[K5_PTS], pv[K5_PTS], acc[K5_PTS][3];
#pragma unroll
    for (int j = 0; j < K5_PTS; j++) {
        int pt = tid + j * K5_THREADS;
        X[j] = (double)(float)coords[pt * 3]; Y[j] = (double)(float)coords[pt * 3 + 1]; Z[j] = (double)(float)coords[pt * 3 + 2];
        pu[j] = (double)(float)pix[pt * 2]; pv[j] = (double)(float)pix[pt * 2 + 1];
        acc[j][0] = acc[j][1] = acc[j][2] = 0;
    }
    const double f = p.f, cx = p.cx, cy = p.cy;
    for (int h = h_begin; h < h_end; h++) {
        __syncthreads();
        if (tid < 39) s_h[tid] = p.s.hypjp[((size_t)frame * p.H + h) * 39 + tid];
        __syncthreads();
        double go = p.s.sog[(size_t)frame * p.H + h];
        if (p.grad_clamp > 0) go = fmax(-p.grad_clamp, fmin(p.grad_clamp, go));   // train_score_softam.lua:97
        const double* R = s_h;       // jp rotation
        const double* t = s_h + 9;
        const double* J = s_h + 12;  // 3x9 Rodrigues Jacobian at rod(R)
        // cv pose of the same hypothesis for the reprojection-error image (getDiffMap on cvHyp, cnn_softam.h:601):
        // cv R = diag(1,-1,-1) R_jp, cv t = (t0,-t1,-t2)  (cv2our never flips for a proper rotation)
        double w6[6] = {0, 0, 0, 0, 0, 0};
#pragma unroll
        for (int j = 0; j < K5_PTS; j++) {
            // --- diffmap entry with the reference's roundings (projection -> float, float diff, double norm, float store)
            double xc = dot3_plain(R[0], X[j], R[1], Y[j], R[2], Z[j], t[0]);
            double yc = dot3_plain(-R[3], X[j], -R[4], Y[j], -R[5], Z[j], -t[1]);
            double zc = dot3_plain(-R[6], X[j], -R[7], Y[j], -R[8], Z[j], -t[2]);
            double iz = zc ? __ddiv_rn(1., zc) : 1;
            float pfu = (float)__dadd_rn(__dmul_rn(__dmul_rn(xc, iz), f), cx), pfv = (float)__dadd_rn(__dmul_rn(__dmul_rn(yc, iz), f), cy);
            float du = __fsub_rn((float)pu[j], pfu), dv = __fsub_rn((float)pv[j], pfv);
            double e = (double)(float)fmin(sqrt(__dadd_rn(__dmul_rn((double)du, (double)du), __dmul_rn((double)dv, (double)dv))), 100.0);
            double g;
            if (p.ext_g) {
                g = p.ext_g[((size_t)frame * p.H + h) * DSAC_N_CONST + tid + j * K5_THREADS];   // backward hook's dDiffMaps[h](y,x)
            } else {
                double sg = 1.0 / (1.0 + exp(-p.beta * ((double)p.thr - e)));
                g = go * (-p.alpha * p.beta * sg * (1.0 - sg));   // dDiffMaps[h](y,x) under the soft-inlier score
            }
            // --- dProjectdObj / dProjectdHyp in the jp convention (cnn_softam.h:404-528)
            double ex = R[0] * X[j] + R[1] * Y[j] + R[2] * Z[j] + t[0];
            double ey = R[3] * X[j] + R[4] * Y[j] + R[5] * Z[j] + t[1];
            double ez = R[6] * X[j] + R[7] * Y[j] + R[8] * Z[j] + t[2];
            if (fabs(ez) < 1e-8) continue;
            double px = -f * ex / ez + cx, py = f * ey / ez + cy;
            double err = sqrt((pu[j] - px) * (pu[j] - px) + (pv[j] - py) * (pv[j] - py));
            if (err > 100.0) continue;
            err += 1e-8;
            double ddx = pu[j] - px, ddy = pv[j] - py;
#pragma unroll
            for (int k = 0; k < 3; k++) {
                double pxd = -f * R[0 * 3 + k] / ez + f * ex / ez / ez * R[2 * 3 + k];
                double pyd = f * R[1 * 3 + k] / ez - f * ey / ez / ez * R[2 * 3 + k];
                acc[j][k] += g * (0.5 / err * (2 * ddx * -pxd + 2 * ddy * -pyd));
            }
            double dN0 = -1 / err * ddx, dN1 = -1 / err * ddy;
            double Xv[3] = {X[j], Y[j], Z[j]};
            double v9[9];
#pragma unroll
            for (int k = 0; k < 3; k++) {
                v9[k] = dN0 * (-f * Xv[k] / ez);
                v9[3 + k] = dN1 * (f * Xv[k] / ez);
                v9[6 + k] = dN0 * (f * ex / ez / ez * Xv[k]) + dN1 * (-f * ey / ez / ez * Xv[k]);
            }
#pragma unroll
            for (int m = 0; m < 3; m++) {
                double s = 0;
#pragma unroll
                for (int k = 0; k < 9; k++) s += v9[k] * J[m * 9 + k];
                w6[m] += g * s;
            }
            w6[3] += g * (dN0 * (-f / ez));
            w6[4] += g * (dN1 * (f / ez));
            w6[5] += g * (dN0 * (f * ex / ez / ez) + dN1 * (-f * ey / ez / ez));
        }
        // sum_i g * dProjectdHyp  (1x6) over the 1600 points
#pragma unroll
        for (int k = 0; k < 6; k++) {
            double v = w6[k];
#pragma unroll
            for (int off = 16; off; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
            if (lane == 0) s_red[warp][k] = v;
        }
        __syncthreads();
        if (tid < 6) {
            double v = 0;
            for (int w = 0; w < K5_WARPS; w++) v += s_red[w][tid];
            s_w[tid] = v;
        }
        __syncthreads();
        // supportPointGradients = w . dPNP_h (1x12) onto the 4 support cells (cnn_softam.h:632-642)
        if (tid < 12) {
            const double* Jp = p.s.dpnp + ((size_t)frame * p.H + h) * 72;
            double s = 0;
            for (int k = 0; k < 6; k++) s += s_w[k] * Jp[k * 12 + tid];
            int c = p.img_idx[((size_t)frame * p.H + h) * 4 + tid / 3];
            if (c >= 0) {
                int x = c % DSAC_GRID_CONST, y = c / DSAC_GRID_CONST;
                int colb = p.fix_q4 ? (y * DSAC_GRID_CONST + x) * 3 : (x * DSAC_GRID_CONST + y) * 3;   // quirk Q4
                row[colb + tid % 3] += s;   // 12 distinct addresses; ordered by the barriers of the h loop
            }
        }
    }
    __syncthreads();
    // direct part: column of point (x,y) -- x-major in the reference (quirk Q4, cnn_softam.h:628)
#pragma unroll
    for (int j = 0; j < K5_PTS; j++) {
        int pt = tid + j * K5_THREADS;
        int x = pt % DSAC_GRID_CONST, y = pt / DSAC_GRID_CONST;
        int colb = p.fix_q4 ? pt * 3 : (x * DSAC_GRID_CONST + y) * 3;
        for (int k = 0; k < 3; k++) row[colb + k] += acc[j][k];
    }
}

// ---- batched Kabsch (Hypothesis::calcRigidBodyTransform, Hypothesis.cpp:145-200): thread = problem.
// b ~ R a + t with R = V diag(1,1,sign) U^T from the SVD of sum (a-ca)(b-cb)^T.
__device__ void sym_eig3(const double S[9], double w[3], double V[9]) {
    double A[9];
    for (int i = 0; i < 9; i++) { A[i] = S[i]; V[i] = (i % 4 == 0) ? 1.0 : 0.0; }
    for (int sweep = 0; sweep < 40; sweep++) {
        double off = fabs(A[1]) + fabs(A[2]) + fabs(A[5]);
        if (off == 0.0) break;
        for (int pq = 0; pq < 3; pq++) {
            const int p = pq == 2 ? 1 : 0, q = pq == 0 ? 1 : 2;
            double apq = A[p * 3 + q];
            if (apq == 0.0) continue;
            double theta = (A[q * 3 + q] - A[p * 3 + p]) / (2.0 * apq);
            double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
            double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
            for (int k = 0; k < 3; k++) {
                double akp = A[k * 3 + p], akq = A[k * 3 + q];
                A[k * 3 + p] = c * akp - s * akq;
                A[k * 3 + q] = s * akp + c * akq;
            }
            for (int k = 0; k < 3; k++) {
                double apk = A[p * 3 + k], aqk = A[q * 3 + k];
                A[p * 3 + k] = c * apk - s * aqk;
                A[q * 3 + k] = s * apk + c * aqk;
            }
            A[p * 3 + q] = A[q * 3 + p] = 0.0;
            for (int k = 0; k < 3; k++) {
                double vkp = V[k * 3 + p], vkq = V[k * 3 + q];
                V[k * 3 + p] = c * vkp - s * vkq;
                V[k * 3 + q] = s * vkp + c * vkq;
            }
        }
    }
    w[0] = A[0]; w[1] = A[4]; w[2] = A[8];
}

__global__ void k_kabsch(int n, int m, const double* __restrict__ a, const double* __restrict__ b, double* R, double* t) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double* pa = a + (size_t)i * m * 3;
    const double* pb = b + (size_t)i * m * 3;
    double cA[3] = {0, 0, 0}, cB[3] = {0, 0, 0};
    for (int k = 0; k < m; k++)
        for (int d = 0; d < 3; d++) { cA[d] += pa[k * 3 + d]; cB[d] += pb[k * 3 + d]; }
    for (int d = 0; d < 3; d++) { cA[d] *= 1.0 / (double)m; cB[d] *= 1.0 / (double)m; }
    double C[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};   // pointsA * pointsB^T
    for (int k = 0; k < m; k++)
        for (int r = 0; r < 3; r++)
            for (int c = 0; c < 3; c++) C[r * 3 + c] += (pa[k * 3 + r] - cA[r]) * (pb[k * 3 + c] - cB[c]);
    // SVD C = U diag(s) V^T through the eigen-decomposition of C^T C (V) and U = C V / s
    double S[9], w[3], V[9];
    for (int r = 0; r < 3; r++)
        for (int c = 0; c < 3; c++) S[r * 3 + c] = C[0 * 3 + r] * C[0 * 3 + c] + C[1 * 3 + r] * C[1 * 3 + c] + C[2 * 3 + r] * C[2 * 3 + c];
    sym_eig3(S, w, V);
    // order eigenvalues descending
    int o[3] = {0, 1, 2};
    if (w[o[0]] < w[o[1]]) { int x = o[0]; o[0] = o[1]; o[1] = x; }
    if (w[o[1]] < w[o[2]]) { int x = o[1]; o[1] = o[2]; o[2] = x; }
    if (w[o[0]] < w[o[1]]) { int x = o[0]; o[0] = o[1]; o[1] = x; }
    double Vs[9], U[9];
    for (int j = 0; j < 3; j++)
        for (int k = 0; k < 3; k++) Vs[k * 3 + j] = V[k * 3 + o[j]];
    for (int j = 0; j < 2; j++) {
        double u[3], nn = 0;
        for (int k = 0; k < 3; k++) { u[k] = C[k * 3] * Vs[0 * 3 + j] + C[k * 3 + 1] * Vs[1 * 3 + j] + C[k * 3 + 2] * Vs[2 * 3 + j]; nn += u[k] * u[k]; }
        nn = nn > 0 ? 1.0 / sqrt(nn) : 0.0;
        for (int k = 0; k < 3; k++) U[k * 3 + j] = u[k] * nn;
    }
    // third left vector: C v3 / s3 when s3 is well above rounding, else completes the right-handed frame
    {
        double u[3], nn = 0;
        for (int k = 0; k < 3; k++) { u[k] = C[k * 3] * Vs[0 * 3 + 2] + C[k * 3 + 1] * Vs[1 * 3 + 2] + C[k * 3 + 2] * Vs[2 * 3 + 2]; nn += u[k] * u[k]; }
        double cr[3] = {U[3] * U[7] - U[6] * U[4], U[6] * U[1] - U[0] * U[7], U[0] * U[4] - U[3] * U[1]};
        if (nn > 1e-24 * (w[o[0]] > 0 ? w[o[0]] : 1.0)) {
            nn = 1.0 / sqrt(nn);
            for (int k = 0; k < 3; k++) U[k * 3 + 2] = u[k] * nn;
        } else {
            for (int k = 0; k < 3; k++) U[k * 3 + 2] = cr[k];
        }
    }
    // sign = det(V U^T) < 0 ? -1 : 1 ; R = V diag(1,1,sign) U^T
    double VUt[9];
    for (int r = 0; r < 3; r++)
        for (int c = 0; c < 3; c++) VUt[r * 3 + c] = Vs[r * 3] * U[c * 3] + Vs[r * 3 + 1] * U[c * 3 + 1] + Vs[r * 3 + 2] * U[c * 3 + 2];
    double det = VUt[0] * (VUt[4] * VUt[8] - VUt[5] * VUt[7]) - VUt[1] * (VUt[3] * VUt[8] - VUt[5] * VUt[6]) + VUt[2] * (VUt[3] * VUt[7] - VUt[4] * VUt[6]);
    double sign = det < 0 ? -1.0 : 1.0;
    double Ro[9];
    for (int r = 0; r < 3; r++)
        for (int c = 0; c < 3; c++) Ro[r * 3 + c] = Vs[r * 3] * U[c * 3] + Vs[r * 3 + 1] * U[c * 3 + 1] + sign * Vs[r * 3 + 2] * U[c * 3 + 2];
    for (int k = 0; k < 9; k++) R[(size_t)i * 9 + k] = Ro[k];
    for (int r = 0; r < 3; r++) t[(size_t)i * 3 + r] = -(Ro[r * 3] * cA[0] + Ro[r * 3 + 1] * cA[1] + Ro[r * 3 + 2] * cA[2]) + cB[r];
}

}  // namespace dsac

int backward_run(dsac_engine* e, int32_t n, const int16_t* coords, const int32_t* pix, int32_t pix_shared,
                 const double* gt_jp, dsac_backward_out* out);
int kabsch_run(dsac_engine* e, int32_t n, int32_t m, const double* a, const double* b, double* R, double* t);
struct dsac_backward_dsac_out;
int backward_dsac_run(dsac_engine* e, int32_t n, dsac_backward_dsac_out* out);
