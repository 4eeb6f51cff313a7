// sampler_split.cuh -- K1 (minimal-set sampling, cnn_softam.h:1010-1060) as a round-based pipeline of flat kernels.
//
// The monolithic k_sample (kernels.cuh) runs one persistent CTA per (frame, stream) that alternates between integer
// work (MT19937 regeneration, candidate boundaries) and fp64 work (filter, full P3P): the fp64 pipe idles during the
// former, block barriers separate the phases and the register budget is the maximum over all of them.  Here every
// phase is its own kernel with its own register budget and its own grid:
//
//   k1_cells   once per call: per-cell record table (scene coordinate, float-rounded normalised pixel, 1/|bearing|)
//   per round r = 0 .. R-1:
//     k1_slot    one CTA per (frame, stream) -- integer only: (a) ordered selection of the previous round's accepted
//                candidates (first `quota` of the stream, in stream order), (b) size of the next round from the
//                observed acceptance rate, (c) MT19937 regeneration + uniform_int_distribution decode + candidate
//                boundaries for that many candidates, written to HBM as 4 cell indices per candidate
//     k1_filter  flat, persistent over (slot, chunk) work items: conservative fp64 filter, one thread per candidate,
//                no barriers in the loop; flagged candidates go to a global queue
//     k1_solve   flat, persistent over the flagged queue: full fp64 P3P with 4 lanes per candidate (one quartic root
//                each), the reference's float-rounded reprojection check, accepted poses to HBM
//   k1_slot (select only), then k_sample in resume mode for streams that still miss hypotheses (normally none).
//
// The candidate stream, the acceptance decisions and the order of the accepted candidates are exactly those of
// k_sample (same device functions), so the sampled indices stay bit-exact; only the scheduling differs.
#pragma once
#include <cuda_runtime.h>

#include "kernels.cuh"

namespace dsac {

#define K1S_THREADS_DEF 256
constexpr int K1S_THREADS = K1S_THREADS_DEF;     // k1_slot
constexpr int K1S_WARPS = K1S_THREADS / 32;
constexpr int K1S_SR = 2048;                     // candidates per generator window (super-round)
constexpr int K1S_WORDS = K1S_SR * 8 + 1024;     // decoded stream words buffered per window
constexpr int K1S_MAX_CAP = 32768;               // candidates per stream and round (flag queue entries hold 15 bits)
constexpr int K1S_IDX_BITS = 15;
constexpr int K1S_SEL_WORDS = K1S_MAX_CAP / 32 / K1S_THREADS_DEF;   // accept-bit words per thread in the selection
constexpr int K1S_ACC_LIST = 1024;               // accepted candidates selected per stream and round (<= quota <= DSAC_MAX_HYPS)
#ifndef K1F_THREADS_DEF
#define K1F_THREADS_DEF 256
#endif
constexpr int K1F_THREADS = K1F_THREADS_DEF;     // k1_filter
constexpr int K1F_MAX_CHUNK = 2048;              // candidates per filter work item (multiple of K1F_THREADS)
constexpr int K1V_THREADS = 128;                 // k1_solve: 32 groups of 4 lanes
constexpr int K1S_MAX_ROUNDS = 16;
#ifndef K1S_CAP_PER_HYP
#define K1S_CAP_PER_HYP 64       /* round capacity in candidates per hypothesis of the stream (cap = 16 384 at 256 hypotheses; 96 measured the same) */
#endif
#ifndef K1S_FIRST_ROUND_FRAC
#define K1S_FIRST_ROUND_FRAC 0.9   /* first round: this fraction of what the previous call's streams needed */
#endif
#ifndef K1S_MARGIN_SIGMA
#define K1S_MARGIN_SIGMA 2.0       /* later rounds: margin in standard deviations of the binomial accept count */
#endif
constexpr int K1S_MAX_SETS = 32;                  // launch sets (portions) per call

struct K1SplitParams {
    SampleParams sp;            // inputs / outputs of k_sample
    K1SlotState* state;         // [slots]
    CellRec* celltab;           // [n][N]
    uint2* cells;               // [slots][cap]   4 x uint16 cell indices per candidate
    uint32_t* endw;             // [slots][cap]   stream position after the candidate
    uint32_t* accbits;          // [slots][cap/32]
    double* pose_out;           // [slots][cap][6] rvec, tvec of accepted candidates
    uint2* wq;                  // filter work items of launch set `qidx`: (slot * 128 + chunk, candidates in the chunk)
    uint32_t* fq;               // flagged candidates: slot << K1S_IDX_BITS | index
    int* wq_n;                  // [K1S_MAX_SETS] per launch set
    int* fq_n;                  // [K1S_MAX_SETS]
    unsigned long long* stats_cur;   // [2] candidates, accepted hypotheses of the streams finished in this call
    const unsigned long long* stats_prev;   // the same of the previous call (prior for the first round's size)
    unsigned long long* dbg;    // [K1S_MAX_ROUNDS][4] or null: active streams, candidates, flagged, accepted per round
    int cap;                    // candidates per stream and round (multiple of 256, <= K1S_MAX_CAP)
    int chunk;                  // candidates per filter work item (multiple of 256)
    int n_slots;
    int round;                  // >= 0; select_only: no generation
    int select_only;
    // A round is generated in portions (launch sets): the first k1_slot of a round selects, sizes the round and generates
    // up to `portion` candidates; the following ones (gen_only) append the next `portion` of the same round.  Every
    // launch set has its own work / flag queue (index qidx), so the generator of set k+1 can run on a second stream
    // while filter and solve work on set k (integer pipe next to the fp64 pipe).
    int gen_only;
    int portion;                // candidates per launch set (multiple of chunk)
    int round_limit;            // candidates a round may have at most (= portion * launch sets of the round)
    int qidx;                   // launch set of this call: index into wq_n / fq_n, wq region qidx * wq_stride
    int wq_stride;
    int fqidx;                  // flag queue of this call: index into fq_n (the sets of a round may share one queue: one k1_solve per round)
    double first_frac;          // first round: this fraction of the expected need (K1S_FIRST_ROUND_FRAC; > 1 for few streams)
    int spec;                   // 1: a speculative window of k1_spec (virtual slot: no work items, no accept bits, no statistics)
};

// ------------------------------------------------------------------ k1_cells
// The FIRST (n_slots + 31) / 32 blocks seed the streams instead: MT19937's seeding recurrence is serial (624 dependent
// steps), so one THREAD per stream does it here, all streams at once and next to the cell records, instead of thread 0 of
// every k1_slot CTA with the other 255 threads waiting (10 us per CTA, two CTA waves).  A warp seeds 32 streams in lockstep
// and hands every 32 steps over through a shared-memory tile, so that the states reach HBM as 128-byte rows.
__global__ void __launch_bounds__(256) k1_cells(K1SplitParams q, int n_frames, int seed_blocks) {
    const SampleParams& p = q.sp;
    __shared__ uint32_t tile[32][33];
    if ((int)blockIdx.x < seed_blocks) {
        if (threadIdx.x >= 32) return;
        const int lane = (int)threadIdx.x, slot0 = (int)blockIdx.x * 32, slot = slot0 + lane;
        // stream s of global frame g: mt19937(seed + g*T + s)   (thread_rand.cpp:52 for g = 0)
        uint32_t v = p.seed + (uint32_t)(p.frame0 * (long long)p.T + slot);
        if (q.n_slots < 32) {   // a few streams: nothing to coalesce, every stream stores its own words
            if (slot < q.n_slots) {
                uint32_t* mt = q.state[slot].mt;
                mt[0] = v;
                for (int i = 1; i < MT_N; i++) {
                    v = 1812433253u * (v ^ (v >> 30)) + (uint32_t)i;
                    mt[i] = v;
                }
            }
            return;
        }
        for (int i0 = 0; i0 < MT_N; i0 += 32) {
#pragma unroll 8
            for (int j = 0; j < 32; j++) {
                const int i = i0 + j;
                if (i > 0) v = 1812433253u * (v ^ (v >> 30)) + (uint32_t)i;
                tile[lane][j] = v;
            }
            __syncwarp();
            if (i0 + lane < MT_N)
                for (int r = 0; r < 32 && slot0 + r < q.n_slots; r++) q.state[slot0 + r].mt[i0 + lane] = tile[r][lane];
            __syncwarp();
        }
        return;
    }
    const int i = ((int)blockIdx.x - seed_blocks) * blockDim.x + threadIdx.x;
    if (i >= n_frames * DSAC_N_CONST) return;
    const int frame = i / DSAC_N_CONST, c = i - frame * DSAC_N_CONST;
    const int16_t* coords = p.coords + (size_t)frame * DSAC_N_CONST * 3;
    const int32_t* pix = p.pix + (size_t)frame * p.pix_stride;
    const double inv_f = 1. / p.f, cx_f = p.cx * inv_f, cy_f = p.cy * inv_f;
    CellRec r;
    r.X = __ldg(coords + c * 3); r.Y = __ldg(coords + c * 3 + 1); r.Z = __ldg(coords + c * 3 + 2); r.pad = 0;
    r.xn = (float)(((double)__ldg(pix + c * 2) - p.cx) * inv_f);       // cv::undistortPoints rounds to float (p3p_pixel)
    r.yn = (float)(((double)__ldg(pix + c * 2 + 1) - p.cy) * inv_f);
    const double mu = r.xn * p.f + p.cx, mv = r.yn * p.f + p.cy;     // float * double
    const double u = inv_f * mu - cx_f, v = inv_f * mv - cy_f;
    r.k = rsqrt(u * u + v * v + 1);
    q.celltab[i] = r;
}

// ------------------------------------------------------------------ k1_slot
template <int NW>
struct K1GSmemT {
    uint32_t st[2 * MT_N];                       // MT19937 state, double-buffered (old / new generation)
    __align__(16) unsigned char vals[K1S_WORDS];  // Lemire value (0..39) of stream word pos+i; 255 = rejected draw
    unsigned short cand_start[K1S_SR + 512];     // word offset (from pos) where candidate i starts
    unsigned short acc_list[K1S_ACC_LIST];       // selection: accepted candidates of the round, in order
    int warp[2][NW];
    uint32_t newpos;
    int n_sr, any_reject, walk_fail;
    uint32_t ev[NW][K1_EV_CAP];
    int ev_n[NW];
    unsigned short brk_ci[K1_BRK_CAP], brk_cur[K1_BRK_CAP];
    int brk_n;
    int sel_total;
};
using K1GSmem = K1GSmemT<K1S_WARPS>;

// Size of the next round: enough candidates for the hypotheses still missing, from the acceptance rate observed so
// far (cpa = candidates per accepted hypothesis) plus a margin of ~2.5 sigma of the binomial count, so that nearly
// every stream finishes in the round.  The first round has no observation of its own: it takes 80 % of what the
// streams of the previous call needed (prior), or 16 candidates per hypothesis.
__device__ __forceinline__ int k1_round_size(int quota, int acc, long long cand_base, int cap, long long cand_left, double prior_cpa, double first_frac) {
    double n;
    if (cand_base == 0) {
        // no previous call to learn from: assume 64 candidates per accepted hypothesis (a wrong guess costs the first call
        // some extra candidates or an extra round, never a different result)
        n = first_frac * ((prior_cpa > 0) ? prior_cpa : 64.0) * quota;
        if (n < 64) n = 64;
    } else if (acc == 0) {
        n = 4.0 * (double)cand_base;
    } else {
        const double need = (double)(quota - acc), cpa = (double)cand_base / (double)acc;
        n = (need + K1S_MARGIN_SIGMA * sqrt(need) + 1.0) * cpa;
    }
    if (n > (double)cap) n = (double)cap;
    if (n > (double)cand_left) n = (double)cand_left;
    int r = (int)n;
    if (r < 1 && cand_left > 0) r = 1;
    return r;
}

// The work of k1_slot for one (frame, stream), by a CTA of NT threads.  tid: thread index.
// TW3: regeneration through mt_twist3 (own words in registers, branch-free: fastest for a lone CTA -- 230 against 388 cycles per
// block -- but ten instructions more per thread, which costs the issue-bound full batch 0.05 ms per step)
template <int NT, bool TW3 = (NT > 256)>
__device__ __forceinline__ void k1_slot_body(const K1SplitParams& q, K1GSmemT<NT / 32>& sm, const int tid, const int s, const int frame,
                                             const int slot_ov = -1) {
    constexpr int NW = NT / 32, SEL_WORDS = K1S_MAX_CAP / 32 / NT;   // warps of the group; accept-bit words per thread in the selection
    static_assert(SEL_WORDS >= 1 && K1S_LEFT_CAP % NT == 0, "k1_slot_body: thread count");
    const SampleParams& p = q.sp;
    const int lane = tid & 31, warp_id = tid >> 5;
    const int slot = (slot_ov >= 0) ? slot_ov : frame * p.T + s;   // slot_ov: a virtual slot of k1_spec (state / candidate arrays of its own)
    K1SlotState& S = q.state[slot];
    int h0, quota;
    stream_chunk(p.H, p.T, s, &h0, &quota);
    const size_t cbase = (size_t)slot * q.cap;
    const long long cand_max = p.max_candidates > 0 ? (long long)p.max_candidates : (1ll << 40);

    uint32_t pos, gen;
    int acc;
    long long cand_base;
    int already = 0;          // candidates of this round generated by earlier launch sets
    if (q.gen_only) {
        // ---------------- a further portion of the current round: restore the generator, nothing to select
        if (quota == 0 || S.done) return;
        already = S.n_round;
        if (already >= S.target) return;
        acc = S.acc;
        cand_base = S.cand_base;
        pos = S.pos;
        gen = S.gen;
        {
            uint32_t* half = sm.st + ((gen / MT_N) & 1u) * MT_N;
            for (int k = tid; k < MT_N; k += NT) half[k] = S.mt[k];
            const int ln = S.left_n;
            for (int k = tid; k < ln; k += NT) sm.vals[k] = S.left[k];
            if (tid == 0) { sm.any_reject = S.any_reject; sm.walk_fail = 0; }
        }
        __syncthreads();
    } else if (q.round == 0) {
        if (quota == 0) {
            if (tid == 0) {
                S.done = 1; S.acc = 0; S.n_round = 0; S.target = 0; S.cand_base = 0; S.left_n = 0; S.any_reject = 0; S.overflow = 0; S.pos = 0; S.gen = 0;
                p.stream_ncand[slot] = 0;
                p.stream_endpos[slot] = 0;
            }
            return;
        }
        // stream s of global frame g: mt19937(seed + g*T + s)   (thread_rand.cpp:52 for g = 0)
        for (int k = tid; k < MT_N; k += NT) sm.st[k] = S.mt[k];   // seeded by k1_cells
        pos = (s == 0) ? p.skip : 0u;
        gen = 0;
        acc = 0;
        cand_base = 0;
        if (tid == 0) { sm.any_reject = 0; sm.walk_fail = 0; }
        __syncthreads();
    } else {
        if (S.done) return;
        // ---------------- selection: the first (quota - acc) accepted candidates of the previous round, in order
        acc = S.acc;
        cand_base = S.cand_base;
        const int n_prev = S.n_round;
        const int n_words = (n_prev + 31) >> 5;          // <= K1S_MAX_CAP / 32
        const uint32_t* ab = q.accbits + (size_t)slot * (q.cap >> 5);
        uint32_t w[SEL_WORDS];
        int mine = 0;
#pragma unroll
        for (int k = 0; k < SEL_WORDS; k++) {
            const int wi = SEL_WORDS * tid + k;
            w[k] = (wi < n_words) ? ab[wi] : 0u;
            mine += __popc(w[k]);
        }
        int tot;
        int rank = block_excl_scan<NW>(mine, &tot, sm.warp[0], tid);
        const int room = quota - acc;
#pragma unroll
        for (int k = 0; k < SEL_WORDS; k++) {
            uint32_t ww = w[k];
            const int base_i = (SEL_WORDS * tid + k) * 32;
            while (ww) {
                const int b = __ffs(ww) - 1;
                ww &= ww - 1;
                if (rank < room) sm.acc_list[rank] = (unsigned short)(base_i + b);
                rank++;
            }
        }
        __syncthreads();
        const int n_emit = min(tot, room);
        for (int k = tid; k < n_emit; k += NT) {
            const int i = sm.acc_list[k];
            const size_t hi = (size_t)frame * p.H + h0 + acc + k;
            const double* po = q.pose_out + (cbase + i) * 6;
            double rvec[3] = {po[0], po[1], po[2]}, tvec[3] = {po[3], po[4], po[5]};
            double* hp = p.hyp_pose + hi * 6;
            hp[0] = rvec[0]; hp[1] = rvec[1]; hp[2] = rvec[2];
            hp[3] = tvec[0]; hp[4] = tvec[1]; hp[5] = tvec[2];
            double Rm[9];
            rodrigues_v2m(rvec, Rm);  // getDiffMap -> cv::projectPoints rebuilds R from rvec
            float4* P = reinterpret_cast<float4*>(p.hyp_P + hi * 12);
            P[0] = make_float4((float)(p.f * Rm[0]), (float)(p.f * Rm[1]), (float)(p.f * Rm[2]), (float)(p.f * tvec[0]));
            P[1] = make_float4((float)(p.f * Rm[3]), (float)(p.f * Rm[4]), (float)(p.f * Rm[5]), (float)(p.f * tvec[1]));
            P[2] = make_float4((float)Rm[6], (float)Rm[7], (float)Rm[8], (float)tvec[2]);
            const uint2 cc = q.cells[cbase + i];
            *reinterpret_cast<int4*>(p.img_idx + hi * 4) =
                make_int4((int)(cc.x & 0xffffu), (int)(cc.x >> 16), (int)(cc.y & 0xffffu), (int)(cc.y >> 16));
            p.cand_idx[hi] = (int32_t)(cand_base + i);
            if (acc + k == quota - 1) {
                p.stream_ncand[slot] = cand_base + i + 1;
                p.stream_endpos[slot] = (unsigned long long)q.endw[cbase + i];
            }
        }
        if (q.dbg && tid == 0) atomicAdd(q.dbg + (size_t)(q.round - 1) * 4 + 3, (unsigned long long)tot);
        if (acc + n_emit >= quota) {
            if (tid == 0) {
                S.done = 1; S.acc = quota; S.cand_base = cand_base + n_prev; S.n_round = 0; S.target = 0;
                atomicAdd(q.stats_cur + 0, (unsigned long long)(cand_base + sm.acc_list[room - 1] + 1));
                atomicAdd(q.stats_cur + 1, (unsigned long long)quota);
            }
            return;
        }
        acc += n_emit;
        cand_base += n_prev;
        if (q.select_only || cand_base >= cand_max) {   // the resume pass of k_sample takes over from here
            if (tid == 0) { S.acc = acc; S.cand_base = cand_base; S.n_round = 0; S.target = 0; }
            return;
        }
        // ---------------- restore the generator
        pos = S.pos;
        gen = S.gen;
        {
            uint32_t* half = sm.st + ((gen / MT_N) & 1u) * MT_N;
            for (int k = tid; k < MT_N; k += NT) half[k] = S.mt[k];
            const int ln = S.left_n;
            for (int k = tid; k < ln; k += NT) sm.vals[k] = S.left[k];
            if (tid == 0) { sm.any_reject = S.any_reject; sm.walk_fail = 0; }
        }
        __syncthreads();
    }

    // the thread's own three words of the current state, carried in registers from one regeneration to the next (mt_twist3)
    uint32_t own[3] = {0u, 0u, 0u};
    if (TW3 && tid < K1_WAVE) {
        const uint32_t* half = sm.st + ((gen / MT_N) & 1u) * MT_N;
        own[0] = half[tid]; own[1] = half[tid + K1_WAVE];
        if (tid + 2 * K1_WAVE < MT_N) own[2] = half[tid + 2 * K1_WAVE];
    }
    // ---------------- size of this round (first launch set of the round), size of this portion
    int round_total;
    if (q.gen_only) {
        round_total = S.target;
    } else {
        double prior = 0;
        if (q.stats_prev && q.stats_prev[1] > 0) prior = (double)q.stats_prev[0] / (double)q.stats_prev[1];
        round_total = k1_round_size(quota, acc, cand_base, min(q.cap, q.round_limit), cand_max - cand_base, prior, q.first_frac);
    }
    const int n_round = min(q.portion, round_total - already);   // candidates this launch generates

    // ---------------- generation: windows of up to K1S_SR candidates (phases A1, A2 and E of k_sample)
    // development aid (DSAC_K1_TIMERS=1): thread-0 cycles per phase of the generator -> phase_cycles[8..13]
    const bool timed = p.phase_cycles != nullptr && tid == 0;
    long long t_mark = timed ? clock64() : 0, t_ph[6] = {0, 0, 0, 0, 0, 0};
#define K1S_PHASE(k) do { if (timed) { const long long t_now = clock64(); t_ph[k] += t_now - t_mark; t_mark = t_now; } } while (0)
    int produced = 0;
    uint32_t st_par = (gen / MT_N) & 1u;   // which half of sm.st holds the current state
    while (produced < n_round) {
        const int n_target = min(K1S_SR, n_round - produced);
        const int w_need = min(K1S_WORDS - 640, n_target * 8 + 768);   // a regeneration may overshoot by 623 words
        // (leftover words [pos, gen) are at vals[0..gen-pos))
        // One barrier per 624-word regeneration: thread t < 227 twists words t, t + 227, t + 454 (each needs the thread's own
        // previous word and OLD neighbours only) and decodes them on the fly.  Measured alternatives (tools/micro/regen_bench.cu,
        // a lone CTA: twist alone 382 cycles per block, twist + decode fused 504, in this kernel 677; twist and decode on
        // separate warps 486 alone but 13 % slower with four CTAs per SM; decode of the previous block by all threads: equal):
        // the block time is the instruction stream of the twisting warps, two per scheduler.
        while ((int)(gen - pos) < w_need) {
            const uint32_t* so = sm.st + st_par * MT_N;           // old state
            uint32_t* sn = sm.st + (st_par ^ 1u) * MT_N;            // new state
            st_par ^= 1u;
            const int base_off = (int)(gen - pos);
            const bool all_in = base_off >= 0 && base_off + MT_N <= K1S_WORDS;   // the usual case: no per-word window test
            if (tid < K1_WAVE) {
                uint32_t x[3];
                bool has3;
                if (TW3) {
                    mt_twist3(so, tid, own, x);
                    own[0] = x[0]; own[1] = x[1]; own[2] = x[2];
                    has3 = tid + 2 * K1_WAVE < MT_N;
                } else {
                    has3 = mt_regenerate_words(so, tid, x) == 3;
                }
                bool rej_any = false;
#pragma unroll
                for (int w = 0; w < 3; w++) {
                    if (w < 2 || has3) {
                        const int k = tid + w * K1_WAVE;
                        sn[k] = x[w];
                        // libstdc++'s Lemire down-scaling of a 32-bit word to [0, 40): value = high half of w * 40,
                        // re-drawn if the low half is < 2^32 mod 40 = 16
                        const uint32_t tv = mt_temper(x[w]);
                        const uint32_t hi = __umulhi(tv, (uint32_t)DSAC_GRID_CONST), lo = tv * (uint32_t)DSAC_GRID_CONST;
                        const bool rej = lo < ((0u - DSAC_GRID_CONST) % DSAC_GRID_CONST);
                        const int off = base_off + k;
                        if (all_in || (off >= 0 && off < K1S_WORDS)) {
                            sm.vals[off] = rej ? (unsigned char)255 : (unsigned char)hi;
                            rej_any |= rej;
                        }
                    }
                }
                if (rej_any) sm.any_reject = 1;
            }
            gen += MT_N;
            __syncthreads();
        }
        K1S_PHASE(0);   // regeneration + decode
        const int w_avail = min((int)(gen - pos), K1S_WORDS);

        // candidate boundaries (see k_sample, phase A2)
        bool a2_done = false;
        if (!sm.any_reject && !p.a2_generic) {
            const unsigned short* pr16 = reinterpret_cast<const unsigned short*>(sm.vals);
            const int scan_end = min(w_avail >> 1, n_target * 4 + 384);
            // Every thread takes 16-byte blocks (8 pairs = 4 words of 2 pairs) and compares each word with the three
            // preceding pairs two pairs at a time (zero-half test on the XOR with the shifted predecessors, ~7
            // instructions per pair); only blocks that contain a repeat (~1 in 60) go through the recording path.
            const uint4* v128 = reinterpret_cast<const uint4*>(sm.vals);
            const int n_blocks = (scan_end + 7) >> 3;
            // (at most 8 warps scan: the walking thread below visits one event list per scanning warp, and with 32 lists the
            // serial walk cost more than the scan gained -- thread-0 cycles per frame 112 k vs 77 k)
            constexpr int NWS = NW < 8 ? NW : 8;
            const int bseg = ((n_blocks + NWS - 1) / NWS + 31) & ~31;   // blocks per warp, contiguous: events stay ordered
            const int bbeg = min(warp_id * bseg, n_blocks), bend = (warp_id < NWS) ? min(bbeg + bseg, n_blocks) : bbeg;
            int cnt = 0;
            for (int b0 = bbeg; b0 < bend; b0 += 32) {
                const int b = b0 + lane;
                uint32_t w[6] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu};   // w[0..1]: the two words before the block
                if (b < bend) {
                    const uint4 cur = v128[b];
                    w[2] = cur.x; w[3] = cur.y; w[4] = cur.z; w[5] = cur.w;
                    if (b > 0) {
                        const uint2 prv = *reinterpret_cast<const uint2*>(sm.vals + 16 * b - 8);
                        w[0] = prv.x; w[1] = prv.y;
                    }
                }
                uint32_t any = 0;
#pragma unroll
                for (int j2 = 2; j2 < 6; j2++) {
                    const uint32_t s1 = __funnelshift_l(w[j2 - 1], w[j2], 16);       // (pair 2j-1, pair 2j)
                    const uint32_t s3 = __funnelshift_l(w[j2 - 2], w[j2 - 1], 16);   // (pair 2j-3, pair 2j-2)
                    const uint32_t x1 = w[j2] ^ s1, x2 = w[j2] ^ w[j2 - 1], x3 = w[j2] ^ s3;
                    any |= ((x1 - 0x00010001u) & ~x1) | ((x2 - 0x00010001u) & ~x2) | ((x3 - 0x00010001u) & ~x3);
                }
                const bool has = (b < bend) && (any & 0x80008000u) != 0u;
                if (__any_sync(0xffffffffu, has)) {   // rare: record (pair index, distance) in pair order
                    uint32_t evs[8];
                    int ne = 0;
                    if (has) {
#pragma unroll
                        for (int h2 = 0; h2 < 8; h2++) {
                            const int k = 8 * b + h2;
                            const uint32_t wj = w[2 + (h2 >> 1)], wp1 = w[1 + (h2 >> 1)], wp2 = w[(h2 >> 1)];
                            uint32_t pk, q1, q2, q3;
                            if (h2 & 1) { pk = wj >> 16; q1 = wj & 0xffffu; q2 = wp1 >> 16; q3 = wp1 & 0xffffu; }
                            else { pk = wj & 0xffffu; q1 = wp1 >> 16; q2 = wp1 & 0xffffu; q3 = wp2 >> 16; }
                            const uint32_t d = (pk == q1) ? 1u : (pk == q2) ? 2u : (pk == q3) ? 3u : 0u;
                            if (d && k < scan_end) evs[ne++] = ((uint32_t)k << 2) | d;
                        }
                    }
                    int incl = ne;
#pragma unroll
                    for (int off = 1; off < 32; off <<= 1) {
                        const int o = __shfl_up_sync(0xffffffffu, incl, off);
                        if (lane >= off) incl += o;
                    }
                    const int tot = __shfl_sync(0xffffffffu, incl, 31);
                    const int at = cnt + incl - ne;
                    for (int e = 0; e < ne; e++)
                        if (at + e < K1_EV_CAP) sm.ev[warp_id][at + e] = evs[e];
                    cnt += tot;
                }
            }
            if (lane == 0 && warp_id < NWS) sm.ev_n[warp_id] = cnt;
            __syncthreads();
            K1S_PHASE(1);   // scan for repeated pairs
            if (tid == 0) {
                int cur = 0, ci = 0, nb = 1, stop_at = -1;
                bool fail = false;
                sm.brk_ci[0] = 0; sm.brk_cur[0] = 0;
                for (int w = 0; w < NWS && !fail && stop_at < 0; w++) {
                    const int n = sm.ev_n[w];
                    if (n > K1_EV_CAP) { fail = true; break; }
                    for (int e = 0; e < n; e++) {
                        const uint32_t evv = sm.ev[w][e];
                        const int k = (int)(evv >> 2), d = (int)(evv & 3u);
                        if (k < cur) continue;                 // inside a candidate already parsed
                        const int j = (k - cur) >> 2, spp = cur + 4 * j;
                        if (k - d < spp) continue;             // the equal pair belongs to the previous candidate
                        if (ci + j >= n_target) { stop_at = n_target; break; }
                        const int np = cand_pairs_len(pr16, spp, scan_end);
                        if (np < 0) { stop_at = ci + j; break; }   // window ends inside this candidate
                        if (nb >= K1_BRK_CAP) { fail = true; break; }
                        ci += j + 1;
                        cur = spp + np;
                        sm.brk_ci[nb] = (unsigned short)ci;
                        sm.brk_cur[nb] = (unsigned short)cur;
                        nb++;
                    }
                }
                int n_ok = ci + ((scan_end - cur) >> 2);       // clean 4-pair candidates after the last break
                if (stop_at >= 0) n_ok = min(n_ok, stop_at);
                sm.n_sr = min(n_ok, n_target);
                sm.brk_n = nb;
                sm.walk_fail = fail ? 1 : 0;
            }
            __syncthreads();
            K1S_PHASE(2);   // thread 0's walk over the events
            if (!sm.walk_fail) {
                const int n_ok = sm.n_sr, nb = sm.brk_n;
                int m = 0;
                for (int i = tid; i <= n_ok; i += NT) {
                    while (m + 1 < nb && (int)sm.brk_ci[m + 1] <= i) m++;
                    sm.cand_start[i] = (unsigned short)(2 * ((int)sm.brk_cur[m] + 4 * (i - (int)sm.brk_ci[m])));
                }
                a2_done = true;
            }
        }
        if (!a2_done) {
            int rp = 0, n_done = 0, par = 0;   // word offset of the chunk, candidates placed so far
            bool out_of_words = false;
            while (n_done < n_target && !out_of_words) {
                const int n_chunk = min(NT, n_target - n_done);
                int extra = 0, start = 0, qn = 0;
                for (;;) {
                    int tot;
                    const int excl = block_excl_scan<NW>(extra, &tot, sm.warp[par], tid);
                    par ^= 1;
                    start = rp + 8 * tid + excl;
                    int cells[4];
                    qn = (tid < n_chunk) ? cand_parse_fast(sm.vals, start, w_avail, cells) : start + 8;
                    const int ne = (qn < 0) ? 0 : (qn - start) - 8;
                    const int changed = (ne != extra);
                    extra = ne;
                    if (!__syncthreads_or(changed)) break;
                }
                int bad = (tid < n_chunk && qn < 0) ? tid : NT;
#pragma unroll
                for (int off = 16; off; off >>= 1) bad = min(bad, __shfl_xor_sync(0xffffffffu, bad, off));
                if (lane == 0) sm.warp[par][tid >> 5] = bad;
                __syncthreads();
                int n_ok = n_chunk;
#pragma unroll
                for (int w = 0; w < NW; w++) n_ok = min(n_ok, sm.warp[par][w]);
                par ^= 1;
                if (tid < n_ok) sm.cand_start[n_done + tid] = (unsigned short)start;
                if (tid == n_ok - 1) sm.newpos = (uint32_t)qn;          // end of the last complete candidate
                __syncthreads();
                if (n_ok > 0) rp = (int)sm.newpos;
                n_done += n_ok;
                out_of_words = (n_ok < n_chunk);
            }
            if (tid == 0) {
                sm.cand_start[n_done] = (unsigned short)rp;
                sm.n_sr = n_done;
            }
        }
        __syncthreads();
        K1S_PHASE(3);   // candidate start offsets
        const int n_sr = sm.n_sr;

        // the window's candidates to HBM
        for (int i = tid; i < n_sr; i += NT) {
            int cells[4];
            cand_parse_fast(sm.vals, sm.cand_start[i], w_avail, cells);
            q.cells[cbase + already + produced + i] = make_uint2((uint32_t)cells[0] | ((uint32_t)cells[1] << 16), (uint32_t)cells[2] | ((uint32_t)cells[3] << 16));
            q.endw[cbase + already + produced + i] = pos + (uint32_t)sm.cand_start[i + 1];
        }

        K1S_PHASE(4);   // candidates to HBM (thread 0's share)
        // advance the stream: the unread tail of the window moves to the front
        {
            const int consumed = sm.cand_start[n_sr];
            const int left = w_avail - consumed;
            unsigned char keep[K1S_LEFT_CAP / NT];
            __syncthreads();
#pragma unroll
            for (int k = 0; k < K1S_LEFT_CAP / NT; k++) {
                const int i = tid + k * NT;
                keep[k] = (i < left) ? sm.vals[consumed + i] : (unsigned char)0;
            }
            __syncthreads();
            bool rej_left = false;
#pragma unroll
            for (int k = 0; k < K1S_LEFT_CAP / NT; k++) {
                const int i = tid + k * NT;
                if (i < left) {
                    sm.vals[i] = keep[k];
                    rej_left |= (keep[k] == 255);
                }
            }
            if (tid == 0) { sm.any_reject = 0; sm.walk_fail = 0; }
            __syncthreads();
            if (rej_left) sm.any_reject = 1;   // a rejected draw carried over into the next window
            if (left > K1S_LEFT_CAP && tid == 0) S.overflow = 1;
            pos += (uint32_t)consumed;
            produced += n_sr;
            __syncthreads();
        }
        K1S_PHASE(5);   // leftover move
        if (n_sr == 0) break;   // (cannot happen: every window holds at least one candidate)
    }
    if (timed)
        for (int k = 0; k < 6; k++) atomicAdd(p.phase_cycles + 8 + k, (unsigned long long)t_ph[k]);
#undef K1S_PHASE

    // ---------------- hand the portion over: state, work items, cleared accept bits
    {
        const int left = min((int)(gen - pos), K1S_LEFT_CAP);
        const uint32_t* half = sm.st + ((gen / MT_N) & 1u) * MT_N;
        for (int k = tid; k < MT_N; k += NT) S.mt[k] = half[k];
        for (int k = tid; k < left; k += NT) S.left[k] = sm.vals[k];
        if (!q.spec) {
            uint32_t* ab = q.accbits + (size_t)slot * (q.cap >> 5) + (already >> 5);   // `already` is a multiple of the chunk size
            for (int k = tid; k < ((produced + 31) >> 5); k += NT) ab[k] = 0u;
        }
        if (tid == 0) {
            S.pos = pos; S.gen = gen; S.acc = acc; S.cand_base = cand_base; S.n_round = already + produced; S.done = 0;
            if (!q.gen_only) S.target = round_total;
            S.left_n = left; S.any_reject = sm.any_reject;
            if (q.round == 0 && !q.gen_only) S.overflow = 0;
            const int n_items = q.spec ? 0 : (produced + q.chunk - 1) / q.chunk;
            if (n_items > 0) {
                const int at = atomicAdd(q.wq_n + q.qidx, n_items);
                uint2* wq = q.wq + (size_t)q.qidx * q.wq_stride;
                const int c0 = already / q.chunk;
                for (int c = 0; c < n_items; c++)
                    wq[at + c] = make_uint2((uint32_t)slot * 128u + (uint32_t)(c0 + c), (uint32_t)min(q.chunk, produced - c * q.chunk));
            }
            if (q.dbg) {
                if (!q.gen_only) atomicAdd(q.dbg + (size_t)q.round * 4 + 0, 1ull);
                atomicAdd(q.dbg + (size_t)q.round * 4 + 1, (unsigned long long)produced);
            }
        }
    }
}

#ifndef K1S_MIN_BLOCKS
#define K1S_MIN_BLOCKS 4
#endif
// NT threads per (frame, stream): 256 (4 CTAs per SM) when there are streams to fill the GPU several times over; 512 or
// 1024 when there are fewer streams than SMs can hold -- a stream's generation is a serial chain of windows, and the time of
// a lone CTA is what a small batch (single-frame latency, strong scaling) waits for.
template <int NT>
__global__ void __launch_bounds__(NT, (NT == K1S_THREADS) ? K1S_MIN_BLOCKS : 1024 / NT) k1_slot_t(K1SplitParams q) {
    __shared__ K1GSmemT<NT / 32> sm;
    k1_slot_body<NT>(q, sm, threadIdx.x, blockIdx.x, blockIdx.y);
}
__global__ void __launch_bounds__(K1S_THREADS, K1S_MIN_BLOCKS) k1_slot(K1SplitParams q) {
    __shared__ K1GSmem sm;
    k1_slot_body<K1S_THREADS>(q, sm, threadIdx.x, blockIdx.x, blockIdx.y);
}

// ------------------------------------------------------------------ k1_spec / k1_stitch: one stream generated by many CTAs
// With a few streams (single-frame latency, BASELINE config 2) a stream's first round is one CTA's serial chain: ~280
// MT19937 state regenerations and 11 windows of decode / scan / walk / write, 236 us for 21 946 candidates.  Here the round is
// cut into windows of K1P_BLOCKS state blocks (W = 8 112 stream words); window j is generated by its own CTAs, which reach
// their part of the stream by twisting the seeded state forward WITHOUT decoding (the cheap part of a regeneration) and
// then run the ordinary generator (k1_slot_body) on a virtual slot for W / 8 + 32 candidates.  Where window j's first
// candidate really starts is known only once window j-1 is parsed (a repeated cell shifts everything after it by two words), so
// windows j >= 1 are generated for all four possible alignments (start = first word of the window + 0, 2, 4, 6 words: candidates
// are sequences of (x, y) pairs, and every alignment falls into step with the true parse at the first candidate boundary it
// shares with it).  k1_stitch then walks the windows in order -- true start of window j+1 = end of the last candidate of window j
// that starts before it -- picks each window's alignment, checks that the boundary really is a candidate start there, and
// gathers the chosen candidates into the stream's ordinary arrays, state and work items.  Any mismatch (a rejected Lemire draw,
// a repeat inside the few candidates around a window boundary, a window too short) abandons the speculation: the stream is left
// at its seeded state and the next, ordinary round generates it.  Same candidates, same order, same stream positions.
constexpr int K1P_BLOCKS = 13;                          // state blocks per window
constexpr int K1P_W = K1P_BLOCKS * MT_N;                // 8 112 stream words per window (a multiple of 8)
constexpr int K1P_NW = K1P_W / 8 + 32;                  // candidates a window CTA generates: covers >= W + 256 words
constexpr int K1P_CAPW = 2048;                          // candidate capacity of a virtual slot
constexpr int K1P_MAX_WIN = 24;
constexpr int K1P_VPER = 1 + 4 * (K1P_MAX_WIN - 1);     // virtual slots per stream
constexpr int K1P_TABLE = 2 + 3 * K1P_MAX_WIN;
constexpr int K1P_TAIL = 96;                            // stream positions staged from the end of every window's list
static_assert(K1P_NW <= K1S_SR && K1P_NW <= K1P_CAPW && K1P_W % 8 == 0, "k1_spec window");

struct K1SpecParams {
    K1SlotState* vstate;   // [slots][K1P_VPER]
    uint2* vcells;         // [slots][K1P_VPER][K1P_CAPW]
    uint32_t* vendw;       // [slots][K1P_VPER][K1P_CAPW]
    int* result;           // [slots] windows stitched (0: speculation abandoned) -- development aid
    int* table;            // [slots][K1P_TABLE]: n_win, then per window (virtual slot, first candidate, base index), then the total: k1_stitch -> k1_gather
};

// windows of the speculative round: the first round's size as k1_round_size would choose it, in windows
__device__ __forceinline__ int k1_spec_windows(const K1SplitParams& q, int quota) {
    double prior = 0;
    if (q.stats_prev && q.stats_prev[1] > 0) prior = (double)q.stats_prev[0] / (double)q.stats_prev[1];
    const double n = q.first_frac * ((prior > 0) ? prior : 64.0) * quota;
    int nw = (int)(n / (K1P_W / 8) + 0.5);
    if (nw > K1P_MAX_WIN) nw = K1P_MAX_WIN;
    if ((long long)nw * K1P_NW > (long long)q.cap) nw = q.cap / K1P_NW;
    return nw < 2 ? 0 : nw;
}

__global__ void __launch_bounds__(K1S_THREADS, K1S_MIN_BLOCKS) k1_spec(K1SplitParams q, K1SpecParams sp) {
    __shared__ K1GSmem sm;
    const SampleParams& p = q.sp;
    const int tid = threadIdx.x, v = blockIdx.x, slot = blockIdx.y;
    const int frame = slot / p.T, s = slot - frame * p.T;
    int h0, quota;
    stream_chunk(p.H, p.T, s, &h0, &quota);
    if (quota == 0) return;
    const int j = (v == 0) ? 0 : 1 + (v - 1) / 4, a = (v == 0) ? 0 : (v - 1) & 3;
    if (j >= k1_spec_windows(q, quota)) return;
    const uint32_t pos0 = (s == 0) ? p.skip : 0u;
    const uint32_t pos_v = pos0 + (uint32_t)j * (uint32_t)K1P_W + 2u * (uint32_t)a;
    const int n_skip = (int)(pos_v / MT_N);                 // state blocks before the one that holds pos_v
    // the seeded state (k1_cells), twisted forward n_skip times: 227 threads, three dependent words each, raw state only
    for (int k = tid; k < MT_N; k += K1S_THREADS) sm.st[k] = q.state[slot].mt[k];
    __syncthreads();
    uint32_t par = 0;
    uint32_t own[3] = {0u, 0u, 0u};
    if (tid < K1_WAVE) {
        own[0] = sm.st[tid]; own[1] = sm.st[tid + K1_WAVE];
        if (tid + 2 * K1_WAVE < MT_N) own[2] = sm.st[tid + 2 * K1_WAVE];
    }
    for (int it = 0; it < n_skip; it++) {
        const uint32_t* so = sm.st + par * MT_N;
        uint32_t* sn = sm.st + (par ^ 1u) * MT_N;
        if (tid < K1_WAVE) {
            uint32_t x[3];
            mt_twist3(so, tid, own, x);
            sn[tid] = x[0];
            sn[tid + K1_WAVE] = x[1];
            if (tid + 2 * K1_WAVE < MT_N) sn[tid + 2 * K1_WAVE] = x[2];
            own[0] = x[0]; own[1] = x[1]; own[2] = x[2];
        }
        par ^= 1u;
        __syncthreads();
    }
    const int vs = slot * K1P_VPER + v;
    K1SlotState& Sv = sp.vstate[vs];
    for (int k = tid; k < MT_N; k += K1S_THREADS) Sv.mt[k] = sm.st[par * MT_N + k];
    if (tid == 0) {
        Sv.pos = pos_v; Sv.gen = (uint32_t)n_skip * (uint32_t)MT_N; Sv.acc = 0; Sv.n_round = 0; Sv.done = 0; Sv.left_n = 0;
        Sv.any_reject = 0; Sv.overflow = 0; Sv.target = 0; Sv.cand_base = 0;
    }
    __threadfence_block();
    __syncthreads();
    // the ordinary generator on the virtual slot: "a later round with nothing to select" restores pos / gen / state from Sv
    K1SplitParams qq = q;
    qq.state = sp.vstate; qq.cells = sp.vcells; qq.endw = sp.vendw; qq.cap = K1P_CAPW;
    qq.round = 1; qq.gen_only = 0; qq.select_only = 0; qq.portion = K1P_NW; qq.round_limit = K1P_NW; qq.spec = 1; qq.dbg = nullptr;
    k1_slot_body<K1S_THREADS, true>(qq, sm, tid, s, frame, vs);
}

struct K1StitchSmem {
    uint32_t head[K1P_VPER][8];            // stream positions after the first 8 candidates of every window list
    int n_list[K1P_VPER];                  // candidates in the list (0: unusable)
    int c_list[K1P_VPER];                  // first candidate of the list that starts at or after the NEXT window (-1: not found in the staged tail)
    uint32_t p_next[K1P_VPER];             // ... and where it starts
    uint32_t start0[K1P_VPER];
    int win_v[K1P_MAX_WIN], win_m[K1P_MAX_WIN], win_c[K1P_MAX_WIN], win_base[K1P_MAX_WIN + 1];
    int n_win, ok, wq_at;
};

constexpr int K1T_THREADS = 1024;
__global__ void __launch_bounds__(K1T_THREADS) k1_stitch(K1SplitParams q, K1SpecParams sp) {
    __shared__ K1StitchSmem sm;
    const SampleParams& p = q.sp;
    const int tid = threadIdx.x, slot = blockIdx.x;
    const int frame = slot / p.T, s = slot - frame * p.T;
    int h0, quota;
    stream_chunk(p.H, p.T, s, &h0, &quota);
    K1SlotState& S = q.state[slot];
    if (quota == 0) {
        if (tid == 0) {
            S.done = 1; S.acc = 0; S.n_round = 0; S.target = 0; S.cand_base = 0; S.left_n = 0; S.any_reject = 0; S.overflow = 0; S.pos = 0; S.gen = 0;
            p.stream_ncand[slot] = 0;
            p.stream_endpos[slot] = 0;
        }
        return;
    }
    const int n_win = k1_spec_windows(q, quota);
    const uint32_t pos0 = (s == 0) ? p.skip : 0u;
    const int n_virt = n_win > 0 ? 1 + 4 * (n_win - 1) : 0;
    const size_t vbase = (size_t)slot * K1P_VPER;
    // per window list, one warp each (all lists in parallel, coalesced): its length, its first 8 stream positions, and the first
    // candidate that starts at or after the next window (searched in the last K1P_TAIL entries: candidate nl - TAIL + t + 1 starts
    // at entry nl - TAIL + t) -- neither depends on where the list is entered, so the chain below is table look-ups only
    {
        const uint32_t FULL = 0xffffffffu;
        const int lane = tid & 31, warp = tid >> 5;
        for (int v = warp; v < n_virt; v += K1T_THREADS / 32) {
            const K1SlotState& Sv = sp.vstate[vbase + v];
            int nl = min(max(Sv.n_round, 0), K1P_CAPW);
            if (Sv.any_reject || Sv.overflow || nl < K1P_TAIL + 8) nl = 0;
            const int jv = (v == 0) ? 0 : 1 + (v - 1) / 4, av = (v == 0) ? 0 : (v - 1) & 3;
            const uint32_t Onext = pos0 + (uint32_t)(jv + 1) * (uint32_t)K1P_W;
            const uint32_t* ew = sp.vendw + (vbase + v) * K1P_CAPW;
            int tc = -1;
            uint32_t pn = 0u;
            if (nl > 0) {
                if (lane < 8) sm.head[v][lane] = ew[lane];
#pragma unroll
                for (int t0 = 0; t0 < K1P_TAIL; t0 += 32) {
                    const uint32_t val = ew[nl - K1P_TAIL + t0 + lane];
                    const uint32_t over = __ballot_sync(FULL, val >= Onext);
                    if (tc < 0 && over) {
                        const int l = __ffs(over) - 1;
                        tc = t0 + l;
                        pn = __shfl_sync(FULL, val, l);
                    }
                }
            }
            if (lane == 0) {
                sm.n_list[v] = nl;
                // tc == 0: the crossing may lie before the staged tail; tc < 0: the list ends before the next window
                const int c = (tc > 0) ? nl - K1P_TAIL + tc + 1 : -1;
                sm.c_list[v] = (c > 0 && c < nl) ? c : -1;
                sm.p_next[v] = pn;
                sm.start0[v] = pos0 + (uint32_t)jv * (uint32_t)K1P_W + 2u * (uint32_t)av;
            }
        }
    }
    __syncthreads();
    if (tid == 0) {   // the chain over the windows
        int ok = n_win >= 2, base = 0;
        uint32_t P = pos0;                       // true start of the current window's first candidate
        for (int j = 0; j < n_win && ok; j++) {
            const uint32_t O = pos0 + (uint32_t)j * (uint32_t)K1P_W;
            const uint32_t rel = P - O;
            if (P < O || (rel & 1u)) { ok = 0; break; }
            const int a = (int)((rel >> 1) & 3u), v = (j == 0) ? 0 : 1 + 4 * (j - 1) + a;
            if (j == 0 && a != 0) { ok = 0; break; }
            const int nl = sm.n_list[v];
            if (nl <= 0) { ok = 0; break; }
            // m: the candidate of this list that starts at P (start_0 = the list's own start, start_i = position after i-1)
            int m = -1;
            if (sm.start0[v] == P) m = 0;
            else
                for (int i = 0; i < 8; i++)
                    if (sm.head[v][i] == P) { m = i + 1; break; }
            if (m < 0) { ok = 0; break; }
            int c = nl;                          // one past the last candidate taken from this window
            if (j + 1 < n_win) {
                c = sm.c_list[v];
                if (c < 0 || c <= m) { ok = 0; break; }
                P = sm.p_next[v];
            }
            sm.win_v[j] = v; sm.win_m[j] = m; sm.win_c[j] = c; sm.win_base[j] = base;
            base += c - m;
        }
        if (ok && base > q.cap) ok = 0;
        sm.win_base[n_win > 0 ? n_win : 0] = base;
        sm.n_win = n_win; sm.ok = ok;
    }
    __syncthreads();
    const size_t cbase = (size_t)slot * q.cap;
    if (!sm.ok) {
        // speculation abandoned: the stream stands at its seeded state, the next (ordinary) round generates it
        if (tid == 0) {
            S.pos = pos0; S.gen = 0; S.acc = 0; S.cand_base = 0; S.n_round = 0; S.target = 0; S.done = 0; S.left_n = 0;
            S.any_reject = 0; S.overflow = 0;
            if (sp.result) sp.result[slot] = 0;
            sp.table[(size_t)slot * K1P_TABLE] = 0;
            sp.table[(size_t)slot * K1P_TABLE + 1] = 0;
        }
        return;
    }
    const int n_total = sm.win_base[sm.n_win];
    {   // the window table for k1_gather (which copies the chosen candidates on many SMs)
        int* tb = sp.table + (size_t)slot * K1P_TABLE;
        if (tid == 0) { tb[0] = sm.n_win; tb[1] = n_total; }
        if (tid < sm.n_win) { tb[2 + 3 * tid] = sm.win_v[tid]; tb[3 + 3 * tid] = sm.win_m[tid]; tb[4 + 3 * tid] = sm.win_base[tid]; }
    }
    {
        const K1SlotState& Sl = sp.vstate[vbase + sm.win_v[sm.n_win - 1]];   // the last window ran to its own end: its state is the round's
        for (int k = tid; k < MT_N; k += K1T_THREADS) S.mt[k] = Sl.mt[k];
        const int ln = min(max(Sl.left_n, 0), K1S_LEFT_CAP);
        for (int k = tid; k < ln; k += K1T_THREADS) S.left[k] = Sl.left[k];
        uint32_t* ab = q.accbits + (size_t)slot * (q.cap >> 5);
        for (int k = tid; k < ((n_total + 31) >> 5); k += K1T_THREADS) ab[k] = 0u;
        {   // filter work items of the round
            const int n_items = (n_total + q.chunk - 1) / q.chunk;
            if (tid == 0) sm.wq_at = atomicAdd(q.wq_n + q.qidx, n_items);
            __syncthreads();
            uint2* wq = q.wq + (size_t)q.qidx * q.wq_stride + sm.wq_at;
            for (int c = tid; c < n_items; c += K1T_THREADS)
                wq[c] = make_uint2((uint32_t)slot * 128u + (uint32_t)c, (uint32_t)min(q.chunk, n_total - c * q.chunk));
        }
        if (tid == 0) {
            S.pos = Sl.pos; S.gen = Sl.gen; S.acc = 0; S.cand_base = 0; S.n_round = n_total; S.target = n_total; S.done = 0;
            S.left_n = ln; S.any_reject = Sl.any_reject; S.overflow = 0;
            if (q.dbg) {
                atomicAdd(q.dbg + 0, 1ull);
                atomicAdd(q.dbg + 1, (unsigned long long)n_total);
            }
            if (sp.result) sp.result[slot] = sm.n_win;
        }
    }
}

// copies the candidates k1_stitch chose from the window lists into the stream's ordinary arrays (blockIdx.y: stream)
constexpr int K1G_THREADS = 256, K1G_PER_CTA = 1024;
__global__ void __launch_bounds__(K1G_THREADS) k1_gather(K1SplitParams q, K1SpecParams sp) {
    __shared__ int tb[K1P_TABLE];
    const int slot = blockIdx.y, tid = threadIdx.x;
    if (tid < K1P_TABLE) tb[tid] = sp.table[(size_t)slot * K1P_TABLE + tid];
    __syncthreads();
    const int n_win = tb[0], n_total = tb[1];
    const int g0 = blockIdx.x * K1G_PER_CTA;
    if (n_win <= 0 || g0 >= n_total) return;
    const size_t cbase = (size_t)slot * q.cap, vbase = (size_t)slot * K1P_VPER;
    uint2 c[K1G_PER_CTA / K1G_THREADS];
    uint32_t e[K1G_PER_CTA / K1G_THREADS];
#pragma unroll
    for (int k = 0; k < K1G_PER_CTA / K1G_THREADS; k++) {
        const int g = g0 + tid + k * K1G_THREADS;
        if (g < n_total) {
            int j = 0;
            while (j + 1 < n_win && tb[4 + 3 * (j + 1)] <= g) j++;
            const size_t src = (vbase + tb[2 + 3 * j]) * K1P_CAPW + (size_t)(tb[3 + 3 * j] + (g - tb[4 + 3 * j]));
            c[k] = sp.vcells[src];
            e[k] = sp.vendw[src];
        }
    }
#pragma unroll
    for (int k = 0; k < K1G_PER_CTA / K1G_THREADS; k++) {
        const int g = g0 + tid + k * K1G_THREADS;
        if (g < n_total) { q.cells[cbase + g] = c[k]; q.endw[cbase + g] = e[k]; }
    }
}

// ------------------------------------------------------------------ k1_pipe: one stream generated by K CTAs in a chain
// For 9 .. ~190 streams (strong scaling: 128 frames per GPU) the four-fold windows of k1_spec do not fit the GPU, but a stream's
// first round is still one CTA's serial chain.  Here K CTAs share a stream: window w (K1P_W stream words) belongs to CTA w mod K.
// Every CTA twists through ALL state blocks (without decoding those of the other CTAs' windows: the cheap part) and decodes,
// scans, parses and writes only its own windows.  The one thing a window needs from its predecessor -- the stream position of its
// first candidate and the number of candidates before it -- is published by the predecessor right after its walk and awaited by
// a spin on a global flag; a stream's CTAs have consecutive block indices in window order, so the CTA that is waited for is
// always dispatched first.  No speculation, nothing to stitch: every candidate is written at its final index.  Any irregularity
// (a rejected Lemire draw, an event-list overflow, a candidate that does not fit its window's margin) aborts the chain: the
// stream is left at its seeded state and the next, ordinary round generates it.
constexpr int K1Q_MARGIN = 256;                           // stream words decoded beyond a window (the straddling candidate)
constexpr int K1Q_MAX_WIN = 32;
struct K1PipeParams {
    uint32_t* chain;      // [slots][K1Q_MAX_WIN + 1][4]: stream position, candidates before, abort, flag (== epoch when valid)
    uint32_t epoch;       // > 0, different for every call of an engine lane
    int K;                // CTAs per stream
};

__device__ __forceinline__ int k1_pipe_windows(const K1SplitParams& q, int quota) {
    double prior = 0;
    if (q.stats_prev && q.stats_prev[1] > 0) prior = (double)q.stats_prev[0] / (double)q.stats_prev[1];
    const double n = q.first_frac * ((prior > 0) ? prior : 64.0) * quota;
    int nw = (int)(n / (K1P_W / 8) + 0.5);
    if (nw > K1Q_MAX_WIN) nw = K1Q_MAX_WIN;
    while (nw > 0 && (long long)nw * (K1P_W / 8 + 8) > (long long)q.cap) nw--;
    return nw < 2 ? 0 : nw;
}

__global__ void __launch_bounds__(K1S_THREADS, K1S_MIN_BLOCKS) k1_pipe(K1SplitParams q, K1PipeParams pp) {
    __shared__ K1GSmem sm;
    __shared__ uint32_t s_P, s_base, s_abort, s_count, s_pnext;
    const SampleParams& p = q.sp;
    const int tid = threadIdx.x, lane = tid & 31, warp_id = tid >> 5;
    const int kk = blockIdx.x, slot = blockIdx.y;
    const int frame = slot / p.T, s = slot - frame * p.T;
    int h0, quota;
    stream_chunk(p.H, p.T, s, &h0, &quota);
    K1SlotState& S = q.state[slot];
    const uint32_t pos0 = (s == 0) ? p.skip : 0u;
    if (quota == 0) {
        if (kk == 0 && tid == 0) {
            S.done = 1; S.acc = 0; S.n_round = 0; S.target = 0; S.cand_base = 0; S.left_n = 0; S.any_reject = 0; S.overflow = 0; S.pos = 0; S.gen = 0;
            p.stream_ncand[slot] = 0;
            p.stream_endpos[slot] = 0;
        }
        return;
    }
    const int n_win = k1_pipe_windows(q, quota);
    if (n_win == 0) {      // not worth it (few hypotheses per stream): the ordinary round generates the stream
        if (kk == 0 && tid == 0) {
            S.pos = pos0; S.gen = 0; S.acc = 0; S.cand_base = 0; S.n_round = 0; S.target = 0; S.done = 0; S.left_n = 0; S.any_reject = 0; S.overflow = 0;
        }
        return;
    }
    volatile uint32_t* chain = pp.chain + (size_t)slot * (K1Q_MAX_WIN + 1) * 4;
    const size_t cbase = (size_t)slot * q.cap;
    // the seeded state (k1_cells); cur_block = regenerations done = first stream word of the next block / 624
    for (int k = tid; k < MT_N; k += K1S_THREADS) sm.st[k] = S.mt[k];
    __syncthreads();
    uint32_t par = 0;
    uint32_t own[3] = {0u, 0u, 0u};
    if (tid < K1_WAVE) {
        own[0] = sm.st[tid]; own[1] = sm.st[tid + K1_WAVE];
        if (tid + 2 * K1_WAVE < MT_N) own[2] = sm.st[tid + 2 * K1_WAVE];
    }
    uint32_t cur_block = 0;
    constexpr int SCAN_END = (K1P_W + K1Q_MARGIN) / 2;        // pairs scanned per window
    constexpr int L_PAIRS = K1P_W / 2;                         // a candidate belongs to the window its first pair lies in
    for (int w = kk; w < n_win; w += pp.K) {
        const uint32_t O = pos0 + (uint32_t)w * (uint32_t)K1P_W;
        if (tid == 0) sm.any_reject = 0;
        __syncthreads();
        // ---- twist to the window (no decode), then twist + decode the words [O, O + W + margin)
        while ((cur_block + 1u) * (uint32_t)MT_N <= O || cur_block * (uint32_t)MT_N < O + (uint32_t)(K1P_W + K1Q_MARGIN)) {
            const bool decode = (cur_block + 1u) * (uint32_t)MT_N > O;
            const uint32_t* so = sm.st + par * MT_N;
            uint32_t* sn = sm.st + (par ^ 1u) * MT_N;
            if (tid < K1_WAVE) {
                uint32_t x[3];
                mt_twist3(so, tid, own, x);
                own[0] = x[0]; own[1] = x[1]; own[2] = x[2];
                const bool has3 = tid + 2 * K1_WAVE < MT_N;
                bool rej_any = false;
#pragma unroll
                for (int ww = 0; ww < 3; ww++) {
                    if (ww < 2 || has3) {
                        const int k = tid + ww * K1_WAVE;
                        sn[k] = x[ww];
                        if (decode) {
                            const uint32_t tv = mt_temper(x[ww]);
                            const uint32_t hi = __umulhi(tv, (uint32_t)DSAC_GRID_CONST), lo = tv * (uint32_t)DSAC_GRID_CONST;
                            const bool rej = lo < ((0u - DSAC_GRID_CONST) % DSAC_GRID_CONST);
                            const int off = (int)(cur_block * (uint32_t)MT_N + (uint32_t)k - O);   // stream word O + off
                            if (off >= 0 && off < K1S_WORDS) {
                                sm.vals[off] = rej ? (unsigned char)255 : (unsigned char)hi;
                                rej_any |= rej;
                            }
                        }
                    }
                }
                if (rej_any) sm.any_reject = 1;
            }
            par ^= 1u;
            cur_block++;
            __syncthreads();
        }
        const int w_avail = min((int)(cur_block * (uint32_t)MT_N - O), K1S_WORDS);   // decoded words from O on (>= W + margin)
        // ---- scan for repeated pairs (as k1_slot_body)
        const unsigned short* pr16 = reinterpret_cast<const unsigned short*>(sm.vals);
        {
            const uint4* v128 = reinterpret_cast<const uint4*>(sm.vals);
            constexpr int n_blocks = (SCAN_END + 7) >> 3;
            constexpr int NWS = K1S_WARPS < 8 ? K1S_WARPS : 8;
            constexpr int bseg = ((n_blocks + NWS - 1) / NWS + 31) & ~31;
            const int bbeg = min(warp_id * bseg, n_blocks), bend = (warp_id < NWS) ? min(bbeg + bseg, n_blocks) : bbeg;
            int cnt = 0;
            for (int b0 = bbeg; b0 < bend; b0 += 32) {
                const int b = b0 + lane;
                uint32_t wv[6] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu};
                if (b < bend) {
                    const uint4 cur = v128[b];
                    wv[2] = cur.x; wv[3] = cur.y; wv[4] = cur.z; wv[5] = cur.w;
                    if (b > 0) {
                        const uint2 prv = *reinterpret_cast<const uint2*>(sm.vals + 16 * b - 8);
                        wv[0] = prv.x; wv[1] = prv.y;
                    }
                }
                uint32_t any = 0;
#pragma unroll
                for (int j2 = 2; j2 < 6; j2++) {
                    const uint32_t s1 = __funnelshift_l(wv[j2 - 1], wv[j2], 16);
                    const uint32_t s3 = __funnelshift_l(wv[j2 - 2], wv[j2 - 1], 16);
                    const uint32_t x1 = wv[j2] ^ s1, x2 = wv[j2] ^ wv[j2 - 1], x3 = wv[j2] ^ s3;
                    any |= ((x1 - 0x00010001u) & ~x1) | ((x2 - 0x00010001u) & ~x2) | ((x3 - 0x00010001u) & ~x3);
                }
                const bool has = (b < bend) && (any & 0x80008000u) != 0u;
                if (__any_sync(0xffffffffu, has)) {
                    uint32_t evs[8];
                    int ne = 0;
                    if (has) {
#pragma unroll
                        for (int h2 = 0; h2 < 8; h2++) {
                            const int k = 8 * b + h2;
                            const uint32_t wj = wv[2 + (h2 >> 1)], wp1 = wv[1 + (h2 >> 1)], wp2 = wv[(h2 >> 1)];
                            uint32_t pk, q1, q2, q3;
                            if (h2 & 1) { pk = wj >> 16; q1 = wj & 0xffffu; q2 = wp1 >> 16; q3 = wp1 & 0xffffu; }
                            else { pk = wj & 0xffffu; q1 = wp1 >> 16; q2 = wp1 & 0xffffu; q3 = wp2 >> 16; }
                            const uint32_t d = (pk == q1) ? 1u : (pk == q2) ? 2u : (pk == q3) ? 3u : 0u;
                            if (d && k < SCAN_END) evs[ne++] = ((uint32_t)k << 2) | d;
                        }
                    }
                    int incl = ne;
#pragma unroll
                    for (int off = 1; off < 32; off <<= 1) {
                        const int o = __shfl_up_sync(0xffffffffu, incl, off);
                        if (lane >= off) incl += o;
                    }
                    const int tot = __shfl_sync(0xffffffffu, incl, 31);
                    const int at = cnt + incl - ne;
                    for (int e = 0; e < ne; e++)
                        if (at + e < K1_EV_CAP) sm.ev[warp_id][at + e] = evs[e];
                    cnt += tot;
                }
            }
            if (lane == 0 && warp_id < NWS) sm.ev_n[warp_id] = cnt;
        }
        __syncthreads();
        // ---- the predecessor's hand-over, the walk from there, the hand-over to the successor
        if (tid == 0) {
            uint32_t P = pos0, base = 0u, abort_ = sm.any_reject ? 1u : 0u;
            if (w > 0) {
                while (chain[w * 4 + 3] != pp.epoch) __nanosleep(40);
                __threadfence();
                P = chain[w * 4 + 0]; base = chain[w * 4 + 1]; abort_ |= chain[w * 4 + 2];
            }
            int cur = (int)(P - O) >> 1, ci = 0, nb = 1, stop_at = -1;
            if (P < O || ((P - O) & 1u) || cur >= 64) abort_ = 1u;
            uint32_t count = 0u, pnext = 0u;
            if (!abort_) {
                constexpr int NWS = K1S_WARPS < 8 ? K1S_WARPS : 8;
                bool fail = false;
                sm.brk_ci[0] = 0; sm.brk_cur[0] = (unsigned short)cur;
                for (int wi = 0; wi < NWS && !fail && stop_at < 0; wi++) {
                    const int n = sm.ev_n[wi];
                    if (n > K1_EV_CAP) { fail = true; break; }
                    for (int e = 0; e < n; e++) {
                        const uint32_t evv = sm.ev[wi][e];
                        const int k = (int)(evv >> 2), d = (int)(evv & 3u);
                        if (k < cur) continue;
                        const int j = (k - cur) >> 2, spp = cur + 4 * j;
                        if (k - d < spp) continue;
                        if (spp >= L_PAIRS + 32) { stop_at = ci + j; break; }   // far enough into the margin
                        const int np = cand_pairs_len(pr16, spp, SCAN_END);
                        if (np < 0) { stop_at = ci + j; break; }
                        if (nb >= K1_BRK_CAP) { fail = true; break; }
                        ci += j + 1;
                        cur = spp + np;
                        sm.brk_ci[nb] = (unsigned short)ci;
                        sm.brk_cur[nb] = (unsigned short)cur;
                        nb++;
                    }
                }
                int n_ok = ci + ((SCAN_END - cur) >> 2);       // clean 4-pair candidates after the last break
                if (stop_at >= 0) n_ok = min(n_ok, stop_at);
                if (fail) abort_ = 1u;
                else {
                    // candidates that START before pair L_PAIRS: in the last break segment that begins before L_PAIRS
                    int m = 0;
                    while (m + 1 < nb && (int)sm.brk_cur[m + 1] < L_PAIRS) m++;
                    int cnt = (int)sm.brk_ci[m] + ((L_PAIRS - (int)sm.brk_cur[m] + 3) >> 2);
                    int start_pair;
                    if (m + 1 < nb && cnt >= (int)sm.brk_ci[m + 1]) { cnt = (int)sm.brk_ci[m + 1]; start_pair = (int)sm.brk_cur[m + 1]; }
                    else start_pair = (int)sm.brk_cur[m] + 4 * (cnt - (int)sm.brk_ci[m]);
                    if (cnt > n_ok || cnt < 1 || start_pair > SCAN_END - 8 || (long long)base + cnt > (long long)q.cap) abort_ = 1u;
                    count = (uint32_t)cnt;
                    pnext = O + 2u * (uint32_t)start_pair;
                    sm.brk_n = nb;
                }
            }
            if (abort_) { count = 0u; pnext = P; }
            // hand over to window w + 1 (the entry after the last window is the round's result, read below by the last CTA itself)
            chain[(w + 1) * 4 + 0] = pnext; chain[(w + 1) * 4 + 1] = base + count; chain[(w + 1) * 4 + 2] = abort_;
            __threadfence();
            chain[(w + 1) * 4 + 3] = pp.epoch;
            s_P = P; s_base = base; s_abort = abort_; s_count = count; s_pnext = pnext;
        }
        __syncthreads();
        const uint32_t base = s_base, count = s_count;
        if (!s_abort) {
            // ---- start offsets and the candidates themselves, at their final index
            const int nb = sm.brk_n;
            int m = 0;
            for (int i = tid; i <= (int)count; i += K1S_THREADS) {
                while (m + 1 < nb && (int)sm.brk_ci[m + 1] <= i) m++;
                sm.cand_start[i] = (unsigned short)(2 * ((int)sm.brk_cur[m] + 4 * (i - (int)sm.brk_ci[m])));
            }
            __syncthreads();
            for (int i = tid; i < (int)count; i += K1S_THREADS) {
                int cells[4];
                cand_parse_fast(sm.vals, sm.cand_start[i], w_avail, cells);
                q.cells[cbase + base + i] = make_uint2((uint32_t)cells[0] | ((uint32_t)cells[1] << 16), (uint32_t)cells[2] | ((uint32_t)cells[3] << 16));
                q.endw[cbase + base + i] = O + (uint32_t)sm.cand_start[i + 1];
            }
        }
        if (w == n_win - 1) {
            // ---- the last window closes the round: state, accept bits, work items (or the fresh state if the chain aborted)
            const int n_total = s_abort ? 0 : (int)(base + count);
            if (s_abort) {
                if (tid == 0) {
                    S.pos = pos0; S.gen = 0; S.acc = 0; S.cand_base = 0; S.n_round = 0; S.target = 0; S.done = 0; S.left_n = 0;
                    S.any_reject = 0; S.overflow = 0;
                }
            } else {
                const uint32_t P_end = s_pnext, gen = cur_block * (uint32_t)MT_N;
                const int left = min((int)(gen - P_end), K1S_LEFT_CAP), left_off = (int)(P_end - O);
                const uint32_t* half = sm.st + par * MT_N;
                for (int k = tid; k < MT_N; k += K1S_THREADS) S.mt[k] = half[k];
                for (int k = tid; k < left; k += K1S_THREADS) S.left[k] = sm.vals[left_off + k];
                uint32_t* ab = q.accbits + (size_t)slot * (q.cap >> 5);
                for (int k = tid; k < ((n_total + 31) >> 5); k += K1S_THREADS) ab[k] = 0u;
                const int n_items = (n_total + q.chunk - 1) / q.chunk;
                if (tid == 0) s_P = (uint32_t)atomicAdd(q.wq_n + q.qidx, n_items);
                __syncthreads();
                uint2* wq = q.wq + (size_t)q.qidx * q.wq_stride + s_P;
                for (int c = tid; c < n_items; c += K1S_THREADS)
                    wq[c] = make_uint2((uint32_t)slot * 128u + (uint32_t)c, (uint32_t)min(q.chunk, n_total - c * q.chunk));
                if (tid == 0) {
                    S.pos = P_end; S.gen = gen; S.acc = 0; S.cand_base = 0; S.n_round = n_total; S.target = n_total; S.done = 0;
                    S.left_n = left; S.any_reject = 0; S.overflow = (int)(gen - P_end) > K1S_LEFT_CAP ? 1 : 0;
                    if (q.dbg) { atomicAdd(q.dbg + 0, 1ull); atomicAdd(q.dbg + 1, (unsigned long long)n_total); }
                }
            }
        }
        __syncthreads();      // vals / event lists are reused by this CTA's next window
    }
}

// ------------------------------------------------------------------ k1_filter
// The filter's inputs straight from the cell table: bearings of points 0..2 from the stored 1/|(u, v, 1)|.
__device__ __forceinline__ bool k1_filter_candidate(const CellRec* cell, const int cells[4], double f, double cx, double cy,
                                                    double inv_f, double cx_f, double cy_f, double thr) {
    double bear[3][3], X[4][3], mu3 = 0, mv3 = 0;
#pragma unroll
    for (int j = 0; j < 4; j++) {
        const CellRec r = cell[cells[j]];
        const double mu = r.xn * f + cx, mv = r.yn * f + cy;
        X[j][0] = (double)r.X; X[j][1] = (double)r.Y; X[j][2] = (double)r.Z;
        if (j < 3) {
            const double u = inv_f * mu - cx_f, v = inv_f * mv - cy_f;
            bear[j][0] = u * r.k; bear[j][1] = v * r.k; bear[j][2] = r.k;
        } else {
            mu3 = mu; mv3 = mv;
        }
    }
    return p3p_quick_core(bear, X, mu3, mv3, f, cx, cy, thr);
}

#ifndef K1F_MAXREG
#define K1F_MAXREG 128   /* measured: 128 registers (no spills) beat 96 (+8 % filter time) even though 96 would leave room for a co-resident generator CTA */
#endif
struct K1FSmem {
    CellRec cell[2][DSAC_N_CONST];            // the frame's cell table, double-buffered: 2 x 38.4 KB
    unsigned short wlist[12][K1F_MAX_CHUNK / 8];   // per warp: flagged candidates of its share of the item (8 used; 12 keeps the measured layout)
    unsigned long long mbar[2];               // one transaction barrier per buffer
};

// The frame's 38 400-byte cell table reaches shared memory by TMA (tma_load_1d, kernels.cuh): one thread issues the bulk
// copy, the CTA waits on the transaction barrier, and the table of the NEXT work item is fetched into the other buffer
// while the warps filter the current one.
// One work item = up to `chunk` consecutive candidates of one stream.  After the cell table is in shared memory the
// warps run independently: a warp filters every (NTHREADS/32)-th group of 32 candidates of the item (coalesced 8-byte
// loads of the cell indices, the next group's prefetched), keeps the flagged ones in its own list and appends them to
// the global queue with one atomic per item.  A group barrier only when moving on to another frame's table.
// The CTA: NTHREADS threads; items first_item, first_item + item_stride, ...  The transaction barriers must have been
// initialised.
template <int NTHREADS>
__device__ __forceinline__ void k1_filter_body(const K1SplitParams& q, K1FSmem& sm, const int tid, const int first_item, const int item_stride) {
    const SampleParams& p = q.sp;
    const int lane = tid & 31, warp_id = tid >> 5;
    const int n_items = q.wq_n[q.qidx];
    const uint2* wq = q.wq + (size_t)q.qidx * q.wq_stride;
    const double inv_f = 1. / p.f, cx_f = p.cx * inv_f, cy_f = p.cy * inv_f;
    unsigned short* wl = sm.wlist[warp_id];
    constexpr uint32_t TABLE_BYTES = (uint32_t)(sizeof(CellRec) * DSAC_N_CONST);
    int cur = 0;
    int frame_in[2] = {-1, -1};          // frame whose table buffer b holds (or is receiving)
    uint32_t parity[2] = {0u, 0u};
    bool pending[2] = {false, false};    // a copy into buffer b has been issued and not yet waited for
    unsigned long long n_flagged = 0;
    int item = first_item;
    if (item < n_items) {
        const int f0 = (int)(wq[item].x >> 7) / p.T;
        if (tid == 0) tma_load_1d(sm.cell[0], q.celltab + (size_t)f0 * DSAC_N_CONST, TABLE_BYTES, &sm.mbar[0]);
        frame_in[0] = f0;
        pending[0] = true;
    }
    for (; item < n_items; item += item_stride) {
        const uint2 it2 = wq[item];
        const uint32_t it = it2.x;
        const int slot = (int)(it >> 7), chunk = (int)(it & 127u);
        const int frame = slot / p.T;           // == frame_in[cur]
        // the next item's table, into the other buffer (free: everybody left it at the last switch)
        const int nxt = item + item_stride;
        int nframe = frame;
        if (nxt < n_items) {
            nframe = (int)(wq[nxt].x >> 7) / p.T;
            if (nframe != frame && frame_in[cur ^ 1] != nframe) {
                if (tid == 0) tma_load_1d(sm.cell[cur ^ 1], q.celltab + (size_t)nframe * DSAC_N_CONST, TABLE_BYTES, &sm.mbar[cur ^ 1]);
                frame_in[cur ^ 1] = nframe;
                pending[cur ^ 1] = true;
            }
        }
        if (pending[cur]) {
            mbar_wait(&sm.mbar[cur], parity[cur]);
            parity[cur] ^= 1u;
            pending[cur] = false;
        }
        const CellRec* cell = sm.cell[cur];
        const int base = chunk * q.chunk;
        const int n_here = (int)it2.y;
        const uint2* cc = q.cells + (size_t)slot * q.cap + base;
        int cnt = 0;
        int i = warp_id * 32 + lane;
        uint2 c = (i < n_here) ? __ldg(cc + i) : make_uint2(0u, 0u);
        for (int i0 = warp_id * 32; i0 < n_here; i0 += NTHREADS) {
            i = i0 + lane;
            const int in = i + NTHREADS;
            const uint2 cn = (in < n_here) ? __ldg(cc + in) : make_uint2(0u, 0u);   // next group's cell indices
            bool need = false;
            if (i < n_here) {
                const int cells[4] = {(int)(c.x & 0xffffu), (int)(c.x >> 16), (int)(c.y & 0xffffu), (int)(c.y >> 16)};
                need = k1_filter_candidate(cell, cells, p.f, p.cx, p.cy, inv_f, cx_f, cy_f, (double)p.thr);
            }
            const uint32_t bits = __ballot_sync(0xffffffffu, need);
            if (need) wl[cnt + __popc(bits & ((1u << lane) - 1u))] = (unsigned short)(base + i);
            cnt += __popc(bits);
            c = cn;
        }
        __syncwarp();
        if (cnt > 0) {
            int at = 0;
            if (lane == 0) at = atomicAdd(q.fq_n + q.fqidx, cnt);
            at = __shfl_sync(0xffffffffu, at, 0);
            for (int k = lane; k < cnt; k += 32) q.fq[at + k] = ((uint32_t)slot << K1S_IDX_BITS) | (uint32_t)wl[k];
            n_flagged += (unsigned long long)cnt;
        }
        __syncwarp();
        if (nframe != frame) {   // moving to the other buffer: the one left behind may be overwritten from the next iteration on
            __syncthreads();
            cur ^= 1;
        }
    }
    if (q.dbg && lane == 0 && n_flagged) atomicAdd(q.dbg + (size_t)q.round * 4 + 2, n_flagged);
}

__global__ void __maxnreg__(K1F_MAXREG) k1_filter(K1SplitParams q) {
    extern __shared__ __align__(128) unsigned char k1f_smem_raw[];
    K1FSmem& sm = *reinterpret_cast<K1FSmem*>(k1f_smem_raw);
    if (threadIdx.x == 0) { mbar_init(&sm.mbar[0]); mbar_init(&sm.mbar[1]); }
    __syncthreads();
    k1_filter_body<K1F_THREADS>(q, sm, threadIdx.x, blockIdx.x, gridDim.x);
}

#ifndef K1V_GROUP
#define K1V_GROUP 1   /* lanes per flagged candidate: 4 = one quartic root per lane, 2 = two roots per lane, 1 = one thread per candidate */
#endif
#ifndef K1V_MIN_BLOCKS
#define K1V_MIN_BLOCKS 4
#endif
template <int GROUP>
__device__ __forceinline__ void k1_solve_body(const K1SplitParams& q) {
    const SampleParams& p = q.sp;
    const int tid = threadIdx.x;
    constexpr int GROUPS = K1V_THREADS / GROUP, ROOTS = 4 / GROUP;
    const int n_q = q.fq_n[q.fqidx];
    const int sub = tid % GROUP;
    for (int base = blockIdx.x * GROUPS; base < n_q; base += gridDim.x * GROUPS) {
        const int qi = base + tid / GROUP;
        bool ok = false, fragile = false;
        double rvec[3], tvec[3];
        double e2 = 1.7976931348623157e308, R[9], t[3];
        float obj[12], img[8];
        int nsol = 0, slot = 0, ci = 0;
        if (qi < n_q) {
            const uint32_t ent = q.fq[qi];
            slot = (int)(ent >> K1S_IDX_BITS);
            ci = (int)(ent & ((1u << K1S_IDX_BITS) - 1u));
            const int frame = slot / p.T;
            const uint2 c = q.cells[(size_t)slot * q.cap + ci];
            const int cells[4] = {(int)(c.x & 0xffffu), (int)(c.x >> 16), (int)(c.y & 0xffffu), (int)(c.y >> 16)};
            const CellRec* cell = q.celltab + (size_t)frame * DSAC_N_CONST;
            const int32_t* pix = p.pix + (size_t)frame * p.pix_stride;
            P3PProblem pr;
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const CellRec r = cell[cells[j]];
                pr.mu[j] = r.xn * p.f + p.cx;   // float * double
                pr.mv[j] = r.yn * p.f + p.cy;
                pr.X[j][0] = (double)r.X; pr.X[j][1] = (double)r.Y; pr.X[j][2] = (double)r.Z;
                obj[j * 3] = (float)pr.X[j][0]; obj[j * 3 + 1] = (float)pr.X[j][1]; obj[j * 3 + 2] = (float)pr.X[j][2];
                img[j * 2] = (float)__ldg(pix + cells[j] * 2);
                img[j * 2 + 1] = (float)__ldg(pix + cells[j] * 2 + 1);
            }
            P3PFront fr;
            p3p_front(pr, p.f, p.cx, p.cy, fr);
            nsol = p3p_full(pr, fr, p.f, p.cx, p.cy, R, t, &e2, sub * ROOTS, (sub + 1) * ROOTS);
            if (nsol == 0) e2 = 1.7976931348623157e308;
        }
        // minimum over the group; ties go to the lower root index, as the sequential loop would
        double be = e2;
        int bl = sub;
#pragma unroll
        for (int off = 1; off < GROUP; off <<= 1) {
            double oe = __shfl_xor_sync(0xffffffffu, be, off);
            int ol = __shfl_xor_sync(0xffffffffu, bl, off);
            if (oe < be || (oe == be && ol < bl)) { be = oe; bl = ol; }
        }
        if (nsol > 0 && bl == sub)
            ok = minimal_set_accept(obj, img, p.f, p.cx, p.cy, p.thr, R, t, e2, rvec, tvec, &fragile);
        if (fragile) atomicAdd(p.n_fragile, 1ull);
        if (ok) {
            double* po = q.pose_out + ((size_t)slot * q.cap + ci) * 6;
            po[0] = rvec[0]; po[1] = rvec[1]; po[2] = rvec[2];
            po[3] = tvec[0]; po[4] = tvec[1]; po[5] = tvec[2];
            atomicOr(q.accbits + (size_t)slot * (q.cap >> 5) + (ci >> 5), 1u << (ci & 31));
        }
    }
}

// one thread per flagged candidate when there are many (a full batch: fewer, fuller warps), four lanes per candidate -- one quartic
// root each, the same minimum with the same tie rule -- when there are few (single-frame latency: the launch lasts as long as one
// candidate's chain, and the four roots are that chain's longest part)
__global__ void __launch_bounds__(K1V_THREADS, K1V_MIN_BLOCKS) k1_solve(K1SplitParams q) { k1_solve_body<K1V_GROUP>(q); }
__global__ void __launch_bounds__(K1V_THREADS, K1V_MIN_BLOCKS) k1_solve4(K1SplitParams q) { k1_solve_body<4>(q); }

}  // namespace dsac
