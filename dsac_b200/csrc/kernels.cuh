// kernels.cuh -- sm_100a kernels of the forward pass.
//
//   k_sample  (K1)  minimal-set sampling: device MT19937 streams -> candidates -> fp64 P3P ->
//                   reprojection check -> ordered compaction of the first H accepted per
//                   stream                           (cnn_softam.h:1010-1060)
//   k_score   (K2)  fused HxN reprojection-error matrix + soft-inlier score; the last CTA of a
//                   frame finishes softmax / entropy / soft-argmax (K3)
//                                                    (cnn_softam.h:1065-1094, :319-362, :535-553, :80-88)
//
// No tensor cores anywhere: the work is point-wise + reductions (see DESIGN.md).
#pragma once
#include <cuda_runtime.h>

#include "pose_math.cuh"
#include "sampler.cuh"

namespace dsac {

// ------------------------------------------------------------------ block helpers
// Exclusive prefix sum over a block of NWARPS warps (+ block total).  One barrier: consecutive calls must
// use different s_warp buffers.
template <int NWARPS>
__device__ __forceinline__ int block_excl_scan(int v, int* total, int* s_warp /* >= NWARPS ints */, int tid = -1) {
    if (tid < 0) tid = threadIdx.x;
    const int lane = tid & 31, warp = tid >> 5;
    int incl = v;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        int n = __shfl_up_sync(0xffffffffu, incl, off);
        if (lane >= off) incl += n;
    }
    if (lane == 31) s_warp[warp] = incl;   // callers alternate between two s_warp buffers
    __syncthreads();
    int base = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < NWARPS; w++) {
        int x = s_warp[w];
        if (w < warp) base += x;
        tot += x;
    }
    *total = tot;
    return base + incl - v;
}

// ------------------------------------------------------------------ TMA staging helpers
// 1-D bulk copy global -> shared memory (cp.async.bulk, SASS UBLKCP) completing on a transaction barrier: one thread
// issues it, everybody who reads the data waits on the barrier.  Sizes and addresses are multiples of 16 bytes.
__device__ __forceinline__ uint32_t smem_addr_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void tma_load_1d(void* dst_smem, const void* src_gmem, uint32_t bytes, unsigned long long* mbar) {
    const uint32_t d = smem_addr_u32(dst_smem), m = smem_addr_u32(mbar);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // earlier generic-proxy reads of the buffer are done (barrier), order them before the async write
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(m), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(d), "l"(src_gmem), "r"(bytes), "r"(m)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* mbar, uint32_t parity) {
    const uint32_t m = smem_addr_u32(mbar);
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "DSAC_MBAR_WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@!p bra DSAC_MBAR_WAIT_%=;\n"
        "}\n" ::"r"(m), "r"(parity)
        : "memory");
}

__device__ __forceinline__ void mbar_init(unsigned long long* mbar) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_addr_u32(mbar)) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

// ------------------------------------------------------------------ K1: sampling
constexpr int K1S_LEFT_CAP = 2048;               // decoded words carried from one round of the split sampler to the next

// Stream state the split sampler (sampler_split.cuh) carries between its rounds, one per (frame, stream); k_sample
// resumes from it (SampleParams::resume) for the streams the rounds left unfinished.
struct K1SlotState {
    uint32_t mt[624];           // MT19937 state that regenerates the stream words [gen, gen + 624)
    uint32_t pos, gen;          // next unread stream word; words generated so far (a multiple of 624)
    int32_t acc;                // hypotheses accepted so far
    int32_t n_round;            // candidates of the current round
    int32_t done;               // quota reached
    int32_t left_n;             // decoded words [pos, gen) kept in left[]
    int32_t any_reject;         // left[] contains a rejected draw (value 255)
    int32_t overflow;           // leftover did not fit (cannot happen with the window sizes used; checked by the host)
    int32_t target;             // candidates the current round shall reach (generated in portions, see sampler_split.cuh)
    int32_t pad_;
    long long cand_base;        // candidates consumed before the current round
    unsigned char left[K1S_LEFT_CAP];
};

struct SampleParams {
    const int16_t* coords;   // [n][N][3]
    const int32_t* pix;      // [n or 1][N][2]
    int pix_stride;          // N*2 or 0 (shared grid)
    double f, cx, cy;
    int H, T, thr;
    uint32_t seed, skip;
    int max_candidates;
    long long frame0;
    double* hyp_pose;        // [n][H][6]
    float* hyp_P;            // [n][H][12]  rows (f*R0|f*t0), (f*R1|f*t1), (R2|t2) in float for K2
    int32_t* img_idx;        // [n][H][4]
    int32_t* cand_idx;       // [n][H]
    long long* stream_ncand; // [n][T]
    unsigned long long* stream_endpos;  // [n][T] stream words consumed when the stream's last hypothesis was accepted
    uint32_t* status;        // [n]
    unsigned long long* n_fragile;  // [1]
    unsigned long long* phase_cycles;  // [8] or null: thread-0 cycles per phase (development aid)
    int a2_generic;                    // 1: always take the general boundary path (test aid, DSAC_K1_A2_GENERIC=1)
    const K1SlotState* resume;         // null: streams start at their seed; else continue the split sampler's streams
};

#ifndef K1_THREADS_DEF
#define K1_THREADS_DEF 384
#endif
constexpr int K1_THREADS = K1_THREADS_DEF;
constexpr int K1_WARPS = K1_THREADS / 32;
#ifndef K1_MIN_BLOCKS
#define K1_MIN_BLOCKS 2
#endif
#ifndef K1_SUPER_CANDS
#define K1_SUPER_CANDS 4096
#endif
static_assert(K1_SUPER_CANDS <= 4096, "phase C packs a super-round's flags in 128 words");
constexpr int K1_SUPER_MAX = K1_SUPER_CANDS / K1_THREADS;  // super-round = up to K1_SUPER_CANDS candidates
constexpr int K1_CANDS = K1_SUPER_MAX * K1_THREADS;       // candidates buffered per super-round
constexpr int K1_WORDS = K1_CANDS * 8 + 1024;             // decoded stream words buffered per super-round
#ifndef K1_GEN624
#define K1_GEN624 1                                       // 1: a whole state regeneration (624 words) per barrier; 0: 227-word waves
#endif
constexpr int K1_WAVE = MT_N - MT_M;                      // 227 MT19937 words are mutually independent
constexpr int K1_EV_CAP = 64;                             // repeated-pair events buffered per warp and super-round (expected: ~4)
constexpr int K1_BRK_CAP = 160;                           // candidates with a repeated cell per super-round (expected: ~16)

// Per-cell record staged in shared memory: scene coordinate (mm) and the float-rounded
// normalised pixel that cv::undistortPoints hands to P3P.
struct __align__(8) CellRec {
    short X, Y, Z, pad;   // scene coordinate, mm
    float xn, yn;         // normalised pixel rounded to float (cv::undistortPoints), see p3p_pixel
    double k;             // 1 / |(u, v, 1)| of the bearing P3P derives from it (used by the filter only)
};

struct K1Smem {
    CellRec cell[DSAC_N_CONST];
#if K1_GEN624
    uint32_t st[2 * MT_N];                      // MT19937 state, double-buffered (old / new generation)
#else
    uint32_t st[1024];                          // sliding window of the raw MT19937 sequence (linear index & 1023)
#endif
    __align__(4) unsigned char vals[K1_WORDS];  // Lemire value (0..39) of stream word pos+i; 255 = rejected draw
    unsigned short cand_start[K1_CANDS + 512];    // word offset (from pos) where candidate i starts
    unsigned short q_idx[K1_CANDS];             // queue of candidates that need the full solve, ascending
    uint32_t flagbits[K1_CANDS / 32];
    uint32_t wordbase[K1_CANDS / 32];
    int warp[2][K1_WARPS];
    uint32_t newpos;
    int q_n, n_sr, any_reject, walk_fail;
    // event-based boundary phase: repeated (x, y) pairs found by each warp in its segment of the window, and the
    // resulting breaks of the 8-words-per-candidate rhythm
    uint32_t ev[K1_WARPS][K1_EV_CAP];           // (pair index << 2) | distance to the equal predecessor (1..3)
    int ev_n[K1_WARPS];
    unsigned short brk_ci[K1_BRK_CAP], brk_cur[K1_BRK_CAP];   // from candidate brk_ci on, candidates start at pair brk_cur + 4*(i - brk_ci)
    int brk_n;
};

// 4 distinct cells (x, y drawn in that order, a repeated cell is re-drawn: cnn_softam.h:1021-1039)
// from the decoded value stream starting at word offset q; returns the offset after the candidate,
// or -1 if the buffered words run out.  255 marks a word libstdc++'s Lemire loop rejects.
__device__ __forceinline__ int cand_parse(const unsigned char* vals, int q, int limit, int cells[4]) {
    int n = 0;
    while (n < 4) {
        int vx, vy;
        do {
            if (q >= limit) return -1;
            vx = vals[q++];
        } while (vx == 255);
        do {
            if (q >= limit) return -1;
            vy = vals[q++];
        } while (vy == 255);
        int c = vy * DSAC_GRID_CONST + vx;
        bool dup = false;
#pragma unroll
        for (int j = 0; j < 3; j++)
            if (j < n && cells[j] == c) dup = true;
        if (!dup) cells[n++] = c;
    }
    return q;
}

// Common case of cand_parse in ~25 instructions: 8 words at an even offset, no rejected draw, 4 distinct
// cells.  Falls back to the generic parser otherwise.
__device__ __forceinline__ int cand_parse_fast(const unsigned char* vals, int q, int limit, int cells[4]) {
    if (q + 8 <= limit && !(q & 1)) {
        const unsigned short* v16 = reinterpret_cast<const unsigned short*>(vals + q);
        const unsigned a0 = v16[0], a1 = v16[1], a2 = v16[2], a3 = v16[3];   // (y << 8) | x
        const unsigned any = a0 | a1 | a2 | a3;      // values are <= 39 or exactly 255: bit 7 set <=> some byte is 255
        const int c0 = (a0 >> 8) * DSAC_GRID_CONST + (a0 & 255), c1 = (a1 >> 8) * DSAC_GRID_CONST + (a1 & 255);
        const int c2 = (a2 >> 8) * DSAC_GRID_CONST + (a2 & 255), c3 = (a3 >> 8) * DSAC_GRID_CONST + (a3 & 255);
        const bool distinct = (c0 != c1) & (c0 != c2) & (c0 != c3) & (c1 != c2) & (c1 != c3) & (c2 != c3);
        if (!(any & 0x8080u) && distinct) {
            cells[0] = c0; cells[1] = c1; cells[2] = c2; cells[3] = c3;
            return q + 8;
        }
    }
    return cand_parse(vals, q, limit, cells);
}

// One CTA per (frame, stream).  Per super-round of up to S x 256 candidates:
//   A  MT19937 in waves of 227 words (one barrier each), every word decoded on the fly to its
//      uniform_int_distribution value; candidate boundaries by a block-wide fixed point over per-thread runs
//   B  cheap conservative filter, one thread per candidate, no block barriers
//   C  queue the ~2% that need the full fp64 P3P, in candidate order
//   D  full solve + reprojection check on the queue, ordered compaction of the accepted
__global__ void __launch_bounds__(K1_THREADS, K1_MIN_BLOCKS) k_sample(SampleParams p) {
    extern __shared__ __align__(16) unsigned char k1_smem_raw[];
    K1Smem& sm = *reinterpret_cast<K1Smem*>(k1_smem_raw);

    const int tid = threadIdx.x, lane = tid & 31;
    const int s = blockIdx.x, frame = blockIdx.y;
    int h0, quota;
    stream_chunk(p.H, p.T, s, &h0, &quota);
    if (quota == 0) {
        if (tid == 0) {
            p.stream_ncand[(size_t)frame * p.T + s] = 0;
            p.stream_endpos[(size_t)frame * p.T + s] = 0;
        }
        return;
    }

    const K1SlotState* rs = p.resume ? p.resume + ((size_t)frame * p.T + s) : nullptr;
    if (rs && rs->done) return;
    if (rs && rs->overflow) rs = nullptr;   // the leftover of a round did not fit the state (cannot happen with the window sizes used): redo the stream from its seed
    // stream s of global frame g: mt19937(seed + g*T + s)   (thread_rand.cpp:52 for g = 0)
    if (!rs && tid == 0) mt_seed(sm.st, p.seed + (uint32_t)((p.frame0 + frame) * (long long)p.T + s));

    const int16_t* coords = p.coords + (size_t)frame * DSAC_N_CONST * 3;
    const int32_t* pix = p.pix + (size_t)frame * p.pix_stride;
    const double k1_inv_f = 1. / p.f, k1_cx_f = p.cx * k1_inv_f, k1_cy_f = p.cy * k1_inv_f;
    {
        for (int c = tid; c < DSAC_N_CONST; c += K1_THREADS) {
            CellRec r;
            r.X = __ldg(coords + c * 3); r.Y = __ldg(coords + c * 3 + 1); r.Z = __ldg(coords + c * 3 + 2); r.pad = 0;
            r.xn = (float)(((double)__ldg(pix + c * 2) - p.cx) * k1_inv_f);       // cv::undistortPoints rounds to float (p3p_pixel)
            r.yn = (float)(((double)__ldg(pix + c * 2 + 1) - p.cy) * k1_inv_f);
            const double mu = r.xn * p.f + p.cx, mv = r.yn * p.f + p.cy;        // float * double
            const double u = k1_inv_f * mu - k1_cx_f, v = k1_inv_f * mv - k1_cy_f;
            r.k = rsqrt(u * u + v * v + 1);
            sm.cell[c] = r;
        }
    }
    if (tid == 0) { sm.any_reject = rs ? rs->any_reject : 0; sm.walk_fail = 0; }
    uint32_t pos = (s == 0) ? p.skip : 0u;  // stream position (output word index) of the next unread word
    uint32_t gen = 0;                       // output words generated so far (linear MT index = gen + 624)
    int acc = 0;                            // hypotheses accepted so far
    long long cand_base = 0;                // candidates consumed so far
#if K1_GEN624
    if (rs) {   // continue where the split sampler's last round stopped
        pos = rs->pos; gen = rs->gen; acc = rs->acc; cand_base = rs->cand_base;
        uint32_t* half = sm.st + ((gen / MT_N) & 1u) * MT_N;
        for (int k = tid; k < MT_N; k += K1_THREADS) half[k] = rs->mt[k];
        const int ln = rs->left_n;
        for (int k = tid; k < ln; k += K1_THREADS) sm.vals[k] = rs->left[k];
    }
#endif
    __syncthreads();

    const long long cand_max = p.max_candidates > 0 ? (long long)p.max_candidates : (1ll << 40);
    int S = 4;                              // x256 candidates in the next super-round (adapted to the acceptance rate)

    auto load_problem = [&](const int cells[4], P3PProblem& pr) {
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const CellRec r = sm.cell[cells[j]];
            pr.mu[j] = r.xn * p.f + p.cx;   // float * double
            pr.mv[j] = r.yn * p.f + p.cy;
            pr.X[j][0] = (double)r.X; pr.X[j][1] = (double)r.Y; pr.X[j][2] = (double)r.Z;
        }
    };
    // the filter's inputs straight from the cell table: bearings of points 0..2 from the stored 1/|(u, v, 1)|
    auto filter_candidate = [&](const int cells[4]) -> bool {
        double bear[3][3], X[4][3], mu3 = 0, mv3 = 0;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const CellRec r = sm.cell[cells[j]];
            const double mu = r.xn * p.f + p.cx, mv = r.yn * p.f + p.cy;
            X[j][0] = (double)r.X; X[j][1] = (double)r.Y; X[j][2] = (double)r.Z;
            if (j < 3) {
                const double u = k1_inv_f * mu - k1_cx_f, v = k1_inv_f * mv - k1_cy_f;
                bear[j][0] = u * r.k; bear[j][1] = v * r.k; bear[j][2] = r.k;
            } else {
                mu3 = mu; mv3 = mv;
            }
        }
        return p3p_quick_core(bear, X, mu3, mv3, p.f, p.cx, p.cy, (double)p.thr);
    };

    long long tA1 = 0, tA2 = 0, tB = 0, tC = 0, tD = 0, tE = 0, tmark = clock64();
#define K1_MARK(var) do { long long _n = clock64(); var += _n - tmark; tmark = _n; } while (0)
    while (acc < quota && cand_base < cand_max) {
        // ---------------- phase A1: generate + decode words until the super-round's window is full
        long long want = (long long)S * K1_THREADS;
        if (cand_max - cand_base < want) want = cand_max - cand_base;
        const int n_target = (int)want;
#if K1_GEN624
        const int w_need = min(K1_WORDS - 640, n_target * 8 + 768);   // a regeneration may overshoot by 623 words
#else
        const int w_need = min(K1_WORDS - 256, n_target * 8 + 768);   // a wave may overshoot by 226 words
#endif
        // (leftover words [pos, gen) were moved to vals[0..gen-pos) at the end of the previous super-round)
#if K1_GEN624
        // One whole regeneration of the MT19937 state (624 words) per barrier (mt_regenerate_words, sampler.cuh): thread
        // t < 227 produces the words t, t+227, t+454 from its own previous result and OLD neighbours, which are read from the
        // other half of the double-buffered state.  No hazard inside the interval, 2.75x fewer barriers than 227-word waves.
        while ((int)(gen - pos) < w_need) {
            const uint32_t* so = sm.st + ((gen / MT_N) & 1u) * MT_N;           // old state
            uint32_t* sn = sm.st + (((gen / MT_N) & 1u) ^ 1u) * MT_N;            // new state
            if (tid < K1_WAVE) {
                uint32_t x[3];
                const bool has3 = mt_regenerate_words(so, tid, x) == 3;
#pragma unroll
                for (int w = 0; w < 3; w++) {
                    if (w < 2 || has3) {
                        const int k = tid + w * K1_WAVE;
                        sn[k] = x[w];
                        const int off = (int)(gen - pos) + k;
                        if (off >= 0 && off < K1_WORDS) {
                            const uint64_t prod = (uint64_t)mt_temper(x[w]) * DSAC_GRID_CONST;
                            const bool rej = (uint32_t)prod < ((0u - DSAC_GRID_CONST) % DSAC_GRID_CONST);  // Lemire: low < 2^32 mod 40
                            sm.vals[off] = rej ? (unsigned char)255 : (unsigned char)(prod >> 32);
                            if (rej) sm.any_reject = 1;
                        }
                    }
                }
            }
            gen += MT_N;
            __syncthreads();
        }
#else
        while ((int)(gen - pos) < w_need) {
            for (int el = tid; el < K1_WAVE; el += K1_THREADS) {
                uint32_t n = gen + MT_N + el;  // linear index of the new element
                uint32_t x = mt_twist(sm.st[(n - MT_N) & 1023], sm.st[(n - MT_N + 1) & 1023], sm.st[(n - K1_WAVE) & 1023]);
                sm.st[n & 1023] = x;
                int off = (int)(gen + el - pos);
                if (off >= 0 && off < K1_WORDS) {
                    uint64_t prod = (uint64_t)mt_temper(x) * DSAC_GRID_CONST;
                    bool rej = (uint32_t)prod < ((0u - DSAC_GRID_CONST) % DSAC_GRID_CONST);  // Lemire: low < 2^32 mod 40
                    sm.vals[off] = rej ? (unsigned char)255 : (unsigned char)(prod >> 32);
                    if (rej) sm.any_reject = 1;
                }
            }
            gen += K1_WAVE;
            __syncthreads();
        }
#endif
        const int w_avail = min((int)(gen - pos), K1_WORDS);
        K1_MARK(tA1);

        // ---------------- phase A2: candidate boundaries.  A candidate is 8 words (4 (x, y) pairs) long unless a cell
        // repeats (+2 words) or a draw is rejected (+1).  Fast path (no rejected draw in the window): every warp scans
        // a segment of the window for pairs equal to one of their three predecessors -- the only way four consecutive
        // pairs can fail to be distinct -- (~30 events per super-round); thread 0 walks the events in order, parses the
        // few candidates that really contain a repeat with the generic parser, and records where the 4-pair rhythm
        // breaks; every thread then derives its candidates' starts from the break list.  Three barriers per
        // super-round.  Windows with a rejected draw (one per ~2000 frames) or an overflowing list take the
        // general fixed-point path below.
        bool a2_done = false;
        if (!sm.any_reject && !p.a2_generic) {
            const unsigned short* pr16 = reinterpret_cast<const unsigned short*>(sm.vals);
            const int scan_end = min(w_avail >> 1, n_target * 4 + 384);
            const int warp_id = tid >> 5;
            const int seg = (((scan_end + K1_WARPS - 1) / K1_WARPS) + 31) & ~31;
            const int wbeg = warp_id * seg, wend = min(wbeg + seg, scan_end);
            int cnt = 0;
            for (int k0 = wbeg; k0 < wend; k0 += 32) {
                const int k = k0 + lane;
                // pair k against its three predecessors: neighbours' values by shuffle, lanes 0..2 fetch theirs
                const unsigned pk = (k < scan_end) ? pr16[k] : 0xffffu;
                unsigned p1 = __shfl_up_sync(0xffffffffu, pk, 1), p2 = __shfl_up_sync(0xffffffffu, pk, 2), p3 = __shfl_up_sync(0xffffffffu, pk, 3);
                if (lane < 3) {
                    if (lane < 1) p1 = (k >= 1) ? pr16[k - 1] : 0xffffu;
                    if (lane < 2) p2 = (k >= 2) ? pr16[k - 2] : 0xffffu;
                    p3 = (k >= 3) ? pr16[k - 3] : 0xffffu;
                }
                unsigned d = 0;
                if (k < wend) d = (pk == p1) ? 1u : (pk == p2) ? 2u : (pk == p3) ? 3u : 0u;
                const unsigned m = __ballot_sync(0xffffffffu, d != 0);
                if (d) {
                    const int slot = cnt + __popc(m & ((1u << lane) - 1u));
                    if (slot < K1_EV_CAP) sm.ev[warp_id][slot] = ((uint32_t)k << 2) | d;
                }
                cnt += __popc(m);
            }
            if (lane == 0) sm.ev_n[warp_id] = cnt;
            __syncthreads();
            if (tid == 0) {
                int cur = 0, ci = 0, nb = 1, stop_at = -1;
                bool fail = false;
                sm.brk_ci[0] = 0; sm.brk_cur[0] = 0;
                for (int w = 0; w < K1_WARPS && !fail && stop_at < 0; w++) {
                    const int n = sm.ev_n[w];
                    if (n > K1_EV_CAP) { fail = true; break; }
                    for (int e = 0; e < n; e++) {
                        const uint32_t evv = sm.ev[w][e];
                        const int k = (int)(evv >> 2), d = (int)(evv & 3u);
                        if (k < cur) continue;                 // inside a candidate already parsed
                        const int j = (k - cur) >> 2, sp = cur + 4 * j;
                        if (k - d < sp) continue;              // the equal pair belongs to the previous candidate
                        if (ci + j >= n_target) { stop_at = n_target; break; }
                        const int np = cand_pairs_len(pr16, sp, scan_end);
                        if (np < 0) { stop_at = ci + j; break; }   // window ends inside this candidate
                        if (nb >= K1_BRK_CAP) { fail = true; break; }
                        ci += j + 1;
                        cur = sp + np;
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
            if (!sm.walk_fail) {
                const int n_ok = sm.n_sr, nb = sm.brk_n;
                int m = 0;
                for (int i = tid; i <= n_ok; i += K1_THREADS) {
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
                const int n_chunk = min(K1_THREADS, n_target - n_done);
                int extra = 0, start = 0, qn = 0;
                for (;;) {
                    int tot;
                    const int excl = block_excl_scan<K1_WARPS>(extra, &tot, sm.warp[par]);
                    par ^= 1;
                    start = rp + 8 * tid + excl;
                    int cells[4];
                    qn = (tid < n_chunk) ? cand_parse_fast(sm.vals, start, w_avail, cells) : start + 8;
                    const int ne = (qn < 0) ? 0 : (qn - start) - 8;
                    const int changed = (ne != extra);
                    extra = ne;
                    if (!__syncthreads_or(changed)) break;
                }
                // (practically never) the buffered words ran out inside this chunk: keep the complete prefix
                int bad = (tid < n_chunk && qn < 0) ? tid : K1_THREADS;
#pragma unroll
                for (int off = 16; off; off >>= 1) bad = min(bad, __shfl_xor_sync(0xffffffffu, bad, off));
                if (lane == 0) sm.warp[par][tid >> 5] = bad;
                __syncthreads();
                int n_ok = n_chunk;
#pragma unroll
                for (int w = 0; w < K1_WARPS; w++) n_ok = min(n_ok, sm.warp[par][w]);
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
        const int n_sr = sm.n_sr;
        K1_MARK(tA2);

        // ---------------- phase B: conservative filter, warps run without block barriers
        for (int i0 = 0; i0 < n_sr; i0 += K1_THREADS) {
            const int i = i0 + tid;
            bool need = false;
            if (i < n_sr) {
                int cells[4];
                cand_parse_fast(sm.vals, sm.cand_start[i], w_avail, cells);
                need = filter_candidate(cells);
            }
            uint32_t bits = __ballot_sync(0xffffffffu, need);
            if (lane == 0) sm.flagbits[i >> 5] = bits;
        }
        __syncthreads();

        K1_MARK(tB);
        // ---------------- phase C: queue of flagged candidates in candidate order
        const int n_words = (n_sr + 31) >> 5;   // <= 128
        if (tid < 32) {
            int cnt[4], sum = 0;
#pragma unroll
            for (int k = 0; k < 4; k++) {
                int w = tid * 4 + k;
                cnt[k] = (w < n_words) ? __popc(sm.flagbits[w]) : 0;
                sum += cnt[k];
            }
            int incl = sum;
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
                int nb = __shfl_up_sync(0xffffffffu, incl, off);
                if (lane >= off) incl += nb;
            }
            int run = incl - sum;
#pragma unroll
            for (int k = 0; k < 4; k++) {
                int w = tid * 4 + k;
                if (w < n_words) sm.wordbase[w] = run;
                run += cnt[k];
            }
            if (tid == 31) sm.q_n = incl;
        }
        __syncthreads();
        for (int i = tid; i < n_sr; i += K1_THREADS) {
            uint32_t wbits = sm.flagbits[i >> 5];
            if ((wbits >> (i & 31)) & 1u)
                sm.q_idx[sm.wordbase[i >> 5] + __popc(wbits & ((1u << (i & 31)) - 1u))] = (unsigned short)i;
        }
        __syncthreads();
        const int q_n = sm.q_n;
        K1_MARK(tC);

        // ---------------- phase D: full fp64 P3P + reprojection check (cnn_softam.h:1041-1059) on the
        //                  queue, then the first `quota` accepted candidates of the stream, in order
        int par = 0;
        constexpr int GROUP = 4;   // lanes per flagged candidate: lane `sub` handles quartic root `sub`
        for (int base = 0; base < q_n && acc < quota; base += K1_THREADS / GROUP, par ^= 1) {
            const int qi = base + tid / GROUP, sub = tid % GROUP;
            bool ok = false, fragile = false;
            double rvec[3], tvec[3];
            int cells[4] = {0, 0, 0, 0};
            long long cand = 0;
            double e2 = 1.7976931348623157e308, R[9], t[3];
            float obj[12], img[8];
            int nsol = 0, ci_keep = 0;
            if (qi < q_n) {
                int ci = sm.q_idx[qi];
                ci_keep = ci;
                cand_parse_fast(sm.vals, sm.cand_start[ci], w_avail, cells);
                cand = cand_base + ci;
                P3PProblem pr;
                load_problem(cells, pr);
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    obj[j * 3] = (float)pr.X[j][0]; obj[j * 3 + 1] = (float)pr.X[j][1]; obj[j * 3 + 2] = (float)pr.X[j][2];
                    img[j * 2] = (float)__ldg(pix + cells[j] * 2);
                    img[j * 2 + 1] = (float)__ldg(pix + cells[j] * 2 + 1);
                }
                P3PFront fr;
                p3p_front(pr, p.f, p.cx, p.cy, fr);
                nsol = p3p_full(pr, fr, p.f, p.cx, p.cy, R, t, &e2, sub, sub + 1);
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
            int tot;
            int rank = acc + block_excl_scan<K1_WARPS>(ok ? 1 : 0, &tot, sm.warp[par]);
            if (ok && rank < quota) {
                size_t hi = (size_t)frame * p.H + h0 + rank;
                double* hp = p.hyp_pose + hi * 6;
                hp[0] = rvec[0]; hp[1] = rvec[1]; hp[2] = rvec[2];
                hp[3] = tvec[0]; hp[4] = tvec[1]; hp[5] = tvec[2];
                double Rm[9];
                rodrigues_v2m(rvec, Rm);  // getDiffMap -> cv::projectPoints rebuilds R from rvec
                float4* P = reinterpret_cast<float4*>(p.hyp_P + hi * 12);
                P[0] = make_float4((float)(p.f * Rm[0]), (float)(p.f * Rm[1]), (float)(p.f * Rm[2]), (float)(p.f * tvec[0]));
                P[1] = make_float4((float)(p.f * Rm[3]), (float)(p.f * Rm[4]), (float)(p.f * Rm[5]), (float)(p.f * tvec[1]));
                P[2] = make_float4((float)Rm[6], (float)Rm[7], (float)Rm[8], (float)tvec[2]);
                *reinterpret_cast<int4*>(p.img_idx + hi * 4) = make_int4(cells[0], cells[1], cells[2], cells[3]);
                p.cand_idx[hi] = (int32_t)cand;
                if (rank == quota - 1) {
                    p.stream_ncand[(size_t)frame * p.T + s] = cand + 1;
                    p.stream_endpos[(size_t)frame * p.T + s] = (unsigned long long)pos + sm.cand_start[ci_keep + 1];
                }
            }
            acc += tot;
        }

        K1_MARK(tD);
        // ---------------- advance the stream: the unread tail of the window moves to the front
        {
            const int consumed = sm.cand_start[n_sr];
            const int left = w_avail - consumed;     // == gen - (pos + consumed) whenever w_avail == gen - pos
            unsigned char keep[(K1_WORDS / K1_THREADS) + 1];
            __syncthreads();
            if (acc < quota) {
#pragma unroll 1
                for (int k = 0, i = tid; i < left; i += K1_THREADS, k++) keep[k] = sm.vals[consumed + i];
            }
            __syncthreads();
            bool rej_left = false;
            if (acc < quota) {
#pragma unroll 1
                for (int k = 0, i = tid; i < left; i += K1_THREADS, k++) {
                    sm.vals[i] = keep[k];
                    rej_left |= (keep[k] == 255);
                }
            }
            if (tid == 0) { sm.any_reject = 0; sm.walk_fail = 0; }
            __syncthreads();
            if (rej_left) sm.any_reject = 1;   // a rejected draw carried over into the next window
            pos += (uint32_t)consumed;
            cand_base += n_sr;
        }
        // next super-round: as many candidates as the observed acceptance rate suggests are still needed
        if (acc < quota) {
            if (acc > 0) {
                double need_c = (double)(quota - acc) * (double)cand_base / (double)acc * 1.1;
                int r = (int)(need_c / K1_THREADS) + 1;
                S = r < 1 ? 1 : (r > K1_SUPER_MAX ? K1_SUPER_MAX : r);
            } else {
                S = K1_SUPER_MAX;
            }
        }
        __syncthreads();
        K1_MARK(tE);
    }
    if (p.phase_cycles && tid == 0) {
        atomicAdd(p.phase_cycles + 0, (unsigned long long)tA1); atomicAdd(p.phase_cycles + 1, (unsigned long long)tA2);
        atomicAdd(p.phase_cycles + 2, (unsigned long long)tB); atomicAdd(p.phase_cycles + 3, (unsigned long long)tC);
        atomicAdd(p.phase_cycles + 4, (unsigned long long)tD); atomicAdd(p.phase_cycles + 5, (unsigned long long)tE);
    }

    if (acc < quota) {  // sampler exhausted: value-encode like a failed PnP (zero pose, cnn_softam.h:66-71)
        for (int r = acc + tid; r < quota; r += K1_THREADS) {
            size_t hi = (size_t)frame * p.H + h0 + r;
            for (int k = 0; k < 6; k++) p.hyp_pose[hi * 6 + k] = 0.0;
            float4* P = reinterpret_cast<float4*>(p.hyp_P + hi * 12);
            P[0] = make_float4((float)p.f, 0.f, 0.f, 0.f);
            P[1] = make_float4(0.f, (float)p.f, 0.f, 0.f);
            P[2] = make_float4(0.f, 0.f, 1.f, 0.f);
            for (int k = 0; k < 4; k++) p.img_idx[hi * 4 + k] = -1;
            p.cand_idx[hi] = -1;
        }
        if (tid == 0) {
            p.stream_ncand[(size_t)frame * p.T + s] = cand_base;
            p.stream_endpos[(size_t)frame * p.T + s] = pos;
            atomicOr(p.status + frame, 1u /* DSAC_ST_SAMPLER_EXHAUSTED */);
        }
    }
}

// ------------------------------------------------------------------ K2: fused scoring
struct ScoreParams {
    const int16_t* coords;   // [n][N][3]
    const int32_t* pix;      // [n or 1][N][2]
    int pix_stride;
    const float* hyp_P;      // [n][H][12]
    const double* hyp_pose;  // [n][H][6]
    float* diffmaps;         // [n][H][N] or null
    double* scores;          // [n][H]
    double* sf;              // [n][H]
    double* entropy;         // [n]
    double* avg_pose;        // [n][6]
    unsigned int* frame_counter;  // [n] zero-initialised, self-resetting
    int H, tile, tiles_per_frame;
    float cxf, cyf;
    float thr, kbeta;        // kbeta = beta * log2(e)
    double alpha;
    int external_scores;     // 1: scores come from the score hook, only the softmax tail runs
};

constexpr int K2_THREADS = 320;  // 10 warps x 5 points per thread = 1600 scene coordinates
constexpr int K2_PTS = 5;   // (the one-reciprocal sigmoid sum in k_score is written out for exactly 5)
constexpr int K2_WARPS = K2_THREADS / 32;
constexpr int K2_MAX_TILE = 256;

// softmax / entropy / soft-argmax over the H hypotheses of one frame, in double
// (softMax cnn_softam.h:535-553, entropy :80-88, averaging :1082-1094).
__device__ void softargmax_tail(const ScoreParams& p, int frame, double* s_red /* >= 8*K2_WARPS doubles */) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const double* sc = p.scores + (size_t)frame * p.H;
    // max
    double m = -1.7976931348623157e308;
    for (int h = tid; h < p.H; h += K2_THREADS) m = fmax(m, __ldcg(sc + h));
#pragma unroll
    for (int off = 16; off; off >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, off));
    if (lane == 0) s_red[warp] = m;
    __syncthreads();
    m = s_red[0];
    for (int w = 1; w < K2_WARPS; w++) m = fmax(m, s_red[w]);
    __syncthreads();
    // sum of exp and exp-weighted poses
    double acc[7] = {0, 0, 0, 0, 0, 0, 0};
    for (int h = tid; h < p.H; h += K2_THREADS) {
        double e = exp(__ldcg(sc + h) - m);
        acc[0] += e;
        const double* hp = p.hyp_pose + ((size_t)frame * p.H + h) * 6;
#pragma unroll
        for (int k = 0; k < 6; k++) acc[1 + k] += e * hp[k];
    }
#pragma unroll
    for (int k = 0; k < 7; k++) {
#pragma unroll
        for (int off = 16; off; off >>= 1) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], off);
        if (lane == 0) s_red[warp * 8 + k] = acc[k];
    }
    __syncthreads();
    double tot[7];
#pragma unroll
    for (int k = 0; k < 7; k++) {
        double t = 0;
        for (int w = 0; w < K2_WARPS; w++) t += s_red[w * 8 + k];
        tot[k] = t;
    }
    __syncthreads();
    // probabilities + entropy
    double ent = 0;
    for (int h = tid; h < p.H; h += K2_THREADS) {
        double pr = exp(__ldcg(sc + h) - m) / tot[0];
        p.sf[(size_t)frame * p.H + h] = pr;
        if (pr > 0) ent -= pr * log2(pr);
    }
#pragma unroll
    for (int off = 16; off; off >>= 1) ent += __shfl_xor_sync(0xffffffffu, ent, off);
    if (lane == 0) s_red[warp] = ent;
    __syncthreads();
    if (tid == 0) {
        double e = 0;
        for (int w = 0; w < K2_WARPS; w++) e += s_red[w];
        p.entropy[frame] = e;
        for (int k = 0; k < 6; k++) p.avg_pose[(size_t)frame * 6 + k] = tot[1 + k] / tot[0];
    }
}

// One warp's share of a tile: the warp's 160 scene coordinates (5 per thread, in registers) against the tile's nh
// hypotheses (3x4 rows in shared memory), 8 hypotheses at a time; writes the error matrix and leaves the warp's
// partial soft-inlier sums in part[0..nh).
//
// Per (hypothesis, point): ONE rsqrt gives the clamped reprojection error,
//   e = |pix - proj| = sqrt(A)/|z|,  A = (pu*z - xs)^2 + (pv*z - ys)^2  ->  e = A * rsqrt(A * z^2).
// A z^2 vanishes for a point exactly on its pixel (A = 0 -> e = 0 through the floor under the rsqrt) or exactly in the
// camera plane (z = 0, where cv::projectPoints substitutes 1/z := 1).  GUARDED = false evaluates the formula without
// the select on z and only records (one FSETP per 5 pairs) whether one of the thread's five z is exactly 0; the
// caller then repeats the warp's tile with GUARDED = true, which overwrites everything the unguarded pass wrote.
// Returns that flag.
//
// Soft inlier sigma(beta (tau - e)) = 1 / (1 + t), t = 2^(kbeta (e - tau)); the thread's five sigmoids share one reciprocal.
// One group of up to 8 hypotheses starting at hb.  FULL = all 8 exist: no per-hypothesis branch, so the eight bodies
// form one basic block and the instruction scheduler can overlap the MUFU tail (rsqrt, ex2, rcp: 13 per hypothesis,
// 8 issue cycles each on the XU pipe) of one hypothesis with the FMA-pipe projection of the next -- with a branch
// between hypotheses the warps of a CTA, which run in step, all queue on the XU pipe at the same time.
template <bool WRITE_DM, bool GUARDED, bool FULL>
__device__ __forceinline__ bool score_group8(const float* s_P, int hb, int nh, const float (&X)[K2_PTS], const float (&Y)[K2_PTS],
                                             const float (&Z)[K2_PTS], const float (&pu)[K2_PTS], const float (&pv)[K2_PTS],
                                             float* dm, float kbeta, float tau_k, float* part, int tid, int lane) {
    bool rare = false;
    float acc[8];
#pragma unroll
    for (int u = 0; u < 8; u++) {
        const int h = hb + u;
        float a = 0.f;
        if (FULL || h < nh) {
            const float4 r0 = *reinterpret_cast<const float4*>(s_P + h * 12);
            const float4 r1 = *reinterpret_cast<const float4*>(s_P + h * 12 + 4);
            const float4 r2 = *reinterpret_cast<const float4*>(s_P + h * 12 + 8);
            float e[K2_PTS], az[K2_PTS];
#pragma unroll
            for (int j = 0; j < K2_PTS; j++)
                e[j] = score_pair_error<GUARDED>(r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w, r2.x, r2.y, r2.z, r2.w, X[j], Y[j], Z[j],
                                                 pu[j], pv[j], &az[j]);
            if (!GUARDED) rare |= (fminf(fminf(fminf(az[0], az[1]), fminf(az[2], az[3])), az[4]) == 0.f);
            if (WRITE_DM) {   // cells 4 tid .. 4 tid + 3 as one 16-byte streaming store, cell 1280 + tid as a 4-byte one
                float* row = dm + (size_t)h * DSAC_N_CONST;
                __stcs(reinterpret_cast<float4*>(row) + tid, make_float4(e[0], e[1], e[2], e[3]));
                __stcs(row + 4 * K2_THREADS + tid, e[4]);
            }
            a = score_sigmoid_sum5(e, kbeta, tau_k);
        }
        acc[u] = a;
    }
    // transposed warp reduction: 8 partials -> lane (4*b4+2*b3+b2) group holds hypothesis sum
#pragma unroll
    for (int half = 4, off = 16; half >= 1; half >>= 1, off >>= 1) {
        const bool up = (lane & off) != 0;
#pragma unroll
        for (int i = 0; i < 4; i++) {
            if (i < half) {
                float send = up ? acc[i] : acc[i + half];
                float keep = up ? acc[i + half] : acc[i];
                acc[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
            }
        }
    }
    float v = acc[0];
    v += __shfl_xor_sync(0xffffffffu, v, 2);
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    if ((lane & 3) == 0) {
        int u = ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1);
        if (FULL || hb + u < nh) part[hb + u] = v;
    }
    return rare;
}

template <bool WRITE_DM, bool GUARDED>
__device__ __forceinline__ bool score_tile(const float* s_P, int nh, const float (&X)[K2_PTS], const float (&Y)[K2_PTS],
                                           const float (&Z)[K2_PTS], const float (&pu)[K2_PTS], const float (&pv)[K2_PTS],
                                           float* dm, float kbeta, float tau_k, float* part, int tid, int lane) {
    static_assert(K2_PTS == 5, "the shared-reciprocal sigmoid sum is written out for 5 points per thread");
    bool rare = false;
    int hb = 0;
    for (; hb + 8 <= nh; hb += 8) rare |= score_group8<WRITE_DM, GUARDED, true>(s_P, hb, nh, X, Y, Z, pu, pv, dm, kbeta, tau_k, part, tid, lane);
    if (hb < nh) rare |= score_group8<WRITE_DM, GUARDED, false>(s_P, hb, nh, X, Y, Z, pu, pv, dm, kbeta, tau_k, part, tid, lane);
    return rare;
}

// the guarded repeat is kept out of line: it runs (practically) never
template <bool WRITE_DM>
__device__ __noinline__ void score_tile_guarded(const float* s_P, int nh, const float (&X)[K2_PTS], const float (&Y)[K2_PTS],
                                                const float (&Z)[K2_PTS], const float (&pu)[K2_PTS], const float (&pv)[K2_PTS],
                                                float* dm, float kbeta, float tau_k, float* part, int tid, int lane) {
    score_tile<WRITE_DM, true>(s_P, nh, X, Y, Z, pu, pv, dm, kbeta, tau_k, part, tid, lane);
}

#ifndef K2_MIN_BLOCKS
#define K2_MIN_BLOCKS 3
#endif
template <bool WRITE_DM>
__global__ void __launch_bounds__(K2_THREADS, K2_MIN_BLOCKS) k_score(ScoreParams p) {
    __shared__ __align__(128) float s_P[K2_MAX_TILE * 12];
    __shared__ __align__(8) unsigned long long s_bar;
    __shared__ float s_part[K2_WARPS][K2_MAX_TILE];
    __shared__ double s_red[8 * K2_WARPS];
    __shared__ unsigned int s_last;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int frame = blockIdx.y, tile_idx = blockIdx.x;
    const int hbeg = tile_idx * p.tile;
    const int nh = min(p.tile, p.H - hbeg);

    if (!p.external_scores) {
        // this thread's 5 scene coordinates (cells 4 tid .. 4 tid + 3 and 1280 + tid) and their (pixel - principal point), as floats
        float X[K2_PTS], Y[K2_PTS], Z[K2_PTS], pu[K2_PTS], pv[K2_PTS];
        {
            const int16_t* c = p.coords + (size_t)frame * DSAC_N_CONST * 3;
            const int2* px = reinterpret_cast<const int2*>(p.pix + (size_t)frame * p.pix_stride);
#pragma unroll
            for (int j = 0; j < K2_PTS; j++) {
                const int pt = (j < 4) ? 4 * tid + j : 4 * K2_THREADS + tid;   // four adjacent cells + one: 16-byte stores of the error rows
                X[j] = (float)__ldg(c + pt * 3);
                Y[j] = (float)__ldg(c + pt * 3 + 1);
                Z[j] = (float)__ldg(c + pt * 3 + 2);
                int2 q = __ldg(px + pt);
                pu[j] = (float)q.x - p.cxf;
                pv[j] = (float)q.y - p.cyf;
            }
        }
        // stage the tile's 3x4 projection rows (48 bytes per hypothesis, contiguous) in shared memory by TMA: one thread
        // issues the bulk copy while the others are still converting their scene coordinates; everybody waits on the barrier
        if (tid == 0) mbar_init(&s_bar);
        __syncthreads();
        if (tid == 0) tma_load_1d(s_P, p.hyp_P + ((size_t)frame * p.H + hbeg) * 12, (uint32_t)nh * 48u, &s_bar);
        mbar_wait(&s_bar, 0u);

        float* dm = WRITE_DM ? p.diffmaps + ((size_t)frame * p.H + hbeg) * DSAC_N_CONST : nullptr;
        const float tau_k = p.thr * p.kbeta;
        const bool rare = score_tile<WRITE_DM, false>(s_P, nh, X, Y, Z, pu, pv, dm, p.kbeta, tau_k, s_part[warp], tid, lane);
        if (__any_sync(0xffffffffu, rare)) {
            __syncwarp();
            score_tile_guarded<WRITE_DM>(s_P, nh, X, Y, Z, pu, pv, dm, p.kbeta, tau_k, s_part[warp], tid, lane);
        }
        __syncthreads();
        // fixed-order cross-warp sum -> score (double from here on, like the reference's vector<double>)
        for (int h = tid; h < nh; h += K2_THREADS) {
            float ssum = 0.f;
#pragma unroll
            for (int w = 0; w < K2_WARPS; w++) ssum += s_part[w][h];
            p.scores[(size_t)frame * p.H + hbeg + h] = p.alpha * (double)ssum;
        }
    }

    // ---- last CTA of the frame runs the softmax / soft-argmax tail
    __threadfence();
    __syncthreads();
    if (tid == 0) {
        unsigned int prev = atomicAdd(p.frame_counter + frame, 1u);
        s_last = (prev == (unsigned int)p.tiles_per_frame - 1u);
        if (s_last) p.frame_counter[frame] = 0u;  // self-reset for the next launch
    }
    __syncthreads();
    if (s_last) {
        __threadfence();
        softargmax_tail(p, frame, s_red);
    }
}

}  // namespace dsac
