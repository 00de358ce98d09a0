// Precision / recall counts for the depth-edge AUC metric (sm_100a).
//
// Replaces (reference root relative):
//   evaluate_boundaries        eval_depth_edges.py:67-145   (threshold loop :117-143)
//   crop of _pred_eval         eval_depth_edges.py:195-197, 206-208
//   per-image sum              eval_depth_edges.py:298-301
//   correspond_pixels          py-bsds500 (not vendored), call sites eval_depth_edges.py:50-52, 130-132
//
// The matcher is an exact maximum-cardinality bipartite matching between predicted and GT boundary
// pixels closer than max_dist * diagonal (SURVEY.md A.3; counts are unique for any maximum matching).
// One persistent CTA per (image, threshold) problem, problems handed out through an atomic counter:
//   scan   the cropped window once (the 2 B/px of algorithmic traffic), compact predicted pixels,
//   greedy nearest-first proposals with 16-bit CAS on the GT side,
//   then phases of { exhaustive alternating-forest BFS from all free predicted pixels, level-synchronous
//   with warp-per-vertex expansion; one vertex-disjoint augmenting path per tree, claimed with CAS }
//   until a phase finds no free GT pixel => no augmenting path exists => maximum.
// Per-pixel state is 16-bit offset codes in an L2-resident per-CTA arena; nothing is allocated.
// With apply_thinning = 1 every problem's window is thinned first (thin_window_kernel below) and the per-problem
// matchers read the thinned bit planes.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "common.cuh"
#include "thin.cuh"

namespace mte {
namespace pr {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr unsigned short kFree = 0xFFFF;
constexpr unsigned short kDead = 0xFFFE;  // predicted pixel without any GT pixel in range
constexpr int kCtasPerSm = 2;

enum { IN_LEVELS = 0, IN_BINARY = 1, IN_F32 = 2, IN_F64 = 3, IN_BITS = 4 };

struct MatchP {
    const void *pred;          // [N,H,W] levels u8 / binary u8 / f32 / f64   (binary mode: [nProblems,H,W])
    const unsigned *bits;      // bits mode: one thinned bit plane of the window per problem of the chunk
    size_t bitsPlane;          // stride of the bit planes in words (h rows of bitsNw words, rounded up)
    int bitsNw;
    int probBase;              // global index of the chunk's first problem (image = g / T, threshold = g % T)
    const unsigned char *gt;   // [N,H,W]   (binary mode: [nProblems,H,W])
    int inMode;
    int N, H, W, T;
    int x0, y0, w, h;          // window
    int nProblems;             // N*T
    const double *thr;         // [T] device (float modes)
    int noff;
    int countsImgStride;       // rows per image in counts: 0 = summed over the images ([T][4]), T = per image ([N][T][4])
    const short2 *off;         // [noff] (dx, dy), nearest first
    const unsigned short *neg; // [noff] index of the negated offset
    unsigned long long *counts;  // [T][4] count_r,sum_r,count_p,sum_p (accumulated)   (pr mode)
    long long *countPerProblem;  // [nProblems] (correspond_pixels mode) or nullptr
    unsigned char *matchA, *matchB;  // optional outputs [nProblems,h,w]
    char *arena;               // kArenas * arenaBytes
    size_t arenaBytes;
    const int *problemList;    // optional indirection: only these problems (the shared-memory kernel's overflow list)
    const unsigned int *listCount;  // device count of problemList entries
    unsigned int *overflowCount;    // written by the shared-memory kernel, reset by the dense kernel
    int *overflowList;
    unsigned int *stats;       // optional profiling counters {phases, levels, expanded vertices, free roots}
    unsigned int *trace;       // debug builds: per-item cycle stamps of the many-root phases of stage 0 (scripts/match_trace.py)
    unsigned int *nextProblem; // dynamic scheduler (self-resetting)
    unsigned int *doneCtas;
};

// Small tables ride in the kernel parameters (graph-capturable, no staging copy); larger ones (radius > 7 px
// or > kParamThr thresholds) are copied into the workspace first.  Either way the CTA stages the offsets in
// shared memory: lanes index them divergently.  kMaxOff holds the largest table build_offsets makes.
constexpr int kParamOff = 256, kParamThr = 160, kMaxOff = 4096;
struct ParamTables {
    short2 off[kParamOff];
    unsigned short neg[kParamOff];
    double thr[kParamThr];
};

struct Arena {
    unsigned short *mateP, *mateQ, *parentQ, *stampQ, *claimP;
    int *plist, *fa, *fb, *ends;
};

__host__ __device__ inline size_t arena_bytes(int h, int w) {
    const size_t px = (size_t)h * w;
    return align_up(px * 2, 256) * 5 + align_up(px * 4, 256) * 4;
}

__device__ inline Arena carve(char *base, int h, int w) {
    const size_t px = (size_t)h * w;
    const size_t s2 = align_up(px * 2, 256), s4 = align_up(px * 4, 256);
    Arena A;
    A.mateP = (unsigned short *)base; base += s2;
    A.mateQ = (unsigned short *)base; base += s2;
    A.parentQ = (unsigned short *)base; base += s2;
    A.stampQ = (unsigned short *)base; base += s2;
    A.claimP = (unsigned short *)base; base += s2;
    A.plist = (int *)base; base += s4;
    A.fa = (int *)base; base += s4;
    A.fb = (int *)base; base += s4;
    A.ends = (int *)base;
    return A;
}

__device__ __forceinline__ unsigned short cas16(unsigned short *addr, unsigned short expected, unsigned short val) {
    return atomicCAS(addr, expected, val);
}

// the binarisation rule of a threshold sweep: level plane -> level <= t, strength map -> pred >= thr[t] in fp64
// (NaN is never set).  o indexes the [N,H,W] plane.
__device__ __forceinline__ bool sweep_pred(const void *pred, int inMode, size_t o, int t, const double *thr) {
    switch (inMode) {
        case IN_LEVELS: return ((const unsigned char *)pred)[o] <= t;
        case IN_F32: return (double)((const float *)pred)[o] >= thr[t];
        default: return ((const double *)pred)[o] >= thr[t];
    }
}

// prob: the problem's index within the launch (bits and binary modes index their planes with it)
__device__ __forceinline__ bool is_pred(const MatchP &P, int img, int t, int prob, int gy, int gx) {
    const size_t o = (size_t)gy * P.W + gx;
    switch (P.inMode) {
        case IN_BINARY: return ((const unsigned char *)P.pred)[(size_t)prob * P.H * P.W + o] != 0;
        case IN_BITS: {
            const int y = gy - P.y0, x = gx - P.x0;
            return (P.bits[(size_t)prob * P.bitsPlane + (size_t)y * P.bitsNw + (x >> 5)] >> (x & 31)) & 1u;
        }
        default: return sweep_pred(P.pred, P.inMode, (size_t)img * P.H * P.W + o, t, P.thr);
    }
}

// ---- pieces the three matcher kernels share (NT: the kernel's threads per CTA)

// stage the offsets (and the inverse-offset indices where sNeg is given, the thresholds where withThr) in shared memory
template <int NT>
__device__ __forceinline__ void stage_tables(const MatchP &P, const ParamTables &tabs, int tablesInParam, bool withThr,
                                             short2 *sOff, unsigned short *sNeg, double *sThr) {
    for (int i = threadIdx.x; i < P.noff; i += NT) {
        sOff[i] = tablesInParam ? tabs.off[i] : P.off[i];
        if (sNeg) sNeg[i] = tablesInParam ? tabs.neg[i] : P.neg[i];
    }
    if (withThr)
        for (int i = threadIdx.x; i < P.T; i += NT) sThr[i] = tablesInParam ? tabs.thr[i] : P.thr[i];
    __syncthreads();
}

// thread 0 draws the next ticket of the dynamic scheduler, all threads return it; through the problem list when
// viaList (a ticket past the list's end returns P.nProblems: nothing left)
__device__ __forceinline__ int next_ticket(const MatchP &P, bool viaList, int &sTicket) {
    if (threadIdx.x == 0) {
        int pr = (int)atomicAdd(P.nextProblem, 1u);
        if (viaList) pr = (pr < (int)*P.listCount) ? P.problemList[pr] : P.nProblems;
        sTicket = pr;
    }
    __syncthreads();
    return sTicket;
}

// problems are ordered image-major so consecutive CTAs share the GT plane in L2
__device__ __forceinline__ void decode_problem(const MatchP &P, int prob, int &img, int &t) {
    const int g = P.probBase + prob;
    img = (P.inMode == IN_BINARY) ? prob : g / P.T;
    t = (P.inMode == IN_BINARY) ? 0 : g - img * P.T;
}

// warp-aggregated append to a shared counter: one atomic per warp; returns this lane's slot (valid where take)
__device__ __forceinline__ int warp_append(int *counter, bool take) {
    const int lane = threadIdx.x & 31;
    const unsigned m = __ballot_sync(MTE_FULL_MASK, take);
    int wbase = 0;
    if (lane == 0 && m) wbase = atomicAdd(counter, __popc(m));
    wbase = __shfl_sync(MTE_FULL_MASK, wbase, 0);
    return wbase + __popc(m & ((1u << lane) - 1));
}

// exclusive prefix sum of one value per thread over the CTA (warp 0 scans the NT partials, NT / 32 per lane)
template <int NT>
__device__ __forceinline__ int block_exclusive_scan(int v, int *sScan) {
    const int lane = threadIdx.x & 31;
    sScan[threadIdx.x] = v;
    __syncthreads();
    if (threadIdx.x < 32) {
        int loc[NT / 32], run = 0;
#pragma unroll
        for (int k = 0; k < NT / 32; k++) { loc[k] = run; run += sScan[lane * (NT / 32) + k]; }
        int incl = run;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int u = __shfl_up_sync(MTE_FULL_MASK, incl, o); if (lane >= o) incl += u; }
        const int excl = incl - run;
#pragma unroll
        for (int k = 0; k < NT / 32; k++) sScan[lane * (NT / 32) + k] = excl + loc[k];
    }
    __syncthreads();
    return sScan[threadIdx.x];
}

// Lane 0 takes the next entry of the shared work queue fa[sHead, sTail) and waits until it is published (slots hold
// kFree until then); -2 once the queue is drained and no vertex is pending (one being expanded may still publish).
// All lanes return the predicted vertex.
__device__ __forceinline__ int queue_pop(int *sHead, const int *sTail, const int *sPending, const unsigned short *fa) {
    int my = -1;
    if ((threadIdx.x & 31) == 0) {
        for (;;) {
            const int hd = *(volatile int *)sHead, tl = *(volatile const int *)sTail;
            if (hd < tl) {
                if (atomicCAS(sHead, hd, hd + 1) == hd) { my = hd; break; }
            } else if (*(volatile const int *)sPending == 0) {
                my = -2;
                break;
            }
        }
        if (my >= 0) {
            int v;
            while ((v = ((volatile const unsigned short *)fa)[my]) == kFree) {}
            my = v;
        }
    }
    return __shfl_sync(MTE_FULL_MASK, my, 0);
}

// flip the augmenting path that ends at free GT vertex q, in compact ids (parentQ: predicted id, mateP: GT id)
__device__ __forceinline__ void flip_path(int q, const unsigned short *parentQ, unsigned short *mateP,
                                          unsigned short *mateQ) {
    for (;;) {
        const int pi = parentQ[q];
        const unsigned short prev = mateP[pi];
        mateP[pi] = (unsigned short)q;
        mateQ[q] = (unsigned short)pi;
        if (prev == kFree) break;
        q = prev;
    }
}

// add one problem's count_r, sum_r, count_p, sum_p to its row of P.counts
__device__ __forceinline__ void add_counts(const MatchP &P, int img, int t, int matched, int nQ, int nP) {
    unsigned long long *c = P.counts + (size_t)(t + img * P.countsImgStride) * 4;
    atomicAdd(c + 0, (unsigned long long)matched);
    atomicAdd(c + 1, (unsigned long long)nQ);
    atomicAdd(c + 2, (unsigned long long)matched);
    atomicAdd(c + 3, (unsigned long long)nP);
}

// last CTA out resets the scheduler so the workspace header is clean for the next launch; the launch over the
// overflow list also clears the count of that list
__device__ __forceinline__ void reset_scheduler(const MatchP &P, bool clearOverflow) {
    if (threadIdx.x == 0) {
        __threadfence();
        const unsigned d = atomicAdd(P.doneCtas, 1u);
        if (d == gridDim.x - 1) {
            *P.nextProblem = 0u;
            *P.doneCtas = 0u;
            if (clearOverflow) *P.overflowCount = 0u;
        }
    }
}

__global__ void __launch_bounds__(kThreads) match_kernel(const __grid_constant__ MatchP Pin,
                                                         const __grid_constant__ ParamTables tabs, int tablesInParam) {
    __shared__ int sProblem, sNP, sNQ, sCntA, sCntB, sEnds, sMatched;
    __shared__ short2 sOff[kMaxOff];
    __shared__ unsigned short sNeg[kMaxOff];
    __shared__ double sThr[MTE_MAX_THRESHOLDS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    MatchP P = Pin;
    const int w = P.w, h = P.h;
    const Arena A = carve(P.arena + (size_t)blockIdx.x * P.arenaBytes, h, w);
    stage_tables<kThreads>(P, tabs, tablesInParam, P.inMode == IN_F32 || P.inMode == IN_F64, sOff, sNeg, sThr);
    P.off = sOff;
    P.neg = sNeg;
    P.thr = sThr;

    for (;;) {
        const int prob = next_ticket(P, P.problemList != nullptr, sProblem);
        if (prob >= P.nProblems) break;
        int img, t;
        decode_problem(P, prob, img, t);
        const unsigned char *gt = P.gt + (size_t)img * P.H * P.W;
        if (threadIdx.x == 0) { sNP = 0; sNQ = 0; sMatched = 0; }
        __syncthreads();

        // ---- scan the window: initialise per-pixel state at boundary pixels, compact predicted pixels
        int myQ = 0;
        for (int base = 0; base < w * h; base += kThreads) {
            const int i = base + threadIdx.x;
            bool isP = false;
            if (i < w * h) {
                const int y = i / w, x = i - y * w;
                const int gy = P.y0 + y, gx = P.x0 + x;
                isP = is_pred(P, img, t, prob, gy, gx);
                if (gt[(size_t)gy * P.W + gx] != 0) {
                    A.mateQ[i] = kFree;
                    A.stampQ[i] = 0;
                    myQ++;
                }
                if (isP) { A.mateP[i] = kFree; A.claimP[i] = 0; }
            }
            const int slot = warp_append(&sNP, isP);
            if (isP) A.plist[slot] = i;
        }
        myQ = __reduce_add_sync(MTE_FULL_MASK, myQ);
        if (lane == 0 && myQ) atomicAdd(&sNQ, myQ);
        __syncthreads();
        const int nP = sNP, nQ = sNQ;

        // ---- greedy start: nearest free GT pixel (warp per predicted pixel, lanes over offsets)
        for (int pi = warp; pi < nP; pi += kWarps) {
            const int p = A.plist[pi];
            const int py = p / w, px = p - py * w;
            bool done = false, anyQ = false;
            for (int k0 = 0; k0 < P.noff && !done; k0 += 32) {
                const int k = k0 + lane;
                bool cand = false;
                int q = 0;
                if (k < P.noff) {
                    const short2 o = P.off[k];
                    const int qy = py + o.y, qx = px + o.x;
                    if (qy >= 0 && qy < h && qx >= 0 && qx < w) {
                        q = qy * w + qx;
                        cand = gt[(size_t)(P.y0 + qy) * P.W + P.x0 + qx] != 0;
                    }
                }
                unsigned m = __ballot_sync(MTE_FULL_MASK, cand);
                anyQ |= m != 0;
                while (m && !done) {  // try candidates nearest first
                    const int l = __ffs(m) - 1;
                    m &= m - 1;
                    int ok = 0;
                    if (lane == l) {
                        ok = cas16(&A.mateQ[q], kFree, P.neg[k]) == kFree;
                        if (ok) A.mateP[p] = (unsigned short)k;
                    }
                    done = __shfl_sync(MTE_FULL_MASK, ok, l) != 0;
                }
            }
            if (done && lane == 0) atomicAdd(&sMatched, 1);
            if (!done && !anyQ && lane == 0) A.mateP[p] = kDead;
        }
        __syncthreads();

        // ---- augmenting phases
        for (unsigned short phase = 1;; phase++) {
            // frontier 0: free (not dead) predicted pixels
            if (threadIdx.x == 0) { sCntA = 0; sEnds = 0; }
            __syncthreads();
            for (int base = 0; base < nP; base += kThreads) {
                const int pi = base + threadIdx.x;
                bool fr = false;
                int p = 0;
                if (pi < nP) { p = A.plist[pi]; fr = A.mateP[p] == kFree; }
                const int slot = warp_append(&sCntA, fr);
                if (fr) A.fa[slot] = p;
            }
            __syncthreads();
            int *cur = A.fa, *nxt = A.fb;
            int nCur = sCntA;
            if (nCur == 0) break;
            if (P.stats && threadIdx.x == 0) { atomicAdd(P.stats + 0, 1u); atomicAdd(P.stats + 3, (unsigned)nCur); }
            // exhaustive alternating-forest BFS
            while (nCur > 0) {
                if (threadIdx.x == 0) sCntB = 0;
                __syncthreads();
                for (int fi = warp; fi < nCur; fi += kWarps) {
                    const int p = cur[fi];
                    const int py = p / w, px = p - py * w;
                    for (int k0 = 0; k0 < P.noff; k0 += 32) {
                        const int k = k0 + lane;
                        if (k >= P.noff) continue;
                        const short2 o = P.off[k];
                        const int qy = py + o.y, qx = px + o.x;
                        if (qy < 0 || qy >= h || qx < 0 || qx >= w) continue;
                        if (gt[(size_t)(P.y0 + qy) * P.W + P.x0 + qx] == 0) continue;
                        const int q = qy * w + qx;
                        const unsigned short s = A.stampQ[q];
                        if (s == phase) continue;
                        if (cas16(&A.stampQ[q], s, phase) != s) continue;  // someone else got it
                        A.parentQ[q] = P.neg[k];
                        const unsigned short mq = A.mateQ[q];
                        if (mq == kFree) {
                            A.ends[atomicAdd(&sEnds, 1)] = q;
                        } else {
                            const short2 om = P.off[mq];
                            nxt[atomicAdd(&sCntB, 1)] = (qy + om.y) * w + (qx + om.x);
                        }
                    }
                }
                __syncthreads();
                nCur = sCntB;
                if (P.stats && threadIdx.x == 0) { atomicAdd(P.stats + 1, 1u); atomicAdd(P.stats + 2, (unsigned)sCntB); }
                int *tmp = cur; cur = nxt; nxt = tmp;
                __syncthreads();
            }
            const int nEnds = sEnds;
            if (nEnds == 0) break;  // no augmenting path anywhere: maximum
            // one vertex-disjoint augmenting path per tree
            for (int ei = threadIdx.x; ei < nEnds; ei += kThreads) {
                const int qEnd = A.ends[ei];
                int q = qEnd;
                bool ok = true;
                for (;;) {  // claim walk (no mate is touched)
                    const short2 o = P.off[A.parentQ[q]];
                    const int qy = q / w, qx = q - qy * w;
                    const int p = (qy + o.y) * w + (qx + o.x);
                    const unsigned short c = A.claimP[p];
                    if (c == phase || cas16(&A.claimP[p], c, phase) != c) { ok = false; break; }
                    const unsigned short mp = A.mateP[p];
                    if (mp == kFree) break;  // reached the root
                    const short2 om = P.off[mp];
                    const int py = qy + o.y, px = qx + o.x;
                    q = (py + om.y) * w + (px + om.x);
                }
                if (!ok) continue;
                q = qEnd;
                for (;;) {  // flip walk
                    const unsigned short pc = A.parentQ[q];
                    const short2 o = P.off[pc];
                    const int qy = q / w, qx = q - qy * w;
                    const int py = qy + o.y, px = qx + o.x;
                    const int p = py * w + px;
                    const unsigned short prev = A.mateP[p];
                    A.mateP[p] = P.neg[pc];
                    A.mateQ[q] = pc;
                    if (prev == kFree) break;
                    const short2 om = P.off[prev];
                    q = (py + om.y) * w + (px + om.x);
                }
                atomicAdd(&sMatched, 1);
            }
            __syncthreads();
            if (phase == 0xFFF0) break;  // unreachable in practice (each phase adds >= 1 match)
        }
        __syncthreads();

        // ---- results
        const int matched = sMatched;
        if (threadIdx.x == 0) {
            if (P.counts) add_counts(P, img, t, matched, nQ, nP);
            if (P.countPerProblem) P.countPerProblem[prob] = matched;
        }
        if (P.matchA || P.matchB) {
            for (int i = threadIdx.x; i < w * h; i += kThreads) {
                const int y = i / w, x = i - y * w;
                const int gy = P.y0 + y, gx = P.x0 + x;
                if (P.matchA) {
                    const bool isP = is_pred(P, img, t, prob, gy, gx);
                    P.matchA[(size_t)prob * w * h + i] = (isP && A.mateP[i] < kDead) ? 1 : 0;
                }
                if (P.matchB) {
                    const bool isQ = gt[(size_t)gy * P.W + gx] != 0;
                    P.matchB[(size_t)prob * w * h + i] = (isQ && A.mateQ[i] != kFree) ? 1 : 0;
                }
            }
        }
        __syncthreads();
    }
    reset_scheduler(P, P.problemList != nullptr);
}

// ---------------------------------------------------------------------------
// Shared-memory matcher: the same algorithm with the whole problem resident on the SM.
//
// State is indexed by COMPACT vertex ids (16 bit): the GT side is a bitmap of the window plus a per-word
// rank (pixel -> id by popcount), the predicted side a list of pixel positions.  A BFS level then costs a few
// shared-memory round trips instead of L2 round trips (profiles/r01_notes.md: ~1000 levels per problem on long
// contours, 15 us each in the L2 version).  Problems that do not fit (window bitmap or vertex counts beyond the
// ~200 KB budget) are appended to an overflow list and solved by match_kernel above.
// ---------------------------------------------------------------------------
constexpr int kSmThreads = 512;
constexpr int kSmWarps = kSmThreads / 32;
constexpr int kSmemTableOff = 1024;  // offsets staged in static shared memory (radius <= 17 px)

struct SmemLayout {
    int nW;          // bitmap words of the window
    int capP, capQ;  // vertex capacities
    unsigned oBits, oRank, oPpix, oMateP, oClaimP, oFa, oFb, oMateQ, oParentQ, oStampQ, oEnds, total;
};

__global__ void __launch_bounds__(kSmThreads, 1) match_smem_kernel(const __grid_constant__ MatchP Pin,
                                                                   const __grid_constant__ ParamTables tabs,
                                                                   int tablesInParam, const SmemLayout SL) {
    extern __shared__ __align__(16) unsigned char dyn[];
    __shared__ int sProblem, sNP, sNQ, sCntA, sEnds, sMatched, sHead, sTail, sPending;
    __shared__ int sScan[kSmThreads];
    __shared__ short2 sOff[kSmemTableOff];
    __shared__ double sThr[MTE_MAX_THRESHOLDS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    MatchP P = Pin;
    const int w = P.w, h = P.h, hw = w * h;
    unsigned *qbits = reinterpret_cast<unsigned *>(dyn + SL.oBits);
    unsigned short *qrank = reinterpret_cast<unsigned short *>(dyn + SL.oRank);
    unsigned *ppix = reinterpret_cast<unsigned *>(dyn + SL.oPpix);
    unsigned short *mateP = reinterpret_cast<unsigned short *>(dyn + SL.oMateP);
    unsigned short *claimP = reinterpret_cast<unsigned short *>(dyn + SL.oClaimP);
    unsigned short *fa = reinterpret_cast<unsigned short *>(dyn + SL.oFa);
    unsigned short *mateQ = reinterpret_cast<unsigned short *>(dyn + SL.oMateQ);
    unsigned short *parentQ = reinterpret_cast<unsigned short *>(dyn + SL.oParentQ);
    unsigned short *stampQ = reinterpret_cast<unsigned short *>(dyn + SL.oStampQ);
    unsigned short *ends = reinterpret_cast<unsigned short *>(dyn + SL.oEnds);
    stage_tables<kSmThreads>(P, tabs, tablesInParam, P.inMode == IN_F32 || P.inMode == IN_F64, sOff, nullptr, sThr);
    P.thr = sThr;
    const int noff = P.noff;

    // GT vertex id of window pixel q (caller has checked the bit)
    auto qid = [&](int q) -> int {
        const unsigned bits = qbits[q >> 5];
        return (int)qrank[q >> 5] + __popc(bits & ((1u << (q & 31)) - 1u));
    };

    for (;;) {
        const int prob = next_ticket(P, false, sProblem);
        if (prob >= P.nProblems) break;
        int img, t;
        decode_problem(P, prob, img, t);
        const unsigned char *gt = P.gt + (size_t)img * P.H * P.W;
        if (threadIdx.x == 0) { sNP = 0; sNQ = 0; sMatched = 0; }
        __syncthreads();

        // ---- scan: GT bitmap (one ballot per 32 window pixels), predicted pixel list; 4 independent
        //      steps per thread so 8 byte loads are in flight before the first ballot
        for (int base = 0; base < SL.nW * 32; base += 4 * kSmThreads) {
            bool isPk[4], isQk[4];
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const int i = base + u * kSmThreads + threadIdx.x;
                isPk[u] = false; isQk[u] = false;
                if (i < hw) {
                    const int y = i / w, x = i - y * w;
                    const int gy = P.y0 + y, gx = P.x0 + x;
                    isPk[u] = is_pred(P, img, t, prob, gy, gx);
                    isQk[u] = gt[(size_t)gy * P.W + gx] != 0;
                }
            }
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const int i = base + u * kSmThreads + threadIdx.x;
                if (base + u * kSmThreads >= SL.nW * 32) break;  // warp-uniform
                const unsigned mq = __ballot_sync(MTE_FULL_MASK, isQk[u]);
                if (lane == 0) {
                    qbits[i >> 5] = mq;
                    if (mq) atomicAdd(&sNQ, __popc(mq));
                }
                const int slot = warp_append(&sNP, isPk[u]);
                if (isPk[u] && slot < SL.capP) { ppix[slot] = (unsigned)i; mateP[slot] = kFree; claimP[slot] = 0; }
            }
        }
        __syncthreads();
        const int nP = sNP, nQ = sNQ;
        if (nP > SL.capP || nQ > SL.capQ || nQ >= 0xFFF0 || nP >= 0xFFF0) {  // does not fit: leave it to the dense kernel
            if (threadIdx.x == 0) P.overflowList[atomicAdd(P.overflowCount, 1u)] = prob;
            __syncthreads();
            continue;
        }
        // ---- rank: exclusive prefix popcount over the bitmap words
        {
            const int per = (SL.nW + kSmThreads - 1) / kSmThreads;
            const int w0 = threadIdx.x * per, w1 = min(w0 + per, SL.nW);
            int sum = 0;
            for (int k = w0; k < w1; k++) sum += __popc(qbits[k]);
            int run = block_exclusive_scan<kSmThreads>(sum, sScan);
            for (int k = w0; k < w1; k++) { qrank[k] = (unsigned short)run; run += __popc(qbits[k]); }
        }
        for (int k = threadIdx.x; k < nQ; k += kSmThreads) { mateQ[k] = kFree; stampQ[k] = 0; }
        __syncthreads();

        // ---- greedy start: nearest free GT pixel (warp per predicted pixel, lanes over offsets)
        for (int pi = warp; pi < nP; pi += kSmWarps) {
            const int p = (int)ppix[pi];
            const int py = p / w, px = p - py * w;
            bool done = false, anyQ = false;
            for (int k0 = 0; k0 < noff && !done; k0 += 32) {
                const int k = k0 + lane;
                bool cand = false;
                int q = 0;
                if (k < noff) {
                    const short2 o = sOff[k];
                    const int qy = py + o.y, qx = px + o.x;
                    if (qy >= 0 && qy < h && qx >= 0 && qx < w) {
                        q = qy * w + qx;
                        cand = (qbits[q >> 5] >> (q & 31)) & 1u;
                    }
                }
                unsigned m = __ballot_sync(MTE_FULL_MASK, cand);
                anyQ |= m != 0;
                while (m && !done) {
                    const int l = __ffs(m) - 1;
                    m &= m - 1;
                    int ok = 0;
                    if (lane == l) {
                        const int qi = qid(q);
                        ok = cas16(&mateQ[qi], kFree, (unsigned short)pi) == kFree;
                        if (ok) mateP[pi] = (unsigned short)qi;
                    }
                    done = __shfl_sync(MTE_FULL_MASK, ok, l) != 0;
                }
            }
            if (done && lane == 0) atomicAdd(&sMatched, 1);
            if (!done && !anyQ && lane == 0) mateP[pi] = kDead;
        }
        __syncthreads();

        // ---- augmenting phases
        for (unsigned short phase = 1;; phase++) {
            if (threadIdx.x == 0) { sCntA = 0; sEnds = 0; }
            __syncthreads();
            for (int base = 0; base < nP; base += kSmThreads) {
                const int pi = base + threadIdx.x;
                const bool fr = pi < nP && mateP[pi] == kFree;
                const int slot = warp_append(&sCntA, fr);
                if (fr) fa[slot] = (unsigned short)pi;
            }
            __syncthreads();
            const int nRoots = sCntA;
            if (nRoots == 0) break;
            if (P.stats && threadIdx.x == 0) { atomicAdd(P.stats + 0, 1u); atomicAdd(P.stats + 3, (unsigned)nRoots); }
            // Exhaustive alternating forest, explored ASYNCHRONOUSLY: the forest only has to be a forest (every GT
            // vertex claimed once, parent = the predicted vertex that claimed it), not a BFS layering, so the warps
            // drain one shared work queue of predicted vertices without any CTA barrier per level.  Every vertex
            // enters the queue at most once per phase (its mate is claimed once), so the queue never wraps.
            for (int i = nRoots + threadIdx.x; i < nP; i += kSmThreads) fa[i] = kFree;  // unpublished slots
            if (threadIdx.x == 0) { sHead = 0; sTail = nRoots; sPending = nRoots; }
            __syncthreads();
            for (;;) {
                const int pi = queue_pop(&sHead, &sTail, &sPending, fa);
                if (pi == -2) break;
                const int p = (int)ppix[pi];
                const int py = p / w, px = p - py * w;
                for (int k = lane; k < noff; k += 32) {
                    const short2 o = sOff[k];
                    const int qy = py + o.y, qx = px + o.x;
                    if (qy < 0 || qy >= h || qx < 0 || qx >= w) continue;
                    const int q = qy * w + qx;
                    if (!((qbits[q >> 5] >> (q & 31)) & 1u)) continue;
                    const int qi = qid(q);
                    const unsigned short s = stampQ[qi];
                    if (s == phase) continue;
                    if (cas16(&stampQ[qi], s, phase) != s) continue;
                    parentQ[qi] = (unsigned short)pi;
                    const unsigned short mq = mateQ[qi];
                    if (mq == kFree) {
                        ends[atomicAdd(&sEnds, 1)] = (unsigned short)qi;
                    } else {
                        atomicAdd(&sPending, 1);
                        const int slot = atomicAdd(&sTail, 1);
                        ((volatile unsigned short *)fa)[slot] = mq;
                    }
                }
                __syncwarp();
                if (lane == 0) {
                    __threadfence_block();
                    atomicSub(&sPending, 1);
                    if (P.stats) atomicAdd(P.stats + 2, 1u);
                }
            }
            __syncthreads();
            const int nEnds = sEnds;
            if (nEnds == 0) break;
            for (int ei = threadIdx.x; ei < nEnds; ei += kSmThreads) {
                const int qEnd = ends[ei];
                int q = qEnd;
                bool ok = true;
                for (;;) {  // claim walk
                    const int pi = parentQ[q];
                    const unsigned short c = claimP[pi];
                    if (c == phase || cas16(&claimP[pi], c, phase) != c) { ok = false; break; }
                    const unsigned short mp = mateP[pi];
                    if (mp == kFree) break;
                    q = mp;
                }
                if (!ok) continue;
                flip_path(qEnd, parentQ, mateP, mateQ);
                atomicAdd(&sMatched, 1);
            }
            __syncthreads();
            if (phase == 0xFFF0) break;
        }
        __syncthreads();

        // ---- results
        const int matched = sMatched;
        if (threadIdx.x == 0) {
            if (P.counts) add_counts(P, img, t, matched, nQ, nP);
            if (P.countPerProblem) P.countPerProblem[prob] = matched;
        }
        if (P.matchA) {
            unsigned char *ma = P.matchA + (size_t)prob * hw;
            for (int i = threadIdx.x; i < hw; i += kSmThreads) ma[i] = 0;
            __syncthreads();
            for (int pi = threadIdx.x; pi < nP; pi += kSmThreads) ma[ppix[pi]] = mateP[pi] < kDead ? 1 : 0;
        }
        if (P.matchB) {
            unsigned char *mb = P.matchB + (size_t)prob * hw;
            for (int i = threadIdx.x; i < hw; i += kSmThreads) {
                const bool isQ = (qbits[i >> 5] >> (i & 31)) & 1u;
                mb[i] = (isQ && mateQ[qid(i)] != kFree) ? 1 : 0;
            }
        }
        __syncthreads();
    }
    reset_scheduler(P, false);
}

// ---------------------------------------------------------------------------
// Threshold-sweep matcher: ONE CTA per image solves all T nested problems incrementally.
//
// The predicted sets are nested in the threshold (level planes: P_t grows with t; strength maps with ascending
// thresholds: P_t shrinks with t), and only the predicted side changes.  Adding predicted pixels to a maximum matching
// and augmenting from the new pixels only gives a maximum matching of the larger problem (a vertex whose search
// failed can never be matched later -- Kuhn's lemma), so the stages s = 0..T-1 (sets growing with s) are solved in
// turn on one persistent state:
//   stage s: greedy nearest-first proposals of the new pixels, then phases of { asynchronous alternating forest
//   from the new pixels that are still free; one CAS-claimed augmenting path per tree } until a phase finds no
//   free GT pixel.  That last forest is closed under alternating reachability and contains no free GT pixel, so no
//   later augmenting path can enter it: its GT vertices are marked DEAD and never explored again.
// Every GT vertex dies at most once, so the whole sweep costs about as much as its largest problem instead of T
// independent solves.  |M_t| after stage s is the count of threshold t_s.  Images whose vertex sets do not fit the
// shared-memory budget hand their T problems to the per-problem kernels through the overflow list.
// ---------------------------------------------------------------------------
constexpr unsigned kDeadStamp = 0xFFFFFFFFu;   // GT stamp word: phase << 16 | root (predicted vertex id of the tree)
constexpr unsigned short kFailed = 0xFFFD;     // predicted pixel whose search failed conclusively (Kuhn: for good)
enum { RF_FOUND = 1u, RF_CLASS_FOUND = 2u };
constexpr int kSwThreads = 512, kSwWarps = kSwThreads / 32;
constexpr int kEndsCap = 2048;  // free GT pixels recorded per phase (further ones wait for the next phase)

struct SweepLayout {
    int nW, capP, capQ;
    unsigned oBits, oRank, oPpix, oMateP, oClassP, oFa, oRootP, oRflag, oMateQ, oParentQ, oStamp, oEnds, total;
};


__global__ void __launch_bounds__(kSwThreads, 1) match_sweep_kernel(const __grid_constant__ MatchP Pin,
                                                                    const __grid_constant__ ParamTables tabs,
                                                                    int tablesInParam, const SweepLayout SL) {
    extern __shared__ __align__(16) unsigned char dyn[];
    __shared__ int sImage, sNP, sNQ, sCntA, sEnds, sMatched, sHead, sTail, sPending;
    __shared__ int sGr[3];   // greedy rounds: rotating append counters (one barrier per round)
#ifdef MTE_DEBUG_KNOBS
    __shared__ int sMaxChain;  // profiling: longest run of hops one warp walked without going back to the queue, per phase
#endif
    __shared__ int sScan[kSwThreads];
    __shared__ int sStage[MTE_MAX_THRESHOLDS + 2];   // histogram, then start offset of every stage
    __shared__ int sCursor[MTE_MAX_THRESHOLDS + 2];
    __shared__ short2 sOff[kSmemTableOff];
    __shared__ double sThr[MTE_MAX_THRESHOLDS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    MatchP P = Pin;
    const int w = P.w, h = P.h, hw = w * h, T = P.T;
    unsigned *qbits = reinterpret_cast<unsigned *>(dyn + SL.oBits);
    unsigned short *qrank = reinterpret_cast<unsigned short *>(dyn + SL.oRank);
    unsigned *ppix = reinterpret_cast<unsigned *>(dyn + SL.oPpix);
    unsigned short *mateP = reinterpret_cast<unsigned short *>(dyn + SL.oMateP);
    unsigned short *fa = reinterpret_cast<unsigned short *>(dyn + SL.oFa);
    unsigned short *classP = reinterpret_cast<unsigned short *>(dyn + SL.oClassP);  // union-find over the roots of a phase
    unsigned short *mateQ = reinterpret_cast<unsigned short *>(dyn + SL.oMateQ);
    unsigned short *parentQ = reinterpret_cast<unsigned short *>(dyn + SL.oParentQ);
    unsigned *stamp = reinterpret_cast<unsigned *>(dyn + SL.oStamp);
    unsigned short *rootP = reinterpret_cast<unsigned short *>(dyn + SL.oRootP);
    unsigned *rflagW = reinterpret_cast<unsigned *>(dyn + SL.oRflag);  // one flag byte per predicted vertex
    unsigned short *ends = reinterpret_cast<unsigned short *>(dyn + SL.oEnds);
    const bool levels = P.inMode == IN_LEVELS;
    stage_tables<kSwThreads>(P, tabs, tablesInParam, !levels, sOff, nullptr, sThr);
    const int noff = P.noff;
#ifdef MTE_DEBUG_KNOBS
    const long long tZero = clock64();
    if (P.trace && blockIdx.x == 0 && threadIdx.x == 0) { P.trace[0] = 0x7ACE7ACEu; P.trace[1] = 0u; }
#endif
    long long tk = 0;
    auto tick = [&](int slot) {  // profiling: cycles (>> 8) per section, accumulated by thread 0
        if (P.stats && threadIdx.x == 0) {
            const long long now = clock64();
            if (slot >= 0) atomicAdd(P.stats + slot, (unsigned)((now - tk) >> 8));
            tk = now;
        }
    };

    auto rflag_get = [&](int pi) -> unsigned { return (((volatile unsigned *)rflagW)[pi >> 2] >> (8 * (pi & 3))) & 0xFFu; };
    auto rflag_or = [&](int pi, unsigned f) -> unsigned {  // returns the flags before the update
        return (atomicOr(&rflagW[pi >> 2], f << (8 * (pi & 3))) >> (8 * (pi & 3))) & 0xFFu;
    };
    // Trees of a phase that run into each other are put into one class (union-find over their roots, path halving,
    // larger id under smaller): what one of them could not enter, the other explored, so a class none of whose trees
    // found a free GT pixel is closed under alternating reachability as a whole (see the phase epilogue).
    auto class_find = [&](int x) -> int {
        volatile unsigned short *cp = classP;
        int p = cp[x];
        while (p != x) {
            const int gp = cp[p];
            if (gp == p) return p;
            cp[x] = (unsigned short)gp;
            x = gp;
            p = cp[x];
        }
        return x;
    };
    auto class_union = [&](int a, int b) {
        for (;;) {
            a = class_find(a);
            b = class_find(b);
            if (a == b) return;
            if (a < b) { const int t = a; a = b; b = t; }
            if (cas16(&classP[a], (unsigned short)a, (unsigned short)b) == (unsigned short)a) return;
        }
    };
    // Is window pixel q a GT pixel, and which id does it have?  The rank is kept per 64 window pixels (two bitmap
    // words); the word pair and the rank are fetched together, before the bit is known: ONE shared-memory round trip
    // on the chain of a hop instead of two (the bitmap is padded to whole 16-byte groups).
    auto qprobe = [&](int q, int &qi) -> bool {
        const uint2 b = *reinterpret_cast<const uint2 *>(qbits + ((q >> 6) << 1));
        const int r0 = (int)qrank[q >> 6];
        const unsigned word = (q & 32) ? b.y : b.x;
        qi = r0 + __popc(word & ((1u << (q & 31)) - 1u)) + ((q & 32) ? __popc(b.x) : 0);
        return (word >> (q & 31)) & 1u;
    };
    // stage at which window pixel (gy, gx) of image img joins the predicted set; T = never
    auto stage_of = [&](int img, int gy, int gx) -> int {
        const size_t o = (size_t)img * P.H * P.W + (size_t)gy * P.W + gx;
        if (levels) {
            const int L = ((const unsigned char *)P.pred)[o];
            return L < T ? L : T;
        }
        const double v = P.inMode == IN_F32 ? (double)((const float *)P.pred)[o] : ((const double *)P.pred)[o];
        // thresholds ascend: count = #{t : v >= thr[t]} by bisection; the pixel belongs to P_t for t < count and the
        // stages run from the largest threshold down
        int lo = 0, hi = T;
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (v >= sThr[mid]) lo = mid + 1; else hi = mid;
        }
        return T - lo;  // lo == 0 (below every threshold, or NaN) -> T = never
    };
    // resident predicted pixels are kept as y << 16 | x: the hop of an alternating chain then needs no division
    auto pack_yx = [&](unsigned i) -> unsigned { const unsigned y = i / (unsigned)w; return (y << 16) | (i - y * (unsigned)w); };
    const short2 off0 = sOff[min(lane, noff - 1)];  // lane's own entry of the first 32 offsets (all of them at KITTI radius)

    for (;;) {
        const int img = next_ticket(P, false, sImage);
        if (img >= P.N) break;
        const unsigned char *gt = P.gt + (size_t)img * P.H * P.W;
        if (threadIdx.x == 0) { sNQ = 0; sMatched = 0; }
#ifdef MTE_DEBUG_KNOBS
        if (threadIdx.x == 0) sMaxChain = 0;
#endif
        for (int i = threadIdx.x; i < T + 2; i += kSwThreads) sStage[i] = 0;
        __syncthreads();
        tick(-1);

        // ---- ONE pass over the window: GT bitmap (atomicOr per GT pixel), stage histogram, and the predicted pixels
        //      appended unsorted as pixel | stage << 24 to a temporary list in this CTA's global arena (written once,
        //      read once).  Level planes are read as 32-bit words (4 pixels) when the layout allows it.
        unsigned *tmpList = reinterpret_cast<unsigned *>(P.arena + (size_t)blockIdx.x * P.arenaBytes);  // hw entries
        unsigned *gpix = tmpList + hw;                                                                 // sorted by stage
        for (int i = threadIdx.x; i < SL.nW; i += kSwThreads) qbits[i] = 0u;
        if (threadIdx.x == 0) sNP = 0;
        __syncthreads();
        auto emit = [&](int i, int stg, bool isQ) {  // window pixel i
            if (isQ) atomicOr(&qbits[i >> 5], 1u << (i & 31));
            if (stg < T) {
                atomicAdd(&sStage[stg], 1);
                const int slot = atomicAdd(&sNP, 1);
                tmpList[slot] = (unsigned)i | ((unsigned)stg << 24);
            }
        };
        const unsigned char *lv = (const unsigned char *)P.pred + (size_t)img * P.H * P.W;
        const bool words = levels && (P.W % 4) == 0 && ((reinterpret_cast<uintptr_t>(lv) | reinterpret_cast<uintptr_t>(gt)) & 3) == 0;
        if (words) {
            const int xa = P.x0 & ~3;                          // first word column
            const int cpr = (P.x0 + w - xa + 3) >> 2;          // words per window row
            const int nChunks = cpr * h;
            // kScanU independent word pairs per thread in flight: the scan is one CTA streaming 0.5 MB, i.e. latency-
            // bound (4 in flight: 31 round trips for the KITTI crop, 80 us of every image's critical path)
            constexpr int kScanU = 12;
            for (int base = 0; base < nChunks; base += kScanU * kSwThreads) {
                unsigned lw[kScanU], gw[kScanU];
#pragma unroll
                for (int u = 0; u < kScanU; u++) {
                    const int c = base + u * kSwThreads + threadIdx.x;
                    lw[u] = 0xFFFFFFFFu; gw[u] = 0u;
                    if (c < nChunks) {
                        const int y = c / cpr, cx = xa + 4 * (c - y * cpr);
                        const size_t o = (size_t)(P.y0 + y) * P.W + cx;
                        lw[u] = *reinterpret_cast<const unsigned *>(lv + o);
                        gw[u] = *reinterpret_cast<const unsigned *>(gt + o);
                    }
                }
#pragma unroll
                for (int u = 0; u < kScanU; u++) {
                    const int c = base + u * kSwThreads + threadIdx.x;
                    if (c >= nChunks) continue;
                    // most words hold neither an edge of any setting nor a GT pixel
                    if (gw[u] == 0u && __vcmpltu4(lw[u], (unsigned)T * 0x01010101u) == 0u) continue;
                    const int y = c / cpr, cx = xa + 4 * (c - y * cpr);
#pragma unroll
                    for (int k = 0; k < 4; k++) {
                        const int x = cx + k - P.x0;
                        if (x < 0 || x >= w) continue;
                        const int L = (lw[u] >> (8 * k)) & 0xFF;
                        const bool isQ = ((gw[u] >> (8 * k)) & 0xFF) != 0;
                        if (L < T || isQ) emit(y * w + x, L < T ? L : T, isQ);
                    }
                }
            }
        } else {
            for (int base = 0; base < hw; base += 4 * kSwThreads) {
                int stg[4];
                bool isQ[4];
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    const int i = base + u * kSwThreads + threadIdx.x;
                    stg[u] = T; isQ[u] = false;
                    if (i < hw) {
                        const int y = i / w, x = i - y * w;
                        stg[u] = stage_of(img, P.y0 + y, P.x0 + x);
                        isQ[u] = gt[(size_t)(P.y0 + y) * P.W + P.x0 + x] != 0;
                    }
                }
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    const int i = base + u * kSwThreads + threadIdx.x;
                    if (i < hw && (stg[u] < T || isQ[u])) emit(i, stg[u], isQ[u]);
                }
            }
        }
        __syncthreads();
        {  // number of GT pixels = population of the bitmap
            int c = 0;
            for (int i = threadIdx.x; i < SL.nW; i += kSwThreads) c += __popc(qbits[i]);
            c = __reduce_add_sync(MTE_FULL_MASK, c);
            if (lane == 0 && c) atomicAdd(&sNQ, c);
        }
        __syncthreads();
        const int nQ = sNQ;
        const int nPall = sNP;
        // stage offsets (T <= 254: one warp scans them)
        if (warp == 0) {
            int run = 0;
            for (int b0 = 0; b0 < T; b0 += 32) {
                const int k = b0 + lane;
                const int c = k < T ? sStage[k] : 0;
                int incl = c;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(MTE_FULL_MASK, incl, o); if (lane >= o) incl += v; }
                if (k < T) { sStage[k] = run + incl - c; sCursor[k] = run + incl - c; }
                run += __shfl_sync(MTE_FULL_MASK, incl, 31);
            }
            if (lane == 0) sStage[T] = run;
        }
        // the predicted side only has to hold the MATCHED pixels (<= nQ) plus a chunk of new ones (see below)
        if (nQ > SL.capQ || nQ >= 0xFFF0 || SL.capP - nQ < 256) {  // does not fit: per-problem kernels
            if (threadIdx.x == 0) {
                const int at = (int)atomicAdd(P.overflowCount, (unsigned)T);
                for (int t = 0; t < T; t++) P.overflowList[at + t] = img * T + t;
            }
            __syncthreads();
            continue;
        }
        __syncthreads();
        // ---- predicted pixels grouped by stage (order inside a stage is arbitrary: counts do not depend on it)
        for (int k0 = threadIdx.x; k0 < nPall; k0 += 4 * kSwThreads) {   // four list entries per thread in flight
            unsigned v[4];
#pragma unroll
            for (int u = 0; u < 4; u++) v[u] = k0 + u * kSwThreads < nPall ? __ldcg(tmpList + k0 + u * kSwThreads) : 0xFFFFFFFFu;
#pragma unroll
            for (int u = 0; u < 4; u++)
                if (k0 + u * kSwThreads < nPall) gpix[atomicAdd(&sCursor[v[u] >> 24], 1)] = v[u] & 0xFFFFFFu;
        }
        __syncthreads();
        // Everything resident at once when it fits.  Otherwise ("compact" mode) the predicted arrays only ever hold the
        // matched pixels plus one chunk of new ones: pixels whose search failed (or that have no GT pixel in range)
        // can never be matched later (Kuhn), are never reached as somebody's mate, and are dropped after every chunk.
        const bool compact = nPall > SL.capP;
        if (!compact)
            for (int k0 = threadIdx.x; k0 < nPall; k0 += 4 * kSwThreads) {
                unsigned v[4];
#pragma unroll
                for (int u = 0; u < 4; u++) v[u] = k0 + u * kSwThreads < nPall ? __ldcg(gpix + k0 + u * kSwThreads) : 0u;
#pragma unroll
                for (int u = 0; u < 4; u++)
                    if (k0 + u * kSwThreads < nPall) { ppix[k0 + u * kSwThreads] = pack_yx(v[u]); mateP[k0 + u * kSwThreads] = kFree; }
            }
        // ---- rank: exclusive prefix popcount over pairs of bitmap words
        {
            const int nW2 = (SL.nW + 1) >> 1;
            const int per = (nW2 + kSwThreads - 1) / kSwThreads;
            const int w0 = threadIdx.x * per, w1 = min(w0 + per, nW2);
            auto pc2 = [&](int k2) { return __popc(qbits[2 * k2]) + (2 * k2 + 1 < SL.nW ? __popc(qbits[2 * k2 + 1]) : 0); };
            int sum = 0;
            for (int k2 = w0; k2 < w1; k2++) sum += pc2(k2);
            int run = block_exclusive_scan<kSwThreads>(sum, sScan);
            for (int k2 = w0; k2 < w1; k2++) { qrank[k2] = (unsigned short)run; run += pc2(k2); }
        }
        for (int k = threadIdx.x; k < nQ; k += kSwThreads) { mateQ[k] = kFree; stamp[k] = 0u; }
        __syncthreads();
        tick(4);

        unsigned short phase = 0;
        int nLive = 0;  // compact mode: matched pixels currently resident
        for (int s = 0; s < T; s++) {
            const long long tStage = (P.stats && threadIdx.x == 0) ? clock64() : 0;
            const int G0 = sStage[s], G1 = sStage[s + 1];  // the pixels that join at this stage (positions in gpix)
            int cur = G0;
            do {
            int p0 = G0, p1 = G1;  // resident index range of the new pixels; [0, p1) is everything resident
            if (compact) {
                const int n = min(G1 - cur, SL.capP - nLive);
                p0 = nLive; p1 = nLive + n;
                for (int k = threadIdx.x; k < n; k += kSwThreads) {
                    ppix[p0 + k] = pack_yx(__ldcg(gpix + cur + k)); mateP[p0 + k] = kFree;
                }
                cur += n;
                __syncthreads();
            } else {
                cur = G1;
            }
            if (p1 > p0) {
                // ---- greedy start: nearest free GT pixel, one THREAD per new predicted pixel, the offsets nearest first
                //      (any greedy start is a valid matching).  The walk is cut into ROUNDS of a few offsets: the pixels
                //      that are still unmatched after a round are compacted into a list for the next one, so that the
                //      few pixels that have to try all offsets do not hold their whole warps for 21 serial probes
                //      (one thread walking everything: 8 rounds x 21 probes per warp, 80 us on the heaviest image).
                //      Lists live in the frontier / root arrays, which are idle until the phases; "saw a GT pixel" is
                //      remembered in the pixel's own mate entry (kSeenQ) until the walk ends.
                {
                    constexpr unsigned short kSeenQ = 0xFFFC;
                    unsigned short *lst[2] = {fa, rootP};
                    if (threadIdx.x < 3) sGr[threadIdx.x] = 0;
                    __syncthreads();
                    int n = p1 - p0, kLo = 0, round = 0;
                    for (; n > 0 && kLo < noff; round++) {
                        const int kHi = min(noff, kLo < 1 ? 1 : (kLo < 5 ? 5 : (kLo < 9 ? 9 : (kLo < 21 ? 21 : kLo + 32))));
                        const int nxt = (round + 1) % 3;
                        const unsigned short *src = lst[round & 1];
                        unsigned short *dst = lst[(round + 1) & 1];
                        if (threadIdx.x == 0) sGr[(round + 2) % 3] = 0;   // next round's append counter (read two rounds ago)
                        for (int i = threadIdx.x; i < n; i += kSwThreads) {
                            const int pi = round == 0 ? p0 + i : (int)src[i];
                            const unsigned p = ppix[pi];
                            const int py = (int)(p >> 16), px = (int)(p & 0xFFFFu);
                            bool done = false;
                            for (int k = kLo; k < kHi && !done; k++) {
                                const short2 o = sOff[k];
                                const int qy = py + o.y, qx = px + o.x;
                                if (qy < 0 || qy >= h || qx < 0 || qx >= w) continue;
                                const int q = qy * w + qx;
                                int qi;
                                if (!qprobe(q, qi)) continue;
                                if (mateP[pi] == kFree) mateP[pi] = kSeenQ;
                                if (((volatile unsigned short *)mateQ)[qi] != kFree) continue;
                                if (cas16(&mateQ[qi], kFree, (unsigned short)pi) == kFree) {
                                    mateP[pi] = (unsigned short)qi;
                                    done = true;
                                }
                            }
                            if (done) atomicAdd(&sMatched, 1);
                            else dst[atomicAdd(&sGr[nxt], 1)] = (unsigned short)pi;
                        }
                        __syncthreads();
                        n = sGr[nxt];
                        kLo = kHi;
                    }
                    // what is left went through every offset: free again if it saw a GT pixel, dead (never matchable) if not
                    const unsigned short *rest = lst[round & 1];
                    for (int i = threadIdx.x; i < n; i += kSwThreads) {
                        const int pi = round == 0 ? p0 + i : (int)rest[i];
                        mateP[pi] = mateP[pi] == kSeenQ ? kFree : kDead;
                    }
                }
                __syncthreads();
                tick(5);
                // ---- augmenting phases rooted at the new pixels that are still free
                for (;;) {
                    phase++;
                    if (threadIdx.x == 0) { sCntA = 0; sEnds = 0; }
                    __syncthreads();
                    for (int base = p0; base < p1; base += kSwThreads) {
                        const int pi = base + threadIdx.x;
                        const bool fr = pi < p1 && mateP[pi] == kFree;
                        const int slot = warp_append(&sCntA, fr);
                        if (fr) {
                            fa[slot] = (unsigned short)pi;
                            rootP[pi] = (unsigned short)pi;
                            classP[pi] = (unsigned short)pi;
                        }
                    }
                    // flag bytes of this stage's pixels (only roots use theirs)
                    for (int i = (p0 >> 2) + threadIdx.x; i <= ((p1 - 1) >> 2); i += kSwThreads) rflagW[i] = 0u;
                    __syncthreads();
                    const int nRoots = sCntA;
                    if (nRoots == 0) break;
                    if (P.stats && threadIdx.x == 0) { atomicAdd(P.stats + 0, 1u); atomicAdd(P.stats + 3, (unsigned)nRoots); }
                    // asynchronous alternating forest (see match_smem_kernel); dead GT vertices are walls.  Every GT
                    // stamp carries the tree (root) that claimed it: a tree that has found a free GT pixel stops
                    // growing; trees that run into each other's vertices are joined into a class.  The trees of a
                    // class without any find have, between them, expanded everything reachable from their roots and
                    // met no free GT pixel: the class is closed under alternating reachability, hence dead for good,
                    // whatever the other trees of the phase do (a single tree that met nobody is the 1-tree case).
                    for (int i = nRoots + threadIdx.x; i < p1; i += kSwThreads) fa[i] = kFree;  // unpublished slots
                    if (threadIdx.x == 0) { sHead = 0; sTail = nRoots; sPending = nRoots; }
                    __syncthreads();
                    tick(6);
                    for (;;) {
#ifdef MTE_DEBUG_KNOBS
                        const long long tWait = (P.trace && lane == 0) ? clock64() : 0;
#endif
                        const int my = queue_pop(&sHead, &sTail, &sPending, fa);
                        if (my == -2) break;
#ifdef MTE_DEBUG_KNOBS   // profiling: queue items (roots + published successors)
                        if (P.stats && lane == 0) atomicAdd(P.stats + 22, 1u);
                        int nHops = 0;
                        const long long tBeg = (P.trace && lane == 0) ? clock64() : 0;
#endif
                        int pi = my;
                        const int root = rootP[pi];  // a successor inherits the tree of its predecessor
                        const unsigned mine = ((unsigned)phase << 16) | (unsigned)root;
                        unsigned p = ppix[pi];
                        unsigned found = rflag_get(root) & RF_FOUND;
                        int lastOther = -1;  // the tree this lane last joined with root's (skips repeated unions)
                        for (;;) {  // a warp keeps ONE successor and goes on with it directly (chains along contours
                                    // would otherwise pay a queue round trip per hop); the others are published.
                                    // The hop is a chain of dependent shared-memory round trips, so everything whose
                                    // address is known early is loaded early: the mate and ITS position next to the
                                    // stamp (the matching does not change during a phase), so the next hop starts with
                                    // its probes; the "tree already found a free GT pixel" flag is only a hint to stop
                                    // growing and is read one hop ahead, off the chain.
                            int keep = -1;
                            unsigned keepP = 0u;
                            const unsigned foundNext = rflag_get(root) & RF_FOUND;
                            if (!found) {
                                const int py = (int)(p >> 16), px = (int)(p & 0xFFFFu);
                                for (int k0 = 0; k0 < noff; k0 += 32) {
                                    const int k = k0 + lane;
                                    int succ = -1;
                                    unsigned succP = 0u;
                                    if (k < noff) {
                                        const short2 o = k0 == 0 ? off0 : sOff[k];
                                        const int qy = py + o.y, qx = px + o.x;
                                        if (qy >= 0 && qy < h && qx >= 0 && qx < w) {
                                            const int q = qy * w + qx;
                                            int qi;
                                            if (qprobe(q, qi)) {
                                                unsigned st = stamp[qi];
                                                const unsigned short mq = mateQ[qi];
                                                if (st != kDeadStamp) {
                                                    if (mq != kFree) succP = ppix[mq];
                                                    bool claimed = false;
                                                    if ((st >> 16) != phase) {
                                                        const unsigned old = atomicCAS(&stamp[qi], st, mine);
                                                        claimed = old == st;
                                                        st = old;  // if somebody else got it first
                                                    }
                                                    if (claimed) {
                                                        parentQ[qi] = (unsigned short)pi;
                                                        if (mq == kFree) {
                                                            // only the FIRST free GT pixel of a tree is recorded: trees are
                                                            // vertex-disjoint, so the recorded paths are too and can be
                                                            // flipped without a claim walk
                                                            if (!(rflag_or(root, RF_FOUND) & RF_FOUND)) {
                                                                const int es = atomicAdd(&sEnds, 1);
                                                                if (es < kEndsCap) ends[es] = (unsigned short)qi;
                                                            }
                                                        } else {
                                                            rootP[mq] = (unsigned short)root;
                                                            succ = mq;
                                                        }
                                                    } else if (st != kDeadStamp && (st & 0xFFFFu) != (unsigned)root) {
                                                        const int other = (int)(st & 0xFFFFu);
                                                        if (other != lastOther) { lastOther = other; class_union(root, other); }
                                                    }
                                                }
                                            }
                                        }
                                    }
                                    unsigned m = __ballot_sync(MTE_FULL_MASK, succ >= 0);
                                    if (m && keep < 0) {
                                        // Which successor the warp keeps is free (any order of exploration is exact): the
                                        // nearest one (lowest lane).  Keeping the FARTHEST one (longer steps along a
                                        // contour) was measured: more queue items (5.1 k -> 7.0 k on the heaviest image)
                                        // and a slower step (1.62 -> 1.70 ms).
                                        const int kl = __ffs(m) - 1;
                                        keep = __shfl_sync(MTE_FULL_MASK, succ, kl);
                                        keepP = __shfl_sync(MTE_FULL_MASK, succP, kl);
                                        m &= ~(1u << kl);
                                    }
                                    if (m) {
                                        int base = 0;
                                        if (lane == 0) {
                                            atomicAdd(&sPending, __popc(m));
                                            base = atomicAdd(&sTail, __popc(m));
                                        }
                                        base = __shfl_sync(MTE_FULL_MASK, base, 0);
                                        __threadfence_block();
                                        if ((m >> lane) & 1u)
                                            ((volatile unsigned short *)fa)[base + __popc(m & ((1u << lane) - 1u))] = (unsigned short)succ;
                                    }
                                }
                            }
                            if (P.stats && lane == 0) atomicAdd(P.stats + 2, 1u);
#ifdef MTE_DEBUG_KNOBS
                            nHops++;
#endif
                            if (keep < 0) break;
                            pi = keep;
                            p = keepP;
                            found = foundNext;
                        }
                        __syncwarp();
                        if (lane == 0) {
                            __threadfence_block();
                            atomicSub(&sPending, 1);
#ifdef MTE_DEBUG_KNOBS
                            if (P.stats) atomicMax(&sMaxChain, nHops);
                            if (P.trace && s == 0 && nRoots >= 16) {
                                const unsigned at = atomicAdd(P.trace + 1, 1u);
                                if (at < 8000u) {
                                    unsigned *e = P.trace + 4 + 4 * at;
                                    e[0] = (unsigned)warp | ((unsigned)(phase & 0xFF) << 8) | ((unsigned)min(nHops, 0xFFFF) << 16);
                                    e[1] = (unsigned)((tWait - tZero) >> 2);
                                    e[2] = (unsigned)((tBeg - tZero) >> 2);
                                    e[3] = (unsigned)((clock64() - tZero) >> 2);
                                }
                            }
#endif
                        }
                    }
                    __syncthreads();
#ifdef MTE_DEBUG_KNOBS   // profiling: explore cycles (>> 8) and phase counts by the number of roots of the phase; the
                         // longest single walk of the phases with 16+ roots summed into slot 31
                    if (P.stats && threadIdx.x == 0) {
                        const int b = nRoots == 1 ? 0 : (nRoots < 4 ? 1 : (nRoots < 16 ? 2 : 3));
                        atomicAdd(P.stats + 23 + b, (unsigned)((clock64() - tk) >> 8));
                        atomicAdd(P.stats + 27 + b, 1u);
                        if (b == 3) atomicAdd(P.stats + 31, (unsigned)sMaxChain);
                        sMaxChain = 0;
                    }
#endif
                    tick(7);
                    const int nEnds = min(sEnds, kEndsCap);
                    // a find anywhere in a class keeps the whole class alive (fa[0..nRoots) still holds the roots: the
                    // queue is append-only)
                    if (nEnds != 0) {
                        for (int i = threadIdx.x; i < nRoots; i += kSwThreads) {
                            const int rp = fa[i];
                            if (rflag_get(rp) & RF_FOUND) rflag_or(class_find(rp), RF_CLASS_FOUND);
                        }
                        __syncthreads();
                    }
                    // wall off the classes that failed conclusively (all of them when the phase found nothing) ...
                    for (int k = threadIdx.x; k < nQ; k += kSwThreads) {
                        const unsigned st = stamp[k];
                        if (st != kDeadStamp && (st >> 16) == phase &&
                            (nEnds == 0 || !(rflag_get(class_find((int)(st & 0xFFFFu))) & RF_CLASS_FOUND)))
                            stamp[k] = kDeadStamp;
                    }
                    // ... and retire their roots
                    for (int i = threadIdx.x; i < nRoots; i += kSwThreads) {
                        const int rp = fa[i];
                        if (nEnds == 0 || !(rflag_get(class_find(rp)) & RF_CLASS_FOUND)) mateP[rp] = kFailed;
                    }
                    __syncthreads();
                    if (nEnds == 0) { tick(8); break; }
                    for (int ei = threadIdx.x; ei < nEnds; ei += kSwThreads) {
                        flip_path(ends[ei], parentQ, mateP, mateQ);  // one path per tree, see above
                        atomicAdd(&sMatched, 1);
                    }
                    __syncthreads();
                    tick(8);
                    if (phase >= 0xFFF0) break;  // unreachable in practice (every phase adds a match or ends the stage)
                }
            }
            __syncthreads();
            if (compact) {
                // ---- drop the pixels that are not matched (in place, stable, one block-wide round of kSwThreads
                //      elements at a time: destinations never run ahead of the round being read) and re-point their mates
                int kept = 0;
                for (int base = 0; base < p1; base += kSwThreads) {
                    const int i = base + threadIdx.x;
                    unsigned px = 0;
                    unsigned short mp = kDead;
                    if (i < p1) { px = ppix[i]; mp = mateP[i]; }
                    const bool keep = mp < kFailed;
                    const unsigned bal = __ballot_sync(MTE_FULL_MASK, keep);
                    if (lane == 0) sScan[warp] = __popc(bal);
                    __syncthreads();
                    int off = kept, tot = 0;
                    for (int wv = 0; wv < kSwWarps; wv++) { const int c = sScan[wv]; if (wv < warp) off += c; tot += c; }
                    if (keep) {
                        const int d = off + __popc(bal & ((1u << lane) - 1u));
                        ppix[d] = px; mateP[d] = mp;
                        mateQ[mp] = (unsigned short)d;
                    }
                    kept += tot;
                    __syncthreads();
                }
                nLive = kept;
            }
            } while (cur < G1);
            __syncthreads();
            // ---- the count of this stage's threshold
            if (P.stats && threadIdx.x == 0) {  // profiling (debug builds): cycles >> 8 and new pixels per stage
                atomicAdd(P.stats + 9 + min(s, 11), (unsigned)((clock64() - tStage) >> 8));
                if (s == 0) atomicAdd(P.stats + 21, (unsigned)(G1 - G0));
            }
            // per-image rows: the image this CTA is sweeping (thread 0 wrote sImage)
            if (threadIdx.x == 0) add_counts(P, sImage, levels ? s : T - 1 - s, sMatched, nQ, G1);
        }
        __syncthreads();
    }
    reset_scheduler(P, false);
}

// ---------------------------------------------------------------------------
// Thinned sweep (apply_thinning = 1): one CTA per (image, threshold) problem of a chunk binarises its window with
// the sweep rule, thins it to convergence with the bit-parallel routine of thin.cuh (zero padding at the WINDOW
// border: the reference crops before it thins) and writes the thinned bit plane to the problem's slot of the slab.
// The per-problem matchers then read the slab in IN_BITS mode.  The two bit planes live in dynamic shared memory when
// they fit (KITTI crop 218 x 1153: 2 x 32.3 KB), else the slab slot and a scratch slot of the workspace are used.
// ---------------------------------------------------------------------------
struct ThinP {
    const void *pred;   // [N,H,W] levels u8 / f32 / f64
    int inMode, H, W, T;
    int x0, y0, w, h, nw;
    size_t plane;       // stride of the bit planes in words: h * nw rounded up to 64 (the words past h * nw are unused)
    unsigned *slab;     // [chunk][plane] thinned planes (out)
    unsigned *scratch;  // [chunk][plane] second plane of the global-memory path
    int probBase;
};
struct ThrTable {
    double v[MTE_MAX_THRESHOLDS];
};

__global__ void __launch_bounds__(thin::kThreads) thin_window_kernel(const __grid_constant__ ThinP Q,
                                                                     const __grid_constant__ ThrTable thr, int inSmem) {
    extern __shared__ __align__(16) unsigned char dyn[];
    const int g = Q.probBase + (int)blockIdx.x;
    const int img = g / Q.T, t = g - img * Q.T;
    unsigned *slab = Q.slab + blockIdx.x * Q.plane;
    unsigned *a = inSmem ? reinterpret_cast<unsigned *>(dyn) : slab;
    unsigned *b = inSmem ? a + Q.plane : Q.scratch + blockIdx.x * Q.plane;
    const size_t imgBase = (size_t)img * Q.H * Q.W;
    const size_t n = (size_t)Q.h * Q.nw;  // the window's words: row y < h only, never the stride's padding
    // binarise: one warp per word, one lane per pixel (bits past w stay zero)
    const int lane = threadIdx.x & 31;
    for (size_t i = threadIdx.x >> 5; i < n; i += thin::kThreads / 32) {
        const int y = (int)(i / Q.nw), x = (int)(i - (size_t)y * Q.nw) * 32 + lane;
        const bool set = x < Q.w && sweep_pred(Q.pred, Q.inMode, imgBase + (size_t)(Q.y0 + y) * Q.W + Q.x0 + x, t, thr.v);
        const unsigned m = __ballot_sync(MTE_FULL_MASK, set);
        if (lane == 0) a[i] = m;
    }
    __syncthreads();
    const unsigned *r = thin::thin_plane(a, b, Q.h, Q.nw, -1);
    if (r != slab)
        for (size_t i = threadIdx.x; i < n; i += thin::kThreads) slab[i] = r[i];
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
struct OffsetTable {
    int n;
    short2 off[kMaxOff];
    unsigned short neg[kMaxOff];
};

static int build_offsets(double radius, OffsetTable &tb) {
    const int r = (int)radius;
    const double r2 = radius * radius;
    tb.n = 0;
    if (r > 31) return MTE_ERR_ARG;  // (2r+1)^2 <= 3969 entries
    for (int d2 = 0; d2 <= 2 * r * r; d2++)
        for (int dy = -r; dy <= r; dy++)
            for (int dx = -r; dx <= r; dx++)
                if (dy * dy + dx * dx == d2 && (double)d2 <= r2) {
                    tb.off[tb.n].x = (short)dx;
                    tb.off[tb.n].y = (short)dy;
                    tb.n++;
                }
    for (int i = 0; i < tb.n; i++)
        for (int j = 0; j < tb.n; j++)
            if (tb.off[j].x == -tb.off[i].x && tb.off[j].y == -tb.off[i].y) tb.neg[i] = (unsigned short)j;
    return MTE_OK;
}

struct Layout {
    size_t offTable, offNeg, offThr, offOverflow, offArena, arenaBytes, total;
    int nArenas;
};

// The dynamic shared memory of the resident matchers, for a w x h window (nW bitmap words).  vertex_cap: the
// capacity, equal for both sides, that the budget leaves after the fixed bytes at perVertex bytes per predicted + GT
// vertex; 0 (the kernel is not used) below 512.  Carve hands out 16 B aligned regions one after another.
static int vertex_cap(int budget, long long fixed, int perVertex) {
    const long long cap = (budget - fixed) / perVertex;
    return cap < 512 ? 0 : (int)(cap > 0xFFF0 ? 0xFFF0 : cap) & ~7;
}
struct Carve {
    unsigned o = 0;
    unsigned take(unsigned bytes) { const unsigned r = o; o += (bytes + 15u) & ~15u; return r; }
};

// capP = capQ = 0 if the window cannot fit
static SmemLayout smem_layout(int h, int w, int budget) {
    SmemLayout S;
    memset(&S, 0, sizeof(S));
    S.nW = (int)(((long long)h * w + 31) / 32);
    // 12 B per predicted vertex + 8 B per GT vertex
    S.capP = S.capQ = vertex_cap(budget, (long long)S.nW * 4 + (((long long)S.nW * 2 + 15) / 16) * 16 + 256, 20);
    if (S.capP == 0) return S;
    Carve C;
    S.oBits = C.take(S.nW * 4);
    S.oRank = C.take(S.nW * 2);
    S.oPpix = C.take(S.capP * 4);
    S.oMateP = C.take(S.capP * 2);
    S.oClaimP = C.take(S.capP * 2);
    S.oFa = C.take(S.capP * 2);
    S.oFb = C.take(S.capP * 2);  // read by nothing, but its 2 B per vertex are part of capP
    S.oMateQ = C.take(S.capQ * 2);
    S.oParentQ = C.take(S.capQ * 2);
    S.oStampQ = C.take(S.capQ * 2);
    S.oEnds = C.take(S.capQ * 2);
    S.total = C.o;
    return S;
}

static SweepLayout sweep_layout(int h, int w, int budget) {
    SweepLayout S;
    memset(&S, 0, sizeof(S));
    S.nW = (int)(((long long)h * w + 31) / 32);
    // 13 B per predicted vertex, 8 B per GT vertex
    S.capP = S.capQ = vertex_cap(budget, (long long)S.nW * 4 + (long long)S.nW + 2 * kEndsCap + 512, 21);
    if (S.capP == 0) return S;
    Carve C;
    S.oBits = C.take(S.nW * 4);
    S.oRank = C.take(((S.nW + 1) / 2) * 2);
    S.oPpix = C.take(S.capP * 4);
    S.oMateP = C.take(S.capP * 2);
    S.oClassP = C.take(S.capP * 2);
    S.oFa = C.take(S.capP * 2);
    S.oRootP = C.take(S.capP * 2);
    S.oRflag = C.take(S.capP + 4);
    S.oMateQ = C.take(S.capQ * 2);
    S.oParentQ = C.take(S.capQ * 2);
    S.oStamp = C.take(S.capQ * 4);
    S.oEnds = C.take(kEndsCap * 2);
    S.total = C.o;
    return S;
}

static Layout layout(int nProblems, int h, int w, int T) {
    Layout L;
    size_t off = MTE_WS_HEADER_BYTES;
    L.offTable = off; off += align_up(sizeof(short2) * kMaxOff, 256);
    L.offNeg = off; off += align_up(sizeof(unsigned short) * kMaxOff, 256);
    L.offThr = off; off += align_up(sizeof(double) * (size_t)(T > 0 ? T : 1), 256);
    L.offOverflow = off; off += align_up(sizeof(int) * (size_t)(nProblems > 0 ? nProblems : 1), 256);
    L.arenaBytes = align_up(arena_bytes(h, w), 256);
    int n = num_sms() * kCtasPerSm;
    if (n > nProblems) n = nProblems;
    if (n < 1) n = 1;
    L.nArenas = n;
    L.offArena = off; off += L.arenaBytes * (size_t)n;
    L.total = off;
    return L;
}

// one bound of a python slice over dim entries: a negative bound counts from the end, then [0, dim] clamps
static int slice_bound(int b, int dim) {
    if (b < 0) b += dim;
    return b < 0 ? 0 : (b > dim ? dim : b);
}

static void clip_crop(const int32_t *crop, int H, int W, int &x0, int &y0, int &w, int &h) {
    int cx0 = 0, cx1 = W, cy0 = 0, cy1 = H;
    if (crop) {
        // python slice semantics of pred[c2:c3, c0:c1], as the reference crops (negative bounds included)
        cx0 = slice_bound(crop[0], W);
        cx1 = slice_bound(crop[1], W);
        cy0 = slice_bound(crop[2], H);
        cy1 = slice_bound(crop[3], H);
    }
    x0 = cx0; y0 = cy0;
    w = cx1 > cx0 ? cx1 - cx0 : 0;
    h = cy1 > cy0 ? cy1 - cy0 : 0;
}

static int launch(MatchP &P, const Layout &L, char *ws, double max_dist, const double *thr_host, cudaStream_t st) {
    OffsetTable tb;
    const double radius = max_dist * sqrt((double)P.h * P.h + (double)P.w * P.w);
    int rc = build_offsets(radius, tb);
    if (rc) return rc;
    static_assert(sizeof(MatchP) + sizeof(ParamTables) + 16 <= 4096, "kernel parameters exceed 4 KB");
    ParamTables pt;
    const bool inParam = tb.n <= kParamOff && (!thr_host || P.T <= kParamThr);
    if (inParam) {
        memcpy(pt.off, tb.off, sizeof(short2) * tb.n);
        memcpy(pt.neg, tb.neg, sizeof(unsigned short) * tb.n);
        if (thr_host) memcpy(pt.thr, thr_host, sizeof(double) * P.T);
    } else {
        // pageable-host async copies are staged by the runtime before they return (not graph-capturable)
        cudaError_t e = cudaMemcpyAsync(ws + L.offTable, tb.off, sizeof(short2) * tb.n, cudaMemcpyHostToDevice, st);
        if (e != cudaSuccess) return (int)e;
        e = cudaMemcpyAsync(ws + L.offNeg, tb.neg, sizeof(unsigned short) * tb.n, cudaMemcpyHostToDevice, st);
        if (e != cudaSuccess) return (int)e;
        if (thr_host && P.T > 0) {
            e = cudaMemcpyAsync(ws + L.offThr, thr_host, sizeof(double) * P.T, cudaMemcpyHostToDevice, st);
            if (e != cudaSuccess) return (int)e;
        }
    }
    P.noff = tb.n;
    P.off = reinterpret_cast<const short2 *>(ws + L.offTable);
    P.neg = reinterpret_cast<const unsigned short *>(ws + L.offNeg);
    P.thr = reinterpret_cast<const double *>(ws + L.offThr);
    P.arena = ws + L.offArena;
    P.arenaBytes = L.arenaBytes;
    WsHeader *hdr = reinterpret_cast<WsHeader *>(ws);
    P.stats = debug_knob("MTE_MATCH_STATS") ? hdr->pad : nullptr;
    P.trace = nullptr;
    if (debug_knob("MTE_MATCH_TRACE") && L.nArenas >= 2)   // the last arena is idle when a single image is matched
        P.trace = reinterpret_cast<unsigned int *>(ws + L.offArena + L.arenaBytes * (size_t)(L.nArenas - 1));
    P.nextProblem = hdr->ticket + 4;
    P.doneCtas = hdr->ticket + 5;
    P.overflowCount = hdr->ticket + 6;
    P.overflowList = reinterpret_cast<int *>(ws + L.offOverflow);
    P.problemList = nullptr;
    P.listCount = nullptr;
    // shared-memory kernel first (one CTA per SM, ~200 KB of state), the dense L2 kernel mops up what did not fit
    const SmemLayout SL = smem_layout(P.h, P.w, smem_budget(match_smem_kernel));
    const bool useSmem = SL.capP > 0 && tb.n <= kSmemTableOff;
    // threshold sweeps (level planes; strength maps with ascending thresholds): one CTA per image solves all T nested
    // problems incrementally; what does not fit falls through to the per-problem kernels via the overflow list
    // (thinned sets are not nested: the bits mode never sweeps)
    bool sweep = useSmem && P.counts && !P.matchA && !P.matchB && P.inMode != IN_BINARY && P.inMode != IN_BITS && P.T > 1;
    if (sweep && P.inMode != IN_LEVELS)
        for (int t = 1; t < P.T; t++)
            if (!(thr_host[t] > thr_host[t - 1])) sweep = false;
    const SweepLayout SW = sweep ? sweep_layout(P.h, P.w, smem_budget(match_sweep_kernel)) : SweepLayout{};
    if (useSmem) {
        if (SW.capP > 0)
            match_sweep_kernel<<<std::min(num_sms(), P.N), kSwThreads, SW.total, st>>>(P, pt, inParam ? 1 : 0, SW);
        else
            match_smem_kernel<<<std::min(num_sms(), P.nProblems), kSmThreads, SL.total, st>>>(P, pt, inParam ? 1 : 0, SL);
        MTE_RETURN_IF_CUDA_ERROR();
        // the overflowed problems (usually none) go to the dense kernel
        P.problemList = P.overflowList;
        P.listCount = P.overflowCount;
    }
    match_kernel<<<L.nArenas, kThreads, 0, st>>>(P, pt, inParam ? 1 : 0);
    MTE_RETURN_IF_CUDA_ERROR();
    return MTE_OK;
}

}  // namespace pr
}  // namespace mte

using namespace mte;
using namespace mte::pr;

extern "C" size_t mte_match_workspace_bytes(int n_problems, int h, int w, double max_dist) {
    if (n_problems < 1 || h < 1 || w < 1) return 0;
    (void)max_dist;
    return layout(n_problems, h, w, 1).total;
}

extern "C" int mte_correspond_pixels(const uint8_t *a, const uint8_t *b, int n_problems, int h, int w,
                                     double max_dist, uint8_t *match_a, uint8_t *match_b, int64_t *count,
                                     void *workspace, size_t ws_bytes, mte_stream_t stream) {
    if (!a || !b || !workspace) return MTE_ERR_NULL;
    if (n_problems < 1 || h < 1 || w < 1) return MTE_ERR_SHAPE;
    if (!(max_dist >= 0.0)) return MTE_ERR_ARG;
    const Layout L = layout(n_problems, h, w, 1);
    if (ws_bytes < L.total) return MTE_ERR_WORKSPACE;
    MatchP P;
    memset(&P, 0, sizeof(P));
    P.pred = a; P.gt = b; P.inMode = IN_BINARY;
    P.N = n_problems; P.H = h; P.W = w; P.T = 1;
    P.x0 = 0; P.y0 = 0; P.w = w; P.h = h;
    P.nProblems = n_problems;
    P.countPerProblem = reinterpret_cast<long long *>(count);
    P.matchA = match_a; P.matchB = match_b;
    return launch(P, L, static_cast<char *>(workspace), max_dist, nullptr, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" size_t mte_pr_workspace_bytes(int n_images, int H, int W, int T, double max_dist) {
    if (n_images < 1 || H < 1 || W < 1 || T < 1) return 0;
    (void)max_dist;
    // sized for the un-cropped window (a crop only shrinks it)
    return layout(n_images * T, H, W, T).total;
}

// The thinned sweep's slab (plus the scratch planes of the global-memory thinning path) follows the matcher's
// workspace.  It is sized for chunks of the uncropped plane with both planes in global memory and kept to about
// kThinSlabBudget, so the thinned planes of a chunk stay in L2 between the thinning and the matching launch; a call
// with a crop or with shared-memory thinning fits more problems into the same bytes.
constexpr size_t kThinSlabBudget = (size_t)64 << 20;

static size_t thin_plane_bytes(int h, int w) { return align_up((size_t)h * thin::words_per_row(w) * 4, 256); }

static size_t thin_region_bytes(int nProblems, int H, int W) {
    const size_t per = 2 * thin_plane_bytes(H, W);
    size_t chunk = kThinSlabBudget / per;
    if (chunk < 1) chunk = 1;
    if (chunk > (size_t)nProblems) chunk = (size_t)nProblems;
    return chunk * per;
}

extern "C" size_t mte_pr_thin_workspace_bytes(int n_images, int H, int W, int T, double max_dist) {
    if (n_images < 1 || H < 1 || W < 1 || T < 1) return 0;
    (void)max_dist;
    return layout(n_images * T, H, W, T).total + thin_region_bytes(n_images * T, H, W);
}

static int pr_counts_thinned(MatchP &P, const Layout &L, char *ws, double max_dist, const double *thr_host,
                             cudaStream_t st) {
    ThinP Q;
    memset(&Q, 0, sizeof(Q));
    Q.pred = P.pred; Q.inMode = P.inMode; Q.H = P.H; Q.W = P.W; Q.T = P.T;
    Q.x0 = P.x0; Q.y0 = P.y0; Q.w = P.w; Q.h = P.h; Q.nw = thin::words_per_row(P.w);
    Q.plane = thin_plane_bytes(P.h, P.w) / 4;
    ThrTable tt;
    memset(&tt, 0, sizeof(tt));
    if (thr_host) memcpy(tt.v, thr_host, sizeof(double) * P.T);
    const size_t smem = 2 * Q.plane * 4;
    bool inSmem = smem <= (size_t)dev_info().smemOptin;
    if (inSmem && opt_in_smem((const void *)thin_window_kernel, (int)smem) != cudaSuccess) {
        cudaGetLastError();
        inSmem = false;
    }
    const size_t region = thin_region_bytes(P.nProblems, P.H, P.W);
    int chunk = (int)std::min(region / ((inSmem ? 1 : 2) * Q.plane * 4), (size_t)P.nProblems);
    Q.slab = reinterpret_cast<unsigned *>(ws + L.total);
    Q.scratch = Q.slab + (size_t)chunk * Q.plane;
    P.inMode = IN_BITS;
    P.bits = Q.slab;
    P.bitsPlane = Q.plane;
    P.bitsNw = Q.nw;
    const int nAll = P.nProblems;
    for (int base = 0; base < nAll; base += chunk) {
        const int n = std::min(chunk, nAll - base);
        Q.probBase = base;
        thin_window_kernel<<<n, thin::kThreads, inSmem ? smem : 0, st>>>(Q, tt, inSmem ? 1 : 0);
        MTE_RETURN_IF_CUDA_ERROR();
        P.probBase = base;
        P.nProblems = n;
        const int rc = launch(P, L, ws, max_dist, nullptr, st);
        if (rc) return rc;
    }
    return MTE_OK;
}

// perImage = 0: counts [T][4] summed over the images; 1: counts [N][T][4], one row per (image, threshold).  Every
// matcher CTA knows its image, so the only difference is the row it adds its four counts to.
static int pr_counts_impl(const void *pred, int pred_dtype, const uint8_t *gt, int N, int H, int W, const int32_t *crop,
                          const double *thresholds, int T, double max_dist, int apply_thinning, int64_t *counts,
                          int perImage, void *workspace, size_t ws_bytes, mte_stream_t stream) {
    if (!pred || !gt || !counts || !workspace) return MTE_ERR_NULL;
    if (N < 1 || H < 1 || W < 1) return MTE_ERR_SHAPE;
    if (T < 1 || T > MTE_MAX_THRESHOLDS) return MTE_ERR_ARG;
    if (!(max_dist >= 0.0)) return MTE_ERR_ARG;
    if (apply_thinning != 0 && apply_thinning != 1) return MTE_ERR_ARG;
    if (pred_dtype != MTE_U8 && !thresholds) return MTE_ERR_NULL;
    const Layout L = layout(N * T, H, W, T);
    const size_t need = apply_thinning ? mte_pr_thin_workspace_bytes(N, H, W, T, max_dist) : L.total;
    if (ws_bytes < need) return MTE_ERR_WORKSPACE;
    MatchP P;
    memset(&P, 0, sizeof(P));
    P.pred = pred; P.gt = gt;
    P.inMode = pred_dtype == MTE_U8 ? IN_LEVELS : (pred_dtype == MTE_F32 ? IN_F32 : IN_F64);
    P.N = N; P.H = H; P.W = W; P.T = T;
    clip_crop(crop, H, W, P.x0, P.y0, P.w, P.h);
    P.nProblems = N * T;
    P.counts = reinterpret_cast<unsigned long long *>(counts);
    P.countsImgStride = perImage ? T : 0;
    if (P.w == 0 || P.h == 0) return MTE_OK;  // empty window: nothing to count
    if (apply_thinning)
        return pr_counts_thinned(P, L, static_cast<char *>(workspace), max_dist, thresholds,
                                 reinterpret_cast<cudaStream_t>(stream));
    return launch(P, L, static_cast<char *>(workspace), max_dist, thresholds, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int mte_pr_counts(const void *pred, int pred_dtype, const uint8_t *gt, int N, int H, int W,
                             const int32_t *crop, const double *thresholds, int T, double max_dist,
                             int apply_thinning, int64_t *counts, void *workspace, size_t ws_bytes,
                             mte_stream_t stream) {
    return pr_counts_impl(pred, pred_dtype, gt, N, H, W, crop, thresholds, T, max_dist, apply_thinning, counts, 0,
                          workspace, ws_bytes, stream);
}

extern "C" int mte_pr_counts_per_image(const void *pred, int pred_dtype, const uint8_t *gt, int N, int H, int W,
                                       const int32_t *crop, const double *thresholds, int T, double max_dist,
                                       int apply_thinning, int64_t *counts, void *workspace, size_t ws_bytes,
                                       mte_stream_t stream) {
    return pr_counts_impl(pred, pred_dtype, gt, N, H, W, crop, thresholds, T, max_dist, apply_thinning, counts, 1,
                          workspace, ws_bytes, stream);
}
