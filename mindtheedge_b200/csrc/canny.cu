// Depth -> edge extraction for evaluation (sm_100a), bit-exact with the reference path
//   edge_from_depth            edge.py:73-93  (twin packnet_code/packnet_sfm/utils/edge.py:64-89)
//   cv2.Canny(u8, low, high)   third-party call at edge.py:88 (aperture 3, L1 gradient), SURVEY.md A.2
//
// Three kernels, all integer work after the quantisation:
//  1. canny_nms_kernel   depth -> u8 (clamp, *255/max, trunc) -> Sobel3 (BORDER_REPLICATE) -> L1 magnitude ->
//                        fixed-point NMS, staged through a shared-memory halo tile; emits per pixel the FIRST
//                        threshold index at which it is a candidate (cl) and at which it is strong (sl).
//  2. canny_uf_hyst_kernel  multi-threshold hysteresis for ALL nested pairs at once: incremental union-find
//                        over the candidate pixels in threshold order; result is one u8 "birth level" plane
//                        E with  E(p) <= t  <=>  p is an edge of cv2.Canny at pair t  (instead of T planes).
//  3. canny_expand_kernel  optional: the T {0,255} planes the reference API returns.

#include <stdlib.h>

#include <algorithm>
#include <type_traits>

#include "common.cuh"

namespace mte {
namespace canny {

constexpr int TG22 = 13573;  // round(tan(22.5 deg) * 2^15)
constexpr int TW = 128, TH = 32, kThreads = 256;
constexpr int kNever = 255;

struct Thresholds {
    int n;
    int low[MTE_MAX_THRESHOLDS];
    int high[MTE_MAX_THRESHOLDS];
};

template <typename T>
__device__ __forceinline__ unsigned char quantise(T d, T lo, T hi, T factor) {
    // edge.py:81-87 (the comparisons leave NaN alone; the uint8 cast of NaN is 0 on x86 and here)
    if (d < lo) d = lo;
    if (d > hi) d = hi;
    const T v = d * factor;
    return (unsigned char)(int)v;
}
template <>
__device__ __forceinline__ unsigned char quantise<unsigned char>(unsigned char d, unsigned char, unsigned char,
                                                                 unsigned char) {
    return d;
}

// One CTA = one 128 x 32 tile.  Three phases through shared memory, four horizontally adjacent pixels per thread
// and step in the two stencil phases (the first version spent ~300 instructions per pixel, most of them
// recomputing the Sobel sums and walking the threshold list per pixel):
//   A  quantise the tile + halo 2 (coordinates clamped = BORDER_REPLICATE) into u8
//   B  Sobel3 + L1 magnitude for the tile + halo 1 from column sums shared by the four pixels; stored as one u16:
//      magnitude (<= 2040, 11 bits) | NMS sector << 11 (0 horizontal, 1 vertical, 2 diagonal s=+1, 3 diagonal s=-1)
//   C  NMS against the two neighbours of the sector; the surviving magnitude indexes a per-CTA table
//      magnitude -> (first candidate level, first strong level) built once per launch (canny_lut_kernel)
constexpr int QS = TW + 8;        // u8 row stride of the quantised tile (word aligned, halo 2 at columns 2..)
constexpr int MS = TW + 4;        // u16 row stride of the magnitude tile (halo 1 at column 1..)
constexpr int kMaxMag = 2040;     // |dx| + |dy| <= 2 * 4 * 255

// magnitude -> (first candidate level | first strong level << 8), once per launch
__global__ void __launch_bounds__(kThreads) canny_lut_kernel(const __grid_constant__ Thresholds thr,
                                                             unsigned short *__restrict__ lut) {
    const int v = blockIdx.x * kThreads + threadIdx.x;
    if (v > kMaxMag) return;
    int first_c = kNever, first_s = kNever;
    for (int t = thr.n - 1; t >= 0; t--) {  // nested pairs: the last hit going down the list is the first index
        if (v > thr.low[t]) first_c = t;
        if (v > thr.high[t]) first_s = t;
    }
    lut[v] = (unsigned short)(first_c | (first_s << 8));
}

template <typename T>
__global__ void __launch_bounds__(kThreads) canny_nms_kernel(const T *__restrict__ depth, int N, int H, int W, T lo,
                                                             T hi, T factor, const unsigned short *__restrict__ glut,
                                                             unsigned char *__restrict__ cl,
                                                             unsigned char *__restrict__ E) {
    __shared__ __align__(16) unsigned char q[TH + 4][QS];
    __shared__ __align__(16) unsigned short mag[TH + 2][MS];
    __shared__ unsigned short lut[kMaxMag + 1];  // first_c | first_s << 8
    const int tilesX = ceil_div(W, TW), tilesY = ceil_div(H, TH);
    const int tile = blockIdx.x % (tilesX * tilesY), img = blockIdx.x / (tilesX * tilesY);
    const int x0 = (tile % tilesX) * TW, y0 = (tile / tilesX) * TH;
    const T *src = depth + (size_t)img * H * W;

    for (int v = threadIdx.x; v <= kMaxMag; v += kThreads) lut[v] = glut[v];
    // A: q[r][c] = pixel (y0 + r - 2, x0 + c - 4), columns 2 .. TW + 5 used.  Groups of four columns: one 128-bit
    //    load and one 32-bit shared store when the group lies inside the image (fp32 planes with W % 4 == 0)
    const bool vec4 = std::is_same<T, float>::value && (W % 4) == 0 && (reinterpret_cast<uintptr_t>(src) & 15) == 0;
    for (int i = threadIdx.x; i < (TH + 4) * (QS / 4); i += kThreads) {
        const int r = i / (QS / 4), c = (i - r * (QS / 4)) * 4;
        const int y = min(max(y0 + r - 2, 0), H - 1), xg = x0 + c - 4;
        const T *row = src + (size_t)y * W;
        unsigned pk = 0;
        if (vec4 && xg >= 0 && xg + 3 < W) {
            const float4 v = __ldg(reinterpret_cast<const float4 *>(row + xg));
            pk = (unsigned)quantise<float>(v.x, (float)lo, (float)hi, (float)factor) |
                 ((unsigned)quantise<float>(v.y, (float)lo, (float)hi, (float)factor) << 8) |
                 ((unsigned)quantise<float>(v.z, (float)lo, (float)hi, (float)factor) << 16) |
                 ((unsigned)quantise<float>(v.w, (float)lo, (float)hi, (float)factor) << 24);
        } else {
#pragma unroll
            for (int k = 0; k < 4; k++)
                pk |= (unsigned)quantise<T>(row[min(max(xg + k, 0), W - 1)], lo, hi, factor) << (8 * k);
        }
        *reinterpret_cast<unsigned *>(&q[r][c]) = pk;
    }
    __syncthreads();
    // B: mag[r][c] = pixel (y0 + r - 1, x0 + c - 2); groups of 4 columns c = 4k .. 4k+3 cover columns 0 .. TW + 3
    for (int i = threadIdx.x; i < (TH + 2) * (MS / 4); i += kThreads) {
        const int r = i / (MS / 4), c = (i - r * (MS / 4)) * 4;
        // q columns c+1 .. c+6 around the four centres c+2 .. c+5 (q column = mag column + 2), rows r .. r+2
        int V[6], D[6];
        unsigned wq[3][2];  // the eight bytes c .. c+7 of the three rows as words (two loads instead of six)
#pragma unroll
        for (int rr = 0; rr < 3; rr++) {
            wq[rr][0] = *reinterpret_cast<const unsigned *>(&q[r + rr][c]);
            wq[rr][1] = *reinterpret_cast<const unsigned *>(&q[r + rr][c + 4]);
        }
        auto qb = [&](int rr, int k) -> int { return (int)((wq[rr][(k + 1) >> 2] >> (8 * ((k + 1) & 3))) & 0xFFu); };
#pragma unroll
        for (int k = 0; k < 6; k++) {
            const int a = qb(0, k), m = qb(1, k), b = qb(2, k);
            V[k] = a + 2 * m + b;   // vertical [1 2 1] column sum
            D[k] = b - a;           // vertical difference
        }
        unsigned short out[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const int dx = V[k + 2] - V[k];
            const int dy = D[k] + 2 * D[k + 1] + D[k + 2];
            const int y = y0 + r - 1, x = x0 + c + k - 2;
            int v = 0;
            if (y >= 0 && y < H && x >= 0 && x < W) {  // outside the image the magnitude is 0
                const int ax = abs(dx), ay = abs(dy) << 15;
                const int tg22x = ax * TG22, tg67x = tg22x + (ax << 16);
                const int sector = ay < tg22x ? 0 : (ay > tg67x ? 1 : (((dx ^ dy) < 0) ? 3 : 2));
                v = (ax + abs(dy)) | (sector << 11);
            }
            out[k] = (unsigned short)v;
        }
        *reinterpret_cast<uint2 *>(&mag[r][c]) = make_uint2(out[0] | ((unsigned)out[1] << 16), out[2] | ((unsigned)out[3] << 16));
    }
    __syncthreads();
    // C: four output pixels per thread and step; tile pixel (r, c) is mag[r + 1][c + 2]
    const bool vec = (W % 4) == 0 && ((reinterpret_cast<uintptr_t>(cl) | reinterpret_cast<uintptr_t>(E)) & 3) == 0;
    for (int i = threadIdx.x; i < TH * (TW / 4); i += kThreads) {
        const int r = i / (TW / 4), c = (i - r * (TW / 4)) * 4;
        const int y = y0 + r, x = x0 + c;
        if (y >= H || x >= W) continue;
        unsigned oc = 0, os = 0;
        // the 3 x 8 neighbourhood (u16 columns c .. c+7 of rows r .. r+2) as six 64-bit loads; the two neighbours of the
        // sector are then SELECTED from registers (no data-dependent addresses, no branches)
        unsigned nb[3][4];
#pragma unroll
        for (int rr = 0; rr < 3; rr++) {
            const uint2 lo2 = *reinterpret_cast<const uint2 *>(&mag[r + rr][c]);
            const uint2 hi2 = *reinterpret_cast<const uint2 *>(&mag[r + rr][c + 4]);
            nb[rr][0] = lo2.x; nb[rr][1] = lo2.y; nb[rr][2] = hi2.x; nb[rr][3] = hi2.y;
        }
        auto at = [&](int rr, int j) -> int { return (int)((nb[rr][j >> 1] >> (16 * (j & 1))) & 0xFFFFu); };
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const int j = k + 2;  // centre column inside the 8
            const int pv = at(1, j), m = pv & 0x7FF, sector = pv >> 11;
            // sector 0: left / right, 1: up / down, 2: up-left / down-right, 3: up-right / down-left
            const int a1 = sector == 0 ? at(1, j - 1) : (sector == 1 ? at(0, j) : (sector == 2 ? at(0, j - 1) : at(0, j + 1)));
            const int a2 = sector == 0 ? at(1, j + 1) : (sector == 1 ? at(2, j) : (sector == 2 ? at(2, j + 1) : at(2, j - 1)));
            const int n1 = a1 & 0x7FF, n2 = a2 & 0x7FF;
            const bool keep = (m > n1) & ((m > n2) | ((sector < 2) & (m == n2)));
            const unsigned e = lut[keep ? m : 0];
            oc |= (e & 0xFFu) << (8 * k);
            os |= (e >> 8) << (8 * k);
        }
        const size_t o = (size_t)img * H * W + (size_t)y * W + x;
        if (vec) {
            *reinterpret_cast<unsigned *>(cl + o) = oc;
            *reinterpret_cast<unsigned *>(E + o) = os;
        } else {
#pragma unroll
            for (int k = 0; k < 4; k++)
                if (x + k < W) { cl[o + k] = (unsigned char)(oc >> (8 * k)); E[o + k] = (unsigned char)(os >> (8 * k)); }
        }
    }
}

// ---------------------------------------------------------------------------
// Multi-threshold hysteresis as incremental connected components (Kruskal order).
//
// cl(p) = first threshold index at which p is a candidate, E(p) initialised to the first index at which p
// is strong (255 = never).  Pair t's edge set is: candidates (cl <= t) 8-connected, through candidates, to a
// strong pixel (sl <= t).  Candidate sets are nested in t, so components only ever merge as t grows: one
// lock-free union-find per image, levels t = 0..T-1 processed in order:
//   (i)   pixels with cl == t join their 8-neighbours with cl <= t         (atomicCAS link, smaller root wins)
//   (ii)  every pixel already an edge (E <= t) flags its root
//   (iii) every unassigned candidate whose root is flagged gets E = t
// => E(p) <= t  <=>  p is an edge of cv2.Canny at pair t, for all pairs at once, with no data-dependent
// iteration count (a relaxation needs one sweep per tile a weak chain crosses: 50-120 grid-wide
// iterations on long object boundaries, profiles/r01_notes.md).  One CTA per image walks the compacted
// candidate list (~2 % of the pixels); parents live in an L2-resident int32 plane.
// ---------------------------------------------------------------------------
constexpr int kUfThreads = 1024;

struct UfP {
    const unsigned char *cl;
    unsigned char *E;
    int N, H, W, T;
    int *parent;          // [N,H,W]
    int *list;            // [N,H,W] candidate pixels, sorted by cl
    int *merged;          // [N,H,W] roots linked away during the current level
    unsigned char *flag;  // [N,H,W] "component holds an edge pixel", valid at roots
    int *todo;            // [N] written by the shared-memory kernel: 1 = image left to the L2 kernel (nullptr = all)
    int cap;              // shared-memory kernel: candidate capacity
    unsigned long long *prof;  // optional per-section cycle counters (MTE_HYST_PROF)
    unsigned oRank, oParent, oFlag, oEc, oPerm, oWork;  // shared-memory kernel: byte offsets of its arrays behind the bitmap
};

// find with path halving (every visited node is re-pointed to its grandparent; lock-free safe: a node only
// ever moves to one of its ancestors, roots change only through the CAS in uf_unite)
__device__ __forceinline__ int uf_find(int *parent, int x) {
    int p = __ldcg(parent + x);
    while (p != x) {
        const int gp = __ldcg(parent + p);
        if (gp == p) return p;
        __stcg(parent + x, gp);
        x = gp;
        p = __ldcg(parent + x);
    }
    return x;
}

// 16 level bytes of one thread-step (128-bit load when the plane allows it)
__device__ __forceinline__ void load16(unsigned char (&v)[16], const unsigned char *cl, int i0, int HW, bool vec) {
    if (vec) {
        *reinterpret_cast<uint4 *>(v) = __ldg(reinterpret_cast<const uint4 *>(cl + i0));
    } else {
#pragma unroll
        for (int k = 0; k < 16; k++) v[k] = (i0 + k < HW) ? cl[i0 + k] : (unsigned char)kNever;
    }
}

__global__ void __launch_bounds__(kUfThreads) canny_uf_hyst_kernel(const UfP P) {
    __shared__ int sHist[256];   // candidates per level, then bucket write cursors
    __shared__ int sEnd[256];    // sEnd[t] = number of candidates with cl <= t (list is sorted by cl)
    __shared__ int sMerged;
    const int img = blockIdx.x;
    if (P.todo && !P.todo[img]) return;  // solved by the shared-memory kernel
    const int HW = P.H * P.W;
    const size_t base = (size_t)img * HW;
    const unsigned char *cl = P.cl + base;
    unsigned char *E = P.E + base;
    int *parent = P.parent + base;
    int *list = P.list + base;
    int *merged = P.merged + base;
    unsigned char *flag = P.flag + base;
    const int T = P.T;
    for (int i = threadIdx.x; i < 256; i += kUfThreads) sHist[i] = 0;
    __syncthreads();
    // counting sort of the candidate pixels by their first-candidate level (two coalesced passes over cl)
    const bool vec = (HW % 16) == 0 && (reinterpret_cast<uintptr_t>(cl) & 15) == 0;
    for (int i0 = threadIdx.x * 16; i0 < HW; i0 += kUfThreads * 16) {
        unsigned char v[16];
        load16(v, cl, i0, HW, vec);
#pragma unroll
        for (int k = 0; k < 16; k++) {
            // warp-aggregated: one shared atomic per distinct level in the warp (most candidates share 1-2 levels)
            const unsigned grp = __match_any_sync(__activemask(), (int)v[k]);
            if (v[k] != kNever && (int)(__ffs(grp) - 1) == (int)(threadIdx.x & 31)) atomicAdd(&sHist[v[k]], __popc(grp));
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int run = 0;
        for (int t = 0; t < 255; t++) {
            const int c = sHist[t];
            sHist[t] = run;  // becomes the write cursor of bucket t
            run += c;
            sEnd[t] = run;
        }
    }
    __syncthreads();
    for (int i0 = threadIdx.x * 16; i0 < HW; i0 += kUfThreads * 16) {
        unsigned char v[16];
        load16(v, cl, i0, HW, vec);
#pragma unroll
        for (int k = 0; k < 16; k++) {
            const unsigned act = __activemask();
            const unsigned grp = __match_any_sync(act, (int)v[k]);
            const int leader = __ffs(grp) - 1, lane = threadIdx.x & 31;
            int slot = 0;
            if (v[k] != kNever && lane == leader) slot = atomicAdd(&sHist[v[k]], __popc(grp));
            slot = __shfl_sync(act, slot, leader);
            if (v[k] != kNever) {
                list[slot + __popc(grp & ((1u << lane) - 1))] = i0 + k;
                parent[i0 + k] = i0 + k;
                flag[i0 + k] = 0;
            }
        }
    }
    __syncthreads();
    const int W = P.W, H = P.H;
    for (int t = 0; t < T; t++) {
        const int begin = t ? sEnd[t - 1] : 0, end = sEnd[t];
        if (threadIdx.x == 0) sMerged = 0;
        __syncthreads();
        // (i) the pixels that become candidates at this level join their neighbours that already are
        for (int k = begin + threadIdx.x; k < end; k += kUfThreads) {
            const int p = list[k];
            const int y = p / W, x = p - y * W;
#pragma unroll
            for (int d = 0; d < 8; d++) {
                const int dy = (d < 3) ? -1 : ((d < 5) ? 0 : 1);
                const int dx = (d == 0 || d == 3 || d == 5) ? -1 : ((d == 1 || d == 6) ? 0 : 1);
                const int yy = y + dy, xx = x + dx;
                if (yy < 0 || yy >= H || xx < 0 || xx >= W) continue;
                const int q = yy * W + xx;
                if (cl[q] > t) continue;
                // unite, remembering every root that loses its root status (its flag must follow it)
                int a = p, b = q;
                for (;;) {
                    a = uf_find(parent, a);
                    b = uf_find(parent, b);
                    if (a == b) break;
                    if (a < b) { const int tmp = a; a = b; b = tmp; }
                    if (atomicCAS(parent + a, a, b) == a) {
                        merged[atomicAdd(&sMerged, 1)] = a;
                        break;
                    }
                }
            }
        }
        __syncthreads();
        // (ii) flags: components that already held an edge keep it across merges; new strong pixels seed theirs
        const int nMerged = sMerged;
        for (int k = threadIdx.x; k < nMerged; k += kUfThreads) {
            const int a = merged[k];
            if (__ldcg(flag + a)) flag[uf_find(parent, a)] = 1;
        }
        for (int k = threadIdx.x; k < end; k += kUfThreads) {
            const int p = list[k];
            if (__ldcg(E + p) == t) flag[uf_find(parent, p)] = 1;  // unassigned pixels still carry their sl
        }
        __syncthreads();
        // (iii) every unassigned candidate of a flagged component becomes an edge at this level
        for (int k = threadIdx.x; k < end; k += kUfThreads) {
            const int p = list[k];
            if (__ldcg(E + p) > t && __ldcg(flag + uf_find(parent, p))) E[p] = (unsigned char)t;
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------
// The same incremental union-find with the whole per-image state in SHARED memory: candidates get compact 16-bit
// ids (raster rank: window bitmap + per-64-pixel rank, as in the matcher), parents are 16-bit shared-memory words,
// component flags one bit each.  A find is then a few 30-cycle shared-memory hops instead of dependent L2 round
// trips (the L2 kernel above spends its time there: ~2 x candidates finds per level).  Per-candidate edge levels
// live in a compact global array in list order (coalesced) and are scattered to the plane at the end.  Images with
// more candidates than fit are left to the L2 kernel through P.todo.
// Bitmap rows are padded to whole 32-bit words (row stride WP = 32 * ceil(W / 32) bits), so any W % 16 == 0 works.
// BIG = true (planes whose bitmaps do not fit next to a useful number of candidates, e.g. DDAD 1216 x 1936): the two
// bitmaps and the rank table live in the image's global scratch (L2-resident, a few hundred KB) instead; they are only
// touched by independent, pipelined accesses (flood frontier, neighbour lookups), while the union-find chains --
// the latency-critical part -- stay in shared memory.
// ---------------------------------------------------------------------------
constexpr int kWorkCap = 4096;  // changed-word worklist entries of the flood (beyond that: one full sweep)

__device__ __forceinline__ int ufs_find(volatile unsigned short *parent, int x) {
    int p = parent[x];
    while (p != x) {
        const int gp = parent[p];
        if (gp == p) return p;
        parent[x] = (unsigned short)gp;
        x = gp;
        p = parent[x];
    }
    return x;
}

template <bool BIG>
__global__ void __launch_bounds__(kUfThreads) canny_uf_hyst_smem_kernel(const UfP P) {
    extern __shared__ __align__(16) unsigned char dyn[];
    __shared__ int sHist[256], sEnd[256], sScan[kUfThreads];
    __shared__ int sCnt[3], sFullA[3];   // flood worklists: three rotating counters (read / append / clear), one barrier per round
    __shared__ unsigned char sRep[256];
    using WL = typename std::conditional<BIG, unsigned, unsigned short>::type;  // worklist entry: a bitmap word index
    const int img = blockIdx.x;
    const int H = P.H, W = P.W, HW = H * W, T = P.T;
    const int WPR = (W + 31) >> 5, WP = WPR * 32;  // words / bits per bitmap row
    const int nW = H * WPR, nW2 = (nW + 1) >> 1;
    const size_t base = (size_t)img * HW;
    const unsigned char *cl = P.cl + base;
    unsigned char *E = P.E + base;
    int *list = P.list + base;
    int *merged = P.merged + base;
    // candidate ids are positions in the level-sorted list: "is a candidate at level t" is id < sEnd[t], the
    // per-candidate state (parent, edge level, flag) is indexed by id in shared memory and the per-level passes touch
    // nothing else; the neighbour lookup of step (i) goes raster rank -> id through a table that is resident too (8
    // scattered reads per candidate: from L2 they were a third of the unite pass)
    unsigned short *perm = reinterpret_cast<unsigned short *>(dyn + P.oPerm);
    unsigned *qbits = BIG ? reinterpret_cast<unsigned *>(merged) : reinterpret_cast<unsigned *>(dyn);
    unsigned short *qrank = BIG ? reinterpret_cast<unsigned short *>(qbits + 2 * nW) : reinterpret_cast<unsigned short *>(dyn + P.oRank);
    unsigned short *parent = reinterpret_cast<unsigned short *>(dyn + P.oParent);
    unsigned *flagW = reinterpret_cast<unsigned *>(dyn + P.oFlag);
    unsigned char *Ec = dyn + P.oEc;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    long long tk = clock64();
    auto tick = [&](int slot) {
        if (P.prof && threadIdx.x == 0) {
            const long long now = clock64();
            atomicAdd(P.prof + slot, (unsigned long long)(now - tk));
            tk = now;
        }
    };
    for (int i = threadIdx.x; i < 256; i += kUfThreads) sHist[i] = 0;
    // sRep[m]: for a set m of neighbour positions (bit d: 0 NW, 1 N, 2 NE, 3 W, 4 E, 5 SW, 6 S, 7 SE), one representative
    // (lowest position) per group of positions that are 8-adjacent to each other.  Neighbours from EARLIER levels that
    // touch each other are already in one component, so a new pixel only has to join one of each group.
    if (threadIdx.x < 256) {
        const int m = threadIdx.x;
        const int ny[8] = {-1, -1, -1, 0, 0, 1, 1, 1}, nx[8] = {-1, 0, 1, -1, 1, -1, 0, 1};
        int lab[8];
        for (int d = 0; d < 8; d++) lab[d] = d;
        for (int it = 0; it < 8; it++)
            for (int a = 0; a < 8; a++)
                for (int b = 0; b < 8; b++)
                    if (((m >> a) & 1) && ((m >> b) & 1) && abs(ny[a] - ny[b]) <= 1 && abs(nx[a] - nx[b]) <= 1 && lab[b] < lab[a])
                        lab[a] = lab[b];
        int r = 0;
        for (int d = 0; d < 8; d++)
            if (((m >> d) & 1) && lab[d] == d) r |= 1 << d;
        sRep[m] = (unsigned char)r;
    }
    __syncthreads();
    const bool vec = (reinterpret_cast<uintptr_t>(cl) & 15) == 0 && (reinterpret_cast<uintptr_t>(E) & 15) == 0;  // W % 16 == 0 (host)
    // ---- pass 1: bitmaps of the candidates (cbits) and of the pixels that are strong at some level (qbits = seed),
    //      one 16-pixel chunk (half a bitmap word; chunks never straddle a row) per thread and step
    unsigned *cbits = BIG ? qbits + nW : reinterpret_cast<unsigned *>(dyn + P.oParent);   // smem: borrowed until the flood is done
    WL *wlA = reinterpret_cast<WL *>(dyn + P.oWork), *wlB = wlA + kWorkCap;
    const int HPR = WPR * 2;  // 16-pixel chunks per bitmap row
    //      (kP1U chunk pairs per thread in flight: one CTA streams the image's two level planes, i.e. the pass is a
    //      chain of round trips -- 30 of them at KITTI size with one chunk per step)
    constexpr int kP1U = 4;
    for (int hc0 = threadIdx.x; hc0 < H * HPR; hc0 += kP1U * kUfThreads) {
        unsigned char v[kP1U][16], sv[kP1U][16];
#pragma unroll
        for (int u = 0; u < kP1U; u++) {
            const int hc = hc0 + u * kUfThreads;
            const int y = hc / HPR, x0 = (hc - y * HPR) * 16;
            if (hc < H * HPR && x0 < W) { load16(v[u], cl, y * W + x0, HW, vec); load16(sv[u], E, y * W + x0, HW, vec); }
            else {
#pragma unroll
                for (int k = 0; k < 16; k++) { v[u][k] = (unsigned char)kNever; sv[u][k] = (unsigned char)kNever; }
            }
        }
#pragma unroll
        for (int u = 0; u < kP1U; u++) {
            const int hc = hc0 + u * kUfThreads;
            if (hc < H * HPR) {   // (H * HPR is even: the two lanes of a bitmap word are in range together)
                const int i0 = hc * 16;  // bit index of the chunk
                unsigned half = 0, shalf = 0;
#pragma unroll
                for (int k = 0; k < 16; k++) {
                    half |= (v[u][k] != kNever ? 1u : 0u) << k;
                    shalf |= (sv[u][k] != kNever ? 1u : 0u) << k;
                }
                const unsigned hi = __shfl_down_sync(__activemask(), half, 1), shi = __shfl_down_sync(__activemask(), shalf, 1);
                if (!(lane & 1)) { cbits[i0 >> 5] = half | (hi << 16); qbits[i0 >> 5] = (shalf | (shi << 16)) & (half | (hi << 16)); }
            }
        }
    }
    if (threadIdx.x < 3) { sCnt[threadIdx.x] = 0; sFullA[threadIdx.x] = 0; }
    __syncthreads();
    // ---- flood: only candidates connected to a strong pixel can ever become edges (the edge sets of the pairs are
    //      nested), and on noisy depth they are a fraction of the candidates (~6 k of ~30 k per KITTI image), so the
    //      union-find below runs on that reachable set R only.  R grows from the strong pixels by bit-parallel
    //      dilation restricted to the candidates: inside a word a Kogge-Stone occluded fill runs along the whole
    //      horizontal run at once; a worklist of changed words keeps an iteration proportional to the frontier.
    auto hfill = [](unsigned seed, unsigned c) -> unsigned {
        unsigned f = seed & c, m = c;
        f |= m & (f << 1); m &= m << 1; f |= m & (f << 2); m &= m << 2; f |= m & (f << 4); m &= m << 4;
        f |= m & (f << 8); m &= m << 8; f |= m & (f << 16);
        m = c;
        f |= m & (f >> 1); m &= m >> 1; f |= m & (f >> 2); m &= m >> 2; f |= m & (f >> 4); m &= m >> 4;
        f |= m & (f >> 8); m &= m >> 8; f |= m & (f >> 16);
        return f;
    };
    for (int i = threadIdx.x; i < nW; i += kUfThreads)
        if (qbits[i]) { const int s = atomicAdd(&sCnt[0], 1); if (s < kWorkCap) wlA[s] = (WL)i; else sFullA[0] = 1; }
    __syncthreads();
    for (int iter = 0;; iter++) {
        // Round `iter` reads list / counter cur, appends to nxt and clears clr, the counter that round iter - 1 read (every
        // thread passed the barrier that ended that round) and that round iter + 1 appends to (after this round's
        // barrier): ONE barrier per round instead of four -- a flood over long contours is a few dozen rounds of a
        // thousand threads.  The two lists alternate: the one appended to now was read in the previous round.
        const int cur = iter % 3, nxt = (iter + 1) % 3, clr = (iter + 2) % 3;
        const int nA = min(sCnt[cur], kWorkCap);
        const bool full = sFullA[cur] != 0;
        if (nA == 0 && !full) break;
        if (threadIdx.x == 0) { sCnt[clr] = 0; sFullA[clr] = 0; }
        const WL *src = (iter & 1) ? wlB : wlA;
        WL *dst = (iter & 1) ? wlA : wlB;
        const int nSrc = full ? nW : nA;
        for (int k = threadIdx.x; k < nSrc; k += kUfThreads) {
            const int wi = full ? k : (int)src[k];
            const unsigned v = ((volatile unsigned *)qbits)[wi];
            if (!v) continue;
            const int r = wi / WPR, c = wi - r * WPR;
            const unsigned h3 = v | (v << 1) | (v >> 1);
#pragma unroll
            for (int dr = -1; dr <= 1; dr++) {
                const int rr = r + dr;
                if (rr < 0 || rr >= H) continue;
#pragma unroll
                for (int dc = -1; dc <= 1; dc++) {
                    const int cc = c + dc;
                    if (cc < 0 || cc >= WPR) continue;
                    const unsigned contrib = dc == 0 ? h3 : (dc < 0 ? ((v & 1u) << 31) : (v >> 31));
                    if (!contrib) continue;
                    const int ti = rr * WPR + cc;
                    const unsigned cm = cbits[ti], cur = ((volatile unsigned *)qbits)[ti];
                    if (!(contrib & cm & ~cur)) continue;
                    const unsigned add = hfill(contrib | cur, cm) & ~cur;
                    const unsigned old = atomicOr(&qbits[ti], add);
                    if (add & ~old) {
                        const int s2 = atomicAdd(&sCnt[nxt], 1);
                        if (s2 < kWorkCap) dst[s2] = (WL)ti; else sFullA[nxt] = 1;
                    }
                }
            }
        }
        __syncthreads();
    }
    tick(0);
    if (T == 1) {
        // a single pair: the flood result IS the edge set (every candidate connected to a strong pixel becomes an
        // edge at level 0) -- no components to track over levels
        for (int wi = threadIdx.x; wi < nW; wi += kUfThreads) {
            unsigned bits = qbits[wi];
            if (!bits) continue;
            const int y = wi / WPR, pbase = y * W + (wi - y * WPR) * 32;
            while (bits) {
                const int b = __ffs(bits) - 1;
                bits &= bits - 1;
                E[pbase + b] = 0;
            }
        }
        if (threadIdx.x == 0) P.todo[img] = 0;
        return;
    }
    // ---- histogram of first-candidate levels over R (sparse: walk the set bits)
    for (int wi = threadIdx.x; wi < nW; wi += kUfThreads) {
        unsigned bits = qbits[wi];
        if (!bits) continue;
        const int y = wi / WPR, pbase = y * W + (wi - y * WPR) * 32;  // pixel of bit 0
        while (bits) {   // four level bytes in flight (one L2 round trip per bit otherwise)
            int lvl[4], n = 0;
#pragma unroll
            for (int j = 0; j < 4; j++)
                if (bits) { lvl[j] = cl[pbase + __ffs(bits) - 1]; bits &= bits - 1; n = j + 1; }
#pragma unroll
            for (int j = 0; j < 4; j++)
                if (j < n) atomicAdd(&sHist[lvl[j]], 1);   // (warp-aggregating the adds with __match_any_sync was measured slower)
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int run = 0;
        for (int t = 0; t < 255; t++) {
            const int c = sHist[t];
            sHist[t] = run;
            run += c;
            sEnd[t] = run;
        }
    }
    __syncthreads();
    const int nCand = sEnd[254];
    if (P.prof && threadIdx.x == 0) atomicAdd(P.prof + 8, (unsigned long long)nCand);
    // parked neighbour ids of the level passes: 16 B per candidate in the image's `merged` scratch (4 B per pixel),
    // behind the global bitmaps when there are any
    const size_t nidOff = BIG ? (((size_t)2 * nW * 4 + (size_t)nW2 * 2 + 15) & ~(size_t)15) : 0;
    uint4 *nidBuf = reinterpret_cast<uint4 *>(reinterpret_cast<unsigned char *>(merged) + nidOff);
    if (nCand > P.cap || nidOff + (size_t)nCand * 16 > (size_t)HW * 4) {  // leave the image to the L2 kernel
        if (threadIdx.x == 0) P.todo[img] = 1;
        return;
    }
    if (threadIdx.x == 0) P.todo[img] = 0;
    // ---- rank: exclusive prefix popcount over pairs of bitmap words
    {
        const int per = (nW2 + kUfThreads - 1) / kUfThreads;
        const int w0 = threadIdx.x * per, w1 = min(w0 + per, nW2);
        auto pc2 = [&](int k2) { return __popc(qbits[2 * k2]) + (2 * k2 + 1 < nW ? __popc(qbits[2 * k2 + 1]) : 0); };
        int sum = 0;
        for (int k2 = w0; k2 < w1; k2++) sum += pc2(k2);
        sScan[threadIdx.x] = sum;
        __syncthreads();
        if (warp == 0) {
            int loc[kUfThreads / 32], run = 0;
#pragma unroll
            for (int q = 0; q < kUfThreads / 32; q++) { loc[q] = run; run += sScan[lane * (kUfThreads / 32) + q]; }
            int incl = run;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(MTE_FULL_MASK, incl, o); if (lane >= o) incl += v; }
            const int excl = incl - run;
#pragma unroll
            for (int q = 0; q < kUfThreads / 32; q++) sScan[lane * (kUfThreads / 32) + q] = excl + loc[q];
        }
        __syncthreads();
        int run = sScan[threadIdx.x];
        for (int k2 = w0; k2 < w1; k2++) { qrank[k2] = (unsigned short)run; run += pc2(k2); }
    }
    // (the candidate bitmap is dead from here on: its storage becomes parent / edge level / flags)
    for (int i = threadIdx.x; i < nCand; i += kUfThreads) parent[i] = (unsigned short)i;
    for (int i = threadIdx.x; i < (nCand + 31) / 32; i += kUfThreads) flagW[i] = 0u;
    __syncthreads();
    auto qid = [&](int q) -> int {
        const unsigned bits = qbits[q >> 5];
        int r = (int)qrank[q >> 6] + __popc(bits & ((1u << (q & 31)) - 1u));
        if (q & 32) r += __popc(qbits[(q >> 5) - 1]);
        return r;
    };
    // ---- pass 2 (sparse): the pixels of R sorted by level, with their ids and strong levels
    for (int wi = threadIdx.x; wi < nW; wi += kUfThreads) {
        unsigned bits = qbits[wi];
        if (!bits) continue;
        int r = (int)qrank[wi >> 1] + ((wi & 1) ? __popc(qbits[wi - 1]) : 0);
        const int y = wi / WPR, pbase = y * W + (wi - y * WPR) * 32;
        while (bits) {   // four pixels' two level bytes in flight
            int px[4], lvl[4], n = 0;
            unsigned char el[4];
#pragma unroll
            for (int j = 0; j < 4; j++)
                if (bits) {
                    px[j] = pbase + __ffs(bits) - 1;
                    bits &= bits - 1;
                    lvl[j] = cl[px[j]];
                    el[j] = E[px[j]];
                    n = j + 1;
                }
#pragma unroll
            for (int j = 0; j < 4; j++)
                if (j < n) {
                    const int at = atomicAdd(&sHist[lvl[j]], 1);
                    list[at] = px[j];
                    perm[r++] = (unsigned short)at;
                    Ec[at] = el[j];
                }
        }
    }
    __syncthreads();
    tick(1);
    volatile unsigned short *vparent = parent;
    for (int t = 0; t < T; t++) {
        const int begin = t ? sEnd[t - 1] : 0, end = sEnd[t];
        // (i) the pixels that become candidates at this level join their 8-neighbours that already are.
        //  (i-a) HOOK: a new pixel points straight at its first raster-preceding neighbour of the same level (W, NW, N,
        //        NE).  New pixels are untouched singletons until this level, and the pointers run strictly backwards in
        //        raster order, so plain stores build a forest: along a thin contour almost every same-level link is
        //        made here without a find or a CAS (a level that holds most of the reachable set -- the strictest pair
        //        on step edges -- otherwise has a thousand threads fighting over the roots of the same few chains:
        //        0.75 M of 0.94 M unite cycles on the densest bench image).  The neighbour ids are parked in the
        //        image's global scratch for (i-b).
        for (int k = begin + threadIdx.x; k < end; k += kUfThreads) {
            const int p = list[k];
            const int y = p / W, x = p - y * W;
            unsigned nid[8];
#pragma unroll
            for (int d = 0; d < 8; d++) {  // all neighbour lookups first: the table reads overlap
                const int dy = (d < 3) ? -1 : ((d < 5) ? 0 : 1);
                const int dx = (d == 0 || d == 3 || d == 5) ? -1 : ((d == 1 || d == 6) ? 0 : 1);
                const int yy = y + dy, xx = x + dx;
                nid[d] = 0xFFFFu;
                if (yy < 0 || yy >= H || xx < 0 || xx >= W) continue;
                const int q = yy * WP + xx;  // bit index
                if ((qbits[q >> 5] >> (q & 31)) & 1u) nid[d] = perm[qid(q)];
            }
            // directions 0 NW, 1 N, 2 NE, 3 W precede the pixel in raster order
            const int hookOrder[4] = {3, 0, 1, 2};
            int hook = -1;
#pragma unroll
            for (int i = 3; i >= 0; i--)
                if ((int)nid[hookOrder[i]] >= begin && (int)nid[hookOrder[i]] < end) hook = hookOrder[i];
            if (hook >= 0) {
                parent[k] = (unsigned short)nid[hook];
                nid[hook] = 0xFFFFu;  // done
            }
            // same-level neighbours that FOLLOW the pixel unite from their own end
#pragma unroll
            for (int d = 4; d < 8; d++)
                if ((int)nid[d] >= begin) nid[d] = 0xFFFFu;
            // of the earlier-level neighbours that touch each other, one is enough
            unsigned mOld = 0;
#pragma unroll
            for (int d = 0; d < 8; d++) mOld |= ((int)nid[d] < begin ? 1u : 0u) << d;
            const unsigned drop = mOld & ~(unsigned)sRep[mOld];
#pragma unroll
            for (int d = 0; d < 8; d++)
                if ((drop >> d) & 1u) nid[d] = 0xFFFFu;
            nidBuf[k] = make_uint4(nid[0] | (nid[1] << 16), nid[2] | (nid[3] << 16), nid[4] | (nid[5] << 16), nid[6] | (nid[7] << 16));
        }
        __syncthreads();
        //  a hook chain is as long as its contour; a few rounds of pointer jumping over a big level (plain loads and
        //  stores: a node only ever moves to one of its ancestors) flatten it before the finds start
        if (end - begin > kUfThreads) {
            for (int round = 0; round < 6; round++) {
                for (int k = begin + threadIdx.x; k < end; k += kUfThreads) vparent[k] = vparent[vparent[k]];
                __syncthreads();
            }
        }
        //  (i-b) the remaining links (earlier levels, junctions) by find + CAS
        for (int k = begin + threadIdx.x; k < end; k += kUfThreads) {
            const uint4 nb = __ldcg(nidBuf + k);
            const unsigned nw[4] = {nb.x, nb.y, nb.z, nb.w};
#pragma unroll
            for (int d = 0; d < 8; d++) {
                const int n = (int)((nw[d >> 1] >> (16 * (d & 1))) & 0xFFFFu);
                if (n >= end) continue;  // not a candidate, a candidate of a later level, or already dealt with
                int a = k, b = n;
                for (;;) {
                    a = ufs_find(vparent, a);
                    b = ufs_find(vparent, b);
                    if (a == b) break;
                    // link by a hashed priority, not by index: neighbouring pixels have consecutive ids, and when a
                    // whole level is united at once "larger under smaller" builds chains as long as the contours
                    if ((unsigned)a * 0x9E3779B1u < (unsigned)b * 0x9E3779B1u) { const int tmp = a; a = b; b = tmp; }
                    if (atomicCAS(parent + a, (unsigned short)a, (unsigned short)b) == (unsigned short)a) break;
                }
            }
        }
        __syncthreads();
        if (P.prof && threadIdx.x == 0 && t < 12)  // per-level unite cycles | level size << 40 (scripts/hyst_levels.py, one image)
            atomicAdd(P.prof + 16 + t, (unsigned long long)(clock64() - tk) + ((unsigned long long)(end - begin) << 40));
        tick(2);
        // (ii) flags follow the roots that were linked away (a node that ever carried a flag hands it to its current
        //      root: no list of merged roots, whose single shared counter serialised the unions); pixels that turn
        //      strong at this level seed theirs
        for (int k = threadIdx.x; k < end; k += kUfThreads) {
            if (Ec[k] == t || ((((volatile unsigned *)flagW)[k >> 5] >> (k & 31)) & 1u)) {
                const int r = ufs_find(vparent, k);
                if (r != k || Ec[k] == t) atomicOr(&flagW[r >> 5], 1u << (r & 31));
            }
        }
        __syncthreads();
        tick(3);
        // (iii) every unassigned candidate of a flagged component becomes an edge at this level
        for (int k = threadIdx.x; k < end; k += kUfThreads) {
            if (Ec[k] > t) {
                const int r = ufs_find(vparent, k);
                if ((((volatile unsigned *)flagW)[r >> 5] >> (r & 31)) & 1u) Ec[k] = (unsigned char)t;
            }
        }
        __syncthreads();
        tick(4);
    }
    for (int k = threadIdx.x; k < nCand; k += kUfThreads) E[list[k]] = Ec[k];
    __syncthreads();
    tick(5);
}

__global__ void canny_expand_kernel(const unsigned char *__restrict__ E, unsigned char *__restrict__ edges, size_t n,
                                    int T) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const int e = E[i];
        for (int t = 0; t < T; t++) edges[(size_t)t * n + i] = (e <= t) ? 255 : 0;
    }
}

struct Layout {
    size_t offCl, offE, offActive, offLut, total;
    int nTiles, tilesX, tilesY;
};

static Layout layout(int N, int H, int W) {
    Layout L;
    L.tilesX = ceil_div(W, TW);
    L.tilesY = ceil_div(H, TH);
    L.nTiles = L.tilesX * L.tilesY * N;
    size_t off = MTE_WS_HEADER_BYTES;
    const size_t plane = align_up((size_t)N * H * W, 256);
    L.offCl = off; off += plane;
    L.offE = off; off += plane;
    L.offActive = off; off += hysteresis_scratch_bytes(N, H, W);
    L.offLut = off; off += align_up((kMaxMag + 1) * sizeof(unsigned short), 256);
    L.total = off;
    return L;
}

// Shared with the DEE post-process (dee.cu).  scratch needs hysteresis_scratch_bytes().
int run_level_hysteresis(const unsigned char *cl, unsigned char *E, int N, int H, int W, int T, void *scratch,
                         cudaStream_t st) {
    UfP P;
    const size_t px = (size_t)N * H * W;
    char *w = static_cast<char *>(scratch);
    P.cl = cl; P.E = E; P.N = N; P.H = H; P.W = W; P.T = T;
    P.parent = reinterpret_cast<int *>(w);
    P.list = reinterpret_cast<int *>(w + align_up(px * 4, 256));
    P.merged = reinterpret_cast<int *>(w + 2 * align_up(px * 4, 256));
    P.flag = reinterpret_cast<unsigned char *>(w + 3 * align_up(px * 4, 256));
    P.todo = nullptr;
    P.cap = 0;
    P.prof = debug_knob("MTE_HYST_PROF") ? reinterpret_cast<unsigned long long *>(w + hysteresis_scratch_bytes(N, H, W) - 256) : nullptr;
    // shared-memory kernel first: bitmaps next to the per-candidate state when they leave room for a useful number of
    // candidates, otherwise (BIG) bitmaps in the image's global scratch and only the per-candidate state resident
    const int budget =
        std::min(smem_budget(canny_uf_hyst_smem_kernel<false>), smem_budget(canny_uf_hyst_smem_kernel<true>));
    const long long nW = (long long)H * ((W + 31) / 32), nW2 = (nW + 1) / 2;  // bitmap rows padded to whole words
    // [reachable-set bitmap][rank][region X][flood worklists]; region X is the candidate bitmap during the flood,
    // then parent (2 B) + edge level (1 B) + flag (1 bit) + rank -> id (2 B) per pixel of the reachable set.  BIG:
    // region X only.
    const long long bitmapB = align_up((size_t)nW * 4, 16), rankB = align_up((size_t)nW2 * 2, 16);
    if ((W % 16) == 0 && budget > 0 && nW * 32 < (1LL << 31) && !debug_knob("MTE_HYST_L2")) {
        long long workB = 2 * kWorkCap * sizeof(unsigned short);
        long long regionX = (long long)budget - (bitmapB + rankB + workB + 64);
        long long cap = regionX * 8 / 41 - 64;
        bool big = !(regionX >= bitmapB && cap >= 8192 && nW < 65536) || debug_knob("MTE_HYST_BIG");
        unsigned oX = (unsigned)(bitmapB + rankB);
        if (big) {
            workB = 2 * kWorkCap * sizeof(unsigned);
            regionX = (long long)budget - (workB + 64);
            cap = regionX * 8 / 41 - 64;
            oX = 0;
        }
        if (cap > 65535) cap = 65535;
        cap &= ~31LL;
        P.cap = (int)cap;
        P.oRank = (unsigned)bitmapB;
        P.oParent = oX;
        P.oFlag = P.oParent + (unsigned)align_up((size_t)cap * 2, 16);
        P.oEc = P.oFlag + (unsigned)align_up((size_t)cap / 8 + 4, 16);
        P.oPerm = P.oEc + (unsigned)align_up((size_t)cap, 16);
        const unsigned endX = P.oParent + (unsigned)(regionX & ~15LL);
        P.oWork = endX;
        const size_t smem = (size_t)endX + workB;
        P.todo = reinterpret_cast<int *>(w + 3 * align_up(px * 4, 256) + align_up(px, 256));
        if (big) canny_uf_hyst_smem_kernel<true><<<N, kUfThreads, smem, st>>>(P);
        else canny_uf_hyst_smem_kernel<false><<<N, kUfThreads, smem, st>>>(P);
        MTE_RETURN_IF_CUDA_ERROR();
    }
    canny_uf_hyst_kernel<<<N, kUfThreads, 0, st>>>(P);
    MTE_RETURN_IF_CUDA_ERROR();
    return MTE_OK;
}
size_t hysteresis_scratch_bytes(int N, int H, int W) {
    const size_t px = (size_t)N * H * W;
    return 3 * align_up(px * 4, 256) + align_up(px, 256) + align_up((size_t)N * sizeof(int), 256) + 256;
}

static int run_pairs(const void *depth, int dtype, int N, int H, int W, double min_depth, double max_depth,
                     const Thresholds &thr, unsigned char *edges, unsigned char *levels, char *ws, const Layout &L,
                     cudaStream_t st) {
    unsigned char *cl = reinterpret_cast<unsigned char *>(ws + L.offCl);
    unsigned char *E = levels ? levels : reinterpret_cast<unsigned char *>(ws + L.offE);
    const int grid1 = L.nTiles;
    const double factor = 255.0 / max_depth;

    unsigned short *lut = reinterpret_cast<unsigned short *>(ws + L.offLut);
    canny_lut_kernel<<<ceil_div(kMaxMag + 1, kThreads), kThreads, 0, st>>>(thr, lut);
    if (dtype == MTE_F32)
        canny_nms_kernel<float><<<grid1, kThreads, 0, st>>>(static_cast<const float *>(depth), N, H, W, (float)min_depth,
                                                           (float)max_depth, (float)factor, lut, cl, E);
    else if (dtype == MTE_F64)
        canny_nms_kernel<double><<<grid1, kThreads, 0, st>>>(static_cast<const double *>(depth), N, H, W, min_depth,
                                                            max_depth, factor, lut, cl, E);
    else
        canny_nms_kernel<unsigned char><<<grid1, kThreads, 0, st>>>(static_cast<const unsigned char *>(depth), N, H, W,
                                                                   0, 0, 0, lut, cl, E);
    MTE_RETURN_IF_CUDA_ERROR();

    int rc = run_level_hysteresis(cl, E, N, H, W, thr.n, ws + L.offActive, st);
    if (rc) return rc;
    int sms = num_sms();
    if (edges) {
        const size_t n = (size_t)N * H * W;
        const int g = (int)((n + 255) / 256 < (size_t)sms * 16 ? (n + 255) / 256 : (size_t)sms * 16);
        canny_expand_kernel<<<g, 256, 0, st>>>(E, edges, n, thr.n);
        MTE_RETURN_IF_CUDA_ERROR();
    }
    return MTE_OK;
}

}  // namespace canny
}  // namespace mte

using namespace mte;
using namespace mte::canny;

extern "C" size_t mte_canny_workspace_bytes(int N, int H, int W, int T) {
    if (N < 1 || H < 1 || W < 1 || T < 1) return 0;
    return layout(N, H, W).total;
}

extern "C" int mte_canny_from_depth(const void *depth, int dtype, int N, int H, int W, double min_depth,
                                    double max_depth, const int32_t *lows, const int32_t *highs, int T,
                                    uint8_t *edges, uint8_t *levels, void *workspace, size_t ws_bytes,
                                    mte_stream_t stream) {
    if (!depth || !lows || !highs || !workspace) return MTE_ERR_NULL;
    if (!edges && !levels) return MTE_ERR_NULL;
    if (N < 1 || H < 1 || W < 1) return MTE_ERR_SHAPE;
    if (T < 1 || T > MTE_MAX_THRESHOLDS) return MTE_ERR_ARG;
    if (dtype != MTE_F32 && dtype != MTE_F64 && dtype != MTE_U8) return MTE_ERR_ARG;
    if (dtype != MTE_U8 && !(max_depth != 0.0)) return MTE_ERR_ARG;
    const Layout L = layout(N, H, W);
    if (ws_bytes < L.total) return MTE_ERR_WORKSPACE;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    char *ws = static_cast<char *>(workspace);

    Thresholds thr;
    thr.n = T;
    bool nested = true;
    for (int t = 0; t < T; t++) {
        int lo = lows[t], hi = highs[t];
        if (lo > hi) { const int s = lo; lo = hi; hi = s; }  // cv2.Canny swaps
        thr.low[t] = lo;
        thr.high[t] = hi;
        if (t > 0 && (thr.low[t] > thr.low[t - 1] || thr.high[t] > thr.high[t - 1])) nested = false;
    }
    if (nested) return run_pairs(depth, dtype, N, H, W, min_depth, max_depth, thr, edges, levels, ws, L, st);
    // arbitrary pair lists: one independent pass per pair (a level plane only exists for nested lists)
    if (levels) return MTE_ERR_NOT_NESTED;
    const size_t n = (size_t)N * H * W;
    for (int t = 0; t < T; t++) {
        Thresholds one;
        one.n = 1; one.low[0] = thr.low[t]; one.high[0] = thr.high[t];
        int rc = run_pairs(depth, dtype, N, H, W, min_depth, max_depth, one, edges + (size_t)t * n, nullptr, ws, L, st);
        if (rc) return rc;
    }
    return MTE_OK;
}
