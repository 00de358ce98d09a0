// Bit-parallel morphological thinning (sm_100a): the one thinning routine of libmte, used by mte_binary_thin
// (thin.cu) and by the thinned threshold sweep of mte_pr_counts (pr_counts.cu).
//
// MATLAB bwmorph('thin', Inf) as restated in oracle/thin.py: two alternating sub-iterations that delete the pixels
// whose zero-padded 3x3 neighbourhood satisfies G1 & G2 & G3 (first) or G1 & G2 & G3' (second) of Lam, Lee & Suen,
// until a sub-iteration deletes nothing.
//
// The plane is a row-aligned bit plane: nw = ceil(w / 32) words per row, bit j of word k of row y is pixel
// (y, 32 k + j), bits past w are zero.  The deletion rule is evaluated for the 32 pixels of a word at once with
// bitwise logic on the eight neighbour vectors, which come from rows y-1, y, y+1 through funnel shifts across
// adjacent words; words outside the plane read as zero, so the plane border is the zero padding.
#pragma once
#include "common.cuh"

namespace mte {
namespace thin {

constexpr int kThreads = 512;

__host__ __device__ inline int words_per_row(int w) { return (w + 31) >> 5; }

// at least two of four bit vectors
__device__ __forceinline__ unsigned two_of_four(unsigned a, unsigned b, unsigned c, unsigned d) {
    return (a & b) | (c & d) | ((a | b) & (c | d));
}

// Deletion mask of one word.  Neighbours x1..x8 start east and run counter-clockwise (oracle/thin.py):
//     x4 x3 x2
//     x5  p x1
//     x6 x7 x8
// n*, c*, s*: words k-1, k, k+1 of rows y-1, y, y+1.  second = the second sub-iteration (G3' instead of G3).
__device__ __forceinline__ unsigned kill_word(unsigned nl, unsigned nc, unsigned nr, unsigned cl, unsigned cc,
                                              unsigned cr, unsigned sl, unsigned sc, unsigned sr, bool second) {
    const unsigned x1 = __funnelshift_r(cc, cr, 1), x5 = __funnelshift_l(cl, cc, 1);
    const unsigned x2 = __funnelshift_r(nc, nr, 1), x3 = nc, x4 = __funnelshift_l(nl, nc, 1);
    const unsigned x8 = __funnelshift_r(sc, sr, 1), x7 = sc, x6 = __funnelshift_l(sl, sc, 1);
    // G1: exactly one a_i = !x_{2i-1} & (x_{2i} | x_{2i+1})   (x9 = x1)
    const unsigned a1 = ~x1 & (x2 | x3), a2 = ~x3 & (x4 | x5), a3 = ~x5 & (x6 | x7), a4 = ~x7 & (x8 | x1);
    const unsigned g1 = (a1 | a2 | a3 | a4) & ~two_of_four(a1, a2, a3, a4);
    // G2: 2 <= min(n1, n2) <= 3 with n1 = #c_i, n2 = #d_i
    const unsigned c1 = x1 | x2, c2 = x3 | x4, c3 = x5 | x6, c4 = x7 | x8;
    const unsigned d1 = x2 | x3, d2 = x4 | x5, d3 = x6 | x7, d4 = x8 | x1;
    const unsigned g2 = two_of_four(c1, c2, c3, c4) & two_of_four(d1, d2, d3, d4) & ~(c1 & c2 & c3 & c4 & d1 & d2 & d3 & d4);
    // G3: !((x2 | x3 | !x8) & x1);  G3': !((x6 | x7 | !x4) & x5)
    const unsigned g3 = second ? ~((x6 | x7 | ~x4) & x5) : ~((x2 | x3 | ~x8) & x1);
    return cc & g1 & g2 & g3;
}

// Thin the h x (nw words) bit plane in `a` with `b` as scratch of the same size (shared or global memory; all threads
// of the block call this, and `a` must be complete and visible to the block on entry).  max_iter < 0: to convergence,
// else at most max_iter iterations of two sub-iterations.  Each sub-iteration writes a & ~kill into the other plane,
// then one barrier; the loop stops at the first sub-iteration that deletes nothing.  Returns the plane that holds the
// result (a or b); it is complete and visible to the block on return.
__device__ inline unsigned *thin_plane(unsigned *a, unsigned *b, int h, int nw, int max_iter) {
    const int n = h * nw;
    for (int it = 0; max_iter < 0 || it < max_iter; it++) {
        for (int s = 0; s < 2; s++) {
            int killed = 0;
            for (int i = threadIdx.x; i < n; i += blockDim.x) {
                const int y = i / nw, k = i - y * nw;
                const bool hasL = k > 0, hasR = k + 1 < nw;
                unsigned nl = 0, nc = 0, nr = 0, sl = 0, sc = 0, sr = 0;
                if (y > 0) {
                    const unsigned *r = a + i - nw;
                    nc = r[0];
                    if (hasL) nl = r[-1];
                    if (hasR) nr = r[1];
                }
                if (y + 1 < h) {
                    const unsigned *r = a + i + nw;
                    sc = r[0];
                    if (hasL) sl = r[-1];
                    if (hasR) sr = r[1];
                }
                const unsigned cc = a[i], cl = hasL ? a[i - 1] : 0u, cr = hasR ? a[i + 1] : 0u;
                const unsigned kill = kill_word(nl, nc, nr, cl, cc, cr, sl, sc, sr, s == 1);
                b[i] = cc & ~kill;
                killed |= kill != 0u;
            }
            if (!__syncthreads_or(killed)) return a;  // nothing deleted: a is the result
            unsigned *t = a; a = b; b = t;
        }
    }
    return a;
}

}  // namespace thin
}  // namespace mte
