// DEE annotation post-process for sm_100a: edge normals, non-maximum suppression, hysteresis.
//
// Replaces (reference root relative):
//   normals block         infer_edge_estimation.py:193-199 (= :244-250)
//   non_max_suppression   packnet_code/packnet_sfm/utils/tools.py:9-46
//   hysteresis + DFS      packnet_code/packnet_sfm/utils/tools.py:49-92
// and the third-party cv2.Sobel(img, CV_64F, dx, dy, ksize=5) they call: separable
// [1,4,6,4,1] x [-1,-2,0,2,1], BORDER_REFLECT_101, row pass first, fp64 accumulation in tap order, the
// column pass folded symmetrically / anti-symmetrically.  Every fp64 operation below is an explicit
// __dmul_rn / __dadd_rn / __fma_rn in exactly that order (no compiler contraction; a fused multiply-add appears only
// where the product is exact -- a tap times an fp32 value, a power of two times a double -- so that it rounds exactly
// like the separate multiply and add), so the Sobel responses are bit-identical to OpenCV's and the orientation bins /
// uint8 normals follow.
//
// Kernels:  dee_tables_kernel    (the 255 level-threshold directions of the normals)
//           dee_front_tma_kernel (fp32 planes: TMA halo tile, Sobel5 + normals + NMS + hysteresis labels out of a register
//                                 window; with NMS a straight-line row loop whose undecided pixels are redone by
//                                 dee_pixel_exact, without NMS a generic row loop that decides each pixel in line)
//           dee_front_kernel     (fp64 planes and odd shapes: shared-memory halo tile, same decisions)
//           canny::run_level_hysteresis (shared 8-connected flood / union-find hysteresis)
//           dee_finish_kernel    (img * labels / max(labels), the reference's normalisation quirk included)
//           dee_convert_kernel   (NMS only, into the other float type)
// Both front kernels call the same __forceinline__ helpers for the Sobel passes, the zero-gradient level and the NMS bin.
#include <cuda.h>
#include <math.h>
#include <string.h>

#include <type_traits>

#include "common.cuh"

namespace mte {
namespace dee {

constexpr int TW = 64, TH = 16, kThreads = 256;

struct ImgStat {
    unsigned long long borderMaxKey;  // order-preserving key of the largest non-NaN border value
    unsigned int anyStrong;           // a strong interior pixel exists (=> max(labels) >= 2)
    unsigned int borderNaN;           // np.max propagates NaN
};

__device__ __forceinline__ int reflect101(int i, int n) {
    if (n == 1) return 0;
    // one reflection covers every halo index of a plane that is at least 3 wide (-n < i < 2n - 1): no division on
    // the hot path (two integer modulos per loaded element were a third of the kernel's instructions)
    int j = i < 0 ? -i : i;
    j = j >= n ? 2 * (n - 1) - j : j;
    if ((unsigned)j < (unsigned)n) return j;
    const int period = 2 * (n - 1);
    i %= period;
    if (i < 0) i += period;
    return i >= n ? period - i : i;
}

__device__ __forceinline__ unsigned long long dkey(double v) {
    const unsigned long long b = (unsigned long long)__double_as_longlong(v);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__host__ __device__ inline double dkey_inv(unsigned long long k) {
    const unsigned long long b = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;
#ifdef __CUDA_ARCH__
    return __longlong_as_double((long long)b);
#else
    double d;
    memcpy(&d, &b, 8);
    return d;
#endif
}

// ---- exact quantisation without atan2 ---------------------------------------------------------------------------
// The u8 normal is trunc(U(atan2(-sy, sx))) with U(a) = ((a * (180/pi) + 180) / 360) * 255 evaluated op by op in
// fp64 (infer_edge_estimation.py:247-249).  U is monotone, so level k starts at theta_k = the smallest double with
// U(theta_k) >= k; dee_tables_kernel finds the 255 thresholds by bisection over the doubles with exactly the
// operations of the slow path, and stores the DIRECTION (cos, sin) of each.  A pixel then takes a candidate level from
// an fp32 atan2f and proves it with two fp64 cross products against the neighbouring threshold directions
// (sin(A - theta) = (Y cos theta - X sin theta) / r); only when a cross product is within 2^-44 of zero relative to
// |X| + |Y| -- i.e. the angle is within ~6e-14 rad of a threshold, where the last bits of atan2 decide -- the pixel
// falls back to the exact double atan2.  The NMS bin (tools.py:24-38) is decided the same way by |sy| against
// |sx| * tan(22.5 deg) / tan(67.5 deg) with a 2^-40 relative guard band.  ~100 fp64 operations per atan2 become ~12.
struct DeeTab {
    double2 dir[256];        // dir[k] = (cos, sin) of theta_k, k = 1..255
    unsigned char zero4[4];  // level of a zero gradient, by the sign bits of (sy, sx)
};

__device__ __forceinline__ double normal_level_value(double ang) {
    return __dmul_rn(__ddiv_rn(__dadd_rn(__dmul_rn(ang, 180.0 / M_PI), 180.0), 360.0), 255.0);
}

__global__ void dee_tables_kernel(DeeTab *tab) {
    const int k = threadIdx.x;
    if (k >= 1 && k < 256) {
        unsigned long long lo = dkey(-M_PI), hi = dkey(M_PI);  // U(lo) < k <= U(hi)
        while (hi - lo > 1ull) {
            const unsigned long long mid = lo + (hi - lo) / 2ull;
            if (normal_level_value(dkey_inv(mid)) >= (double)k) hi = mid; else lo = mid;
        }
        const double th = dkey_inv(hi);
        tab->dir[k] = make_double2(cos(th), sin(th));
    }
    if (k == 0) tab->dir[0] = make_double2(-1.0, 0.0);
    if (k < 4) {
        const double sy = (k & 1) ? -0.0 : 0.0, sx = (k & 2) ? -0.0 : 0.0;
        tab->zero4[k] = (unsigned char)(int)normal_level_value(atan2(-sy, sx));
    }
}

// ---- arithmetic shared by the front kernels ---------------------------------------------------------------------
// cv2.Sobel's row pass over five consecutive values, tap by tap: d with the derivative taps, m with the smoothing taps.
// FUSED: the inputs are fp32 values, so every product with a tap (0, +-1, +-2, 4, 6) is EXACT in fp64 and a fused
// multiply-add rounds exactly once, like the separate add of the exact product: bit-identical to the mul + add sequence
// (signs of zero and NaN / Inf included; tests/test_oracle_cpu.py::test_sobel5_fused_taps), half the instructions.
// dee_front_kernel keeps the mul + add form for both input types: for an fp64 value 6 * a is not exact.
template <bool FUSED>
__device__ __forceinline__ void sobel5_row(double a0, double a1, double a2, double a3, double a4, double &d, double &m) {
    if (FUSED) {
        d = __fma_rn(-2.0, a1, -a0);
        d = __fma_rn(0.0, a2, d);
        d = __fma_rn(2.0, a3, d);
        d = __dadd_rn(d, a4);
        m = __fma_rn(4.0, a1, a0);
        m = __fma_rn(6.0, a2, m);
        m = __fma_rn(4.0, a3, m);
        m = __dadd_rn(m, a4);
    } else {
        d = __dmul_rn(-1.0, a0);
        d = __dadd_rn(d, __dmul_rn(-2.0, a1));
        d = __dadd_rn(d, __dmul_rn(0.0, a2));
        d = __dadd_rn(d, __dmul_rn(2.0, a3));
        d = __dadd_rn(d, __dmul_rn(1.0, a4));
        m = __dmul_rn(1.0, a0);
        m = __dadd_rn(m, __dmul_rn(4.0, a1));
        m = __dadd_rn(m, __dmul_rn(6.0, a2));
        m = __dadd_rn(m, __dmul_rn(4.0, a3));
        m = __dadd_rn(m, __dmul_rn(1.0, a4));
    }
}

// cv2.Sobel's column pass over the row-pass results of five consecutive rows, D(i) / S(i) for i = 0 .. 4 (S(2) has tap
// 0): symmetric on the derivative rows (-> sx), anti-symmetric on the smoothed rows (-> sy); returns (sx, sy).  FUSED:
// products with a power of two are exact for any double, so they fuse as well (6 * D(2) is rounded on its own, as in
// OpenCV).  The rows come through accessors so that each is read where the arithmetic uses it.
template <bool FUSED, class RowD, class RowS>
__device__ __forceinline__ double2 sobel5_col(RowD D, RowS S) {
    double sx, sy;
    if (FUSED) {
        sx = __fma_rn(4.0, __dadd_rn(D(3), D(1)), __dmul_rn(6.0, D(2)));
        sx = __dadd_rn(sx, __dadd_rn(D(4), D(0)));
        sy = __fma_rn(2.0, __dsub_rn(S(3), S(1)), __dsub_rn(S(4), S(0)));
    } else {
        sx = __dmul_rn(6.0, D(2));
        sx = __dadd_rn(sx, __dmul_rn(4.0, __dadd_rn(D(3), D(1))));
        sx = __dadd_rn(sx, __dmul_rn(1.0, __dadd_rn(D(4), D(0))));
        sy = __dmul_rn(2.0, __dsub_rn(S(3), S(1)));
        sy = __dadd_rn(sy, __dmul_rn(1.0, __dsub_rn(S(4), S(0))));
    }
    return make_double2(sx, sy);
}

// level of a zero gradient, by the sign bits of (sy, sx)
__device__ __forceinline__ int zero_level(double sx, double sy, const unsigned char *sZero) {
    return sZero[(int)(__double2hiint(sy) < 0) | ((int)(__double2hiint(sx) < 0) << 1)];
}

// NMS bin of atan2(sy, sx): 0 = [0, 22.5) u [157.5, 180], 1 = [22.5, 67.5), 2 = [67.5, 112.5), 3 = [112.5, 157.5),
// 4 = none.  |sy| against |sx| tan(22.5 / 67.5 deg) in fp64 with a 2^-40 guard band, and inside that band (or for NaN,
// Inf / Inf) the reference's own expression (tools.py:12-17, 24-38)
__device__ __forceinline__ int bin_exact(double sx, double sy) {
    const double ax = fabs(sx), ay = fabs(sy);
    const double t1 = ax * 0.41421356237309503, t2 = ax * 2.4142135623730951;   // tan 22.5, tan 67.5
    constexpr double lo = 1.0 - 0x1p-40, hi = 1.0 + 0x1p-40;
    if (ax == 0.0 && ay == 0.0) return 0;   // atan2(+-0, +-0) is 0 or +-pi: bin 0 either way
    if (ay < t1 * lo) return 0;
    if (ay > t1 * hi && ay < t2 * lo) return ((sx < 0.0) != (sy < 0.0)) ? 3 : 1;
    if (ay > t2 * hi) return 2;
    double a = __dmul_rn(atan2(sy, sx), 180.0 / M_PI);
    if (a < 0.0) a = __dadd_rn(a, 180.0);
    if ((0.0 <= a && a < 22.5) || (157.5 <= a && a <= 180.0)) return 0;
    if (22.5 <= a && a < 67.5) return 1;
    if (67.5 <= a && a < 112.5) return 2;
    if (112.5 <= a && a < 157.5) return 3;
    return 4;
}

// T = type of the input map (the reference passes float32 network outputs; float64 accepted)
template <typename T>
__global__ void __launch_bounds__(kThreads) dee_front_kernel(const DeeTab *__restrict__ tab,
                                                             const T *__restrict__ img, int N, int H, int W, int doNms,
                                                             int doHyst, double tLow, double tHigh,
                                                             unsigned char *__restrict__ normals,
                                                             T *__restrict__ nmsOut, unsigned char *__restrict__ cl,
                                                             unsigned char *__restrict__ E, ImgStat *stats) {
    __shared__ double s[TH + 4][TW + 4];
    __shared__ double rowD[TH + 4][TW];  // row pass with the derivative taps  (-> sobel x)
    __shared__ double rowS[TH + 4][TW];  // row pass with the smoothing taps   (-> sobel y)
    __shared__ double2 sDir[256];
    __shared__ unsigned char sZero[4];
    if (normals) {  // the table is only built (and only needed) for the normals
        sDir[threadIdx.x & 255] = tab->dir[threadIdx.x & 255];
        if (threadIdx.x < 4) sZero[threadIdx.x] = tab->zero4[threadIdx.x];
    }
    const int tilesX = ceil_div(W, TW), tilesY = ceil_div(H, TH);
    const int tile = blockIdx.x % (tilesX * tilesY), im = blockIdx.x / (tilesX * tilesY);
    const int x0 = (tile % tilesX) * TW, y0 = (tile / tilesX) * TH;
    const T *src = img + (size_t)im * H * W;
    const bool needSobel = (normals != nullptr) || doNms;

    // halo tile: a thread keeps ONE column (its reflected x is computed once) and walks the rows; the four halo
    // columns are a second, small step.  (A flat index costs a division and two reflections per element.)
    {
        const int c = threadIdx.x & (TW - 1), rg = threadIdx.x / TW;   // TW columns x (kThreads / TW) row groups
        const int x = reflect101(x0 + c - 2, W);
        for (int r = rg; r < TH + 4; r += kThreads / TW) {
            const int y = reflect101(y0 + r - 2, H);
            s[r][c] = (double)src[(size_t)y * W + x];
        }
        if (threadIdx.x < 4 * (TH + 4)) {
            const int r = threadIdx.x >> 2, c2 = TW + (threadIdx.x & 3);
            const int y = reflect101(y0 + r - 2, H), x2 = reflect101(x0 + c2 - 2, W);
            s[r][c2] = (double)src[(size_t)y * W + x2];
        }
    }
    __syncthreads();
    if (needSobel) {
        for (int i = threadIdx.x; i < (TH + 4) * TW; i += kThreads) {
            const int r = i / TW, c = i - r * TW;
            double d, m;
            sobel5_row<false>(s[r][c], s[r][c + 1], s[r][c + 2], s[r][c + 3], s[r][c + 4], d, m);
            rowD[r][c] = d;
            rowS[r][c] = m;
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < TH * TW; i += kThreads) {
        const int r = i / TW, c = i - r * TW;
        const int y = y0 + r, x = x0 + c;
        if (y >= H || x >= W) continue;
        const size_t o = (size_t)im * H * W + (size_t)y * W + x;
        const T v = (T)s[r + 2][c + 2];   // the tile holds the exact input value
        double sx = 0.0, sy = 0.0;
        if (needSobel) {
            const double2 grad = sobel5_col<false>([&](int i) { return rowD[r + i][c]; }, [&](int i) { return rowS[r + i][c]; });
            sx = grad.x;
            sy = grad.y;
        }
        if (normals) {
            const double X = sx, Y = -sy;
            int lvl = -1;
            if (X == 0.0 && Y == 0.0) {
                lvl = zero_level(sx, sy, sZero);
            } else {
                const float a32 = atan2f((float)Y, (float)X);
                const int k0 = min(max((int)((a32 * 57.29577951f + 180.f) * (255.f / 360.f)), 0), 255);
                const double m = (fabs(X) + fabs(Y)) * 0x1p-44;
                bool ok = true;
                if (k0 >= 1) { const double2 d = sDir[k0]; ok = (Y * d.x - X * d.y) > m; }                // theta_k0 < A
                if (k0 <= 254) { const double2 d = sDir[k0 + 1]; ok = ok && (Y * d.x - X * d.y) < -m; }   // A < theta_k0+1
                if (ok) lvl = k0;
            }
            if (lvl < 0) lvl = (int)normal_level_value(atan2(-sy, sx));  // within ~6e-14 rad of a threshold, NaN / Inf
            normals[o] = (unsigned char)lvl;
        }
        const bool interior = y >= 1 && y < H - 1 && x >= 1 && x < W - 1;
        T keep = v;
        if (doNms) {
            keep = (T)0;
            if (interior) {
                const int bin = bin_exact(sx, sy);
                T q = (T)1, rr = (T)1;  // tools.py:22-23: no bin (NaN angle) compares against 1
                const int cr = r + 2, cc = c + 2;
                if (bin == 0) { q = (T)s[cr][cc + 1]; rr = (T)s[cr][cc - 1]; }
                else if (bin == 1) { q = (T)s[cr - 1][cc - 1]; rr = (T)s[cr + 1][cc + 1]; }
                else if (bin == 2) { q = (T)s[cr + 1][cc]; rr = (T)s[cr - 1][cc]; }
                else if (bin == 3) { q = (T)s[cr + 1][cc - 1]; rr = (T)s[cr - 1][cc + 1]; }
                if (v >= q && v >= rr) keep = v;
            }
        }
        if (nmsOut) nmsOut[o] = keep;
        if (doHyst) {
            unsigned char c_l = 255, e_l = 255;
            const double kv = (double)keep;
            if (interior) {
                if (kv > tHigh) { c_l = 0; e_l = 0; }
                else if (!(kv < tLow)) c_l = 0;
                if (e_l == 0) atomicOr(&stats[im].anyStrong, 1u);
            } else {
                // border pixels keep their raw value as "label" (tools.py:54-55 never touches them)
                if (kv != kv) atomicOr(&stats[im].borderNaN, 1u);
                else atomicMax(&stats[im].borderMaxKey, dkey(kv));
            }
            cl[o] = c_l;
            E[o] = e_l;
        }
    }
}

// ---------------------------------------------------------------------------
// Front kernel, B200 form (fp32 input, W % 4 == 0, H, W >= 4): the halo tile arrives by ONE bulk-tensor copy (TMA,
// cp.async.bulk.tensor.3d + mbarrier; out-of-image cells zero-filled by the copy engine and, on border tiles only,
// patched with the REFLECT_101 values from inside the tile), and the separable Sobel runs out of a REGISTER window:
// a thread owns one column, walks down the tile rows, computes the two fp64 row filters of a row from five shared
// floats and keeps the last five results in registers for the column filter -- no fp64 round trip through shared
// memory, no per-element index arithmetic.  With the NMS the row loop is straight-line code that only flags the pixels
// its fp32 candidates cannot decide, and dee_pixel_exact redoes them after the loop; without it (normals only, or the
// hysteresis of the raw map) a generic row loop decides each pixel in line.  Both use the shared Sobel passes and exact
// decisions, so they make dee_front_kernel's decisions; that kernel stays for fp64 inputs and odd shapes.
// ---------------------------------------------------------------------------
// The innermost box coordinate of a bulk-tensor copy must be 16-byte aligned (x0 - 2 traps with "illegal
// instruction"; probed with scripts/ubench/tma_test.cu), so the box starts at x0 - 4 and is 8 columns wider than the tile.
constexpr int XW = 128, XH = 31, XROWS = XH + 4, XPAD = 4, XCOLS = XW + 2 * XPAD, kXThreads = XW;   // 35 tile rows = 7 groups of 5
static_assert(XROWS % 5 == 0, "the register window rotates with period 5");
constexpr int kXMinBlocks = 6;   // CTAs per SM the TMA front is compiled for: at most 80 registers a thread

__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
// cond ? a : b as a real SELP (keeps ptxas from turning value selections into divergent branches)
__device__ __forceinline__ unsigned selp(bool cond, unsigned a, unsigned b) {
    unsigned r;
    asm("{\n\t.reg .pred p;\n\tsetp.ne.s32 p, %3, 0;\n\tselp.u32 %0, %1, %2, p;\n\t}" : "=r"(r) : "r"(a), "r"(b), "r"((int)cond));
    return r;
}

// Branch-free fp32 atan2 (octant reduction + odd minimax polynomial; |error| < 3e-6 rad for components in [1e-30, 1e30],
// tests/test_host_cpu.py::test_atan2_candidate_error_bound): only a CANDIDATE; the exact fp64 decisions take over
// whenever it lies too close to a boundary to decide.
__device__ __forceinline__ float atan2_candidate(float y, float x) {
    const float ax = fabsf(x), ay = fabsf(y);
    const float mx = fmaxf(ax, ay), mn = fminf(ax, ay);
    float rc;   // the caller discards candidates whose larger component is outside [1e-30, 1e30]: no denormal handling
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rc) : "f"(mx));
    const float t = mn * rc;
    const float t2 = t * t;
    float p = fmaf(t2, -0.0117212f, 0.05265332f);
    p = fmaf(p, t2, -0.11643287f);
    p = fmaf(p, t2, 0.19354346f);
    p = fmaf(p, t2, -0.33262347f);
    p = fmaf(p, t2, 0.99997726f);
    // fmaxf / fminf drop a NaN operand: x * 0 + y * 0 carries a NaN (or an Inf, as NaN) into the result, so that
    // the exact decisions see a candidate they cannot prove and take the reference's own expression
    p = fmaf(p, t, fmaf(x, 0.f, y * 0.f));
    p = ay > ax ? 1.57079637f - p : p;
    p = x < 0.f ? 3.14159274f - p : p;
    return y < 0.f ? -p : p;
}

// angle of the normal, atan2(-sy, sx), as an fp32 CANDIDATE (|error| < 3e-6 rad on [1e-30, 1e30]:
// tests/test_host_cpu.py::test_atan2_candidate_error_bound).  Outside that range the fast division flushes or
// overflows: the candidate becomes NaN and every decision takes its exact path.
__device__ __forceinline__ float angle_candidate(double sx, double sy) {
    const float fx = (float)sx, fy = (float)-sy;
    const float big = fmaxf(fabsf(fx), fabsf(fy));
    const float a32 = atan2_candidate(fy, fx);
    return (big > 1e-30f && big < 1e30f) ? a32 : __int_as_float(0x7fc00000);
}

// level = trunc(lv(A)), lv(A) = A * 255 / (2 pi) + 127.5, from the fp32 candidate a32.  The candidate level decides
// alone (`decided`) when its fractional part is at least 1e-3 away from an integer (8x the candidate's 1.2e-4 levels of
// error + the fp32 rounding of lv); the rest (0.2 % of the pixels, zero gradients, NaN / Inf) is proved by
// dee_level_exact.  `valid` is false for a NaN candidate.
__device__ __forceinline__ int level_candidate(float a32, bool &decided, bool &valid) {
    const float lv = fmaf(a32, 40.5845105f, 127.5f);
    const int k0 = (int)lv;
    const float fl = lv - (float)k0;
    decided = fl >= 1e-3f && fl <= 1.f - 1e-3f && (unsigned)k0 <= 254u;
    valid = fl == fl;
    return k0;
}

// The exact decisions of the pixels whose fp32 candidate is too close to a boundary (or is NaN: zero gradient, NaN /
// Inf, values outside the fast division's range).  Rare, so they are real calls: ten inlined copies of the double
// atan2 made the row loop 60 KB of code.
__device__ __noinline__ int dee_level_exact(double sx, double sy, int k0, const double2 *sDir, const unsigned char *sZero) {
    if (sx == 0.0 && sy == 0.0) return zero_level(sx, sy, sZero);
    const double X = sx, Y = -sy;
    const int kc = min(max(k0, 0), 255);
    const double m = (fabs(X) + fabs(Y)) * 0x1p-44;
    // k0 >= 0: a valid candidate (within 1.2e-4 levels of the truth), possibly one level off next to a threshold:
    // try kc, kc - 1, kc + 1.  Two fp64 cross products against the neighbouring threshold DIRECTIONS prove a level
    // (sin(A - theta) = (Y cos theta - X sin theta) / r) -- ONLY for an angle known to lie near theta: the sign of a
    // sine says nothing half a turn away, so without a candidate (k0 < 0) the reference's expression decides.
    // dee_front_kernel proves its candidate with its own copy of these products, which loads only the directions it
    // needs: neither form as a shared helper compiles both kernels to the same code as their own copies.
    for (int t = 0; t < 3 && k0 >= 0; t++) {
        const int kk = kc + (t == 0 ? 0 : (t == 1 ? -1 : 1));
        if (kk < 0 || kk > 255) continue;
        const double2 dl = sDir[max(kk, 1)], dh = sDir[min(kk + 1, 255)];
        const bool okLo = kk < 1 || (Y * dl.x - X * dl.y) > m;       // theta_kk < A
        const bool okHi = kk > 254 || (Y * dh.x - X * dh.y) < -m;    // A < theta_kk+1
        if (okLo && okHi) return kk;
    }
    return (int)normal_level_value(atan2(-sy, sx));  // inside a 2^-44 guard band, NaN / Inf: the reference's expression
}

__device__ __noinline__ int dee_bin_exact(double sx, double sy) { return bin_exact(sx, sy); }

// One output pixel entirely by the exact paths, straight from the halo tile (tile rows j .. j + 4 around output row j,
// tile columns c + XPAD - 2 .. + 2): used by the straight-line row loop for the few pixels its fp32 candidate could not
// decide.  Same operation order as the loop (cv2.Sobel's), same decisions as dee_front_kernel.  Returns "strong".
template <bool NRM, bool HYST>
__device__ __noinline__ bool dee_pixel_exact(const float *tile, int j, int c, bool interior, float thF, float tlF,
                                             const double2 *sDir, const unsigned char *sZero, unsigned char *nrmB,
                                             float *nmsB, unsigned char *clB, unsigned char *eB, unsigned off) {
    double d[5], m[5];
#pragma unroll
    for (int r = 0; r < 5; r++) {
        const float *tr = tile + (j + r) * XCOLS + c + XPAD - 2;
        sobel5_row<true>(tr[0], tr[1], tr[2], tr[3], tr[4], d[r], m[r]);
    }
    const double2 grad = sobel5_col<true>([&](int i) { return d[i]; }, [&](int i) { return m[i]; });
    const double sx = grad.x, sy = grad.y;
    if (NRM) nrmB[off] = (unsigned char)dee_level_exact(sx, sy, -1, sDir, sZero);
    const int cr = j + 2, cc = c + XPAD;
    const float v = tile[cr * XCOLS + cc];
    float keep = 0.f;
    if (interior) {
        const int bin = dee_bin_exact(sx, sy);
        const int dy = bin == 0 ? 0 : (bin == 1 ? -1 : 1);
        const int dx = bin == 0 ? 1 : (bin == 2 ? 0 : -1);
        float q = tile[(cr + dy) * XCOLS + cc + dx], rr = tile[(cr - dy) * XCOLS + cc - dx];
        if (bin == 4) { q = 1.f; rr = 1.f; }
        if (v >= q && v >= rr) keep = v;
    }
    if (nmsB) nmsB[off] = keep;
    bool strong = false;
    if (HYST) {
        strong = interior && keep > thF;
        const bool weak = keep < tlF && !strong;
        clB[off] = (interior && !weak) ? 0 : 255;
        eB[off] = strong ? 0 : 255;
    }
    return strong;
}

template <bool NRM, bool NMS, bool HYST>
__global__ void __launch_bounds__(kXThreads, kXMinBlocks) dee_front_tma_kernel(const __grid_constant__ CUtensorMap tmap,
                                                                  const DeeTab *__restrict__ tab, int N, int H, int W,
                                                                  double tLow, double tHigh,
                                                                  unsigned char *__restrict__ normals,
                                                                  float *__restrict__ nmsOut, unsigned char *__restrict__ cl,
                                                                  unsigned char *__restrict__ E, ImgStat *stats) {
    __shared__ __align__(128) float tile[XROWS][XCOLS];
    __shared__ __align__(8) unsigned long long mbar;
    __shared__ double2 sDir[256];
    __shared__ unsigned char sZero[4];
    const int tilesX = ceil_div(W, XW), tilesY = ceil_div(H, XH);
    const int t = blockIdx.x % (tilesX * tilesY), im = blockIdx.x / (tilesX * tilesY);
    const int x0 = (t % tilesX) * XW, y0 = (t / tilesX) * XH;
    const unsigned bar = smem_u32(&mbar);
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"((unsigned)sizeof(tile)) : "memory");
        asm volatile(
            "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
            ::"r"(smem_u32(&tile[0][0])), "l"(reinterpret_cast<unsigned long long>(&tmap)), "r"(x0 - XPAD), "r"(y0 - 2), "r"(im),
              "r"(bar)
            : "memory");
    }
    if (NRM) {  // overlaps the copy
        sDir[threadIdx.x] = tab->dir[threadIdx.x];
        sDir[threadIdx.x + 128] = tab->dir[threadIdx.x + 128];
        if (threadIdx.x < 4) sZero[threadIdx.x] = tab->zero4[threadIdx.x];
    }
    {  // wait for the tile (phase 0)
        unsigned done = 0;
        while (!done)
            asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\tselp.b32 %0, 1, 0, p;\n\t}"
                         : "=r"(done) : "r"(bar) : "memory");
    }
    // border tiles: the zero-filled cells within two pixels of the image get their REFLECT_101 value, which lies
    // inside this tile (in-image cells are never written, so one pass suffices)
    if (x0 == 0 || y0 == 0 || x0 + XW + 2 > W || y0 + XH + 2 > H) {
        for (int i = threadIdx.x; i < XROWS * XCOLS; i += kXThreads) {
            const int r = i / XCOLS, c = i - r * XCOLS;
            const int y = y0 - 2 + r, x = x0 - XPAD + c;
            const bool out = y < 0 || y >= H || x < 0 || x >= W;
            if (out && y >= -2 && y <= H + 1 && x >= -2 && x <= W + 1) {
                const int yy = reflect101(y, H), xx = reflect101(x, W);
                tile[r][c] = tile[yy - (y0 - 2)][xx - (x0 - XPAD)];
            }
        }
    }
    __syncthreads();

    const int c = threadIdx.x, x = x0 + c;
    const bool colIn = x < W;
    const bool xInterior = x >= 1 && x < W - 1;
    const int jEnd = min(XH, H - y0);   // output rows of this tile
    // the hysteresis labels compare an fp32 value with fp64 thresholds: keep > tHigh <=> keep > (largest float <=
    // tHigh), keep < tLow <=> keep < (smallest float >= tLow) -- exact for every threshold incl. +-Inf / NaN
    const float thF = __double2float_rd(tHigh), tlF = __double2float_ru(tLow);
    double wD[5], wS[5];   // row-filter results of the last five tile rows, slot = tile row % 5
    float f[5][3];         // the fp32 values at columns x - 1, x, x + 1 of the same rows (NMS neighbours, centre value)
    bool anyStrong = false;
    // output addresses = a CTA-uniform base + ONE 32-bit running offset (x + row * W), formed by a single wide
    // multiply-add per store (four running 64-bit pointers cost 16 instructions per pixel in adds and pair moves)
    const size_t o0 = (size_t)im * H * W + (size_t)y0 * W;
    unsigned char *const nrmB = NRM ? normals + o0 : nullptr;
    float *const nmsB = nmsOut ? nmsOut + o0 : nullptr;
    unsigned char *const clB = HYST ? cl + o0 : nullptr, *const eB = HYST ? E + o0 : nullptr;
    unsigned oi = (unsigned)x;
    auto st8 = [](unsigned char *base, unsigned off, unsigned v) {
        asm volatile("{\n\t.reg .u64 a;\n\tmad.wide.u32 a, %0, 1, %1;\n\tst.global.u8 [a], %2;\n\t}" ::"r"(off), "l"(base), "r"(v) : "memory");
    };
    auto st32 = [](float *base, unsigned off, float v) {
        asm volatile("{\n\t.reg .u64 a;\n\tmad.wide.u32 a, %0, 4, %1;\n\tst.global.f32 [a], %2;\n\t}" ::"r"(off), "l"(base), "f"(v) : "memory");
    };
    const float *tr = &tile[0][c + XPAD - 2];               // columns x - 2 .. x + 2 of the current tile row
    if constexpr (NMS) {
        // ---- straight-line form (every variant that runs the NMS): no branch in the body of a row except the final
        // stores, so the scheduler interleaves the five unrolled rows (the kernel is bound by dependent-issue latency:
        // ncu `wait` 2.3 per issue at 20-24 warps per SM).  Pixels whose candidate cannot decide are only FLAGGED here
        // and redone by dee_pixel_exact after the loop; zero gradients (flat regions, common) are decided in line.
        // Border pixels: the NMS leaves 0 there (tools.py:19-20), so their raw "label" is 0 for every tile that
        // touches the border: one atomicMax per CTA instead of one per pixel.
        auto row_pass = [&](int u) {
            const float t0 = tr[0], t1 = tr[1], t2 = tr[2], t3 = tr[3], t4 = tr[4];
            tr += XCOLS;
            f[u][0] = t1; f[u][1] = t2; f[u][2] = t3;
            sobel5_row<true>(t0, t1, t2, t3, t4, wD[u], wS[u]);
        };
        unsigned long long flagged = 0ull;
        const float zl0 = (float)sZero[0], zl1 = (float)sZero[1], zl2 = (float)sZero[2], zl3 = (float)sZero[3];
        auto out_row = [&](int u, int j, unsigned &gmask) {   // output row j of the tile; tile row j + 4 is in slot u
            const int y = y0 + j;
            const float v = f[(u + 3) % 5][1];
            // rows j .. j+4 of the row filters sit in slots (u+1)%5 .. (u+5)%5
            const double2 grad = sobel5_col<true>([&](int i) { return wD[(u + 1 + i) % 5]; },
                                                  [&](int i) { return wS[(u + 1 + i) % 5]; });
            const double sx = grad.x, sy = grad.y;
            const float a32 = angle_candidate(sx, sy);
            const bool zero = sx == 0.0 && sy == 0.0;
            bool decided = true;
            int lvl = 0;
            if (NRM) {
                bool valid;
                const int k0 = level_candidate(a32, decided, valid);
                // zero gradient: level by the signs of the two zeros (sZero), picked with selects
                const bool ny = __double2hiint(sy) < 0, nx = __double2hiint(sx) < 0;
                const float zl = nx ? (ny ? zl3 : zl2) : (ny ? zl1 : zl0);
                lvl = zero ? (int)zl : k0;
            }
            // bin of atan2(sy, sx) = -a32 (mod pi): in units of pi / 4 shifted by half a bin the boundaries are the
            // integers and the bins repeat with period 4: the fp32 candidate decides when it is at least 5e-5 (4e-5 rad,
            // > 10x its error) away from every boundary
            const float uu = fmaf(-a32, 1.27323954f, 4.5f);   // in (0.5, 8.5)
            const int iu = (int)uu;
            const float fu = uu - (float)iu;
            decided = decided && fu >= 5e-5f && fu <= 1.f - 5e-5f;
            const int bin = zero ? 0 : (iu & 3);
            const bool need = !zero && !decided;
            const bool interior = xInterior && y >= 1 && y < H - 1;
            const float(&up)[3] = f[(u + 2) % 5];
            const float(&md)[3] = f[(u + 3) % 5];
            const float(&dn)[3] = f[(u + 4) % 5];
            float q = dn[0], rr = up[2];                       // bin 3 (SW, NE)
            q = bin == 2 ? dn[1] : q; rr = bin == 2 ? up[1] : rr;   // (S, N)
            q = bin == 1 ? up[0] : q; rr = bin == 1 ? dn[2] : rr;   // (NW, SE)
            q = bin == 0 ? md[2] : q; rr = bin == 0 ? md[0] : rr;   // (E, W)
            const float keep = (interior && v >= q && v >= rr) ? v : 0.f;
            const bool strong = interior && keep > thF;
            const bool weak = keep < tlF && !strong;
            const bool ok = j < jEnd && colIn;
            anyStrong = anyStrong || (strong && !need && ok);
            gmask |= (need && ok) ? (1u << u) : 0u;
            if (ok) {
                if (NRM) st8(nrmB, oi, (unsigned)lvl);
                if (nmsOut) st32(nmsB, oi, keep);
                if (HYST) {
                    st8(clB, oi, (interior && !weak) ? 0u : 255u);
                    st8(eB, oi, strong ? 0u : 255u);
                }
            }
            oi += (unsigned)W;
        };
        unsigned gm = 0u;
#pragma unroll
        for (int u = 0; u < 4; u++) row_pass(u);   // tile rows 0 .. 3: no output row is complete yet
        row_pass(4);
        out_row(4, 0, gm);
        flagged = (unsigned long long)(gm >> 4);
#pragma unroll 1
        for (int g = 1; g < XROWS / 5; g++) {
            gm = 0u;
#pragma unroll
            for (int u = 0; u < 5; u++) {
                row_pass(u);
                out_row(u, g * 5 + u - 4, gm);
            }
            flagged |= (unsigned long long)gm << (g * 5 - 4);
        }
        // ---- the flagged pixels, exactly
        while (flagged) {
            const int j = __ffsll((long long)flagged) - 1;
            flagged &= flagged - 1ull;
            const int y = y0 + j;
            const bool interior = xInterior && y >= 1 && y < H - 1;
            const bool st = dee_pixel_exact<NRM, HYST>(&tile[0][0], j, c, interior, thF, tlF, sDir, sZero, nrmB, nmsB, clB, eB,
                                                       (unsigned)x + (unsigned)j * (unsigned)W);
            anyStrong = anyStrong || st;
        }
        if (HYST) {
            if (threadIdx.x == 0 && (x0 == 0 || y0 == 0 || x0 + XW >= W || y0 + XH >= H))
                atomicMax(&stats[im].borderMaxKey, dkey(0.0));
            if (__syncthreads_or(anyStrong ? 1 : 0) && threadIdx.x == 0) atomicOr(&stats[im].anyStrong, 1u);
        }
    } else {
    // ---- generic form (no NMS: normals only, or hysteresis of the raw map, whose border labels are the raw values)
#pragma unroll 1
    for (int g = 0; g < XROWS / 5; g++) {
#pragma unroll
        for (int u = 0; u < 5; u++, tr += XCOLS) {
            const int k = g * 5 + u;   // tile row k = image row y0 - 2 + k
            {
                const float t0 = tr[0], t1 = tr[1], t2 = tr[2], t3 = tr[3], t4 = tr[4];
                f[u][1] = t2;
                if (NRM) sobel5_row<true>(t0, t1, t2, t3, t4, wD[u], wS[u]);
            }
            const int j = k - 4;           // output row of the tile, image row y0 + j; its centre is tile row k - 2
            if (j >= 0 && j < jEnd && colIn) {
                const int y = y0 + j;
                const float keep = f[(u + 3) % 5][1];   // no NMS: the raw value
                if (NRM) {
                    // rows j .. j+4 of the row filters sit in slots (u+1)%5 .. (u+5)%5
                    const double2 grad = sobel5_col<true>([&](int i) { return wD[(u + 1 + i) % 5]; },
                                                          [&](int i) { return wS[(u + 1 + i) % 5]; });
                    const double sx = grad.x, sy = grad.y;
                    bool decided, valid;
                    int lvl = level_candidate(angle_candidate(sx, sy), decided, valid);
                    if (!decided) {
                        // flat regions (zero gradient) are common in real maps: decided here, without the call
                        if (sx == 0.0 && sy == 0.0) lvl = zero_level(sx, sy, sZero);
                        else lvl = dee_level_exact(sx, sy, valid ? lvl : -1, sDir, sZero);   // NaN candidate: none
                    }
                    st8(nrmB, oi, (unsigned)lvl);
                }
                const bool interior = xInterior && y >= 1 && y < H - 1;
                if (nmsOut) st32(nmsB, oi, keep);
                if (HYST) {
                    if (interior) {
                        const bool strong = keep > thF;
                        const bool weak = keep < tlF && !strong;   // label 0; everything else (NaN too) is a candidate
                        anyStrong = anyStrong || strong;
                        st8(clB, oi, selp(weak, 255u, 0u));
                        st8(eB, oi, selp(strong, 0u, 255u));
                    } else {
                        // border pixels keep their raw value as "label" (tools.py:54-55 never touches them)
                        const double kv = (double)keep;
                        if (kv != kv) atomicOr(&stats[im].borderNaN, 1u);
                        else atomicMax(&stats[im].borderMaxKey, dkey(kv));
                        st8(clB, oi, 255u);
                        st8(eB, oi, 255u);
                    }
                }
                oi += (unsigned)W;
            }
        }
    }
    if (HYST && __syncthreads_or(anyStrong ? 1 : 0) && threadIdx.x == 0) atomicOr(&stats[im].anyStrong, 1u);
    }
}

// out = img * (labels / max(labels))  in the dtype the reference computes in (C = float or double).  One image per
// blockIdx.y; a thread handles kFinG groups of four consecutive pixels, all loads issued before the first use.  labels /
// max takes only two values inside the image (2 / max at kept pixels, 0 / max elsewhere): computed ONCE per CTA with the
// same division the reference does per pixel -- only the one-pixel border (label = the raw value) divides per pixel.
constexpr int kFinG = 4, kFinThreads = 256, kFinPx = kFinG * kFinThreads * 4;
template <typename T, typename C, typename O>
__global__ void __launch_bounds__(kFinThreads) dee_finish_kernel(const T *__restrict__ val, const unsigned char *__restrict__ E,
                                                                 int N, int H, int W, const ImgStat *__restrict__ stats,
                                                                 O *__restrict__ out) {
    __shared__ C sNorm[3];   // 2 / max, 0 / max, max
    const int im = blockIdx.y;
    const int plane = H * W;
    if (threadIdx.x == 0) {
        const ImgStat st = stats[im];
        // np.max over {0, 2 at kept pixels, raw border values}; NaN wins
        double mx = (H > 2 && W > 2) ? 0.0 : -INFINITY;
        if (st.anyStrong) mx = 2.0;
        if (st.borderMaxKey != 0ull) { const double b = dkey_inv(st.borderMaxKey); mx = b > mx ? b : mx; }
        if (st.borderNaN) mx = NAN;
        const C cm = (C)mx;
        sNorm[0] = (C)2 / cm;
        sNorm[1] = (C)0 / cm;
        sNorm[2] = cm;
    }
    const size_t base = (size_t)im * plane;
    const bool vecOk = sizeof(T) == 4 && sizeof(O) == 4 && (plane & 3) == 0 && (W & 3) == 0 &&
                       (reinterpret_cast<uintptr_t>(val) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0 &&
                       (reinterpret_cast<uintptr_t>(E) & 3) == 0;
    const int j00 = blockIdx.x * kFinPx + threadIdx.x * 4;
    if (vecOk) {
        // rows of whole float4s: a group never straddles a row, the border is its first / last pixel or a whole row
        float4 v[kFinG];
        unsigned e[kFinG];
#pragma unroll
        for (int g = 0; g < kFinG; g++) {
            const int j0 = j00 + g * kFinThreads * 4;
            v[g] = make_float4(0.f, 0.f, 0.f, 0.f);
            e[g] = 0xFFFFFFFFu;
            if (j0 < plane) {
                v[g] = __ldcs(reinterpret_cast<const float4 *>(reinterpret_cast<const float *>(val) + base + j0));
                e[g] = __ldcs(reinterpret_cast<const unsigned *>(E + base + j0));
            }
        }
        __syncthreads();
        const C n2 = sNorm[0], n0 = sNorm[1], cm = sNorm[2];
#pragma unroll
        for (int g = 0; g < kFinG; g++) {
            const int j0 = j00 + g * kFinThreads * 4;
            if (j0 >= plane) continue;
            const int y = j0 / W, x = j0 - y * W;
            const float in[4] = {v[g].x, v[g].y, v[g].z, v[g].w};
            float r[4];
            const bool rowBorder = y == 0 || y == H - 1;
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const C cv = (C)in[k];
                const C norm = ((e[g] >> (8 * k)) & 0xFFu) == 0u ? n2 : n0;
                r[k] = (float)(cv * norm);
            }
            if (rowBorder || x == 0 || x + 4 == W) {   // the border keeps its raw value as label: value * (value / max)
#pragma unroll
                for (int k = 0; k < 4; k++)
                    if (rowBorder || x + k == 0 || x + k == W - 1) { const C cv = (C)in[k]; r[k] = (float)(cv * (cv / cm)); }
            }
            __stcs(reinterpret_cast<float4 *>(reinterpret_cast<float *>(out) + base + j0), make_float4(r[0], r[1], r[2], r[3]));
        }
        return;
    }
    __syncthreads();
    const C n2 = sNorm[0], n0 = sNorm[1], cm = sNorm[2];
    for (int g = 0; g < kFinG; g++) {
        const int j0 = j00 + g * kFinThreads * 4;
        for (int k = 0; k < 4 && j0 + k < plane; k++) {
            const int j = j0 + k, y = j / W, x = j - y * W;
            const bool interior = y >= 1 && y < H - 1 && x >= 1 && x < W - 1;
            const C cv = (C)val[base + j];
            const C norm = interior ? (E[base + j] == 0 ? n2 : n0) : cv / cm;
            out[base + j] = (O)(cv * norm);
        }
    }
}

template <typename T, typename O>
__global__ void dee_convert_kernel(const T *__restrict__ in, O *__restrict__ out, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        out[i] = (O)in[i];
}

struct Layout {
    size_t offStats, offTab, offVal, offCl, offE, offActive, total;
};

// cuTensorMapEncodeTiled through the runtime's driver entry point (libmte.so does not link libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = [] {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            p = nullptr;
        cudaGetLastError();
        return reinterpret_cast<EncodeTiledFn>(p);
    }();
    return fn;
}

// [N, H, W] fp32 planes as a 3-D tensor map with a (XCOLS, XROWS, 1) box; out-of-bounds cells read as zero
static bool make_plane_map(CUtensorMap &m, const float *base, int N, int H, int W) {
    EncodeTiledFn fn = encode_tiled_fn();
    if (!fn || (W % 4) || H < 4 || W < 4 || (reinterpret_cast<uintptr_t>(base) & 15u)) return false;
    const cuuint64_t dims[3] = {(cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
    const cuuint64_t strides[2] = {(cuuint64_t)W * 4, (cuuint64_t)W * H * 4};
    const cuuint32_t box[3] = {(cuuint32_t)XCOLS, (cuuint32_t)XROWS, 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    return fn(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float *>(base), dims, strides, box, estr,
              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

static Layout layout(int N, int H, int W) {
    Layout L;
    size_t off = MTE_WS_HEADER_BYTES;
    L.offStats = off; off += align_up(sizeof(ImgStat) * (size_t)N, 256);
    L.offTab = off; off += align_up(sizeof(DeeTab), 256);
    L.offVal = off; off += align_up((size_t)N * H * W * sizeof(double), 256);
    L.offCl = off; off += align_up((size_t)N * H * W, 256);
    L.offE = off; off += align_up((size_t)N * H * W, 256);
    L.offActive = off; off += canny::hysteresis_scratch_bytes(N, H, W);
    L.total = off;
    return L;
}

template <typename T>
static int run(const T *prob, int N, int H, int W, int do_nms, int do_hyst, double t_low, double t_high,
               unsigned char *normals, void *out, int out_dtype, char *ws, const Layout &L, cudaStream_t st) {
    ImgStat *stats = reinterpret_cast<ImgStat *>(ws + L.offStats);
    T *val = reinterpret_cast<T *>(ws + L.offVal);
    unsigned char *cl = reinterpret_cast<unsigned char *>(ws + L.offCl);
    unsigned char *E = reinterpret_cast<unsigned char *>(ws + L.offE);
    const int tiles = ceil_div(W, TW) * ceil_div(H, TH) * N;
    cudaError_t e = cudaMemsetAsync(stats, 0, sizeof(ImgStat) * (size_t)N, st);
    if (e != cudaSuccess) return (int)e;
    // fp32 inputs are compared against fp32-rounded thresholds when no NMS ran (NumPy weak-scalar promotion:
    // tools.py:58-61 then sees a float32 array); after NMS the array is float64
    double lo = t_low, hi = t_high;
    if (!do_nms && sizeof(T) == 4) { lo = (double)(float)t_low; hi = (double)(float)t_high; }
    const bool wantVal = out != nullptr;
    T *nmsDst = wantVal ? val : nullptr;
    // NMS only, fp32 out of fp32 in (or fp64/fp64): write straight to the output
    if (wantVal && !do_hyst && ((out_dtype == MTE_F32 && sizeof(T) == 4) || (out_dtype == MTE_F64 && sizeof(T) == 8)))
        nmsDst = static_cast<T *>(out);
    DeeTab *tab = reinterpret_cast<DeeTab *>(ws + L.offTab);
    if (normals) dee_tables_kernel<<<1, 256, 0, st>>>(tab);  // 255 bisections, a few microseconds, no host state
    bool tma = false;
    if constexpr (sizeof(T) == 4) {
        CUtensorMap map;
        if (make_plane_map(map, reinterpret_cast<const float *>(prob), N, H, W)) {
            // indexed by NRM * 4 + NMS * 2 + HYST.  No entry 0: without normals the edges are asked for, and
            // mte_dee_postprocess rejects edges without NMS or hysteresis.
            static constexpr decltype(&dee_front_tma_kernel<true, true, true>) kFront[8] = {
                nullptr,
                dee_front_tma_kernel<false, false, true>, dee_front_tma_kernel<false, true, false>,
                dee_front_tma_kernel<false, true, true>, dee_front_tma_kernel<true, false, false>,
                dee_front_tma_kernel<true, false, true>, dee_front_tma_kernel<true, true, false>,
                dee_front_tma_kernel<true, true, true>};
            const int xt = ceil_div(W, XW) * ceil_div(H, XH) * N;
            const int v = (normals != nullptr) * 4 + (do_nms != 0) * 2 + (do_hyst && wantVal);
            kFront[v]<<<xt, kXThreads, 0, st>>>(map, tab, N, H, W, lo, hi, normals, reinterpret_cast<float *>(nmsDst), cl,
                                                E, stats);
            tma = true;
        }
    }
    if (!tma)
        dee_front_kernel<T><<<tiles, kThreads, 0, st>>>(tab, prob, N, H, W, do_nms, do_hyst && wantVal, lo, hi, normals,
                                                        nmsDst, cl, E, stats);
    MTE_RETURN_IF_CUDA_ERROR();
    if (!wantVal) return MTE_OK;
    const size_t n = (size_t)N * H * W;
    const int grid = (int)((n + 255) / 256 < (size_t)num_sms() * 16 ? (n + 255) / 256 : (size_t)num_sms() * 16);
    if (do_hyst) {
        int rc = canny::run_level_hysteresis(cl, E, N, H, W, 1, ws + L.offActive, st);
        if (rc) return rc;
        // the reference computes in float64 once NMS has run (its output array is float64), else in the input type
        auto finish = [&](auto computeType) {
            using C = decltype(computeType);
            // one image per blockIdx.y: batches beyond the grid's y limit go in slices
            for (int n0 = 0; n0 < N; n0 += 65535) {
                const int nn = N - n0 < 65535 ? N - n0 : 65535;
                const size_t po = (size_t)n0 * H * W;
                const dim3 fg((unsigned)ceil_div(H * W, kFinPx), (unsigned)nn);
                if (out_dtype == MTE_F64) dee_finish_kernel<T, C, double><<<fg, kFinThreads, 0, st>>>(val + po, E + po, nn, H, W, stats + n0, (double *)out + po);
                else dee_finish_kernel<T, C, float><<<fg, kFinThreads, 0, st>>>(val + po, E + po, nn, H, W, stats + n0, (float *)out + po);
            }
        };
        if (do_nms) finish(0.0);
        else finish(T(0));
        MTE_RETURN_IF_CUDA_ERROR();
    } else if (nmsDst == val) {
        // NMS only: the reference returns float64 whatever the input type (tools.py:15 np.zeros((H, W))); an output in
        // the input type was written in place above, so this converts into the other float type
        using O = std::conditional_t<sizeof(T) == 4, double, float>;
        dee_convert_kernel<T, O><<<grid, 256, 0, st>>>(val, static_cast<O *>(out), n);
        MTE_RETURN_IF_CUDA_ERROR();
    }
    return MTE_OK;
}

}  // namespace dee
}  // namespace mte

using namespace mte;

extern "C" size_t mte_dee_workspace_bytes(int N, int H, int W) {
    if (N < 1 || H < 1 || W < 1) return 0;
    return dee::layout(N, H, W).total;
}

extern "C" int mte_dee_postprocess(const void *prob, int in_dtype, int N, int H, int W, int do_nms, int do_hyst,
                                   double t_low, double t_high, uint8_t *normals_out, void *edges_out, int out_dtype,
                                   void *workspace, size_t ws_bytes, mte_stream_t stream) {
    if (!prob || !workspace) return MTE_ERR_NULL;
    if (!normals_out && !edges_out) return MTE_ERR_NULL;
    if (N < 1 || H < 1 || W < 1) return MTE_ERR_SHAPE;
    if (in_dtype != MTE_F32 && in_dtype != MTE_F64) return MTE_ERR_ARG;
    if (edges_out && out_dtype != MTE_F32 && out_dtype != MTE_F64) return MTE_ERR_ARG;
    if (edges_out && !do_nms && !do_hyst) return MTE_ERR_ARG;
    const dee::Layout L = dee::layout(N, H, W);
    if (ws_bytes < L.total) return MTE_ERR_WORKSPACE;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    char *ws = static_cast<char *>(workspace);
    if (in_dtype == MTE_F32)
        return dee::run<float>(static_cast<const float *>(prob), N, H, W, do_nms, do_hyst, t_low, t_high, normals_out,
                               edges_out, out_dtype, ws, L, st);
    return dee::run<double>(static_cast<const double *>(prob), N, H, W, do_nms, do_hyst, t_low, t_high, normals_out,
                            edges_out, out_dtype, ws, L, st);
}
