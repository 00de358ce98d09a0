// Edge-loss kernels (templates).  See edge_loss.cu for the host API and the reference map.
//
// Design (HBM-bound stencil + reduction, no tensor cores):
//  * one launch covers every image of up to 4 pyramid scales;
//  * a warp owns a strip of 32 lanes x VEC px (VEC=4: 128-bit coalesced loads); the strips of the
//    stencil kernels overlap by one lane on each side (two for the VEC=1 non-stash backward), so
//    horizontal neighbours always come from a warp shuffle and vertical ones from a rolling row window;
//  * forward (edge_loss_fwd_kernel): persistent warps, each over an equal, cost-balanced range of strip
//    rows fed by a cp.async shared-memory row ring: 3x3 responses -> pick by quantised normal -> sigmoid
//    -> soft-label BCE terms; warp sums -> per-image 2^32 fixed-point integer atomics -> the last CTA
//    (atomic ticket) computes the per-image class balance alpha and writes the loss: single launch, no
//    host sync, bit-reproducible run to run.  It also writes the grad map and, for directional
//    responses, a 1 B/px stash (picked direction + sign of the response);
//  * backward from the stash (edge_loss_bwd_ring_kernel at VEC=4 on the forward's unit ranges,
//    edge_loss_bwd_stash_kernel at VEC=1 on fixed work items): reads grad map, edge and stash, looks the
//    3x3 adjoint up in a 16-entry table and scatters it into three rolling output rows;
//  * backward without a stash (edge_loss_bwd_kernel, e.g. magnitude responses or a resized scale):
//    recomputes the responses from depth / edge / normal and gathers the 3x3 adjoint from registers +
//    shuffles.
#pragma once
#include <math.h>
#include <stdlib.h>

#include "common.cuh"

namespace mte {
namespace loss {

constexpr int kWarps = 8;
constexpr int kThreads = kWarps * 32;
constexpr int kAcc = 8;
enum { A_WP = 0, A_WN, A_SPU, A_SNU, A_SPM, A_SNM, A_SUMM, A_FLAGS };
enum { F_HAS0 = 1u, F_HAS1 = 2u, F_OTHER = 4u, F_NONFINITE = 8u };
enum { MODE_NONE = 0, MODE_MAG = 1, MODE_DIR = 2 };

constexpr int kBwdRH = 8;   // output rows per work item of edge_loss_bwd_kernel / edge_loss_bwd_stash_kernel
// the streaming (ring) kernels: warps per CTA, CTAs per SM, ring depths -- tuning knobs.  Measured on B200 at the
// config-3 loss shape (bench.py, us per fwd+bwd step): 2 CTAs x 8 warps, depths 8/6: 43.4; 1 CTA x 16 warps: depths
// 8/6 43.4, 7/5 41.7, 5/4 40.8, 4/4 39.9, 3/3 39.2, 3/2 38.5, 3/1 41.3; 24 warps 42.0.  Shallow rings win: deeper
// queues only add memory latency and let warps drift apart (the kernel ends with its slowest warp).
#ifndef MTE_LOSS_WARPS
#define MTE_LOSS_WARPS 16
#endif
#ifndef MTE_LOSS_MINB
#define MTE_LOSS_MINB 1
#endif
#ifndef MTE_FWD_D
#define MTE_FWD_D 3
#endif
#ifndef MTE_BWD_D
#define MTE_BWD_D 2
#endif
#ifndef MTE_LOSS_GRIDB
#define MTE_LOSS_GRIDB MTE_LOSS_MINB
#endif
// kRMinB caps the registers (launch bounds), kRGridB is the number of persistent CTAs launched per SM: launching
// fewer than fit leaves room for the CTAs of the NEXT kernel to become resident early (programmatic dependent launch)
constexpr int kRWarps = MTE_LOSS_WARPS, kRThreads = kRWarps * 32, kRMinB = MTE_LOSS_MINB, kRGridB = MTE_LOSS_GRIDB;
#ifndef MTE_SEGCOST_F
#define MTE_SEGCOST_F 4
#endif
#ifndef MTE_SEGCOST_B
#define MTE_SEGCOST_B 5
#endif
constexpr int kSegCost = MTE_SEGCOST_F;     // forward partition: cost of opening a segment, in rows
constexpr int kHaloLanes = 30;  // writing lanes of an overlapped strip (one halo lane per side)
// The backward needs the coefficient of the neighbouring pixel, i.e. depth two columns out: with
// VEC=1 that is two halo lanes per side.
__host__ __device__ constexpr int bwd_halo(int vec) { return vec == 1 ? 2 : 1; }
__host__ __device__ constexpr int bwd_lanes(int vec) { return 32 - 2 * bwd_halo(vec); }

constexpr float kEps = 0.001f;  // grad_loss.py:167,180
constexpr float kLn2 = 0.6931471805599453f;

struct ScaleP {
    const float *x, *e, *n, *m;
    float *g, *dx;
    unsigned char *stash;  // 1 B/px: bits 0-1 picked direction, bits 2-3 sign of the response (1:+ 2:- 0:zero)
    int B, H, W;
    int strips;
    int rowBlocks, items, ctasPerImage, ctaBase;  // work items of edge_loss_bwd_kernel / edge_loss_bwd_stash_kernel only
    int imgBase;
    int unitBase;  // forward / ring backward: first unit (strip row) of this scale in the global unit order
    float scaleWeight;
};

struct LossP {
    ScaleP s[MTE_MAX_SCALES];
    int nScales, totalCtas, totalImages;
    float T, weight, p2n;
    int totalUnits;                // forward / ring backward: units over all scales and images
    unsigned long long *accum;     // forward: [totalImages][kAcc] fixed-point (2^32) per-image sums, zero at launch
    unsigned *ticket;              // forward: [1] finished-CTA counter, [0] kept zero (both self-resetting)
    float *lossOut;         // [1+nScales]
    float *ctx;             // [totalImages] alpha, then per scale {coef, maskBinary}
    const float *gradLoss;  // bwd: [1+nScales]
};

// fp32-rounded k*pi/8, exactly the constants torch compares against (grad_loss.py:80-93)
#define MTE_B1 ((float)(1 * M_PI / 8))
#define MTE_B3 ((float)(3 * M_PI / 8))
#define MTE_B5 ((float)(5 * M_PI / 8))
#define MTE_B7 ((float)(7 * M_PI / 8))

// Quantised normal direction 0:h 1:rl 2:v 3:lr (grad_loss.py:80-93).  The reference bands are
// [B3,B5)->v [B1,B3)->rl [B5,B7)->lr for theta >= 0 and [-B5,-B3)->v [-B7,-B5)->rl [-B3,-B1)->lr for
// theta < 0, everything else (incl. NaN) -> h.  With u = |theta| the negative side is the mirrored
// table with the closed end on the other side, so u is stepped down one ulp there (u > B <=> pred(u) >= B)
// and four compares decide both signs exactly.
__device__ __forceinline__ int dir_index(float t) {
    const bool neg = t < 0.f;
    const int ub = (__float_as_int(t) & 0x7fffffff) - (neg ? 1 : 0);
    const float u = __int_as_float(ub);
    // count in floating point: FSET + FADD per limit (an integer count costs a predicated move pair each)
    const float n = ((u >= MTE_B1) ? 1.f : 0.f) + ((u >= MTE_B3) ? 1.f : 0.f) + ((u >= MTE_B5) ? 1.f : 0.f) +
                    ((u >= MTE_B7) ? 1.f : 0.f);
    const int ni = __float2int_rz(neg ? 4.f - n : n);
    return ni & 3;
}

// cond ? a : b as a real SELP: keeps ptxas from turning value selections into divergent branches
__device__ __forceinline__ float fsel(bool cond, float a, float b) {
    float r;
    asm("{\n\t.reg .pred p;\n\tsetp.ne.s32 p, %3, 0;\n\tselp.f32 %0, %1, %2, p;\n\t}" : "=f"(r) : "f"(a), "f"(b), "r"((int)cond));
    return r;
}

__device__ __forceinline__ float rcp_approx(float x) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
// 1/d correctly rounded for d in the normal range (two FMA Newton steps on MUFU.RCP), branch-free.
__device__ __forceinline__ float rcp_rn_normal(float d) {
    float r = rcp_approx(d);
    float e = fmaf(-d, r, 1.0f);
    r = fmaf(r, e, r);
    e = fmaf(-d, r, 1.0f);
    return fmaf(r, e, r);
}
// torch.clamp(min=1e-6) keeps a NaN (utils/depth.py:104-121), fmaxf would swallow it: max.NaN propagates
__device__ __forceinline__ float fmax_nan(float a, float b) {
    float r;
    asm("max.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
    return r;
}
__device__ __forceinline__ float inv_to_depth(float v) { return rcp_rn_normal(fmax_nan(v, 1e-6f)); }

// Forward: the loss is a mean over millions of terms; MUFU-accuracy sigmoid is far inside 1e-5.
__device__ __forceinline__ float ex2_approx(float x) {
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
// Backward: p(1-p)/(1-p+eps) amplifies the last bits of p where the sigmoid saturates, so p is
// computed the way eager PyTorch does (accurate expf, correctly rounded divide): the gradient then
// reproduces the reference's own rounding, not only the underlying math.
__device__ __forceinline__ float sigmoid_ref(float z) { return rcp_rn_normal(1.0f + expf(-z)); }

template <int VEC>
struct Row {
    float c[VEC];
    float l, r;
    __device__ __forceinline__ float at(int v) const { return v < 0 ? l : (v >= VEC ? r : c[v]); }
};

template <int VEC>
__device__ __forceinline__ void load_vec(float (&out)[VEC], const float *img, int row, int H, int W, int col0,
                                         bool cached) {
    const bool ok = (row >= 0) && (row < H) && (col0 >= 0) && (col0 < W);
    const float *p = img + (size_t)(ok ? row : 0) * W + (ok ? col0 : 0);
    if (VEC == 4) {
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (ok) v = cached ? ld_cached4(p) : ld_stream4(p);
        out[0] = v.x; out[1 % VEC] = v.y; out[2 % VEC] = v.z; out[3 % VEC] = v.w;
    } else {
        float v = 0.f;
        if (ok) v = cached ? __ldg(p) : __ldcs(p);
        out[0] = v;
    }
}

// Centre values of one depth row; out-of-image reads give 0 (the zero padding of conv2d(padding=1)).
template <int VEC, bool INV>
__device__ __forceinline__ void load_row(Row<VEC> &R, const float *img, int row, int H, int W, int col0) {
    load_vec<VEC>(R.c, img, row, H, W, col0, true);
    if (INV) {
        const bool ok = (row >= 0) && (row < H) && (col0 >= 0) && (col0 < W);
#pragma unroll
        for (int v = 0; v < VEC; v++) R.c[v] = ok ? inv_to_depth(R.c[v]) : 0.f;
    }
}
// Horizontal neighbours across the lane boundary (lanes 0 / 31 get don't-care values: they are halo lanes).
template <int VEC>
__device__ __forceinline__ void exchange_row(Row<VEC> &R) {
    R.l = __shfl_up_sync(MTE_FULL_MASK, R.c[VEC - 1], 1);
    R.r = __shfl_down_sync(MTE_FULL_MASK, R.c[0], 1);
}

// Separable parts of the four zero-padded 3x3 cross-correlations of grad_loss.py:20-31 at column v of
// the middle row:  c_v = P + dv,  c_h = R + Dm,  c_lr = P + R,  c_rl = R - P.
template <int VEC>
__device__ __forceinline__ void stencil_parts(const Row<VEC> &up, const Row<VEC> &mid, const Row<VEC> &dn, int v,
                                              float &P, float &R, float &Dm, float &dv) {
    const float tl = up.at(v - 1), tc = up.at(v), tr = up.at(v + 1);
    const float ml = mid.at(v - 1), mr = mid.at(v + 1);
    const float bl = dn.at(v - 1), bc = dn.at(v), br = dn.at(v + 1);
    P = (bl + bc + br) - (tl + tc + tr);
    Dm = mr - ml;
    R = (tr - tl) + Dm + (br - bl);
    dv = bc - tc;
}
// Response of direction k (0:h 1:rl 2:v 3:lr) by operand selection: no divergent branches.
__device__ __forceinline__ float pick_response(int k, float P, float R, float Dm, float dv) {
    const float a = fsel(k < 2, R, P);
    const float b = fsel(k == 0, Dm, fsel(k == 1, -P, fsel(k == 2, dv, R)));
    return a + b;
}

// ---------------------------------------------------------------------------
// Forward
// ---------------------------------------------------------------------------
// Persistent warps, each over one equal, cost-balanced range of strip rows (see fwd_segment), cut into segments at
// strip ends.  A segment's partial sums are reduced in the warp (fixed order) and added to per-image 2^32
// fixed-point int64 accumulators with integer atomics: the result does not depend on the order in which segments
// finish, so the loss is bit-reproducible without any per-CTA partial buffer or barrier.  The last CTA to finish
// (atomic ticket) folds the per-image sums into alpha and the loss.
constexpr double kFix = 4294967296.0;  // 2^32

// Run by the LAST CTA to finish (all of its warps): warp k folds scale k -- one image per lane, plain butterflies in
// a fixed order (reproducible) -- into alpha, the normalisers and the scale's loss; thread 0 then combines the scales.
// It is the serial tail of the kernel, so the dependent chain is kept short: one L2 round trip for the sums, three
// butterflies, two divisions.
template <bool MASK>
static __device__ __forceinline__ void finalize_loss(const LossP &P, double *sLoss /* [MTE_MAX_SCALES] shared */) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int k = warp; k < P.nScales; k += kRWarps) {
        const ScaleP &S = P.s[k];
        const double npix = (double)S.H * (double)S.W;
        double sumM = 0.0;
        unsigned fl = 0;
        // the mask's value set and sum decide the normaliser before the per-image pass; the non-finite flag (a NaN /
        // Inf anywhere in the scale's inputs or sums: the reference's loss is NaN then) rides in the same word
        for (int base = 0; base < S.B; base += 32) {
            const int i = base + lane;
            const unsigned long long *a = P.accum + (size_t)(S.imgBase + i) * kAcc;
            const bool in = i < S.B;
            if (MASK) sumM += in ? (double)(long long)__ldcg(a + A_SUMM) / kFix : 0.0;
            fl |= in ? (unsigned)__ldcg(a + A_FLAGS) : 0u;
        }
        if (MASK) sumM = warp_sum(sumM);
        fl = warp_or(fl);
        const bool nonFinite = (fl & F_NONFINITE) != 0u;
        fl &= ~(unsigned)F_NONFINITE;
        // grad_loss.py:183-187: the mask only masks when its value set is exactly {0,1}
        const bool binary = MASK && fl == (F_HAS0 | F_HAS1);
        // one image per lane; the three sums are independent butterflies (they overlap), the degenerate
        // "no negatives anywhere" variant (all alpha = 1, grad_loss.py:175-176) rides along as acc1
        double acc = 0.0, acc1 = 0.0, wnSum = 0.0;
        for (int base = 0; base < S.B; base += 32) {
            const int i = base + lane;
            if (i < S.B) {
                unsigned long long *a = P.accum + (size_t)(S.imgBase + i) * kAcc;
                const double wp = (double)(long long)__ldcg(a + A_WP) / kFix;
                const double wn = MASK ? (double)(long long)__ldcg(a + A_WN) / kFix : (npix - wp);
                const double sp = (double)(long long)__ldcg(a + (binary ? A_SPM : A_SPU)) / kFix;
                const double sn = (double)(long long)__ldcg(a + (binary ? A_SNM : A_SNU)) / kFix;
                const float alpha = (float)(wn / (wp + wn));  // grad_loss.py:178
                P.ctx[S.imgBase + i] = alpha;
                acc += -(double)P.p2n * (double)alpha * sp - (1.0 - (double)alpha) * sn;
                acc1 += -(double)P.p2n * sp;
                wnSum += wn;
#pragma unroll
                for (int q = 0; q < kAcc; q++)
                    if (MASK || q == A_WP || q == A_SPU || q == A_SNU || q == A_FLAGS) a[q] = 0ull;  // leave the accumulators clean
            }
        }
        acc = warp_sum(acc);
        acc1 = warp_sum(acc1);
        wnSum = warp_sum(wnSum);
        if (wnSum == 0.0) {
            acc = acc1;
            for (int base = 0; base < S.B; base += 32)
                if (base + lane < S.B) P.ctx[S.imgBase + base + lane] = 1.0f;
        }
        acc *= (double)kLn2;
        const double valid = binary ? sumM : npix * (double)S.B;
        const double lossK = nonFinite ? (double)__int_as_float(0x7fc00000) : (double)P.weight * (acc / valid);
        if (lane == 0) {
            sLoss[k] = lossK;
            P.lossOut[1 + k] = (float)lossK;
            P.ctx[P.totalImages + 2 * k] = (float)((double)P.weight / valid);
            P.ctx[P.totalImages + 2 * k + 1] = binary ? 1.0f : 0.0f;
        }
    }
}

// One depth row as the stencils consume it: centre values plus the horizontal 3-sum and difference, computed once
// when the row enters the window and reused by the three output rows it takes part in.
template <int VEC>
struct PRow {
    float c[VEC], s3[VEC], d[VEC];
};
template <int VEC, int MODE>
__device__ __forceinline__ void prep_row(PRow<VEC> &R, const float (&x)[VEC]) {
#pragma unroll
    for (int v = 0; v < VEC; v++) R.c[v] = x[v];
    if (MODE != MODE_NONE) {
        // horizontal neighbours across the lane boundary (lanes 0 / 31 are halo lanes: their outer values are unused)
        const float l = __shfl_up_sync(MTE_FULL_MASK, x[VEC - 1], 1);
        const float r = __shfl_down_sync(MTE_FULL_MASK, x[0], 1);
#pragma unroll
        for (int v = 0; v < VEC; v++) {
            const float xl = v == 0 ? l : x[(v + VEC - 1) % VEC];
            const float xr = v == VEC - 1 ? r : x[(v + 1) % VEC];
            R.s3[v] = (xl + x[v]) + xr;
            R.d[v] = xr - xl;
        }
    }
}

// base + 4 * off as ONE 64-bit multiply-add (opaque to the optimiser, which otherwise re-associates the plane
// offset into every access)
template <typename T>
__device__ __forceinline__ T *elem_addr(T *base, unsigned off) {
    unsigned long long a;
    asm("mad.wide.u32 %0, %1, 4, %2;" : "=l"(a) : "r"(off), "l"((unsigned long long)base));
    return reinterpret_cast<T *>(a);
}

// Directional response + stash code of one pixel with the instruction selection pinned (the compiler's version of
// the same logic spends ~10 more instructions per pixel on predicate spills and integer re-materialisation):
//   band compares f_k = [u >= B_k] (nested) on the ulp-stepped u = |theta| (see dir_index) -> X = f1^f5, Y = f3^f7
//   bit0 = X^Y (odd count), bit1 = theta<0 ? X : Y (the mirrored table) ; direction 0:h 1:rl 2:v 3:lr
//   c = (bit1 ? Pv : Rh) + (bit1 ? (bit0 ? Rh : dv) : (bit0 ? -Pv : Dm))
//   code = direction | 4 << signbit(c)   (bits 2-3: 1 = "+", 2 = "-"; a zero response is recognised by the
//   backward from the grad map itself, |c| == 0)
__device__ __forceinline__ void pick_directional(float th, float Pv, float Rh, float Dm, float dv, float &c,
                                                 unsigned &code) {
    asm("{\n\t"
        ".reg .pred n, x, y, b0, b1, t1, t2;\n\t"
        ".reg .b32 ub, sg, cd;\n\t"
        ".reg .f32 a, bh, bl, b, np;\n\t"
        "and.b32 ub, %2, 0x7fffffff;\n\t"
        "setp.lt.f32 n, %2, 0f00000000;\n\t"
        "@n add.s32 ub, ub, -1;\n\t"
        "setp.ge.f32 x, ub, %9;\n\t"
        "setp.ge.xor.f32 x, ub, %7, x;\n\t"
        "setp.ge.f32 y, ub, %10;\n\t"
        "setp.ge.xor.f32 y, ub, %8, y;\n\t"
        "xor.pred b0, x, y;\n\t"
        "and.pred t1, x, n;\n\t"
        "not.pred t2, n;\n\t"
        "and.pred t2, y, t2;\n\t"
        "or.pred b1, t1, t2;\n\t"
        "selp.f32 a, %3, %4, b1;\n\t"
        "neg.f32 np, %3;\n\t"
        "selp.f32 bh, %4, %6, b0;\n\t"
        "selp.f32 bl, np, %5, b0;\n\t"
        "selp.f32 b, bh, bl, b1;\n\t"
        "add.f32 %0, a, b;\n\t"
        "selp.u32 cd, 6, 4, b1;\n\t"
        "@b0 add.u32 cd, cd, 1;\n\t"
        "mov.b32 sg, %0;\n\t"
        "shr.u32 sg, sg, 31;\n\t"
        "mad.lo.u32 %1, sg, 4, cd;\n\t"
        "}"
        : "=&f"(c), "=r"(code)
        : "f"(th), "f"(Pv), "f"(Rh), "f"(Dm), "f"(dv), "f"(MTE_B1), "f"(MTE_B3), "f"(MTE_B5), "f"(MTE_B7));
}

__device__ __forceinline__ float lg2_approx(float x) {  // arguments here are >= 1e-3: no denormal path needed
    float r;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

// ---- programmatic dependent launch (PDL): the kernels are launched with programmatic stream serialisation, so their
// launch latency, CTA scheduling and index prologue overlap the tail of the previous kernel in the stream / graph;
// pdl_wait() blocks until that kernel has completed and its writes are visible and precedes every global access.
// (Measured on B200 inside the bench's CUDA graphs: no difference with MTE_NO_PDL=1 -- a 512-thread CTA at 96
// registers leaves no room for a dependent CTA to become resident early, and register-capped variants that do leave
// room lose more than the overlap gains.  Kept because it is free and helps behind short foreign kernels.)
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

template <typename K>
static void launch_pdl(K kernel, int grid, int block, int smem, cudaStream_t st, const LossP &P) {
    const bool noPdl = debug_knob("MTE_NO_PDL") != nullptr;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3((unsigned)block);
    cfg.dynamicSmemBytes = (size_t)smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = noPdl ? 0 : 1;
    cudaLaunchKernelEx(&cfg, kernel, P);
}

// ---- asynchronous global -> shared row ring (cp.async / LDGSTS) ----------------------------------------------
// Every lane copies its own VEC*4 bytes of a row into its own slot of the warp's ring and later reads only that slot
// back, so no cross-lane synchronisation is needed: cp.async.wait_group orders a thread's own copies.  The ring
// keeps kRingDepth rows per warp in flight without holding registers (a register ring of that depth would not fit).
template <int VEC>
__device__ __forceinline__ void cp_async_vec(unsigned dst, const void *src, bool ok) {  // !ok: zero-fill
    const unsigned n = ok ? VEC * 4u : 0u;
    if (VEC == 4) asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(n) : "memory");
    else asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(dst), "l"(src), "r"(n) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
template <int VEC>
__device__ __forceinline__ void lds_vec(float (&out)[VEC], const unsigned char *p) {
    if (VEC == 4) {
        const float4 v = *reinterpret_cast<const float4 *>(p);
        out[0] = v.x; out[1 % VEC] = v.y; out[2 % VEC] = v.z; out[3 % VEC] = v.w;
    } else {
        out[0] = *reinterpret_cast<const float *>(p);
    }
}

__host__ __device__ constexpr int fwd_planes(int mode, bool mask) { return 2 + (mode == MODE_DIR ? 1 : 0) + (mask ? 1 : 0); }
constexpr int kFwdRingDepth = MTE_FWD_D;
__host__ __device__ constexpr int fwd_smem_bytes(int vec, int mode, bool mask) {
    return kRWarps * kFwdRingDepth * fwd_planes(mode, mask) * 32 * vec * 4;
}

// Forward work decomposition: the unit is one row of one strip (32 lanes x VEC px, LANES of them writing) of one
// image of one scale; units are ordered scale, image, strip, row and every warp of the persistent grid owns one
// contiguous, equally long range of them (the cost of a unit does not depend on its content), cut into segments
// at strip ends.  A segment streams its rows through a 3-row register window fed by the shared-memory row ring.
template <int VEC, int MODE, bool MASK, bool INV, bool SIG>
__device__ __forceinline__ void fwd_segment(const LossP &P, const ScaleP &S, int img, int strip, int row0, int nrows,
                                            int lane, unsigned char *ring, float (&la)[kAcc - 1], unsigned &lflags,
                                            float &poison) {
    constexpr int D = kFwdRingDepth;
    constexpr int NPL = fwd_planes(MODE, MASK);
    constexpr unsigned PLB = 32 * VEC * 4;     // bytes of one plane row in a slot
    constexpr unsigned SLB = NPL * PLB;        // bytes of a slot
    constexpr int OFF = (MODE == MODE_NONE) ? 0 : 1;
    constexpr int LANES = (MODE == MODE_NONE) ? 32 : kHaloLanes;
    // out-of-image depth reads as 0 (zero padding of conv2d): the copies zero-fill; with the fused inv2depth the
    // fill must be a huge inverse depth whose reciprocal flushes to exactly 0, selected when the row is consumed
    constexpr float kFill = INV ? 3.0e38f : 0.f;
    const int H = S.H;
    const unsigned W = (unsigned)S.W;
    const int col0 = (strip * LANES + lane - OFF) * VEC;
    const bool colOk = col0 >= 0 && col0 < (int)W;
    const bool writer = colOk && (MODE == MODE_NONE || (lane >= 1 && lane <= kHaloLanes));
    // per-lane plane pointers at (row 0, clamped col0); rows are reached with one 32-bit element offset shared by
    // all planes (one IMAD.WIDE per access)
    const size_t lo = (size_t)img * H * W + (colOk ? col0 : 0);
    const float *xP = S.x + lo, *eP = S.e + lo, *nP = S.n + lo, *mP = S.m + lo;
    float *gP = S.g + lo;
    unsigned char *sP = S.stash + lo;
    const bool writeG = writer && S.g != nullptr, writeS = writer && (MODE == MODE_DIR) && S.stash != nullptr;
    const float kT = P.T * 1.4426950408889634f;
    unsigned char *slot0 = ring + lane * (VEC * 4);
    const unsigned ringS = (unsigned)__cvta_generic_to_shared(slot0);
    constexpr int PL_E = 1, PL_N = 2, PL_M = (MODE == MODE_DIR) ? 3 : 2;

    // copies of everything output row j needs that is not in the window yet: depth row row0 + j + OFF, target rows
    // row0 + j (writer lanes only; the others never look at their slots)
    auto issue = [&](unsigned so, int j) {
        const int rx = row0 + j + OFF;
        cp_async_vec<VEC>(ringS + so, elem_addr(xP, (unsigned)min(rx, H - 1) * W), colOk && rx < H);
        if (writer) {
            const unsigned ro = (unsigned)(row0 + j) * W;
            cp_async_vec<VEC>(ringS + so + PL_E * PLB, elem_addr(eP, ro), true);
            if (MODE == MODE_DIR) cp_async_vec<VEC>(ringS + so + PL_N * PLB, elem_addr(nP, ro), true);
            if (MASK) cp_async_vec<VEC>(ringS + so + PL_M * PLB, elem_addr(mP, ro), true);
        }
    };
    auto pad_x = [&](float (&x)[VEC], int row) {
        if (INV) {
            const bool ok = colOk && row >= 0 && row < H;
#pragma unroll
            for (int v = 0; v < VEC; v++) x[v] = ok ? x[v] : kFill;
        }
    };
    auto to_depth = [&](float (&x)[VEC]) {
        if (INV) {
#pragma unroll
            for (int v = 0; v < VEC; v++) x[v] = inv_to_depth(x[v]);
        }
    };

    // x * 0 is NaN exactly when x is NaN or +-Inf: one FFMA per loaded pixel carries "a non-finite prediction was
    // seen" to the end of the segment (the reference's conv2d turns any such pixel into a NaN loss: 0 * inf)
    auto taint = [&](const float (&x)[VEC]) {
#pragma unroll
        for (int v = 0; v < VEC; v++) poison = fmaf(x[v], 0.f, poison);
    };
    PRow<VEC> win[3];  // win[d % 3] holds depth row row0 - OFF + d
    float xa[VEC], xc[VEC];
#pragma unroll
    for (int v = 0; v < VEC; v++) { xa[v] = 0.f; xc[v] = 0.f; }
    if (MODE != MODE_NONE) {  // the two rows that open the window: plain loads
        if (colOk && row0 >= 1) {
            const float *p = elem_addr(xP, (unsigned)(row0 - 1) * W);
            if (VEC == 4) { const float4 v = ld_cached4(p); xa[0] = v.x; xa[1 % VEC] = v.y; xa[2 % VEC] = v.z; xa[3 % VEC] = v.w; }
            else xa[0] = __ldg(p);
        }
        if (colOk) {
            const float *p = elem_addr(xP, (unsigned)row0 * W);
            if (VEC == 4) { const float4 v = ld_cached4(p); xc[0] = v.x; xc[1 % VEC] = v.y; xc[2 % VEC] = v.z; xc[3 % VEC] = v.w; }
            else xc[0] = __ldg(p);
        }
    }
#pragma unroll
    for (int k = 0; k < D; k++) {
        if (k < nrows) issue(k * SLB, k);
        cp_async_commit();
    }
    if (MODE != MODE_NONE) {
        pad_x(xa, row0 - 1);
        pad_x(xc, row0);
        to_depth(xa);
        to_depth(xc);
        taint(xa);
        taint(xc);
        prep_row<VEC, MODE>(win[0], xa);
        prep_row<VEC, MODE>(win[1], xc);
    }
    unsigned so = 0;  // ring slot (byte offset) of the row being consumed
#pragma unroll 1
    for (int jj = 0; jj < nrows; jj += 3) {
#pragma unroll
        for (int u = 0; u < 3; u++) {
            const int j = jj + u;
            if (j < nrows) {  // warp-uniform
                cp_async_wait<D - 1>();
                float xn[VEC], e[VEC], th[VEC], m[VEC];
                lds_vec<VEC>(xn, slot0 + so);
                lds_vec<VEC>(e, slot0 + so + PL_E * PLB);
                if (MODE == MODE_DIR) lds_vec<VEC>(th, slot0 + so + PL_N * PLB);
                if (MASK) lds_vec<VEC>(m, slot0 + so + PL_M * PLB);
                if (j + D < nrows) issue(so, j + D);  // refill the slot just read
                cp_async_commit();
                so = (so + SLB == D * SLB) ? 0u : so + SLB;
                PRow<VEC> &dn = win[(MODE == MODE_NONE) ? 0 : (u + 2) % 3];
                pad_x(xn, row0 + j + OFF);
                to_depth(xn);
                taint(xn);
                prep_row<VEC, MODE>(dn, xn);
                const PRow<VEC> &up = win[(MODE == MODE_NONE) ? 0 : u % 3];
                const PRow<VEC> &mid = win[(MODE == MODE_NONE) ? 0 : (u + 1) % 3];
                float g[VEC];
                unsigned code = 0u;
#pragma unroll
                for (int v = 0; v < VEC; v++) {
                    if (MODE == MODE_NONE) {
                        g[v] = dn.c[v];
                    } else {
                        // separable parts of the four zero-padded 3x3 cross-correlations of grad_loss.py:20-31:
                        // c_v = Pv + dv, c_h = Rh + Dm, c_lr = Pv + Rh, c_rl = Rh - Pv
                        const float Pv = dn.s3[v] - up.s3[v];
                        const float Dm = mid.d[v];
                        const float Rh = (up.d[v] + Dm) + dn.d[v];
                        const float dv = dn.c[v] - up.c[v];
                        if (MODE == MODE_MAG) {
                            const float cv = Pv + dv, ch = Rh + Dm;
                            g[v] = sqrtf(cv * cv + ch * ch + 1e-6f);
                        } else {
                            float c;
                            unsigned cd;
                            pick_directional(th[v], Pv, Rh, Dm, dv, c, cd);
                            g[v] = fabsf(c);
                            code |= cd << (8 * v);
                        }
                    }
                    const float p = SIG ? rcp_approx(1.0f + ex2_approx(fmaf(g[v], -1.4426950408889634f, kT))) : g[v];
                    const float ee = e[v];
                    const float ne = 1.0f - ee;
                    const float lp = lg2_approx(p + kEps);
                    const float ln = lg2_approx((1.0f - p) + kEps);
                    la[A_SPU] = fmaf(ee, lp, la[A_SPU]);
                    la[A_SNU] = fmaf(ne, ln, la[A_SNU]);
                    if (MASK) {
                        const float mm = m[v];
                        la[A_WP] = fmaf(ee, mm, la[A_WP]);
                        la[A_WN] = fmaf(ne, mm, la[A_WN]);
                        la[A_SUMM] += mm;
                        const bool keep = mm != 0.f;
                        la[A_SPM] += keep ? ee * lp : 0.f;
                        la[A_SNM] += keep ? ne * ln : 0.f;
                        lflags |= (mm == 0.f) ? F_HAS0 : ((mm == 1.f) ? F_HAS1 : F_OTHER);
                    } else {
                        la[A_WP] += ee;
                    }
                }
                const unsigned ro = (unsigned)(row0 + j) * W;
                if (writeG) {
                    float *gp = elem_addr(gP, ro);
                    if (VEC == 4) st_stream4(gp, make_float4(g[0], g[1 % VEC], g[2 % VEC], g[3 % VEC]));
                    else __stcs(gp, g[0]);
                }
                if (writeS) {
                    if (VEC == 4) __stcs(reinterpret_cast<unsigned *>(sP + ro), code);
                    else __stcs(sP + ro, (unsigned char)code);
                }
            }
        }
    }
    cp_async_wait<0>();
    if (!writer) {  // halo / out-of-image lanes: discard (select, no NaN propagation)
#pragma unroll
        for (int k = 0; k < kAcc - 1; k++) la[k] = 0.f;
        lflags = 0;
    }
}

// The next segment of a warp's unit range [u0, u1) (u0 advances past it).  A strip is H rows plus COST virtual units
// that stand for the cost of opening a segment (window prologue + pipeline fill), so ranges that span several strips
// are charged for it; nrows <= 0: the range held only virtual units (img and strip are left unset).
struct UnitSeg {
    int si, img, strip, row0, nrows;
};
template <int COST>
__device__ __forceinline__ UnitSeg unit_segment(const LossP &P, int &u0, int u1) {
    UnitSeg s;
    s.si = 0;
#pragma unroll
    for (int k = 1; k < MTE_MAX_SCALES; k++)
        if (k < P.nScales && u0 >= P.s[k].unitBase) s.si = k;
    const ScaleP &S = P.s[s.si];
    const int local = u0 - S.unitBase;
    const int HV = S.H + COST;
    const int t = local / HV;  // (image, strip)
    const int r = local - t * HV;
    const int take = min(HV - r, u1 - u0);
    s.row0 = max(r - COST, 0);
    s.nrows = max(r + take - COST, 0) - s.row0;
    u0 += take;
    if (s.nrows > 0) {
        s.img = t / S.strips;
        s.strip = t - s.img * S.strips;
    }
    return s;
}

template <int VEC, int MODE, bool MASK, bool INV, bool SIG>
__global__ void __launch_bounds__(kRThreads, kRMinB) edge_loss_fwd_kernel(const __grid_constant__ LossP P) {
    extern __shared__ __align__(16) unsigned char fwdRing[];
    const int lane = threadIdx.x & 31;
    const int nWarps = gridDim.x * kRWarps;
    const int gw = blockIdx.x * kRWarps + (threadIdx.x >> 5);
    unsigned char *ring = fwdRing + (threadIdx.x >> 5) * (fwd_smem_bytes(VEC, MODE, MASK) / kRWarps);
    int u0 = (int)((long long)P.totalUnits * gw / nWarps);
    const int u1 = (int)((long long)P.totalUnits * (gw + 1) / nWarps);
    pdl_launch_dependents();
    pdl_wait();
    while (u0 < u1) {
        const UnitSeg sg = unit_segment<kSegCost>(P, u0, u1);
        if (sg.nrows <= 0) continue;
        const ScaleP &S = P.s[sg.si];
        float la[kAcc - 1];
#pragma unroll
        for (int k = 0; k < kAcc - 1; k++) la[k] = 0.f;
        unsigned lflags = 0;
        float poison = 0.f;
        fwd_segment<VEC, MODE, MASK, INV, SIG>(P, S, sg.img, sg.strip, sg.row0, sg.nrows, lane, ring, la, lflags, poison);
        bool bad = __any_sync(MTE_FULL_MASK, !(poison == 0.f));
        // order-independent accumulation: warp tree (fixed) -> 2^32 fixed point -> integer atomics
        unsigned long long *acc = P.accum + (size_t)(S.imgBase + sg.img) * kAcc;
#pragma unroll
        for (int k = 0; k < kAcc - 1; k++) {
            if (MASK || k == A_WP || k == A_SPU || k == A_SNU) {
                const float v = warp_sum(la[k]);
                bad = bad || !isfinite(v);  // __double2ll_rn(NaN / Inf) would be a finite garbage contribution
                if (lane == 0) atomicAdd(acc + k, (unsigned long long)__double2ll_rn((double)v * kFix));
            }
        }
        if (MASK) lflags = warp_or(lflags);
        if (bad) lflags |= F_NONFINITE;
        if (lane == 0 && lflags) atomicOr(acc + A_FLAGS, (unsigned long long)lflags);
    }
    // the last CTA to leave finalises (its warps share the scales)
    __shared__ double sLoss[MTE_MAX_SCALES];
    __shared__ int sLast;
    // grid-wide "last CTA" detection in the cooperative-groups grid-sync style: the CTA barrier orders every warp's
    // accumulator atomics before thread 0's cumulative fence + ticket
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        sLast = atomicAdd(P.ticket + 1, 1u) == gridDim.x - 1u;
        __threadfence();
    }
    __syncthreads();
    if (sLast) {
        finalize_loss<MASK>(P, sLoss);
        __syncthreads();
        if (threadIdx.x == 0) {
            double total = 0.0;
            for (int k = 0; k < P.nScales; k++) total += (double)P.s[k].scaleWeight * sLoss[k];
            P.lossOut[0] = (float)total;
            P.ticket[0] = 0u;  // leave the workspace header clean for the next launch
            P.ticket[1] = 0u;
        }
    }
}

// ---------------------------------------------------------------------------
// Backward
// ---------------------------------------------------------------------------
// Adjoint coefficients of one response pixel n: its contribution to the 3x3 neighbourhood is U / V
// on the two diagonals, A2 above/below, C2 left/right -- from
// K_d[a][b] = alpha*a*(1+beta*(1-|b|)) + gamma*b*(1+beta*(1-|a|)),  a,b in {-1,0,1}.
struct Coef {
    float U, V, A2, C2;
};

template <int VEC>
struct CoefRow {
    Coef c[VEC];
    Coef l, r;
    __device__ __forceinline__ const Coef &at(int v) const { return v < 0 ? l : (v >= VEC ? r : c[v]); }
};

struct BwdImg {
    float cp, cn;  // -G*coef*lambda*alpha , G*coef*(1-alpha)
    bool maskBinary;
};

template <bool MASK, bool SIG>
__device__ __forceinline__ float dloss_dg(float g, float ee, float mm, const BwdImg &I, float T) {
    const float p = SIG ? sigmoid_ref(g - T) : g;
    const float q = 1.0f - p;
    float d = I.cp * ee * rcp_approx(p + kEps) + I.cn * (1.0f - ee) * rcp_approx(q + kEps);
    if (MASK) d = (I.maskBinary && mm == 0.f) ? 0.f : d;
    return SIG ? d * p * q : d;
}

// Coefficients of image img of scale si: the upstream gradient of the total and of the scale's loss, the scale's
// normaliser and mask flag and the image's alpha, all left in ctx by the forward.
template <bool MASK>
__device__ __forceinline__ BwdImg bwd_img(const LossP &P, const ScaleP &S, int si, int img) {
    const float G = __ldg(P.gradLoss) * S.scaleWeight + __ldg(P.gradLoss + 1 + si);
    const float coef = __ldg(P.ctx + P.totalImages + 2 * si) * G;
    const float alpha = __ldg(P.ctx + S.imgBase + img);
    BwdImg I;
    I.cp = -coef * P.p2n * alpha;
    I.cn = coef * (1.0f - alpha);
    I.maskBinary = MASK && (__ldg(P.ctx + P.totalImages + 2 * si + 1) != 0.f);
    return I;
}

template <int VEC, int MODE, bool MASK, bool INV, bool SIG>
__global__ void __launch_bounds__(kThreads, 2) edge_loss_bwd_kernel(const __grid_constant__ LossP P) {
    static_assert(MODE != MODE_NONE, "pointwise backward has its own kernel");
    constexpr int RH = kBwdRH;
    constexpr int PD = 2;  // rows prefetched ahead of the one being consumed (register budget: 128)
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int si = 0;
#pragma unroll
    for (int k = 1; k < MTE_MAX_SCALES; k++)
        if (k < P.nScales && (int)blockIdx.x >= P.s[k].ctaBase) si = k;
    const ScaleP &S = P.s[si];
    const int local = blockIdx.x - S.ctaBase;
    const int img = local / S.ctasPerImage;
    const int item0 = (local - img * S.ctasPerImage) * kWarps + warp;
    const int H = S.H, W = S.W;
    const BwdImg I = bwd_img<MASK>(P, S, si, img);

    for (int item = item0; item < S.items; item += S.ctasPerImage * kWarps) {  // warp-uniform
    const int strip = item / S.rowBlocks;
    const int rb = item - strip * S.rowBlocks;
    const int row0 = rb * RH;
    // writing lanes in the middle of the strip; the outer lanes only supply halo depth / coefficients
    constexpr int HALO = bwd_halo(VEC), LANES = bwd_lanes(VEC);
    const int col0 = (strip * LANES + lane - HALO) * VEC;
    const size_t plane = (size_t)img * H * W;
    const float *x = S.x + plane;
    const bool colOk = col0 >= 0 && col0 < W;
    const bool writer = lane >= HALO && lane < HALO + LANES && colOk;

    // Software pipeline over coefficient rows j = 0..RH+1 (image row row0-1+j).  Depth rows are indexed
    // d = 0..RH+3 (image row row0-2+d); coefficient row j needs depth rows j, j+1, j+2.
    Row<VEC> xr[3];                       // rolling depth window, xr[d % 3]
    Row<VEC> pfx[PD];                     // prefetched depth rows (centre values only)
    float pfe[PD][VEC], pft[PD][VEC], pfm[PD][VEC];
    float oacc[3][VEC];                   // rolling output accumulators, oacc[o % 3]
    load_row<VEC, INV>(xr[0], x, row0 - 2, H, W, col0);
    load_row<VEC, INV>(xr[1], x, row0 - 1, H, W, col0);
#pragma unroll
    for (int k = 0; k < PD; k++) {
        load_row<VEC, INV>(pfx[k], x, row0 + k, H, W, col0);
        load_vec<VEC>(pfe[k], S.e + plane, row0 - 1 + k, H, W, col0, false);
        if (MODE == MODE_DIR) load_vec<VEC>(pft[k], S.n + plane, row0 - 1 + k, H, W, col0, false);
        if (MASK) load_vec<VEC>(pfm[k], S.m + plane, row0 - 1 + k, H, W, col0, false);
    }
    exchange_row<VEC>(xr[0]);
    exchange_row<VEC>(xr[1]);
#pragma unroll
    for (int o = 0; o < 3; o++)
#pragma unroll
        for (int v = 0; v < VEC; v++) oacc[o][v] = 0.f;

#pragma unroll
    for (int j = 0; j < RH + 2; j++) {
        const int row = row0 - 1 + j;
        // consume the prefetched row, refill the slot PD rows ahead
        float e[VEC], th[VEC], m[VEC];
        xr[(j + 2) % 3] = pfx[j % PD];
#pragma unroll
        for (int v = 0; v < VEC; v++) {
            e[v] = pfe[j % PD][v];
            th[v] = (MODE == MODE_DIR) ? pft[j % PD][v] : 0.f;
            m[v] = MASK ? pfm[j % PD][v] : 1.f;
        }
        if (j + PD < RH + 2) {
            load_row<VEC, INV>(pfx[j % PD], x, row0 + j + PD, H, W, col0);
            load_vec<VEC>(pfe[j % PD], S.e + plane, row + PD, H, W, col0, false);
            if (MODE == MODE_DIR) load_vec<VEC>(pft[j % PD], S.n + plane, row + PD, H, W, col0, false);
            if (MASK) load_vec<VEC>(pfm[j % PD], S.m + plane, row + PD, H, W, col0, false);
        }
        exchange_row<VEC>(xr[(j + 2) % 3]);
        const Row<VEC> &up = xr[j % 3], &mid = xr[(j + 1) % 3], &dn = xr[(j + 2) % 3];
        const bool live = colOk && row >= 0 && row < H;
        CoefRow<VEC> C;
#pragma unroll
        for (int v = 0; v < VEC; v++) {
            float sP, sR, sDm, sdv;
            stencil_parts<VEC>(up, mid, dn, v, sP, sR, sDm, sdv);
            Coef k;
            if (MODE == MODE_MAG) {
                const float cv = sP + sdv, ch = sR + sDm;
                const float g = sqrtf(cv * cv + ch * ch + 1e-6f);
                const float d = dloss_dg<MASK, SIG>(g, e[v], m[v], I, P.T);
                const float rg = d * rcp_rn_normal(g);
                const float sv = rg * cv, sh = rg * ch;
                k.U = sv + sh; k.V = sv - sh; k.A2 = 2.f * sv; k.C2 = 2.f * sh;
            } else {
                const int di = dir_index(th[v]);
                const float c = pick_response(di, sP, sR, sDm, sdv);
                const float d = dloss_dg<MASK, SIG>(fabsf(c), e[v], m[v], I, P.T);
                const float s = fsel(c > 0.f, d, fsel(c < 0.f, -d, 0.f));
                const float s2 = 2.f * s;
                // h: U=s V=-s A2=0 C2=2s | rl: U=0 V=-2s A2=-s C2=s | v: U=s V=s A2=2s C2=0 | lr: U=2s V=0 A2=s C2=s
                k.U = fsel(di == 1, 0.f, fsel(di == 3, s2, s));
                k.V = fsel(di == 0, -s, fsel(di == 1, -s2, fsel(di == 2, s, 0.f)));
                k.A2 = fsel(di == 0, 0.f, fsel(di == 1, -s, fsel(di == 2, s2, s)));
                k.C2 = fsel(di == 0, s2, fsel(di == 2, 0.f, s));
            }
            C.c[v].U = live ? k.U : 0.f;
            C.c[v].V = live ? k.V : 0.f;
            C.c[v].A2 = live ? k.A2 : 0.f;
            C.c[v].C2 = live ? k.C2 : 0.f;
        }
        C.l.U = __shfl_up_sync(MTE_FULL_MASK, C.c[VEC - 1].U, 1);
        C.l.V = __shfl_up_sync(MTE_FULL_MASK, C.c[VEC - 1].V, 1);
        C.l.C2 = __shfl_up_sync(MTE_FULL_MASK, C.c[VEC - 1].C2, 1);
        C.r.U = __shfl_down_sync(MTE_FULL_MASK, C.c[0].U, 1);
        C.r.V = __shfl_down_sync(MTE_FULL_MASK, C.c[0].V, 1);
        C.r.C2 = __shfl_down_sync(MTE_FULL_MASK, C.c[0].C2, 1);
        C.l.A2 = 0.f;
        C.r.A2 = 0.f;
        // scatter this coefficient row into the output rows o = j-2 (as "down"), j-1 ("mid"), j ("up")
#pragma unroll
        for (int v = 0; v < VEC; v++) {
            const float asUp = C.at(v - 1).U + C.c[v].A2 + C.at(v + 1).V;
            const float asMid = C.at(v - 1).C2 - C.at(v + 1).C2;
            const float asDn = C.at(v - 1).V + C.c[v].A2 + C.at(v + 1).U;
            oacc[j % 3][v] = asUp;              // first contribution of output row j (overwrites the retired slot)
            if (j >= 1) oacc[(j + 2) % 3][v] += asMid;   // output row j-1
            if (j >= 2) oacc[(j + 1) % 3][v] -= asDn;    // output row j-2 (now complete)
        }
        if (j >= 2) {
            const int o = j - 2;
            const int orow = row0 + o;
            float out[VEC];
#pragma unroll
            for (int v = 0; v < VEC; v++) {
                float d = oacc[o % 3][v];
                if (INV) {
                    // d depth / d inv = -depth^2 where the clamp passes (inv > 1e-6 <=> depth < 1e6), else 0
                    const float dep = xr[j % 3].c[v];  // depth row index j == image row row0 + o
                    d = (dep < 1e6f) ? -d * dep * dep : 0.f;
                }
                out[v] = d;
            }
            if (writer && orow < H) {
                float *op = S.dx + plane + (size_t)orow * W + col0;
                if (VEC == 4) st_stream4(op, make_float4(out[0], out[1 % VEC], out[2 % VEC], out[3 % VEC]));
                else __stcs(op, out[0]);
            }
        }
    }
    }  // item loop
}

// ---------------------------------------------------------------------------
// Backward from the stash (MODE_DIR only): the forward left |c| (the grad map, an output anyway) and one byte
// per pixel (direction + sign), so the backward needs neither the 3x3 stencil nor the normals: per pixel it
// recomputes p = sigmoid(g - T) the reference-faithful way, d loss/d g, looks the four adjoint coefficients up
// in a 16-entry shared-memory table and scatters them into three rolling output rows.
// Traffic: g 4 + edge 4 + stash 1 (+ inverse depth 4 when fused) in, gradient 4 out.  This is the VEC=1 kernel (rows
// that are not whole float4s); at VEC=4 edge_loss_bwd_ring_kernel runs.
// ---------------------------------------------------------------------------
// Entry `code` (direction | sign << 2) of the 16-entry adjoint table: (A, C, A2, C2) for s = 1.
__device__ __forceinline__ float4 adjoint_entry(int code) {
    const int di = code & 3, sg = code >> 2;
    const float sgn = sg == 1 ? 1.f : (sg == 2 ? -1.f : 0.f);
    const float a = (di == 2 || di == 3) ? 1.f : (di == 1 ? -1.f : 0.f);  // h:0 rl:-1 v:1 lr:1
    const float c = (di == 2) ? 0.f : 1.f;                                // h:1 rl:1 v:0 lr:1
    const float bb = (di & 1) ? 1.f : 2.f;                                // axis stencils weigh the centre twice
    return make_float4(sgn * a, sgn * c, sgn * a * bb, sgn * c * bb);
}

// What one row of adjoint coefficients (A, C, A2, C2 per pixel; horizontal neighbours from the adjacent lanes) adds to
// the three output rows it touches: `up` to the row it acts as "up" for, `mid` to the one above, and `dn` (to be
// subtracted) to the one above that, which it completes.
template <int VEC>
struct AdjointRows {
    float up[VEC], mid[VEC], dn[VEC];
};
template <int VEC>
__device__ __forceinline__ AdjointRows<VEC> adjoint_rows(const float (&A)[VEC], const float (&C)[VEC],
                                                         const float (&A2)[VEC], const float (&C2)[VEC]) {
    const float Al = __shfl_up_sync(MTE_FULL_MASK, A[VEC - 1], 1), Ar = __shfl_down_sync(MTE_FULL_MASK, A[0], 1);
    const float Cl = __shfl_up_sync(MTE_FULL_MASK, C[VEC - 1], 1), Cr = __shfl_down_sync(MTE_FULL_MASK, C[0], 1);
    const float C2l = __shfl_up_sync(MTE_FULL_MASK, C2[VEC - 1], 1), C2r = __shfl_down_sync(MTE_FULL_MASK, C2[0], 1);
    AdjointRows<VEC> R;
#pragma unroll
    for (int v = 0; v < VEC; v++) {
        const float a_l = v == 0 ? Al : A[(v + VEC - 1) % VEC], a_r = v == VEC - 1 ? Ar : A[(v + 1) % VEC];
        const float c_l = v == 0 ? Cl : C[(v + VEC - 1) % VEC], c_r = v == VEC - 1 ? Cr : C[(v + 1) % VEC];
        const float c2_l = v == 0 ? C2l : C2[(v + VEC - 1) % VEC], c2_r = v == VEC - 1 ? C2r : C2[(v + 1) % VEC];
        const float SA = (a_l + a_r) + A2[v], DC = c_l - c_r;
        R.up[v] = SA + DC;
        R.mid[v] = c2_l - c2_r;
        R.dn[v] = SA - DC;
    }
    return R;
}

template <bool MASK, bool INV, bool SIG>
__global__ void __launch_bounds__(kThreads, 2) edge_loss_bwd_stash_kernel(const __grid_constant__ LossP P) {
    constexpr int VEC = 1;
    constexpr int RH = kBwdRH;
    constexpr int PD = 3;
    __shared__ float4 sLut[16];  // per code: (A, C, A2, C2) for s = 1
    if (threadIdx.x < 16) sLut[threadIdx.x] = adjoint_entry(threadIdx.x);
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int si = 0;
#pragma unroll
    for (int k = 1; k < MTE_MAX_SCALES; k++)
        if (k < P.nScales && (int)blockIdx.x >= P.s[k].ctaBase) si = k;
    const ScaleP &S = P.s[si];
    const int local = blockIdx.x - S.ctaBase;
    const int img = local / S.ctasPerImage;
    const int item0 = (local - img * S.ctasPerImage) * kWarps + warp;
    const int H = S.H, W = S.W;
    const BwdImg I = bwd_img<MASK>(P, S, si, img);
    const size_t plane = (size_t)img * H * W;

    for (int item = item0; item < S.items; item += S.ctasPerImage * kWarps) {  // warp-uniform
        const int strip = item / S.rowBlocks;
        const int rb = item - strip * S.rowBlocks;
        const int row0 = rb * RH;
        // one halo lane per side is enough here (coefficients are pointwise): lanes 1..30 write
        const int col0 = (strip * kHaloLanes + lane - 1) * VEC;
        const bool colOk = col0 >= 0 && col0 < W;
        const bool writer = lane >= 1 && lane <= kHaloLanes && colOk;

        float pfg[PD][VEC], pfe[PD][VEC], pfm[PD][VEC], pfx[PD][VEC];
        unsigned pfc[PD];
        auto fetch = [&](int slot, int row) {
            load_vec<VEC>(pfg[slot], S.g + plane, row, H, W, col0, false);
            load_vec<VEC>(pfe[slot], S.e + plane, row, H, W, col0, false);
            if (MASK) load_vec<VEC>(pfm[slot], S.m + plane, row, H, W, col0, false);
            if (INV) load_vec<VEC>(pfx[slot], S.x + plane, row, H, W, col0, false);
            const bool ok = row >= 0 && row < H && colOk;
            pfc[slot] = ok ? (unsigned)__ldcs(S.stash + plane + (size_t)row * W + col0) : 0u;
        };
#pragma unroll
        for (int k = 0; k < PD; k++) fetch(k, row0 - 1 + k);
        float oacc[3][VEC], xrow[3][VEC];
#pragma unroll
        for (int o = 0; o < 3; o++)
#pragma unroll
            for (int v = 0; v < VEC; v++) { oacc[o][v] = 0.f; xrow[o][v] = 0.f; }

#pragma unroll
        for (int j = 0; j < RH + 2; j++) {
            const int row = row0 - 1 + j;
            float g[VEC], e[VEC], m[VEC];
            const unsigned codes = pfc[j % PD];
#pragma unroll
            for (int v = 0; v < VEC; v++) {
                g[v] = pfg[j % PD][v];
                e[v] = pfe[j % PD][v];
                m[v] = MASK ? pfm[j % PD][v] : 1.f;
                if (INV) xrow[j % 3][v] = pfx[j % PD][v];
            }
            if (j + PD < RH + 2) fetch(j % PD, row + PD);
            const bool live = colOk && row >= 0 && row < H;
            float A[VEC], C[VEC], A2[VEC], C2[VEC];
#pragma unroll
            for (int v = 0; v < VEC; v++) {
                float d = dloss_dg<MASK, SIG>(g[v], e[v], m[v], I, P.T);
                d = (live && g[v] != 0.f) ? d : 0.f;  // sign(0) = 0: a zero response passes no gradient
                const float4 k = sLut[(codes >> (8 * v)) & 15u];
                A[v] = d * k.x; C[v] = d * k.y; A2[v] = d * k.z; C2[v] = d * k.w;
            }
            const AdjointRows<VEC> R = adjoint_rows<VEC>(A, C, A2, C2);
#pragma unroll
            for (int v = 0; v < VEC; v++) {
                oacc[j % 3][v] = R.up[v];                           // output row j   (this row acts as "up")
                if (j >= 1) oacc[(j + 2) % 3][v] += R.mid[v];       // output row j-1 ("mid")
                if (j >= 2) oacc[(j + 1) % 3][v] -= R.dn[v];        // output row j-2 ("down"), now complete
            }
            if (j >= 2) {
                const int o = j - 2, orow = row0 + o;
                float out[VEC];
#pragma unroll
                for (int v = 0; v < VEC; v++) {
                    float d = oacc[o % 3][v];
                    if (INV) {
                        // pred was an inverse depth: chain through depth = 1/clamp(inv, 1e-6); coefficient row j-1
                        // carried the inverse depth of image row orow
                        const float inv = xrow[(j + 2) % 3][v];
                        const float dep = inv_to_depth(inv);
                        d = (dep < 1e6f) ? -d * dep * dep : 0.f;
                    }
                    out[v] = d;
                }
                if (writer && orow < H) __stcs(S.dx + plane + (size_t)orow * W + col0, out[0]);
            }
        }
    }
}

// ---------------------------------------------------------------------------
// Backward from the stash, streaming version (VEC = 4): same decomposition as the forward -- persistent warps, each
// owning an equal, cost-balanced range of strip rows, fed by a cp.async shared-memory row ring -- around the
// per-pixel work of edge_loss_bwd_stash_kernel.  Rows / columns outside the image are zero-filled by the copies:
// a zero stash byte selects the all-zero table entry, so padding needs no predicates in the row loop.
// ---------------------------------------------------------------------------
constexpr int kSegCostB = MTE_SEGCOST_B;
constexpr int kBwdRingDepth = MTE_BWD_D;
__host__ __device__ constexpr int bwd_slot_bytes(bool mask, bool inv) { return (2 + (mask ? 1 : 0) + (inv ? 1 : 0)) * 512 + 128; }
__host__ __device__ constexpr int bwd_smem_bytes(bool mask, bool inv) { return kRWarps * kBwdRingDepth * bwd_slot_bytes(mask, inv); }

template <bool MASK, bool INV, bool SIG>
__global__ void __launch_bounds__(kRThreads, kRMinB) edge_loss_bwd_ring_kernel(const __grid_constant__ LossP P) {
    constexpr int VEC = 4;
    constexpr int D = kBwdRingDepth;
    constexpr unsigned PLB = 512, SLB = bwd_slot_bytes(MASK, INV);
    constexpr unsigned O_G = 0, O_E = PLB, O_M = 2 * PLB, O_X = (MASK ? 3 : 2) * PLB, O_S = SLB - 128;
    extern __shared__ __align__(16) unsigned char bwdRing[];
    __shared__ float4 sLut[16];  // per code: (A, C, A2, C2) for s = 1
    if (threadIdx.x < 16) sLut[threadIdx.x] = adjoint_entry(threadIdx.x);
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned char *ring = bwdRing + warp * (D * SLB);
    unsigned char *slot0 = ring + lane * 16, *slotS = ring + O_S + lane * 4;
    const unsigned ringS = (unsigned)__cvta_generic_to_shared(slot0);
    const unsigned ringSS = (unsigned)__cvta_generic_to_shared(slotS);
    const int nWarps = gridDim.x * kRWarps;
    const int gw = blockIdx.x * kRWarps + warp;
    int u0 = (int)((long long)P.totalUnits * gw / nWarps);
    const int u1 = (int)((long long)P.totalUnits * (gw + 1) / nWarps);
    pdl_launch_dependents();
    pdl_wait();
    while (u0 < u1) {
        const UnitSeg sg = unit_segment<kSegCostB>(P, u0, u1);
        if (sg.nrows <= 0) continue;
        const ScaleP &S = P.s[sg.si];
        const int img = sg.img, strip = sg.strip, row0 = sg.row0, nrows = sg.nrows;
        const int H = S.H;
        const unsigned W = (unsigned)S.W;
        const BwdImg I = bwd_img<MASK>(P, S, sg.si, img);
        // one halo lane per side (the coefficients are pointwise): lanes 1..30 write
        const int col0 = (strip * kHaloLanes + lane - 1) * VEC;
        const bool colOk = col0 >= 0 && col0 < (int)W;
        const bool writer = lane >= 1 && lane <= kHaloLanes && colOk;
        const size_t lo = (size_t)img * H * W + (colOk ? col0 : 0);
        const float *gP = S.g + lo, *eP = S.e + lo, *mP = S.m + lo, *xP = S.x + lo;
        const unsigned char *sP = S.stash + lo;
        float *dP = S.dx + lo;

        // coefficient row j of the segment is image row row0 - 1 + j, j = 0 .. nrows + 1
        const int ncoef = nrows + 2;
        auto issue = [&](unsigned so, int j) {
            const int row = row0 - 1 + j;
            const bool ok = colOk && row >= 0 && row < H;
            const unsigned ro = (unsigned)min(max(row, 0), H - 1) * W;
            cp_async_vec<4>(ringS + so + O_G, elem_addr(gP, ro), ok);
            cp_async_vec<4>(ringS + so + O_E, elem_addr(eP, ro), ok);
            if (MASK) cp_async_vec<4>(ringS + so + O_M, elem_addr(mP, ro), ok);
            if (INV) cp_async_vec<4>(ringS + so + O_X, elem_addr(xP, ro), ok);
            cp_async_vec<1>(ringSS + so, sP + ro, ok);
        };
#pragma unroll
        for (int k = 0; k < D; k++) {
            if (k < ncoef) issue(k * SLB, k);
            cp_async_commit();
        }
        float oacc[3][VEC], xrow[3][VEC];
#pragma unroll
        for (int o = 0; o < 3; o++)
#pragma unroll
            for (int v = 0; v < VEC; v++) { oacc[o][v] = 0.f; xrow[o][v] = 0.f; }
        unsigned so = 0;
#pragma unroll 1
        for (int jj = 0; jj < ncoef; jj += 3) {
#pragma unroll
            for (int u = 0; u < 3; u++) {
                const int j = jj + u;
                if (j < ncoef) {  // warp-uniform
                    cp_async_wait<D - 1>();
                    float g[VEC], e[VEC], m[VEC];
                    lds_vec<VEC>(g, slot0 + so + O_G);
                    lds_vec<VEC>(e, slot0 + so + O_E);
                    if (MASK) lds_vec<VEC>(m, slot0 + so + O_M);
                    if (INV) lds_vec<VEC>(xrow[u], slot0 + so + O_X);
                    const unsigned codes = *reinterpret_cast<const unsigned *>(slotS + so);
                    if (j + D < ncoef) issue(so, j + D);
                    cp_async_commit();
                    so = (so + SLB == D * SLB) ? 0u : so + SLB;
                    float A[VEC], C[VEC], A2[VEC], C2[VEC];
#pragma unroll
                    for (int v = 0; v < VEC; v++) {
                        float d = dloss_dg<MASK, SIG>(g[v], e[v], MASK ? m[v] : 1.f, I, P.T);
                        d = (g[v] != 0.f) ? d : 0.f;  // sign(0) = 0: a zero response passes no gradient
                        const float4 k = sLut[(codes >> (8 * v)) & 15u];
                        A[v] = d * k.x; C[v] = d * k.y; A2[v] = d * k.z; C2[v] = d * k.w;
                    }
                    // this coefficient row acts as "up" for output row j (image row row0 - 1 + j ... stored as
                    // segment output o = j), as "mid" for o = j - 1 and as "down" for o = j - 2, which it completes
                    const AdjointRows<VEC> R = adjoint_rows<VEC>(A, C, A2, C2);
#pragma unroll
                    for (int v = 0; v < VEC; v++) {
                        oacc[u][v] = R.up[v];
                        oacc[(u + 2) % 3][v] += R.mid[v];
                        oacc[(u + 1) % 3][v] -= R.dn[v];
                    }
                    if (j >= 2) {
                        float out[VEC];
#pragma unroll
                        for (int v = 0; v < VEC; v++) {
                            float d = oacc[(u + 1) % 3][v];
                            if (INV) {
                                // pred was an inverse depth: chain through depth = 1/clamp(inv, 1e-6); the inverse depth
                                // of this output row came with coefficient row j - 1
                                const float inv = xrow[(u + 2) % 3][v];
                                const float dep = rcp_approx(fmaxf(inv, 1e-6f));
                                d = (inv > 1e-6f) ? -d * dep * dep : 0.f;
                            }
                            out[v] = d;
                        }
                        if (writer)
                            st_stream4(elem_addr(dP, (unsigned)(row0 + j - 2) * W), make_float4(out[0], out[1], out[2], out[3]));
                    }
                }
            }
        }
        cp_async_wait<0>();
    }
}

template <bool MASK, bool INV, bool SIG>
static void launch_bwd_ring_one(const LossP &P, cudaStream_t st) {
    constexpr int smem = bwd_smem_bytes(MASK, INV);
    opt_in_smem((const void *)edge_loss_bwd_ring_kernel<MASK, INV, SIG>, smem);
    launch_pdl(edge_loss_bwd_ring_kernel<MASK, INV, SIG>, P.totalCtas, kRThreads, smem, st, P);
}

// the forward's row ring lives in dynamic shared memory (> 48 KB: opt in once per instantiation)
template <int VEC, int MODE, bool MASK, bool INV, bool SIG>
static void launch_fwd_one(const LossP &P, cudaStream_t st) {
    constexpr int smem = fwd_smem_bytes(VEC, MODE, MASK);
    opt_in_smem((const void *)edge_loss_fwd_kernel<VEC, MODE, MASK, INV, SIG>, smem);
    launch_pdl(edge_loss_fwd_kernel<VEC, MODE, MASK, INV, SIG>, P.totalCtas, kRThreads, smem, st, P);
}

// launchers implemented one translation unit per (direction, VEC) / kernel family so they compile in parallel
void launch_fwd_v4(const LossP &P, int mode, bool mask, bool inv, bool sig, cudaStream_t st);
void launch_fwd_v1(const LossP &P, int mode, bool mask, bool inv, bool sig, cudaStream_t st);
void launch_bwd_v4(const LossP &P, int mode, bool mask, bool inv, bool sig, cudaStream_t st);
void launch_bwd_v1(const LossP &P, int mode, bool mask, bool inv, bool sig, cudaStream_t st);
void launch_bwd_ring(const LossP &P, bool mask, bool inv, bool sig, cudaStream_t st);   // VEC=4
void launch_bwd_stash(const LossP &P, bool mask, bool inv, bool sig, cudaStream_t st);  // VEC=1

#define MTE_LOSS_DISPATCH_BOOL(flag, NAME, ...) \
    if (flag) { constexpr bool NAME = true; __VA_ARGS__ } else { constexpr bool NAME = false; __VA_ARGS__ }

}  // namespace loss
}  // namespace mte
