// Edge loss, ONE PASS: loss + grad map + d loss / d pred in a single launch (shipped configuration: directional
// responses, no mask, prediction at the target size, rows of whole float4s).
//
// Why one pass is possible: the class balance alpha_b = Wn_b / (Wp_b + Wn_b) (grad_loss.py:169-178) depends only on
// the TARGETS (Wp_b = sum of the soft edge labels of image b), not on the prediction.  So the kernel
//   phase 1  sums the edge plane (every warp over the rows it will process: 4 B/px, and the lines stay in L2),
//   -------- grid barrier (persistent cooperative grid, one CTA per SM) --------
//   phase 2  streams depth / edge / normal rows once through the per-warp cp.async ring: 3x3 directional response ->
//            |c| (grad map out) -> p = sigmoid(|c| - T) -> the two log terms (loss sums, order-independent fixed-point
//            atomics as in edge_loss_fwd_kernel) AND d loss / d|c| with the now-known alpha -> the 3x3 adjoint scatter
//            into three rolling output rows -> d loss / d pred out (inv2depth chain rule fused),
// for the upstream gradient the caller EXPECTS (1 for loss.backward(); the value of the previous step otherwise).
// The autograd backward is then mte_edge_loss_grad_rescale: a kernel that exits at once when the actual upstream
// gradient equals the expected one and rescales in place otherwise.
// HBM traffic: 12 B/px in + 8 B/px out = 20 B/px instead of 34 B/px over two launches with a stash round trip.
//
// No halo ROWS: a segment (a warp's run of rows in one strip) computes only the response rows it owns.  The 3x3
// adjoint of its first / last response row also reaches the output rows just outside, and its own first / last output
// rows lack the contribution of the neighbouring segment's response row: those four rows per segment are written by
// BOTH segments with a vector red.add onto rows that phase 1 zeroed (the grid barrier orders zero < add).  Segments
// start on even rows, so every such output row has exactly two contributors and 0 + a + b = 0 + b + a bit for bit:
// the result does not depend on the order of arrival.  (Recomputing one halo row above and below, as the two-kernel
// path does, cost 2 of ~20 rows per segment.)
//
// Reference arithmetic preserved: packnet_code/packnet_sfm/losses/grad_loss.py:65-95 (responses, band pick),
// :122-159 (sigmoid, weight), :161-219 (class-balanced BCE); backward = SURVEY.md A.1.
#include <string.h>

#include "edge_loss_kernels.cuh"

namespace mte {
namespace loss {

#ifndef MTE_FUSED_D
#define MTE_FUSED_D 3
#endif
constexpr int kFusedD = MTE_FUSED_D;
#ifndef MTE_FUSED_SEGCOST
#define MTE_FUSED_SEGCOST 2
#endif
constexpr int kSegCostFused = MTE_FUSED_SEGCOST;  // units are ROW PAIRS; a segment start costs the window prologue + the boundary adds
#ifndef MTE_FUSED_REGS
#define MTE_FUSED_REGS 120
#endif
#ifndef MTE_FUSED_P1ROWS
#define MTE_FUSED_P1ROWS 16
#endif
constexpr int kP1Rows = MTE_FUSED_P1ROWS;  // edge rows a lane keeps in flight in phase 1 (one DRAM round trip per batch)
__host__ __device__ constexpr int fused_smem_bytes() { return kRWarps * kFusedD * 3 * 512; }

__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned *p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned ld_relaxed_u32(const unsigned *p) {
    unsigned v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned atom_add_acq_rel_u32(unsigned *p, unsigned v) {
    unsigned old;
    asm volatile("atom.acq_rel.gpu.global.add.u32 %0, [%1], %2;" : "=r"(old) : "l"(p), "r"(v) : "memory");
    return old;
}

// The grid barrier (all CTAs of the cooperative, co-resident grid, once per launch) in two halves, so that the first
// segment's opening loads go out between them.  Memory model: what every CTA must see after the barrier is what the
// CTAs wrote in phase 1, the fixed-point atomics into `accum` (phase 2 reads them with __ldcg) and the plain zero
// stores of the seam rows (other CTAs red.add onto them later).  __syncthreads() orders every thread's phase-1
// writes before thread 0's arrival, and a release is cumulative, so the release add publishes all of them: its
// fence (MEMBAR.ALL.GPU, not the sequentially consistent MEMBAR.SC.GPU of __threadfence) waits until they have been
// performed.  The waiter polls with relaxed loads (no L1 invalidate per poll), and one acquire load after it has seen
// the full count synchronises with every arrival (they form one release sequence on the counter); __syncthreads()
// passes that on to the CTA.  The counter is reset by the last CTA of the launch (every CTA has left the barrier
// before it takes its final ticket).
__device__ __forceinline__ void grid_arrive(unsigned *ctr) {
    __syncthreads();
    if (threadIdx.x == 0) asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(ctr) : "memory");
}
__device__ __forceinline__ void grid_wait(const unsigned *ctr, unsigned nCtas) {
    if (threadIdx.x == 0) {
#ifdef MTE_FUSED_NOSLEEP
        while (ld_relaxed_u32(ctr) < nCtas) {}
#else
        while (ld_relaxed_u32(ctr) < nCtas) __nanosleep(20);
#endif
        (void)ld_acquire_u32(ctr);
    }
    __syncthreads();
}

#ifdef MTE_FUSED_TRACE
// timing build only (scripts/trace_fused.py): per-phase time stamps folded over all CTAs into ten u64 slots at byte
// 1032 of the workspace header (min via max of the complement).  Breaks the zero-header invariant: never in a release.
__device__ __forceinline__ unsigned long long gtime() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
#define MTE_TRACE(slot, isMin)                                                                                   \
    do {                                                                                                         \
        __syncthreads();                                                                                         \
        if (threadIdx.x == 0) {                                                                                  \
            const unsigned long long t_ = gtime();                                                               \
            atomicMax(reinterpret_cast<unsigned long long *>(F.barrier) + 128 + (slot), (isMin) ? ~t_ : t_); \
        }                                                                                                        \
    } while (0)
#else
#define MTE_TRACE(slot, isMin) do {} while (0)
#endif

struct FusedP {
    LossP L;
    const float *expectG;   // device [1 + nScales] upstream gradient the caller expects, or nullptr = {1, 0, ...}
    unsigned *barrier;      // grid barrier counter (workspace header, self-resetting)
};

// decode the unit range [u0, u1) into its next segment; returns false when the slice holds no rows
struct Seg {
    int si, img, strip, row0, nrows;
};
__device__ __forceinline__ bool next_segment(const LossP &P, int &u0, int u1, Seg &s) {
    int si = 0;
#pragma unroll
    for (int k = 1; k < MTE_MAX_SCALES; k++)
        if (k < P.nScales && u0 >= P.s[k].unitBase) si = k;
    const ScaleP &S = P.s[si];
    const int local = u0 - S.unitBase;
    const int HV = ((S.H + 1) >> 1) + kSegCostFused;  // row pairs of a strip + the virtual units of opening a segment
    const int t = local / HV;  // (image, strip)
    const int r = local - t * HV;
    const int take = min(HV - r, u1 - u0);
    s.row0 = 2 * max(r - kSegCostFused, 0);   // segments start on even rows (see the header: two contributors per row)
    s.nrows = min(2 * max(r + take - kSegCostFused, 0), S.H) - s.row0;
    u0 += take;
    s.si = si;
    s.img = t / S.strips;
    s.strip = t - s.img * S.strips;
    return s.nrows > 0;
}

__device__ __forceinline__ void red_add4(float *p, float4 v) {
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// ---- packed fp32 (sm_100a FADD2 / FMUL2 / FFMA2): the row loop is issue-bound (ncu: warps mostly "not selected",
// ALU + FMA + XU pipes at 30-45 %), and one packed instruction does the work of two for the same pipe time, so every
// per-pixel float operation that has both pixels of a pair in an aligned register pair is issued once per TWO pixels.
// A lane's four pixels are two pairs; the quantities of a pixel's adjoint (A, C) / (A2, C2) are paired per pixel.
__device__ __forceinline__ float2 f2(float s) { return make_float2(s, s); }
__device__ __forceinline__ float2 f2add(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 f2mul(float2 a, float2 b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ float2 f2fma(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ float2 f2sub(float2 a, float2 b) { return __ffma2_rn(b, f2(-1.f), a); }  // a - b, exact
// 1 / d correctly rounded for normal d (see rcp_rn_normal), two at a time
__device__ __forceinline__ float2 rcp_rn_normal2(float2 d) {
    float2 r = make_float2(rcp_approx(d.x), rcp_approx(d.y));
    const float2 nd = f2mul(d, f2(-1.f));
    float2 e = f2fma(nd, r, f2(1.f));
    r = f2fma(r, e, r);
    e = f2fma(nd, r, f2(1.f));
    return f2fma(r, e, r);
}

struct PRow2 {   // one depth row as the stencils consume it, pixel pairs (0,1) and (2,3)
    float2 c[2], s3[2], d[2];
};
__device__ __forceinline__ void prep_row2(PRow2 &R, const float2 (&x)[2]) {
    // horizontal neighbours across the lane boundary (lanes 0 / 31 are halo lanes: their outer values are unused)
    const float l = __shfl_up_sync(MTE_FULL_MASK, x[1].y, 1);
    const float r = __shfl_down_sync(MTE_FULL_MASK, x[0].x, 1);
    R.c[0] = x[0];
    R.c[1] = x[1];
    // the shifted rows are not pair-aligned, so these stay scalar
    R.s3[0] = make_float2((l + x[0].x) + x[0].y, (x[0].x + x[0].y) + x[1].x);
    R.s3[1] = make_float2((x[0].y + x[1].x) + x[1].y, (x[1].x + x[1].y) + r);
    R.d[0] = make_float2(x[0].y - l, x[1].x - x[0].x);
    R.d[1] = make_float2(x[1].y - x[0].y, r - x[1].x);
}

// The loads that open a segment (first D ring rows + the depth rows above / at the first response row), as a function
// of their own: the FIRST segment of every warp issues them BEFORE the grid barrier, so the DRAM round trip that
// refills the pipeline after phase 1 overlaps the barrier instead of following it.
__device__ __forceinline__ void fused_prologue(const ScaleP &S, const Seg &sg, int lane, unsigned char *ring,
                                               float2 (&xa)[2], float2 (&xc)[2]) {
    constexpr int D = kFusedD;
    constexpr unsigned PLB = 512, SLB = 3 * PLB;
    const int H = S.H, row0 = sg.row0, niter = sg.nrows;
    const unsigned W = (unsigned)S.W;
    const int col0 = (sg.strip * kHaloLanes + lane - 1) * 4;
    const bool colOk = col0 >= 0 && col0 < (int)W;
    const size_t lo = (size_t)sg.img * H * W + (colOk ? col0 : 0);
    const float *xP = S.x + lo, *eP = S.e + lo, *nP = S.n + lo;
    const unsigned ringS = (unsigned)__cvta_generic_to_shared(ring + lane * 16);
    auto load_plain = [&](float2 (&x)[2], int row) {
        x[0] = make_float2(0.f, 0.f);
        x[1] = make_float2(0.f, 0.f);
        if (colOk && row >= 0 && row < H) {
            const float4 t = ld_cached4(elem_addr(xP, (unsigned)row * W));
            x[0] = make_float2(t.x, t.y);
            x[1] = make_float2(t.z, t.w);
        }
    };
    load_plain(xa, row0 - 1);
    load_plain(xc, row0);
#pragma unroll
    for (int k = 0; k < D; k++) {
        if (k < niter) {   // response row row0 + k (inside the image): depth row below it, its own target rows
            const int rx = row0 + 1 + k;
            cp_async_vec<4>(ringS + k * SLB, elem_addr(xP, (unsigned)min(rx, H - 1) * W), colOk && rx < H);
            const unsigned ro = (unsigned)(row0 + k) * W;
            cp_async_vec<4>(ringS + k * SLB + PLB, elem_addr(eP, ro), colOk);
            cp_async_vec<4>(ringS + k * SLB + 2 * PLB, elem_addr(nP, ro), colOk);
        }
        cp_async_commit();
    }
}

template <bool INV, bool SIG>
__device__ __forceinline__ void fused_segment(const LossP &P, const ScaleP &S, const Seg &sg, int lane,
                                              unsigned char *ring, const float4 *sLut, float cp, float cn,
                                              float2 (&la)[2], float &poison, float2 (&xa)[2], float2 (&xc)[2]) {
    constexpr int D = kFusedD;
    constexpr unsigned PLB = 512, SLB = 3 * PLB;
    constexpr float kFill = INV ? 3.0e38f : 0.f;  // its reciprocal flushes to exactly 0 (the conv zero padding)
    const int H = S.H, row0 = sg.row0, nrows = sg.nrows;
    const unsigned W = (unsigned)S.W;
    const int col0 = (sg.strip * kHaloLanes + lane - 1) * 4;
    const bool colOk = col0 >= 0 && col0 < (int)W;
    const bool writer = colOk && lane >= 1 && lane <= kHaloLanes;
    const size_t lo = (size_t)sg.img * H * W + (colOk ? col0 : 0);
    const float *xP = S.x + lo, *eP = S.e + lo, *nP = S.n + lo;
    float *gP = S.g + lo, *dP = S.dx + lo;
    const bool writeG = writer && S.g != nullptr;
    const float2 mT = f2(-P.T), cp2 = f2(cp), cn2 = f2(cn), eps2 = f2(kEps), one2 = f2(1.f), m1 = f2(-1.f);
    unsigned char *slot0 = ring + lane * 16;
    const unsigned ringS = (unsigned)__cvta_generic_to_shared(slot0);

    // iteration j = 0 .. nrows - 1 handles RESPONSE row r = row0 + j, a row this segment owns: it needs depth row
    // r + 1 (rows r - 1 and r are in the window) and the target rows r
    auto issue = [&](unsigned so, int j) {
        const int rx = row0 + 1 + j;
        cp_async_vec<4>(ringS + so, elem_addr(xP, (unsigned)min(rx, H - 1) * W), colOk && rx < H);
        const unsigned ro = (unsigned)(row0 + j) * W;
        cp_async_vec<4>(ringS + so + PLB, elem_addr(eP, ro), colOk);
        cp_async_vec<4>(ringS + so + 2 * PLB, elem_addr(nP, ro), colOk);
    };
    auto fix_row = [&](float2 (&x)[2], int row) {  // padding, inv2depth, non-finite tracking
        if (INV) {
            const bool ok = colOk && row >= 0 && row < H;
#pragma unroll
            for (int h = 0; h < 2; h++) {
                // torch.clamp(min=1e-6) keeps a NaN (max.NaN), then the correctly rounded reciprocal
                const float2 v = make_float2(fmax_nan(ok ? x[h].x : kFill, 1e-6f), fmax_nan(ok ? x[h].y : kFill, 1e-6f));
                x[h] = rcp_rn_normal2(v);
            }
        }
        // x * 0 is NaN exactly when x is NaN or +-Inf (the reference's conv2d turns such a pixel into a NaN loss)
        const float2 t = f2fma(x[0], f2(0.f), f2mul(x[1], f2(0.f)));
        poison += t.x + t.y;
    };
    auto lds2 = [&](float2 (&x)[2], const unsigned char *p) {
        const float4 t = *reinterpret_cast<const float4 *>(p);
        x[0] = make_float2(t.x, t.y);
        x[1] = make_float2(t.z, t.w);
    };

    const int niter = nrows;
    PRow2 win[3];  // win[d % 3] holds depth row row0 - 1 + d; xa / xc and the first D ring rows come from fused_prologue
    fix_row(xa, row0 - 1);
    fix_row(xc, row0);
    prep_row2(win[0], xa);
    prep_row2(win[1], xc);
    float oacc[3][4];
#pragma unroll
    for (int o = 0; o < 3; o++)
#pragma unroll
        for (int v = 0; v < 4; v++) oacc[o][v] = 0.f;
    // one output row (accumulator slot `slot`, depth row `dep` for the inv2depth chain rule) to memory: complete rows are
    // stored, rows shared with the neighbouring segment are added onto the zeroed row (see the header)
    auto emit = [&](const float (&acc)[4], const PRow2 &dep, int row, bool shared) {
        float out[4];
#pragma unroll
        for (int v = 0; v < 4; v++) {
            float d = acc[v];
            if (INV) {
                // pred was an inverse depth: chain through depth = 1 / clamp(inv, 1e-6) (utils/depth.py:104-121)
                const float dp = (v & 1) ? dep.c[v >> 1].y : dep.c[v >> 1].x;
                d = (dp < 1e6f) ? -d * dp * dp : 0.f;
            }
            out[v] = d;
        }
        if (writer) {
            float *o = elem_addr(dP, (unsigned)row * W);
            if (shared) red_add4(o, make_float4(out[0], out[1], out[2], out[3]));
            else st_stream4(o, make_float4(out[0], out[1], out[2], out[3]));
        }
    };

    unsigned so = 0;
#pragma unroll 1
    for (int jj = 0; jj < niter; jj += 3) {
#pragma unroll
        for (int u = 0; u < 3; u++) {
            const int j = jj + u;
            if (j < niter) {  // warp-uniform
                cp_async_wait<D - 1>();
                float2 xn[2], e[2], th[2];
                lds2(xn, slot0 + so);
                lds2(e, slot0 + so + PLB);
                lds2(th, slot0 + so + 2 * PLB);
                if (j + D < niter) issue(so, j + D);  // refill the slot just read
                cp_async_commit();
                so = (so + SLB == D * SLB) ? 0u : so + SLB;
                const int r = row0 + j;
                PRow2 &dn = win[(u + 2) % 3];
                fix_row(xn, r + 1);
                prep_row2(dn, xn);
                const PRow2 &up = win[u % 3];
                const PRow2 &mid = win[(u + 1) % 3];
                float g[4];
                float2 X[4], Z[4];   // per pixel: (A, C) and (A2, C2) of the adjoint
#pragma unroll
                for (int h = 0; h < 2; h++) {
                    // separable parts of the four zero-padded 3x3 cross-correlations of grad_loss.py:20-31:
                    // c_v = Pv + dv, c_h = Rh + Dm, c_lr = Pv + Rh, c_rl = Rh - Pv
                    const float2 Pv = f2sub(dn.s3[h], up.s3[h]);
                    const float2 Dm = mid.d[h];
                    const float2 Rh = f2add(f2add(up.d[h], Dm), dn.d[h]);
                    const float2 dv = f2sub(dn.c[h], up.c[h]);
                    float c0, c1;
                    unsigned cd0, cd1;
                    pick_directional(th[h].x, Pv.x, Rh.x, Dm.x, dv.x, c0, cd0);
                    pick_directional(th[h].y, Pv.y, Rh.y, Dm.y, dv.y, c1, cd1);
                    const float2 gg = make_float2(fabsf(c0), fabsf(c1));
                    g[2 * h] = gg.x;
                    g[2 * h + 1] = gg.y;
                    // p the reference-faithful way (accurate expf, correctly rounded reciprocal): the gradient term
                    // p(1-p)/(1-p+eps) amplifies the last bits of p where the sigmoid saturates
                    float2 p = gg;
                    if (SIG) {
                        const float2 nz = f2sub(f2(P.T), gg);   // -(g - T), exactly as g - T negated
                        p = rcp_rn_normal2(f2add(make_float2(expf(nz.x), expf(nz.y)), one2));
                    }
                    const float2 q = f2fma(p, m1, one2);       // 1 - p
                    const float2 pe = f2add(p, eps2), qe = f2add(q, eps2);
                    const float2 ee = e[h], ne = f2fma(ee, m1, one2);
                    la[0] = f2fma(ee, make_float2(lg2_approx(pe.x), lg2_approx(pe.y)), la[0]);
                    la[1] = f2fma(ne, make_float2(lg2_approx(qe.x), lg2_approx(qe.y)), la[1]);
                    float2 d = f2mul(f2mul(cp2, ee), make_float2(rcp_approx(pe.x), rcp_approx(pe.y)));
                    d = f2fma(f2mul(cn2, ne), make_float2(rcp_approx(qe.x), rcp_approx(qe.y)), d);
                    if (SIG) d = f2mul(f2mul(d, p), q);
                    // sign(0) = 0; pixels outside the image do not exist
                    const float d0 = (colOk && gg.x != 0.f) ? d.x : 0.f, d1 = (colOk && gg.y != 0.f) ? d.y : 0.f;
                    const float4 k0 = sLut[cd0 & 15u], k1 = sLut[cd1 & 15u];
                    X[2 * h] = f2mul(f2(d0), make_float2(k0.x, k0.y));
                    Z[2 * h] = f2mul(f2(d0), make_float2(k0.z, k0.w));
                    X[2 * h + 1] = f2mul(f2(d1), make_float2(k1.x, k1.y));
                    Z[2 * h + 1] = f2mul(f2(d1), make_float2(k1.z, k1.w));
                }
                if (writeG) st_stream4(elem_addr(gP, (unsigned)r * W), make_float4(g[0], g[1], g[2], g[3]));
                // neighbours across the lane boundary: (A, C) and C2 of the adjacent pixel
                const float2 Xl = make_float2(__shfl_up_sync(MTE_FULL_MASK, X[3].x, 1), __shfl_up_sync(MTE_FULL_MASK, X[3].y, 1));
                const float2 Xr = make_float2(__shfl_down_sync(MTE_FULL_MASK, X[0].x, 1), __shfl_down_sync(MTE_FULL_MASK, X[0].y, 1));
                const float C2l = __shfl_up_sync(MTE_FULL_MASK, Z[3].y, 1), C2r = __shfl_down_sync(MTE_FULL_MASK, Z[0].y, 1);
                // response row r acts as "up" for output row r + 1 (first contribution: overwrites the retired slot),
                // as "mid" for output row r and as "down" for output row r - 1, which it completes
#pragma unroll
                for (int v = 0; v < 4; v++) {
                    const float2 xl = v == 0 ? Xl : X[(v + 3) % 4], xr = v == 3 ? Xr : X[(v + 1) % 4];
                    const float c2_l = v == 0 ? C2l : Z[(v + 3) % 4].y, c2_r = v == 3 ? C2r : Z[(v + 1) % 4].y;
                    // (a_l + a_r, c_l - c_r) in one packed add: the right neighbour enters as (A, -C)
                    const float2 U = f2add(xl, make_float2(xr.x, -xr.y));
                    const float SA = U.x + Z[v].x, DC = U.y;
                    oacc[u][v] = SA + DC;
                    oacc[(u + 2) % 3][v] += c2_l - c2_r;
                    oacc[(u + 1) % 3][v] -= SA - DC;
                }
                // output row r - 1 has all it gets from this segment: rows row0 - 1 (the neighbour's) and row0 (missing
                // the neighbour's response row) are shared, the rest is complete
                if (r >= 1) emit(oacc[(u + 1) % 3], up, r - 1, j < 2);
                if (j == niter - 1) {   // the last response row: rows r and r + 1 are shared with the segment below
                    emit(oacc[(u + 2) % 3], mid, r, true);
                    if (r + 1 < H) emit(oacc[u], dn, r + 1, true);
                }
            }
        }
    }
    cp_async_wait<0>();
    if (!writer) {  // halo / out-of-image lanes: their pixels belong to the neighbouring strips
        la[0] = f2(0.f);
        la[1] = f2(0.f);
    }
}

// 120 registers x 512 threads leave 4 K registers of the SM free: room for one 128-thread CTA of the (tiny) rescale
// kernel that follows, so its programmatic dependent launch can become resident while this grid is still running.
template <bool INV, bool SIG>
__global__ void __maxnreg__(MTE_FUSED_REGS) edge_loss_fused_kernel(const __grid_constant__ FusedP F) {
    extern __shared__ __align__(16) unsigned char fusedRing[];
    __shared__ float4 sLut[16];  // per stash code (direction | 4 << sign): adjoint coefficients (A, C, A2, C2) for s = 1
    __shared__ double sLoss[MTE_MAX_SCALES];
    __shared__ int sLast;
    const LossP &P = F.L;
    if (threadIdx.x < 16) sLut[threadIdx.x] = adjoint_entry(threadIdx.x);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nWarps = gridDim.x * kRWarps;
    const int gw = blockIdx.x * kRWarps + warp;
    unsigned char *ring = fusedRing + warp * (fused_smem_bytes() / kRWarps);
    const int uBeg = (int)((long long)P.totalUnits * gw / nWarps);
    const int uEnd = (int)((long long)P.totalUnits * (gw + 1) / nWarps);
    pdl_launch_dependents();   // the rescale kernel behind us may take its place on the SMs now (it waits for our end)
    MTE_TRACE(0, true);    // first CTA starts
    MTE_TRACE(1, false);   // last CTA starts

    // ---- phase 1: Wp_b = sum of the edge labels, every warp over the rows it owns (the lines stay in L2 for phase 2)
#ifndef MTE_FUSED_TIMING_NO_PHASE1   // timing experiments only (results are wrong without it)
    {
        int u0 = uBeg;
        while (u0 < uEnd) {
            Seg sg;
            if (!next_segment(P, u0, uEnd, sg)) continue;
            const ScaleP &S = P.s[sg.si];
            const unsigned W = (unsigned)S.W;
            const int col0 = (sg.strip * kHaloLanes + lane - 1) * 4;
            const bool writer = col0 >= 0 && col0 < (int)W && lane >= 1 && lane <= kHaloLanes;
            const float *eP = S.e + (size_t)sg.img * S.H * W + (writer ? col0 : 0);
            if (writer) {   // the two output rows this segment shares with its neighbours start at zero (see the header)
                float *dP = S.dx + (size_t)sg.img * S.H * W + col0;
                const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
                *reinterpret_cast<float4 *>(elem_addr(dP, (unsigned)sg.row0 * W)) = z;
                *reinterpret_cast<float4 *>(elem_addr(dP, (unsigned)(sg.row0 + sg.nrows - 1) * W)) = z;
            }
            float s0 = 0.f, s1 = 0.f;
#pragma unroll 1
            for (int j0 = 0; j0 < sg.nrows; j0 += kP1Rows) {
                float4 t[kP1Rows];
#pragma unroll
                for (int k = 0; k < kP1Rows; k++) {
                    t[k] = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (writer && j0 + k < sg.nrows)
                        t[k] = *reinterpret_cast<const float4 *>(elem_addr(eP, (unsigned)(sg.row0 + j0 + k) * W));
                }
#pragma unroll
                for (int k = 0; k < kP1Rows; k += 2) {
                    s0 += (t[k].x + t[k].y) + (t[k].z + t[k].w);
                    s1 += (t[k + 1].x + t[k + 1].y) + (t[k + 1].z + t[k + 1].w);
                }
            }
            const float v = warp_sum(s0 + s1);
            unsigned long long *acc = P.accum + (size_t)(S.imgBase + sg.img) * kAcc;
            if (lane == 0) {
                atomicAdd(acc + A_WP, (unsigned long long)__double2ll_rn((double)v * kFix));
                if (!isfinite(v)) atomicOr(acc + A_FLAGS, (unsigned long long)F_NONFINITE);
            }
        }
    }
    MTE_TRACE(2, true);    // first CTA done with phase 1
    MTE_TRACE(3, false);   // last CTA done with phase 1 (the last arrival follows)
    grid_arrive(F.barrier);
    // the first segment's opening loads go out while the other CTAs arrive
    int u0 = uBeg;
    Seg sg;
    bool have = false;
    while (u0 < uEnd && !have) have = next_segment(P, u0, uEnd, sg);
    float2 xa[2], xc[2];
    if (have) fused_prologue(P.s[sg.si], sg, lane, ring, xa, xc);
    grid_wait(F.barrier, gridDim.x);
    MTE_TRACE(8, true);    // first CTA out of the barrier
    MTE_TRACE(4, false);   // last CTA out of the barrier
#else
    __syncthreads();
    int u0 = uBeg;
    Seg sg;
    bool have = false;
    while (u0 < uEnd && !have) have = next_segment(P, u0, uEnd, sg);
    float2 xa[2], xc[2];
    if (have) fused_prologue(P.s[sg.si], sg, lane, ring, xa, xc);
#endif

    // ---- phase 2
    while (have) {
        const ScaleP &S = P.s[sg.si];
        // class balance and normaliser of this image, exactly as finalize_loss / the two-kernel backward form them
        const double npix = (double)S.H * (double)S.W;
        float alpha;
        {
            const double wp = (double)(long long)__ldcg(P.accum + (size_t)(S.imgBase + sg.img) * kAcc + A_WP) / kFix;
            const double wn = npix - wp;
            alpha = (float)(wn / (wp + wn));
            if (wn == 0.0) {  // rare: "no negatives anywhere in the batch" -> all alpha = 1 (grad_loss.py:175-176)
                double wnSum = 0.0;
                for (int b = 0; b < S.B; b++)
                    wnSum += npix - (double)(long long)__ldcg(P.accum + (size_t)(S.imgBase + b) * kAcc + A_WP) / kFix;
                if (wnSum == 0.0) alpha = 1.0f;
            }
        }
        float G = F.expectG ? (__ldg(F.expectG) * S.scaleWeight + __ldg(F.expectG + 1 + sg.si)) : S.scaleWeight;
        if (G == 0.f) G = 1.f;  // a zero expectation could not be rescaled later
        const float coef = (float)((double)P.weight / (npix * (double)S.B)) * G;
        const float cp = -coef * P.p2n * alpha, cn = coef * (1.0f - alpha);
        float2 la[2] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
        float poison = 0.f;
        fused_segment<INV, SIG>(P, S, sg, lane, ring, sLut, cp, cn, la, poison, xa, xc);
        bool bad = __any_sync(MTE_FULL_MASK, !(poison == 0.f));
        unsigned long long *acc = P.accum + (size_t)(S.imgBase + sg.img) * kAcc;
        const float vp = warp_sum(la[0].x + la[0].y), vn = warp_sum(la[1].x + la[1].y);
        bad = bad || !isfinite(vp) || !isfinite(vn);
        if (lane == 0) {
            atomicAdd(acc + A_SPU, (unsigned long long)__double2ll_rn((double)vp * kFix));
            atomicAdd(acc + A_SNU, (unsigned long long)__double2ll_rn((double)vn * kFix));
            if (bad) atomicOr(acc + A_FLAGS, (unsigned long long)F_NONFINITE);
        }
        have = false;
        while (u0 < uEnd && !have) have = next_segment(P, u0, uEnd, sg);
        if (have) fused_prologue(P.s[sg.si], sg, lane, ring, xa, xc);
    }
    MTE_TRACE(5, true);    // first CTA done with phase 2
    MTE_TRACE(6, false);   // last CTA done with phase 2
    // ---- the last CTA to leave folds alpha, the normalisers and the loss (same code as the two-kernel forward).  The
    // election needs only the accumulator atomics of every CTA ordered before its ticket; __syncthreads() + the
    // release half of thread 0's acq_rel add publish them (MEMBAR.ALL.GPU, no sequentially consistent fence), and the
    // acquire half lets the last CTA read the sums.  The grad_pred / grad_map stores are published by the kernel's end.
    __syncthreads();
    if (threadIdx.x == 0) sLast = atom_add_acq_rel_u32(P.ticket + 1, 1u) == gridDim.x - 1u;
    __syncthreads();
    if (sLast) {
        MTE_TRACE(9, false);   // the last CTA is elected
        finalize_loss<false>(P, sLoss);
        __syncthreads();
        if (threadIdx.x == 0) {
            double total = 0.0;
            for (int k = 0; k < P.nScales; k++) {
                total += (double)P.s[k].scaleWeight * sLoss[k];
                float G = F.expectG ? (F.expectG[0] * P.s[k].scaleWeight + F.expectG[1 + k]) : P.s[k].scaleWeight;
                if (G == 0.f) G = 1.f;
                P.ctx[P.totalImages + 2 * MTE_MAX_SCALES + k] = G;  // the factor grad_pred carries now
            }
            reinterpret_cast<unsigned *>(P.ctx + P.totalImages + 3 * MTE_MAX_SCALES)[0] = 0u;  // rescale ticket
            P.lossOut[0] = (float)total;
            P.ticket[0] = 0u;
            P.ticket[1] = 0u;
            *F.barrier = 0u;
        }
        MTE_TRACE(7, false);   // the loss is written
    }
}

// d loss / d pred was produced for the expected upstream gradient; bring it to the actual one.  Exits at once when
// they agree (the common case: loss.backward() with the expectation 1, or a steady training loop).
// One wave of one CTA per SM: at <= 32 registers x 128 threads a CTA fits in the 4 K registers the fused kernel leaves
// free, so every CTA is resident (waiting in pdl_wait) before the fused grid ends and none is scheduled after it.
constexpr int kRescaleThreads = 128;
constexpr int kRescaleVec = 4;   // float4 per thread in flight per iteration (the rescaling path streams grad_pred)
__global__ void __launch_bounds__(kRescaleThreads, 65536 / (kRescaleThreads * 32))
edge_loss_rescale_kernel(const __grid_constant__ LossP P, const float *gradLoss, float *ctx, float *expectedOut) {
    pdl_wait();   // launched as a programmatic dependent of the kernel that produces ctx and grad_pred
    float *cur = ctx + P.totalImages + 2 * MTE_MAX_SCALES;
    unsigned *done = reinterpret_cast<unsigned *>(ctx + P.totalImages + 3 * MTE_MAX_SCALES);
    bool any = false;
    for (int k = 0; k < P.nScales; k++) any = any || (gradLoss[0] * P.s[k].scaleWeight + gradLoss[1 + k] != cur[k]);
    if (!any) {  // every CTA sees the same values: nothing to rescale, nothing to record
        if (expectedOut && blockIdx.x == 0 && threadIdx.x <= P.nScales) expectedOut[threadIdx.x] = gradLoss[threadIdx.x];
        return;
    }
    for (int k = 0; k < P.nScales; k++) {
        const ScaleP &S = P.s[k];
        const float G = gradLoss[0] * S.scaleWeight + gradLoss[1 + k];
        const float c = cur[k];
        if (G == c) continue;
        const float f = G / c;
        const size_t n4 = (size_t)S.B * S.H * S.W / 4;
        float4 *d = reinterpret_cast<float4 *>(S.dx);
        const size_t step = (size_t)gridDim.x * kRescaleThreads * kRescaleVec;
        for (size_t i0 = (size_t)blockIdx.x * kRescaleThreads * kRescaleVec + threadIdx.x; i0 < n4; i0 += step) {
            float4 v[kRescaleVec];
#pragma unroll
            for (int u = 0; u < kRescaleVec; u++)
                if (i0 + u * kRescaleThreads < n4) v[u] = d[i0 + u * kRescaleThreads];
#pragma unroll
            for (int u = 0; u < kRescaleVec; u++)
                if (i0 + u * kRescaleThreads < n4) {
                    v[u].x *= f; v[u].y *= f; v[u].z *= f; v[u].w *= f;
                    d[i0 + u * kRescaleThreads] = v[u];
                }
        }
    }
    // the last CTA records what grad_pred carries now (every CTA has read `cur` before taking its ticket)
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(done, 1u) == gridDim.x - 1u) {
            for (int k = 0; k < P.nScales; k++) cur[k] = gradLoss[0] * P.s[k].scaleWeight + gradLoss[1 + k];
            if (expectedOut)
                for (int k = 0; k < 1 + P.nScales; k++) expectedOut[k] = gradLoss[k];
            __threadfence();
            *done = 0u;
        }
    }
}

template <bool INV, bool SIG>
static int launch_fused_one(const FusedP &F, int grid, cudaStream_t st) {
    constexpr int smem = fused_smem_bytes();
    const void *fn = (const void *)edge_loss_fused_kernel<INV, SIG>;
    if (opt_in_smem(fn, smem) != cudaSuccess) return (int)cudaGetLastError();
    // the grid barrier needs every CTA resident at once: cap the grid at the co-resident maximum and launch
    // cooperatively, so the driver never runs a partial grid next to another cooperative kernel
    int perSm = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSm, edge_loss_fused_kernel<INV, SIG>, kRThreads, smem);
    if (perSm < 1) return MTE_ERR_ARG;
    const int maxGrid = perSm * num_sms();
    if (grid > maxGrid) grid = maxGrid;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3((unsigned)kRThreads);
    cfg.dynamicSmemBytes = (size_t)smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeCooperative;
    at[0].val.cooperative = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, edge_loss_fused_kernel<INV, SIG>, F);
    return e == cudaSuccess ? MTE_OK : (int)e;
}

int launch_fused(const FusedP &F, int grid, bool inv, bool sig, cudaStream_t st) {
    if (inv) return sig ? launch_fused_one<true, true>(F, grid, st) : launch_fused_one<true, false>(F, grid, st);
    return sig ? launch_fused_one<false, true>(F, grid, st) : launch_fused_one<false, false>(F, grid, st);
}

}  // namespace loss
}  // namespace mte

using namespace mte;
using namespace mte::loss;

static bool fused_supported(const mte_loss_scale_t *sc, int n, const mte_loss_attrs_t *at) {
    if (!sc || !at || n < 1 || n > MTE_MAX_SCALES) return false;
    if (!at->is_grad) return false;
    for (int i = 0; i < n; i++) {
        const mte_loss_scale_t &s = sc[i];
        if (!s.pred || !s.edge || !s.normal || s.mask) return false;
        if (s.h != s.H || s.w != s.W || s.B < 1 || s.H < 1 || s.W < 4 || (s.W % 4)) return false;
        const void *ptrs[] = {s.pred, s.edge, s.normal, s.grad_map, s.grad_pred};
        for (const void *p : ptrs)
            if (!aligned16(p)) return false;
    }
    return true;
}

extern "C" int mte_edge_loss_fused_supported(const mte_loss_scale_t *sc, int n, const mte_loss_attrs_t *at) {
    return fused_supported(sc, n, at) ? 1 : 0;
}

extern "C" int mte_edge_loss_fwd_grad(const mte_loss_scale_t *sc, int n, const mte_loss_attrs_t *at,
                                      const float *expected_grad_loss, float *loss_out, void *ctx, void *ws,
                                      size_t ws_bytes, mte_stream_t stream) {
    if (!sc || !at || !loss_out || !ctx || !ws) return MTE_ERR_NULL;
    if (!fused_supported(sc, n, at)) return MTE_ERR_ARG;
    for (int i = 0; i < n; i++)
        if (!sc[i].grad_pred) return MTE_ERR_NULL;
    if (ws_bytes < MTE_WS_HEADER_BYTES) return MTE_ERR_WORKSPACE;
    FusedP F;
    memset(&F, 0, sizeof(F));
    LossP &P = F.L;
    int img = 0;
    long long unitBase = 0;
    for (int i = 0; i < n; i++) {
        ScaleP &S = P.s[i];
        S.B = sc[i].B; S.H = sc[i].H; S.W = sc[i].W;
        S.x = sc[i].pred; S.e = sc[i].edge; S.n = sc[i].normal; S.m = nullptr;
        S.g = sc[i].grad_map; S.dx = sc[i].grad_pred; S.stash = nullptr;
        S.strips = ceil_div(S.W, kHaloLanes * 4);
        S.imgBase = img;
        S.unitBase = (int)unitBase;
        unitBase += (long long)S.strips * (((S.H + 1) >> 1) + kSegCostFused) * S.B;   // units are row pairs
        S.scaleWeight = sc[i].scale_weight;
        img += S.B;
    }
    if (unitBase > 0x7fffffffLL || img > kWsMaxLossImages) return MTE_ERR_SHAPE;
    P.nScales = n; P.totalImages = img; P.totalUnits = (int)unitBase;
    P.T = at->sigmoid_thresh; P.weight = at->weight; P.p2n = at->pos_to_neg;
    char *w = static_cast<char *>(ws);
    WsHeader *hdr = reinterpret_cast<WsHeader *>(w);
    P.accum = reinterpret_cast<unsigned long long *>(w + kWsAccumOffset);
    P.ticket = hdr->ticket;
    P.lossOut = loss_out;
    P.ctx = static_cast<float *>(ctx);
    F.expectG = expected_grad_loss;
    F.barrier = hdr->ticket + 2;
    int grid = num_sms();
    const int minUnits = 2;   // row pairs per warp below which a smaller grid is better
    if ((long long)grid * kRWarps * minUnits > unitBase) grid = (int)((unitBase + kRWarps * minUnits - 1) / (kRWarps * minUnits));
    if (grid < 1) grid = 1;
    return launch_fused(F, grid, at->pred_is_inverse != 0, at->is_sigmoid != 0, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int mte_edge_loss_grad_rescale(const mte_loss_scale_t *sc, int n, const float *grad_loss, void *ctx,
                                          float *expected_out, mte_stream_t stream) {
    if (!sc || !grad_loss || !ctx) return MTE_ERR_NULL;
    if (n < 1 || n > MTE_MAX_SCALES) return MTE_ERR_ARG;
    LossP P;
    memset(&P, 0, sizeof(P));
    int img = 0;
    for (int i = 0; i < n; i++) {
        if (!sc[i].grad_pred) return MTE_ERR_NULL;
        if (!aligned16(sc[i].grad_pred) || (sc[i].W % 4)) return MTE_ERR_ALIGN;
        P.s[i].B = sc[i].B; P.s[i].H = sc[i].H; P.s[i].W = sc[i].W;
        P.s[i].dx = sc[i].grad_pred;
        P.s[i].scaleWeight = sc[i].scale_weight;
        img += sc[i].B;
    }
    P.nScales = n; P.totalImages = img;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)num_sms());
    cfg.blockDim = dim3((unsigned)kRescaleThreads);
    cfg.stream = reinterpret_cast<cudaStream_t>(stream);
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, edge_loss_rescale_kernel, P, grad_loss, static_cast<float *>(ctx), expected_out);
    return e == cudaSuccess ? MTE_OK : (int)e;
}
