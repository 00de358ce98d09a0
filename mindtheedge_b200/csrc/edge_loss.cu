// Training edge loss for sm_100a: host side of the C ABI + the rarely-used helper kernels.
//
// Replaces (reference paths relative to the reference root):
//   GradLayer.forward           packnet_code/packnet_sfm/losses/grad_loss.py:65-95
//   GradLoss.forward            packnet_code/packnet_sfm/losses/grad_loss.py:122-159
//   GradLoss.comp_cross_entropy packnet_code/packnet_sfm/losses/grad_loss.py:161-219
//   the per-scale loop          packnet_code/packnet_sfm/models/SemiSupEdgeModel.py:164-198
//   inv2depth (optional fuse)   packnet_code/packnet_sfm/utils/depth.py:104-121
// and the autograd backward of that chain (SURVEY.md A.1).  The hot kernels live in
// edge_loss_kernels.cuh and are instantiated in edge_loss_{fwd,bwd}_v{4,1}.cu.
#include <stdlib.h>
#include <string.h>

#include "edge_loss_kernels.cuh"

namespace mte {
namespace loss {

// is_grad == 0 (DEE-training mode, EdgeEstimationLIDARModel.py:139-144): the loss acts on the map
// itself, the backward is pointwise.
template <bool MASK>
__global__ void __launch_bounds__(kThreads) edge_loss_bwd_pointwise_kernel(const __grid_constant__ LossP P,
                                                                           int isSigmoid, int predInv) {
    for (int si = 0; si < P.nScales; si++) {
        const ScaleP &S = P.s[si];
        const size_t npix = (size_t)S.H * S.W;
        const size_t n = npix * S.B;
        const float G = __ldg(P.gradLoss) * S.scaleWeight + __ldg(P.gradLoss + 1 + si);
        const float coef = __ldg(P.ctx + P.totalImages + 2 * si) * G;
        const bool binary = MASK && (__ldg(P.ctx + P.totalImages + 2 * si + 1) != 0.f);
        for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
            const int img = (int)(i / npix);
            const float alpha = __ldg(P.ctx + S.imgBase + img);
            BwdImg I{-coef * P.p2n * alpha, coef * (1.0f - alpha), binary};
            const float xv = S.x[i];
            const float dep = predInv ? inv_to_depth(xv) : xv;
            const float mm = MASK ? S.m[i] : 1.f;
            float d = isSigmoid ? dloss_dg<MASK, true>(dep, S.e[i], mm, I, P.T)
                                : dloss_dg<MASK, false>(dep, S.e[i], mm, I, P.T);
            if (predInv) d = (dep < 1e6f) ? -d * dep * dep : 0.f;
            S.dx[i] = d;
        }
    }
}

// ---------------------------------------------------------------------------
// Bilinear resize (F.interpolate(mode='bilinear', align_corners=False),
// grad_loss.py:127) -- only used when the prediction and target sizes differ.
// ---------------------------------------------------------------------------
// fp32 source coordinate, rounded once (fused multiply-add): this is what the reference's fp32 interpolation yields
// (oracle bilinear_matrix restates it); at non-dyadic scales a second rounding moves the weights by up to 1e-4.
__device__ __forceinline__ void src_index(int o, float scale, int n, int &i0, int &i1, float &f) {
    float s = fmaf(scale, (float)o + 0.5f, -0.5f);
    s = s < 0.f ? 0.f : s;
    i0 = min((int)s, n - 1);
    i1 = min(i0 + 1, n - 1);
    f = s - (float)i0;
}

__global__ void resize_fwd_kernel(const float *__restrict__ in, float *__restrict__ out, int B, int h, int w, int H,
                                  int W) {
    const float sy = (float)h / (float)H, sx = (float)w / (float)W;
    const size_t n = (size_t)B * H * W;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const int X = (int)(i % W), Y = (int)((i / W) % H), b = (int)(i / ((size_t)W * H));
        int y0, y1, x0, x1;
        float fy, fx;
        src_index(Y, sy, h, y0, y1, fy);
        src_index(X, sx, w, x0, x1, fx);
        const float *p = in + (size_t)b * h * w;
        out[i] = (1.f - fy) * ((1.f - fx) * p[(size_t)y0 * w + x0] + fx * p[(size_t)y0 * w + x1]) +
                 fy * ((1.f - fx) * p[(size_t)y1 * w + x0] + fx * p[(size_t)y1 * w + x1]);
    }
}

// Deterministic adjoint: every source pixel gathers from the destination pixels that read it.
__global__ void resize_bwd_kernel(const float *__restrict__ gout, float *__restrict__ gin, int B, int h, int w, int H,
                                  int W) {
    const float sy = (float)h / (float)H, sx = (float)w / (float)W;
    const size_t n = (size_t)B * h * w;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const int x = (int)(i % w), y = (int)((i / w) % h), b = (int)(i / ((size_t)w * h));
        // destination rows/cols whose source interval can touch (y, x)
        int Y0 = (int)floorf(((float)y - 1.0f + 0.5f) / sy - 0.5f) - 1, Y1 = (int)ceilf(((float)y + 1.0f + 0.5f) / sy - 0.5f) + 1;
        int X0 = (int)floorf(((float)x - 1.0f + 0.5f) / sx - 0.5f) - 1, X1 = (int)ceilf(((float)x + 1.0f + 0.5f) / sx - 0.5f) + 1;
        if (y == 0) Y0 = 0;
        if (x == 0) X0 = 0;
        if (y == h - 1) Y1 = H - 1;
        if (x == w - 1) X1 = W - 1;
        Y0 = max(Y0, 0); X0 = max(X0, 0); Y1 = min(Y1, H - 1); X1 = min(X1, W - 1);
        const float *g = gout + (size_t)b * H * W;
        // fp64 sum: a large upsampling gathers thousands of terms of both signs into one source pixel (1x1 -> 96x97:
        // 9312), where an fp32 running sum drifts by ~5e-5 of the result
        double acc = 0.0;
        for (int Y = Y0; Y <= Y1; Y++) {
            int a0, a1; float fy;
            src_index(Y, sy, h, a0, a1, fy);
            float wy = 0.f;
            if (a0 == y) wy += 1.f - fy;
            if (a1 == y) wy += fy;
            if (wy == 0.f) continue;
            for (int X = X0; X <= X1; X++) {
                int b0, b1; float fx;
                src_index(X, sx, w, b0, b1, fx);
                float wx = 0.f;
                if (b0 == x) wx += 1.f - fx;
                if (b1 == x) wx += fx;
                if (wx != 0.f) acc += (double)(wy * wx) * (double)g[(size_t)Y * W + X];
            }
        }
        gin[i] = (float)acc;
    }
}

// ---------------------------------------------------------------------------
// Host side
// ---------------------------------------------------------------------------
constexpr int kFwdCtaWaves = 2, kBwdCtaWaves = 16;

struct Plan {
    LossP P;
    bool vec, hasNormal, hasMask, isGrad;
    size_t offAccum, accumBytes, offResize[MTE_MAX_SCALES], offResizeDx[MTE_MAX_SCALES], total;
    int fwdGrid;
    bool resized[MTE_MAX_SCALES];
};

static int validate(const mte_loss_scale_t *sc, int n) {
    if (!sc) return MTE_ERR_NULL;
    if (n < 1 || n > MTE_MAX_SCALES) return MTE_ERR_ARG;
    for (int i = 0; i < n; i++) {
        if (!sc[i].pred || !sc[i].edge) return MTE_ERR_NULL;
        if (sc[i].B < 1 || sc[i].h < 1 || sc[i].w < 1 || sc[i].H < 1 || sc[i].W < 1) return MTE_ERR_SHAPE;
        if ((sc[i].normal != nullptr) != (sc[0].normal != nullptr)) return MTE_ERR_ARG;
        if ((sc[i].mask != nullptr) != (sc[0].mask != nullptr)) return MTE_ERR_ARG;
        const void *ptrs[] = {sc[i].pred, sc[i].edge, sc[i].normal, sc[i].mask, sc[i].grad_map, sc[i].grad_pred};
        for (const void *p : ptrs)
            if (reinterpret_cast<uintptr_t>(p) & 3u) return MTE_ERR_ALIGN;
    }
    return MTE_OK;
}

// Lay out CTAs / workspace.  bwd == true uses the overlapped 30-lane strips.
static bool can_use_stash(const mte_loss_scale_t *sc, int n, const mte_loss_attrs_t *at) {
    if (!at || !at->is_grad || debug_knob("MTE_LOSS_NO_STASH")) return false;
    for (int i = 0; i < n; i++) {
        if (!sc[i].stash || !sc[i].grad_map || !sc[i].normal) return false;
        if (sc[i].h != sc[i].H || sc[i].w != sc[i].W) return false;
    }
    return true;
}

static int make_plan(Plan &pl, const mte_loss_scale_t *sc, int n, const mte_loss_attrs_t *at, bool bwd) {
    int rc = validate(sc, n);
    if (rc) return rc;
    LossP &P = pl.P;
    memset(&P, 0, sizeof(P));
    pl.hasNormal = sc[0].normal != nullptr;
    pl.hasMask = sc[0].mask != nullptr;
    pl.isGrad = at ? at->is_grad != 0 : true;
    pl.vec = true;
    for (int i = 0; i < n; i++) {
        if (sc[i].W % 4) pl.vec = false;
        // the kernels read the (possibly resized) prediction at target resolution
        const void *ptrs[] = {sc[i].edge, sc[i].normal, sc[i].mask, sc[i].grad_map};
        for (const void *p : ptrs)
            if (!aligned16(p)) pl.vec = false;
        if (reinterpret_cast<uintptr_t>(sc[i].stash) & 3u) pl.vec = false;
        const bool rs = sc[i].h != sc[i].H || sc[i].w != sc[i].W;
        if (!rs && (!aligned16(sc[i].pred) || (bwd && !aligned16(sc[i].grad_pred)))) pl.vec = false;
    }
    const int VEC = pl.vec ? 4 : 1;
    const int RH = bwd ? kBwdRH : kFwdRH;
    const bool stashBwd = bwd && can_use_stash(sc, n, at);
    const int lanesOut = !pl.isGrad ? 32 : ((bwd && !stashBwd) ? bwd_lanes(VEC) : kHaloLanes);
    int cta = 0, img = 0;
    long long unitBase = 0;
    for (int i = 0; i < n; i++) {
        ScaleP &S = P.s[i];
        S.B = sc[i].B; S.H = sc[i].H; S.W = sc[i].W;
        S.e = sc[i].edge; S.n = sc[i].normal; S.m = sc[i].mask; S.g = sc[i].grad_map; S.dx = sc[i].grad_pred;
        S.stash = sc[i].stash;
        S.x = sc[i].pred;
        S.strips = ceil_div(S.W, lanesOut * VEC);
        S.rowBlocks = ceil_div(S.H, RH);
        S.items = S.strips * S.rowBlocks;
        S.ctasPerImage = ceil_div(S.items, kWarps);  // capped below: warps loop over several items
        S.ctaBase = cta; S.imgBase = img;
        S.unitBase = (int)unitBase;
        unitBase += (long long)S.strips * (S.H + (bwd ? kSegCostB : kSegCost)) * S.B;
        S.scaleWeight = sc[i].scale_weight;
        cta += S.ctasPerImage * S.B;
        img += S.B;
        pl.resized[i] = sc[i].h != sc[i].H || sc[i].w != sc[i].W;
    }
    // Cap the grid near kCtaWaves resident waves so the per-CTA epilogue (partials, ticket) is amortised over
    // several items per warp; every scale keeps at least one CTA per image.
    // measured on B200 (profiles/r01_notes.md): the forward (per-CTA reduction epilogue) likes ~2 resident waves,
    // the backward (no epilogue) only needs enough CTAs for the hardware scheduler to balance the tail
    int waves = bwd ? kBwdCtaWaves : kFwdCtaWaves;
    if (const char *e = debug_knob("MTE_CTA_WAVES")) waves = atoi(e) > 0 ? atoi(e) : waves;  // tuning knob
    const int cap = num_sms() * 2 * waves;
    if (cta > cap) {
        const double shrink = (double)cap / (double)cta;
        cta = 0;
        for (int i = 0; i < n; i++) {
            ScaleP &S = P.s[i];
            int c = (int)(S.ctasPerImage * shrink);
            S.ctasPerImage = c < 1 ? 1 : c;
            S.ctaBase = cta;
            cta += S.ctasPerImage * S.B;
        }
    }
    P.nScales = n; P.totalCtas = cta; P.totalImages = img;
    if (unitBase > 0x7fffffffLL) return MTE_ERR_SHAPE;
    P.totalUnits = (int)unitBase;
    // forward: persistent CTAs (2 per SM), every warp owns an equal contiguous range of strip rows (at least a few
    // rows each, so the window prologue is amortised)
    pl.fwdGrid = num_sms() * kRGridB;
    const int minRows = 4;
    if ((long long)pl.fwdGrid * kRWarps * minRows > unitBase) pl.fwdGrid = (int)((unitBase + kRWarps * minRows - 1) / (kRWarps * minRows));
    if (pl.fwdGrid < 1) pl.fwdGrid = 1;
    if (at) {
        P.T = at->sigmoid_thresh; P.weight = at->weight; P.p2n = at->pos_to_neg;
    }
    size_t off = MTE_WS_HEADER_BYTES;
    // forward: the per-image fixed-point accumulators live in the zero-initialised workspace header and are left
    // zero by the kernel (no memset node per launch)
    pl.offAccum = kWsAccumOffset;
    pl.accumBytes = (size_t)img * kAcc * sizeof(unsigned long long);
    if (img > kWsMaxLossImages) return MTE_ERR_SHAPE;
    for (int i = 0; i < n; i++) {
        const size_t planeBytes = align_up((size_t)sc[i].B * sc[i].H * sc[i].W * sizeof(float), 256);
        pl.offResize[i] = off;
        if (pl.resized[i]) off += planeBytes;
        pl.offResizeDx[i] = off;
        if (pl.resized[i]) off += planeBytes;
    }
    pl.total = off;
    return MTE_OK;
}

}  // namespace loss
}  // namespace mte

using namespace mte;
using namespace mte::loss;

extern "C" size_t mte_edge_loss_workspace_bytes(const mte_loss_scale_t *sc, int n) {
    Plan pl;
    if (make_plan(pl, sc, n, nullptr, false)) return 0;
    return pl.total;
}

extern "C" size_t mte_edge_loss_ctx_bytes(const mte_loss_scale_t *sc, int n) {
    if (validate(sc, n)) return 0;
    size_t imgs = 0;
    for (int i = 0; i < n; i++) imgs += sc[i].B;
    // alpha per image, {coef, maskBinary} per scale, then (one-pass variant) the factor grad_pred carries per scale and
    // the rescale kernel's ticket
    return align_up((imgs + 3 * MTE_MAX_SCALES + 4) * sizeof(float), 16);
}

extern "C" int mte_edge_loss_fwd(const mte_loss_scale_t *sc, int n, const mte_loss_attrs_t *at, float *loss_out,
                                 void *ctx, void *ws, size_t ws_bytes, mte_stream_t stream) {
    if (!at || !loss_out || !ctx || !ws) return MTE_ERR_NULL;
    Plan pl;
    int rc = make_plan(pl, sc, n, at, false);
    if (rc) return rc;
    if (ws_bytes < pl.total) return MTE_ERR_WORKSPACE;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    char *w = static_cast<char *>(ws);
    LossP &P = pl.P;
    P.accum = reinterpret_cast<unsigned long long *>(w + pl.offAccum);
    P.ticket = reinterpret_cast<WsHeader *>(w)->ticket;
    P.totalCtas = pl.fwdGrid;
    P.lossOut = loss_out;
    P.ctx = static_cast<float *>(ctx);
    for (int i = 0; i < n; i++) {
        if (pl.resized[i]) {
            float *tmp = reinterpret_cast<float *>(w + pl.offResize[i]);
            const size_t npx = (size_t)sc[i].B * sc[i].H * sc[i].W;
            const int grid = (int)((npx + 255) / 256 < 148 * 16 ? (npx + 255) / 256 : 148 * 16);
            resize_fwd_kernel<<<grid, 256, 0, st>>>(sc[i].pred, tmp, sc[i].B, sc[i].h, sc[i].w, sc[i].H, sc[i].W);
            P.s[i].x = tmp;
        }
    }
    const int mode = !at->is_grad ? MODE_NONE : (pl.hasNormal ? MODE_DIR : MODE_MAG);
    // a resized prediction is already a depth map in the workspace only if inv2depth is applied after the
    // resize, as the reference does not: inv2depth precedes the head (SemiSupEdgeModel.py:166,187)
    for (int i = 0; i < n; i++)
        if (pl.resized[i] && at->pred_is_inverse) return MTE_ERR_ARG;
    if (pl.vec) launch_fwd_v4(P, mode, pl.hasMask, at->pred_is_inverse != 0, at->is_sigmoid != 0, st);
    else launch_fwd_v1(P, mode, pl.hasMask, at->pred_is_inverse != 0, at->is_sigmoid != 0, st);
    MTE_RETURN_IF_CUDA_ERROR();
    return MTE_OK;
}

extern "C" int mte_edge_loss_bwd(const mte_loss_scale_t *sc, int n, const mte_loss_attrs_t *at,
                                 const float *grad_loss, const void *ctx, void *ws, size_t ws_bytes,
                                 mte_stream_t stream) {
    if (!at || !grad_loss || !ctx || !ws) return MTE_ERR_NULL;
    Plan pl;
    int rc = make_plan(pl, sc, n, at, true);
    if (rc) return rc;
    for (int i = 0; i < n; i++)
        if (!sc[i].grad_pred) return MTE_ERR_NULL;
    if (ws_bytes < pl.total) return MTE_ERR_WORKSPACE;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    char *w = static_cast<char *>(ws);
    LossP &P = pl.P;
    P.ctx = const_cast<float *>(static_cast<const float *>(ctx));
    P.gradLoss = grad_loss;
    for (int i = 0; i < n; i++) {
        if (pl.resized[i]) {
            // recompute the resized prediction (the workspace is not carried from the forward)
            float *tmp = reinterpret_cast<float *>(w + pl.offResize[i]);
            const size_t npx = (size_t)sc[i].B * sc[i].H * sc[i].W;
            const int grid = (int)((npx + 255) / 256 < 148 * 16 ? (npx + 255) / 256 : 148 * 16);
            resize_fwd_kernel<<<grid, 256, 0, st>>>(sc[i].pred, tmp, sc[i].B, sc[i].h, sc[i].w, sc[i].H, sc[i].W);
            P.s[i].x = tmp;
        }
    }
    // resized scales: the gradient is produced at target resolution, then pulled back by the resize adjoint
    for (int i = 0; i < n; i++)
        if (pl.resized[i]) P.s[i].dx = reinterpret_cast<float *>(w + pl.offResizeDx[i]);
    for (int i = 0; i < n; i++)
        if (pl.resized[i] && at->pred_is_inverse) return MTE_ERR_ARG;
    if (!at->is_grad) {
        if (pl.hasMask)
            edge_loss_bwd_pointwise_kernel<true><<<num_sms() * 8, kThreads, 0, st>>>(P, at->is_sigmoid, at->pred_is_inverse);
        else
            edge_loss_bwd_pointwise_kernel<false><<<num_sms() * 8, kThreads, 0, st>>>(P, at->is_sigmoid, at->pred_is_inverse);
    } else {
        const int mode = pl.hasNormal ? MODE_DIR : MODE_MAG;
        if (can_use_stash(sc, n, at)) {
            if (pl.vec && !debug_knob("MTE_LOSS_BWD_OLD")) {
                P.totalCtas = pl.fwdGrid;  // persistent grid over the cost-balanced unit ranges
                launch_bwd_ring_v4(P, pl.hasMask, at->pred_is_inverse != 0, at->is_sigmoid != 0, st);
            } else if (pl.vec) launch_bwd_stash_v4(P, pl.hasMask, at->pred_is_inverse != 0, at->is_sigmoid != 0, st);
            else launch_bwd_stash_v1(P, pl.hasMask, at->pred_is_inverse != 0, at->is_sigmoid != 0, st);
        } else if (pl.vec) launch_bwd_v4(P, mode, pl.hasMask, at->pred_is_inverse != 0, at->is_sigmoid != 0, st);
        else launch_bwd_v1(P, mode, pl.hasMask, at->pred_is_inverse != 0, at->is_sigmoid != 0, st);
    }
    MTE_RETURN_IF_CUDA_ERROR();
    for (int i = 0; i < n; i++) {
        if (pl.resized[i]) {
            const size_t npx = (size_t)sc[i].B * sc[i].h * sc[i].w;
            const int grid = (int)((npx + 255) / 256 < 148 * 16 ? (npx + 255) / 256 : 148 * 16);
            resize_bwd_kernel<<<grid, 256, 0, st>>>(P.s[i].dx, sc[i].grad_pred, sc[i].B, sc[i].h, sc[i].w, sc[i].H,
                                                   sc[i].W);
        }
    }
    MTE_RETURN_IF_CUDA_ERROR();
    return MTE_OK;
}
