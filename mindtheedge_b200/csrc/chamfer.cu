// In-training "light" edge metric (sm_100a): chamfer_distance
//   packnet_code/packnet_sfm/utils/edge.py:20-62, called twice per Canny setting (pred->gt, gt->pred) by
//   ModelWrapper.compute_edge_metrics, packnet_code/packnet_sfm/models/model_wrapper.py:376-442
// The reference runs scipy.ndimage.distance_transform_edt over the whole plane and then only looks at the distances
// under the predicted pixels.  Here the exact squared Euclidean distance is computed only THERE:
//   1. col_dist_kernel   per column, the vertical distance g(y, x) to the nearest GT pixel of that column (two
//                        sequential sweeps per column, coalesced across columns), u16, 0xFFFF = none
//   2. row_eval_kernel   per predicted pixel, min over x' of (x - x')^2 + g(y, x')^2 searched outwards from x and cut
//                        off as soon as k^2 >= best (exact); integer d^2, then sqrt in fp64 as scipy does; the sum,
//                        the pixel count and the "closer than thresh" count are reduced per row in a fixed order
//   3. finish_kernel     per image, the row partials in a fixed order -> out[N,4]
// An image without any GT pixel reproduces scipy's convention (scipy 1.x: as if one background sample sat at row -1, column 0).
#include "common.cuh"

namespace mte {
namespace chamfer {

constexpr unsigned short kNone = 0xFFFF;
constexpr int kThreads = 256;

__device__ __forceinline__ bool is_set(unsigned char v) { return v >= 128; }  // v / 255 > 0.5  (edge.py:30-31, 39-40)

__global__ void __launch_bounds__(kThreads) col_dist_kernel(const unsigned char *__restrict__ gt,
                                                            unsigned short *__restrict__ g, int *__restrict__ hasGt,
                                                            int N, int H, int W) {
    const int idx = blockIdx.x * kThreads + threadIdx.x;
    if (idx >= N * W) return;
    const int img = idx / W, x = idx - img * W;
    const unsigned char *src = gt + (size_t)img * H * W + x;
    unsigned short *dst = g + (size_t)img * H * W + x;
    unsigned d = kNone;
    bool any = false;
    for (int y = 0; y < H; y++) {
        const bool s = is_set(src[(size_t)y * W]);
        any |= s;
        d = s ? 0u : (d >= kNone - 1u ? (unsigned)kNone : d + 1u);
        dst[(size_t)y * W] = (unsigned short)d;
    }
    d = kNone;
    for (int y = H - 1; y >= 0; y--) {
        const bool s = is_set(src[(size_t)y * W]);
        d = s ? 0u : (d >= kNone - 1u ? (unsigned)kNone : d + 1u);
        const unsigned old = dst[(size_t)y * W];
        if (d < old) dst[(size_t)y * W] = (unsigned short)d;
    }
    if (any) atomicOr(hasGt + img, 1);
}

__global__ void __launch_bounds__(kThreads) row_eval_kernel(const unsigned char *__restrict__ pred,
                                                            const unsigned short *__restrict__ g,
                                                            const int *__restrict__ hasGt, int H, int W, double thresh,
                                                            double *__restrict__ partial, signed char *__restrict__ cond) {
    extern __shared__ unsigned short sg[];  // this row of g
    __shared__ double sSum[kThreads / 32];
    __shared__ long long sCnt[kThreads / 32], sClose[kThreads / 32];
    const int y = blockIdx.x, img = blockIdx.y;
    const size_t row = ((size_t)img * H + y) * W;
    for (int x = threadIdx.x; x < W; x += kThreads) sg[x] = g[row + x];
    __syncthreads();
    const bool any = hasGt[img] != 0;
    double sum = 0.0;
    long long cnt = 0, close = 0;
    for (int x = threadIdx.x; x < W; x += kThreads) {
        signed char c = -1;
        if (is_set(pred[row + x])) {
            unsigned long long best;
            if (!any) {
                best = (unsigned long long)(y + 1) * (y + 1) + (unsigned long long)x * x;
            } else {
                best = ~0ull;
                const unsigned g0 = sg[x];
                if (g0 != kNone) best = (unsigned long long)g0 * g0;
                for (unsigned long long k = 1; k * k < best; k++) {
                    const long long xl = (long long)x - (long long)k, xr = (long long)x + (long long)k;
                    if (xl < 0 && xr >= W) break;
                    if (xl >= 0) {
                        const unsigned gv = sg[xl];
                        if (gv != kNone) { const unsigned long long c2 = k * k + (unsigned long long)gv * gv; if (c2 < best) best = c2; }
                    }
                    if (xr < W) {
                        const unsigned gv = sg[xr];
                        if (gv != kNone) { const unsigned long long c2 = k * k + (unsigned long long)gv * gv; if (c2 < best) best = c2; }
                    }
                }
            }
            const double dist = sqrt((double)best);
            sum += dist;
            cnt++;
            const bool cl = dist < thresh;  // edge.py:53
            close += cl ? 1 : 0;
            c = cl ? 1 : 0;
        }
        if (cond) cond[row + x] = c;
    }
    // fixed-order reduction: lanes (butterfly), then warps in order
    sum = warp_sum(sum);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        cnt += __shfl_xor_sync(MTE_FULL_MASK, cnt, o);
        close += __shfl_xor_sync(MTE_FULL_MASK, close, o);
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) { sSum[warp] = sum; sCnt[warp] = cnt; sClose[warp] = close; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0;
        long long c = 0, k = 0;
        for (int i = 0; i < kThreads / 32; i++) { s += sSum[i]; c += sCnt[i]; k += sClose[i]; }
        double *p = partial + ((size_t)img * H + y) * 3;
        p[0] = s; p[1] = (double)c; p[2] = (double)k;
    }
}

__global__ void __launch_bounds__(32) finish_kernel(const double *__restrict__ partial, int H, double *__restrict__ out) {
    const int img = blockIdx.x, lane = threadIdx.x;
    double s = 0.0, c = 0.0, k = 0.0;
    for (int y = lane; y < H; y += 32) {
        const double *p = partial + ((size_t)img * H + y) * 3;
        s += p[0]; c += p[1]; k += p[2];
    }
    s = warp_sum(s); c = warp_sum(c); k = warp_sum(k);
    if (lane == 0) {
        out[(size_t)img * 4 + 0] = s;
        out[(size_t)img * 4 + 1] = c;
        out[(size_t)img * 4 + 2] = k;
        out[(size_t)img * 4 + 3] = 0.0;
    }
}

struct Layout {
    size_t offG, offHas, offPartial, total;
};
static Layout layout(int N, int H, int W) {
    Layout L;
    size_t off = MTE_WS_HEADER_BYTES;
    L.offG = off; off += align_up((size_t)N * H * W * sizeof(unsigned short), 256);
    L.offHas = off; off += align_up((size_t)N * sizeof(int), 256);
    L.offPartial = off; off += align_up((size_t)N * H * 3 * sizeof(double), 256);
    L.total = off;
    return L;
}

}  // namespace chamfer
}  // namespace mte

using namespace mte;
using namespace mte::chamfer;

extern "C" size_t mte_chamfer_workspace_bytes(int N, int H, int W) {
    if (N < 1 || H < 1 || W < 1) return 0;
    return layout(N, H, W).total;
}

extern "C" int mte_chamfer_counts(const uint8_t *pred, const uint8_t *gt, int N, int H, int W, double thresh,
                                  double *out, int8_t *cond_out, void *workspace, size_t ws_bytes,
                                  mte_stream_t stream) {
    if (!pred || !gt || !out || !workspace) return MTE_ERR_NULL;
    if (N < 1 || H < 1 || W < 1) return MTE_ERR_SHAPE;
    if (H >= 0xFFFE || W > 24 * 1024) return MTE_ERR_SHAPE;  // u16 column distances; one row of them in shared memory
    const Layout L = layout(N, H, W);
    if (ws_bytes < L.total) return MTE_ERR_WORKSPACE;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    char *w = static_cast<char *>(workspace);
    unsigned short *g = reinterpret_cast<unsigned short *>(w + L.offG);
    int *has = reinterpret_cast<int *>(w + L.offHas);
    double *partial = reinterpret_cast<double *>(w + L.offPartial);
    cudaError_t e = cudaMemsetAsync(has, 0, (size_t)N * sizeof(int), st);
    if (e != cudaSuccess) return (int)e;
    // a row of u16 distances plus the kernel's static reduction buffers passes the 48 KB a launch gets without the
    // opt-in from W = 24,481 on; opting in below that is harmless
    const size_t rowSmem = (size_t)W * sizeof(unsigned short);
    if (rowSmem > 32 * 1024) {
        e = opt_in_smem((const void *)row_eval_kernel, (int)rowSmem);
        if (e != cudaSuccess) return (int)e;
    }
    col_dist_kernel<<<ceil_div(N * W, kThreads), kThreads, 0, st>>>(gt, g, has, N, H, W);
    MTE_RETURN_IF_CUDA_ERROR();
    row_eval_kernel<<<dim3((unsigned)H, (unsigned)N), kThreads, rowSmem, st>>>(
        pred, g, has, H, W, thresh, partial, reinterpret_cast<signed char *>(cond_out));
    MTE_RETURN_IF_CUDA_ERROR();
    finish_kernel<<<N, 32, 0, st>>>(partial, H, out);
    MTE_RETURN_IF_CUDA_ERROR();
    return MTE_OK;
}
