// On-device preparation of the loss targets from their on-disk encoding (sm_100a), SURVEY.md 8(f) rank 2.
//   decode_normals_kernel        u8 PNG value -> edge-normal angle:  (360.*(v/255.) - 180)*(np.pi/180) in float64, then
//                                float32 (packnet_code/packnet_sfm/datasets/gta_dataset.py:413, 421; to_tensor_sample,
//                                datasets/augmentations.py:226-251)
//   resize_depth_preserve (datasets/augmentations.py:58-100) of a u8 edge map to any shape: every valid (> 0) source
//   pixel lands on (int(y*H/h), int(x*W/w)), the LAST one in raster order wins; then the "/255 if max > 1" rule of
//   resize_sample (:193-199) on the max of each RESIZED map, and the float32 cast.
//   same shape                   edge_max_kernel + edge_resize_preserve_kernel: the scatter is the identity, so the
//                                input max is the output max; one pass copies and applies the rule
//   other shapes                 edge_gather_kernel + edge_scale_kernel: each output pixel walks its source block
//                                backwards and the raw values are written, with a mark per image that has a value > 1;
//                                then the rule.  A downsample can drop every value > 1 of an image (a later pixel of
//                                its block wins), so the input max is not the one the rule needs here.
// The cv2.resize of the normal maps (:201-202, 213-217) is NOT reproduced: it runs in float64, where the resize rule
// of resize.cu is not pinned against cv2.resize (DESIGN.md section 2); the reference's own pipeline reads per-scale
// normal PNGs when they exist
// (gta_dataset.py:416-422), which is the case this covers.
#include <math.h>

#include "common.cuh"

namespace mte {
namespace targets {

constexpr int kThreads = 256;

__device__ __forceinline__ float decode_theta(unsigned v) {
    // every step individually rounded as NumPy does (no FMA contraction)
    const double q = __ddiv_rn((double)v, 255.0);
    const double deg = __dadd_rn(__dmul_rn(360.0, q), -180.0);
    return (float)__dmul_rn(deg, M_PI / 180.0);
}

__global__ void __launch_bounds__(kThreads) decode_normals_kernel(const unsigned char *__restrict__ in,
                                                                  float *__restrict__ out, size_t n) {
    __shared__ float lut[256];
    lut[threadIdx.x] = decode_theta(threadIdx.x);
    __syncthreads();
    for (size_t i = (size_t)blockIdx.x * kThreads + threadIdx.x; i < n; i += (size_t)gridDim.x * kThreads) out[i] = lut[in[i]];
}

__global__ void __launch_bounds__(kThreads) edge_max_kernel(const unsigned char *__restrict__ in, int B, size_t hw,
                                                            int *__restrict__ maxOut) {
    const int img = blockIdx.y;
    const unsigned char *p = in + (size_t)img * hw;
    int m = 0;
    for (size_t i = (size_t)blockIdx.x * kThreads + threadIdx.x; i < hw; i += (size_t)gridDim.x * kThreads) m = max(m, (int)p[i]);
    m = __reduce_max_sync(MTE_FULL_MASK, m);
    if ((threadIdx.x & 31) == 0 && m > 0) atomicMax(maxOut + img, m);
}

// first / last source index s in [0, n) with (int)(s * scale) == D, or an empty range
__device__ __forceinline__ void source_range(int D, double scale, int n, int &lo, int &hi) {
    int a = (int)((double)D / scale) - 2, b = (int)((double)(D + 1) / scale) + 2;
    a = max(a, 0); b = min(b, n - 1);
    lo = n; hi = -1;
    for (int s = a; s <= b; s++) {
        if ((int)__dmul_rn((double)s, scale) == D) { lo = min(lo, s); hi = s; }
    }
}

// "if np.max(sample[key]) > 1: sample[key] = sample[key] / 255" in float64, then FloatTensor
__device__ __forceinline__ float apply_max_rule(int v, int mx) { return mx > 1 ? (float)__ddiv_rn((double)v, 255.0) : (float)v; }

// same shape: maxIn[img] is the image's max (edge_max_kernel)
__global__ void __launch_bounds__(kThreads) edge_resize_preserve_kernel(const unsigned char *__restrict__ in, int B, int h,
                                                                        int w, float *__restrict__ out, int H, int W,
                                                                        const int *__restrict__ maxIn) {
    const size_t hw = (size_t)H * W, n = B * hw;
    for (size_t i = (size_t)blockIdx.x * kThreads + threadIdx.x; i < n; i += (size_t)gridDim.x * kThreads)
        out[i] = apply_max_rule(in[i], maxIn[i / hw]);
}

// other shapes: raw values out; mark[img] > 1 once some output value of the image is > 1 (zeroed before)
__global__ void __launch_bounds__(kThreads) edge_gather_kernel(const unsigned char *__restrict__ in, int B, int h, int w,
                                                               float *__restrict__ out, int H, int W,
                                                               int *__restrict__ mark) {
    const double sy = (double)H / (double)h, sx = (double)W / (double)w;  // shape[0] / h, shape[1] / w (:92-93)
    const size_t n = (size_t)B * H * W;
    int marked = -1;                                          // last image this thread has marked
    for (size_t i = (size_t)blockIdx.x * kThreads + threadIdx.x; i < n; i += (size_t)gridDim.x * kThreads) {
        const int X = (int)(i % W), Y = (int)((i / W) % H), img = (int)(i / ((size_t)W * H));
        const unsigned char *src = in + (size_t)img * h * w;
        int v = 0, y0, y1, x0, x1;
        source_range(Y, sy, h, y0, y1);
        source_range(X, sx, w, x0, x1);
        for (int y = y1; y >= y0 && v == 0; y--)              // last valid source pixel in raster order wins (:98)
            for (int x = x1; x >= x0; x--) {
                const int s = src[(size_t)y * w + x];
                if (s > 0) { v = s; break; }
            }
        out[i] = (float)v;
        if (v > 1 && img != marked) { atomicMax(mark + img, v); marked = img; }
    }
}

__global__ void __launch_bounds__(kThreads) edge_scale_kernel(float *__restrict__ out, size_t n, size_t hw,
                                                              const int *__restrict__ mark) {
    for (size_t i = (size_t)blockIdx.x * kThreads + threadIdx.x; i < n; i += (size_t)gridDim.x * kThreads) {
        const int m = mark[i / hw];
        if (m > 1) out[i] = apply_max_rule((int)out[i], m);
    }
}

static int grid_for(size_t n) {
    const size_t b = (n + kThreads - 1) / kThreads;
    return (int)(b < (size_t)num_sms() * 8 ? (b ? b : 1) : (size_t)num_sms() * 8);
}

}  // namespace targets
}  // namespace mte

using namespace mte;
using namespace mte::targets;

extern "C" int mte_decode_normals(const uint8_t *normal_u8, float *theta_out, size_t n, mte_stream_t stream) {
    if (!normal_u8 || !theta_out) return MTE_ERR_NULL;
    if (n == 0) return MTE_ERR_SHAPE;
    decode_normals_kernel<<<grid_for(n), kThreads, 0, reinterpret_cast<cudaStream_t>(stream)>>>(normal_u8, theta_out, n);
    MTE_RETURN_IF_CUDA_ERROR();
    return MTE_OK;
}

extern "C" size_t mte_edge_resize_workspace_bytes(int B) {
    return B < 1 ? 0 : MTE_WS_HEADER_BYTES + align_up((size_t)B * sizeof(int), 256);
}

extern "C" int mte_edge_resize_preserve(const uint8_t *edge_u8, int B, int h, int w, float *edge_out, int H, int W,
                                        void *workspace, size_t ws_bytes, mte_stream_t stream) {
    if (!edge_u8 || !edge_out || !workspace) return MTE_ERR_NULL;
    if (B < 1 || h < 1 || w < 1 || H < 1 || W < 1) return MTE_ERR_SHAPE;
    if (ws_bytes < mte_edge_resize_workspace_bytes(B)) return MTE_ERR_WORKSPACE;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    int *mx = reinterpret_cast<int *>(static_cast<char *>(workspace) + MTE_WS_HEADER_BYTES);
    cudaError_t e = cudaMemsetAsync(mx, 0, (size_t)B * sizeof(int), st);
    if (e != cudaSuccess) return (int)e;
    const size_t n = (size_t)B * H * W;
    if (H == h && W == w) {
        const size_t hw = (size_t)h * w;
        edge_max_kernel<<<dim3((unsigned)min((size_t)64, (hw + kThreads - 1) / kThreads), (unsigned)B), kThreads, 0, st>>>(edge_u8, B, hw, mx);
        edge_resize_preserve_kernel<<<grid_for(n), kThreads, 0, st>>>(edge_u8, B, h, w, edge_out, H, W, mx);
    } else {
        edge_gather_kernel<<<grid_for(n), kThreads, 0, st>>>(edge_u8, B, h, w, edge_out, H, W, mx);
        edge_scale_kernel<<<grid_for(n), kThreads, 0, st>>>(edge_out, n, (size_t)H * W, mx);
    }
    MTE_RETURN_IF_CUDA_ERROR();
    return MTE_OK;
}
