// Bilinear resize of predicted depth to the GT size (sm_100a): cv2.resize(depth, (W, H), interpolation=INTER_LINEAR)
// of edge.py:76-78, bit for bit as the opencv-python 4.13.0 wheel computes it for float32 (IPP HAL on, the default;
// DESIGN.md section 2).  Per axis with n_in source and n_out output pixels, output index d:
//   f = (d + 0.5) * (n_in / n_out) - 0.5 in fp64,  s = floor(f),  a = (float)(f - s),  s1 = s + 1;
//   s < 0 or s >= n_in - 1 is a BORDER tap: s and s1 clamp to the nearest source index.
// Horizontal pass first, R = border x ? S[s0x] : fma(S[s1x] - S[s0x], ax, S[s0x]); then the vertical pass,
// out = fma(R[s1y] - R[s0y], ay, R[s0y]) on interior rows, R[s0y] on border rows, and fma(R - R, 0, R) where both taps
// are border taps (an Inf there becomes NaN, as in OpenCV).  Every step is written with an explicit _rn intrinsic so
// that nvcc's contraction cannot change the rounding sequence (oracle/csrc/resize.c restates it on the host).
//
// resize_linear_kernel<VEC>: a thread owns 4 adjacent output columns (their taps computed once) and walks kRowSteps
// rows of one image; VEC = one 16-byte store per row (W % 4 == 0 and a 16-byte aligned output), otherwise 4 scalar
// stores with a tail guard.  Source reads go through the read-only cache (neighbouring threads share taps).
// The same shape is a cudaMemcpyAsync (cv2.resize copies too).
#include <math.h>

#include "common.cuh"

namespace mte {
namespace resize {

constexpr int kColThreads = 64;                 // x: 64 threads x 4 columns = 256 output columns per block
constexpr int kRowThreads = 4;                  // y
constexpr int kRowSteps = 8;                    // rows per thread
constexpr int kBlockRows = kRowThreads * kRowSteps;
constexpr int kMaxGridYZ = 65535;

struct Tap {
    int s0, s1;
    float a;
    bool border;
};

__device__ __forceinline__ Tap tap(int d, int n_in, double scale) {
    const double f = __dadd_rn(__dmul_rn(__dadd_rn((double)d, 0.5), scale), -0.5);
    const double fl = floor(f);
    Tap t;
    t.s0 = (int)fl;
    t.s1 = t.s0 + 1;
    t.a = __double2float_rn(__dsub_rn(f, fl));
    t.border = false;
    if (t.s0 < 0) { t.s0 = t.s1 = 0; t.a = 0.0f; t.border = true; }
    if (t.s0 >= n_in - 1) { t.s0 = t.s1 = n_in - 1; t.a = 0.0f; t.border = true; }
    return t;
}

__device__ __forceinline__ float lerp_h(const float *__restrict__ row, const Tap &t) {
    const float v0 = __ldg(row + t.s0);
    return t.border ? v0 : __fmaf_rn(__fsub_rn(__ldg(row + t.s1), v0), t.a, v0);
}

__device__ __forceinline__ float lerp_v(float r0, float r1, const Tap &ty, const Tap &tx) {
    if (!ty.border) return __fmaf_rn(__fsub_rn(r1, r0), ty.a, r0);
    return tx.border ? __fmaf_rn(__fsub_rn(r0, r0), 0.0f, r0) : r0;
}

template <bool VEC>
__global__ void __launch_bounds__(kColThreads *kRowThreads)
    resize_linear_kernel(const float *__restrict__ src, int N, int h, int w, float *__restrict__ dst, int H, int W,
                         double scale_y, double scale_x) {
    const int X0 = (blockIdx.x * kColThreads + threadIdx.x) * 4;
    if (X0 >= W) return;
    Tap tx[4];
#pragma unroll
    for (int k = 0; k < 4; k++) tx[k] = tap(min(X0 + k, W - 1), w, scale_x);
    const size_t plane_in = (size_t)h * w, plane_out = (size_t)H * W;
    for (int img = blockIdx.z; img < N; img += gridDim.z) {
        const float *S = src + (size_t)img * plane_in;
        float *O = dst + (size_t)img * plane_out;
        for (int Yb = blockIdx.y * kBlockRows; Yb < H; Yb += gridDim.y * kBlockRows) {
#pragma unroll 2
            for (int r = 0; r < kRowSteps; r++) {
                const int Y = Yb + r * kRowThreads + threadIdx.y;
                if (Y >= H) break;
                const Tap ty = tap(Y, h, scale_y);
                const float *a0 = S + (size_t)ty.s0 * w, *a1 = S + (size_t)ty.s1 * w;
                float o[4];
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    const float r0 = lerp_h(a0, tx[k]);
                    const float r1 = ty.border ? r0 : lerp_h(a1, tx[k]);
                    o[k] = lerp_v(r0, r1, ty, tx[k]);
                }
                float *out = O + (size_t)Y * W + X0;
                if (VEC) {
                    st_stream4(out, make_float4(o[0], o[1], o[2], o[3]));
                } else {
#pragma unroll
                    for (int k = 0; k < 4; k++)
                        if (X0 + k < W) out[k] = o[k];
                }
            }
        }
    }
}

}  // namespace resize
}  // namespace mte

using namespace mte;
using namespace mte::resize;

extern "C" int mte_resize_linear(const void *src, int dtype, int n_images, int h, int w, void *dst, int H, int W,
                                 mte_stream_t stream) {
    if (!src || !dst) return MTE_ERR_NULL;
    if (n_images < 1 || h < 1 || w < 1 || H < 1 || W < 1) return MTE_ERR_SHAPE;
    if (dtype != MTE_F32) return MTE_ERR_ARG;                 // fp64 is not pinned against cv2.resize (DESIGN.md)
    if (h < 2 || w < 2) return MTE_ERR_SHAPE;                 // one-row / one-column sources: not pinned either
    if ((reinterpret_cast<uintptr_t>(src) & 3u) || (reinterpret_cast<uintptr_t>(dst) & 3u)) return MTE_ERR_ALIGN;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    if (h == H && w == W) {
        const cudaError_t e = cudaMemcpyAsync(dst, src, sizeof(float) * (size_t)n_images * h * w,
                                              cudaMemcpyDeviceToDevice, st);
        return e == cudaSuccess ? MTE_OK : (int)e;
    }
    const double scale_y = (double)h / (double)H, scale_x = (double)w / (double)W;
    const dim3 block(kColThreads, kRowThreads);
    const dim3 grid((unsigned)(((size_t)W + 4 * kColThreads - 1) / (4 * kColThreads)),
                    (unsigned)min(((size_t)H + kBlockRows - 1) / kBlockRows, (size_t)kMaxGridYZ), (unsigned)min(n_images, kMaxGridYZ));
    const float *s = static_cast<const float *>(src);
    float *d = static_cast<float *>(dst);
    if (W % 4 == 0 && aligned16(dst))
        resize_linear_kernel<true><<<grid, block, 0, st>>>(s, n_images, h, w, d, H, W, scale_y, scale_x);
    else
        resize_linear_kernel<false><<<grid, block, 0, st>>>(s, n_images, h, w, d, H, W, scale_y, scale_x);
    MTE_RETURN_IF_CUDA_ERROR();
    return MTE_OK;
}
