// Morphological thinning for sm_100a.
//
// Replaces py-bsds500 `thin.binary_thin` (not vendored; reference call sites eval_depth_edges.py:45, 125):
// MATLAB bwmorph('thin', Inf) -- two alternating sub-iterations that delete the pixels whose zero-padded 3x3
// neighbourhood satisfies G1 & G2 & G3 (first) or G1 & G2 & G3' (second) of Lam, Lee & Suen, until a
// sub-iteration deletes nothing.  PARITY UNPINNED (restated from the published algorithm, see oracle/thin.py).
//
// One CTA per image: the byte plane is packed into a bit plane, thinned by the bit-parallel routine of thin.cuh and
// unpacked again.  The two bit planes live in dynamic shared memory when they fit (384 x 1280: 2 x 61.4 KB), else in
// the CTA's slice of the workspace.
#include "thin.cuh"

namespace mte {
namespace thin {

__global__ void __launch_bounds__(kThreads) binary_thin_kernel(const unsigned char *__restrict__ in,
                                                               unsigned char *__restrict__ out, unsigned *planes,
                                                               int H, int W, int max_iter, int inSmem) {
    extern __shared__ __align__(16) unsigned dyn[];
    const int nw = words_per_row(W);
    const size_t pw = (size_t)H * nw;
    unsigned *a = inSmem ? dyn : planes + blockIdx.x * 2 * pw;
    unsigned *b = a + pw;
    const size_t plane = (size_t)H * W;
    const unsigned char *src = in + blockIdx.x * plane;
    // pack: one warp per word, one lane per pixel (bits past W stay zero)
    const int lane = threadIdx.x & 31;
    for (size_t i = threadIdx.x >> 5; i < pw; i += kThreads / 32) {
        const int y = (int)(i / nw), x = (int)(i - (size_t)y * nw) * 32 + lane;
        const unsigned m = __ballot_sync(MTE_FULL_MASK, x < W && src[(size_t)y * W + x] != 0);
        if (lane == 0) a[i] = m;
    }
    __syncthreads();
    const unsigned *r = thin_plane(a, b, H, nw, max_iter);
    unsigned char *dst = out + blockIdx.x * plane;
    for (size_t i = threadIdx.x; i < plane; i += kThreads) {
        const int y = (int)(i / W), x = (int)(i - (size_t)y * W);
        dst[i] = (unsigned char)((r[(size_t)y * nw + (x >> 5)] >> (x & 31)) & 1u);
    }
}

static size_t planes_bytes(int H, int W) { return (size_t)2 * H * words_per_row(W) * sizeof(unsigned); }

}  // namespace thin
}  // namespace mte

using namespace mte;

// covers the global-memory bit planes of every image (the shared-memory path needs none of it)
extern "C" size_t mte_thin_workspace_bytes(int N, int H, int W) {
    if (N < 1 || H < 1 || W < 1) return 0;
    return MTE_WS_HEADER_BYTES + align_up((size_t)N * thin::planes_bytes(H, W), 256);
}

extern "C" int mte_binary_thin(const uint8_t *in, uint8_t *out, int N, int H, int W, int max_iter, void *workspace,
                               size_t ws_bytes, mte_stream_t stream) {
    if (!in || !out || !workspace) return MTE_ERR_NULL;
    if (N < 1 || H < 1 || W < 1) return MTE_ERR_SHAPE;
    if (ws_bytes < mte_thin_workspace_bytes(N, H, W)) return MTE_ERR_WORKSPACE;
    const size_t smem = thin::planes_bytes(H, W);
    bool inSmem = smem <= (size_t)dev_info().smemOptin;
    if (inSmem && opt_in_smem((const void *)thin::binary_thin_kernel, (int)smem) != cudaSuccess) {
        cudaGetLastError();
        inSmem = false;
    }
    unsigned *planes = reinterpret_cast<unsigned *>(static_cast<char *>(workspace) + MTE_WS_HEADER_BYTES);
    thin::binary_thin_kernel<<<N, thin::kThreads, inSmem ? smem : 0, reinterpret_cast<cudaStream_t>(stream)>>>(
        in, out, planes, H, W, max_iter, inSmem ? 1 : 0);
    MTE_RETURN_IF_CUDA_ERROR();
    return MTE_OK;
}
