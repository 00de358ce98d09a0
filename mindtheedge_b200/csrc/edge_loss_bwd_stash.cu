// Instantiations of the stash-based edge-loss backward (VEC=1).
#include "edge_loss_kernels.cuh"
namespace mte { namespace loss {
void launch_bwd_stash(const LossP &P, bool mask, bool inv, bool sig, cudaStream_t st) {
    MTE_LOSS_DISPATCH_BOOL(mask, MASK, MTE_LOSS_DISPATCH_BOOL(inv, INV, MTE_LOSS_DISPATCH_BOOL(sig, SIG,
        edge_loss_bwd_stash_kernel<MASK, INV, SIG><<<P.totalCtas, kThreads, 0, st>>>(P);)))
}
}}  // namespace mte::loss
