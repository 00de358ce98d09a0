// Instantiations of the streaming (ring) edge-loss backward from the stash (VEC=4).
#include "edge_loss_kernels.cuh"
namespace mte { namespace loss {
void launch_bwd_ring(const LossP &P, bool mask, bool inv, bool sig, cudaStream_t st) {
    MTE_LOSS_DISPATCH_BOOL(mask, MASK, MTE_LOSS_DISPATCH_BOOL(inv, INV, MTE_LOSS_DISPATCH_BOOL(sig, SIG,
        launch_bwd_ring_one<MASK, INV, SIG>(P, st);)))
}
}}  // namespace mte::loss
