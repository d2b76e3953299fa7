// K5 sampler kernels of kernel family 2 (Matern-5/2): see ensemble_kernel.cuh
#include "ensemble_kernel.cuh"

int ab_ens_launch_k2(ab_gp* h, EnsArgs& A, int n_half, int p, bool small_cta, int ws) {
    return launch_ens_kind<2>(h, A, n_half, p, small_cta, ws);
}
