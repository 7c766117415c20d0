// likelihood_kernels.cuh -- declarations of the kernels of likelihood_kernels.cu (launched by rbo_api.cu).
#pragma once
#include "rbo_device.cuh"

namespace rbo {

// Matrices of the likelihood are padded to NP = a multiple of RBO_LK_B rows (identity on the padding: K_pad = diag(K, I)), row-major
// with pitch NP; every kernel below works on whole RBO_LK_B x RBO_LK_B tiles.
#define RBO_LK_B 64
#define RBO_LK_THREADS 256
// dynamic shared memory of rbo_lik_potrf_diag_kernel: the block and its inverse
#define RBO_LK_DIAG_SMEM (2 * RBO_LK_B * (RBO_LK_B + 1) * 8)

__global__ void rbo_lik_assemble_kernel(const double* Xpts, int d, int N, int NP, KernelSpec kern, double kdiag, double* A);
__global__ void rbo_lik_potrf_diag_kernel(double* A, int NP, int kb, double* Dinv, double* diagL, int* status);
__global__ void rbo_lik_panel_kernel(double* A, int NP, int kb, const double* Dinv);
__global__ void rbo_lik_update_kernel(double* A, int NP, int kb);
__global__ void rbo_lik_trinv_row_kernel(const double* A, int NP, int i, const double* Dinv, double* W);
__global__ void rbo_lik_lauum_kernel(const double* W, int NP, double* Kinv);
__global__ void rbo_lik_grad_kernel(const double* Xpts, int d, int N, int NP, KernelSpec kern, const double* a, const double* Kinv, double* partial);
__global__ void rbo_lik_final_kernel(const double* y, const double* a, const double* diagL, int N, const double* partial, int ntiles, int nk,
                                     double* out);
__global__ void rbo_lik_to_colmajor_kernel(const double* A, int NP, int N, double* L);

}  // namespace rbo
