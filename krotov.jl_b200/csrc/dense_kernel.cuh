// Dense-generator engine (FP64 DMMA complex GEMM per Chebyshev term) -- interface.
#pragma once
#include <cuda_runtime.h>

#include <complex>
#include <string>
#include <vector>

#include "../../include/krotov_cuda.h"

namespace kr {
struct DenseEngine;
struct DenseComm {  // per-iteration view of the rank mailboxes (see krotov_comm_connect)
    int rank = 0, world = 1;
    double *mbox[8] = {};
    int *err_flag = nullptr;
    long long timeout_cycles = 0;
};
void dense_set_comm(DenseEngine *e, const DenseComm &c);
// Non-linear control amplitudes on the device (krotov_set_amplitudes, krotov_set_amplitude_saturation); every pointer
// null = linear controls.
constexpr int kAmpDeg = 4;
struct AmpDev {
    const double *amp_old = nullptr;  // [L][N_T] a_l(eps_old): coefficients of the generator under the known pulses
    const double *dfac = nullptr;     // [L][N_T] a_l'(eps_old): factor of mu_l (src/optimize.jl:337-346)
    const double *poly = nullptr;     // [L][kAmpDeg+1] polynomial coefficients, ascending powers
    const double *shape = nullptr;    // [L][N_T] per-interval factor
    const double *sat = nullptr;      // [L] s_l > 0: the polynomial is evaluated at tanh(s_l eps) (bounded amplitudes)
    double *amp_new = nullptr;        // [L][N_T] a_l(eps_new), written by the pulse update (launch-per-term stream)
    // Tied control terms (krotov_set_control_terms): [L] control of every term (as doubles), then [L][N_T] a_t'(eps_old).
    // nullptr: every term is its own control.
    const double *tie = nullptr;
};
void dense_set_amp(DenseEngine *e, const AmpDev &a);
// Sparse generators (d > 32): ELL description with one shared pattern, slot 0 = diagonal.
struct SparseDesc {
    int W = 0, nnz_union = 0;
    bool hermitian = true;
    const std::vector<int> *cols = nullptr;                     // [d][W]
    const std::vector<std::complex<double>> *vals_f = nullptr;  // [n_gen][1+L][d][W]
    const std::vector<std::complex<double>> *vals_b = nullptr;  // adjoint terms (unused when hermitian)
};
DenseEngine *dense_create(int d, int N, int L, int N_T, int n_gen, const std::vector<std::complex<double>> &Hdense,
                          const std::vector<int> &gen_of_traj, const double *psi0, const double *target, int store_fw,
                          cudaStream_t stream, std::string &err, const SparseDesc *sp = nullptr);
void dense_destroy(DenseEngine *e);
void dense_info(DenseEngine *e, krotov_info *out);
bool dense_set_cheby(DenseEngine *e, int direction, int ndtc, const std::vector<int> &dtc_of_step,
                     const std::vector<double> &E_min, const std::vector<double> &Delta, const std::vector<int> &m,
                     const std::vector<double> &coef, int m_max, const std::vector<std::complex<double>> &phase,
                     std::string &err);
bool dense_seed(DenseEngine *e, double2 *d_tau, std::string &err);
bool dense_forward(DenseEngine *e, const double *d_eps, double2 *d_tau, long long &launches, std::string &err);
bool dense_iterate(DenseEngine *e, const double *d_eps_old, double *d_eps_new, const double *d_alpha,
                   const double *d_dt, double *d_ga, const double2 *d_chi_coef, double2 *d_tau, long long &launches,
                   std::string &err);
bool dense_set_chi(DenseEngine *e, const double *chi_host, std::string &err);
bool dense_get_states(DenseEngine *e, double *states_host, std::string &err);
bool dense_get_storage(DenseEngine *e, int which, int k, int n0, int n1, double *out_host, std::string &err);
}  // namespace kr
