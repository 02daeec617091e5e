// libkrotov_cuda: C ABI (include/krotov_cuda.h) + host-side preparation for the sm_100a kernels.
//
// Host work done here (all of it outside the per-time-step path):
//   * union sparsity pattern of all generator terms, slot assignment (per-diagonal when possible)
//   * per-direction row tables P_t = 2c (H_t - beta delta_t0) rebuilt whenever the Chebyshev
//     polynomial changes (krotov_set_cheby)
//   * launch configuration of the persistent kernel, exchange-array reset, CUDA-event timing
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <complex>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <set>
#include <string>
#include <vector>

#include <thread>

#include "../../include/krotov_cuda.h"
#include "dense_kernel.cuh"
#include "device_buffer.cuh"
#include "warp_kernel.cuh"
#include "warp2_kernel.cuh"
#include "tiny_kernel.cuh"
#include "kernel_table.h"

using cplx = std::complex<double>;

constexpr int kXaccMaxStride = 16;  // accumulator words of the cross-rank sum at most one 128-byte line apart

namespace {

thread_local std::string g_create_error = "";

// KROTOV_TRACE=1 prints host-side timings of the non-hot-path entry points to stderr
struct Trace {
    const char *what;
    std::chrono::steady_clock::time_point t0;
    bool on;
    explicit Trace(const char *w) : what(w), t0(std::chrono::steady_clock::now()), on(getenv("KROTOV_TRACE") != nullptr) {}
    void lap(const char *label) {
        if (!on) return;
        auto t1 = std::chrono::steady_clock::now();
        fprintf(stderr, "[krotov trace] %s: %s %.3f ms\n", what, label, std::chrono::duration<double, std::milli>(t1 - t0).count());
        t0 = t1;
    }
};

using kr::DevBuf;

struct HostSparse {  // ELL description of a sparse generator family (d > 32), slot 0 = diagonal
    int W = 0, nnz_union = 0;
    bool hermitian = true;
    std::vector<int> cols;
    std::vector<cplx> vals_f, vals_b;
};

struct ChebyTables {  // one direction
    bool set = false;
    int ndtc = 0, mmax = 0, m_max_used = 0;
    std::vector<double> E_min, Delta;
    DevBuf coef, m, phase, dtc;
    std::vector<int> dtc_of_step;
    std::vector<int> m_host;
    std::vector<double> coef_host;
    std::vector<cplx> phase_host;
};

// the handle's stream and timing events: a base of krotov_handle_s, so they are destroyed after every member
struct HandleStream {
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    ~HandleStream() {
        if (ev0) cudaEventDestroy(ev0);
        if (ev1) cudaEventDestroy(ev1);
        if (stream) cudaStreamDestroy(stream);
    }
};

}  // namespace

struct krotov_handle_s : HandleStream {
    int d = 0, N = 0, L = 0, N_T = 0, n_gen = 0, functional = 0, N_global = 0, store_fw = 0, device = 0;
    int path = 0;
    std::vector<double> tlist, dt;
    std::vector<int> gen_of_traj;
    std::vector<double> weight;
    bool has_target = false;
    // generator, dense host copy per (g, term): row-major d*d
    std::vector<cplx> Hdense;  // [n_gen][1+L][d][d]
    // ---- warp path
    int W = 0;   // off-diagonal slots actually needed
    int Wt = 0;  // template width serving it
    int nnz_union = 0;
    bool preg = false;
    bool pair = false;  // two trajectories of one generator per warp (warp2_kernel.cuh)
    bool mu_hermitian = false;
    bool taylor = false;  // krotov_problem.propagator == KROTOV_PROP_EXPMV: cheb[] holds Taylor tables (krotov_set_taylor)
    int lpt = 32;  // threads (= padded rows) per trajectory on the warp path: 32, 64 or 128
    bool tiny = false;  // d <= 4, N <= 32, L <= 2: one thread per trajectory, everything in registers (tiny_kernel.cuh)
    bool tiny_imag[2] = {false, false};  // every prepared term of the direction is purely imaginary (real Hamiltonian)
    std::vector<int> cols;  // [Wt][lpt]
    std::vector<char> slot_valid;  // [Wt][32] slot holds a real matrix entry (i, cols[s][i])
    int wpc = 1, tpw = 1, nCTA = 1;
    DevBuf d_cols, d_Pf, d_Pb, d_inv_s, d_gen, d_dt, d_alpha, d_eps_old, d_eps_new, d_ga, d_X, d_Phi, d_psi0,
        d_target, d_chiT, d_chicoef, d_psif, d_tau, d_R, d_err, d_weight, d_prof, d_Tf, d_Tb, d_acc,
        d_rawf, d_rawb, d_rowscale, d_envamps, d_envout;  // unscaled generator rows of both directions + per-generator (fy, beta): rows are scaled on the device
    DevBuf d_mbox[2];
    ChebyTables cheb[2];
    bool chiT_valid = false, chicoef_valid = false, swept = false;
    // comm
    int rank = 0, world = 1;
    double *peer_mbox[2][kr::kMaxRanks] = {};
    size_t mail_bytes = 0, xacc_bytes = 0;  // d_mbox[par] = mailboxes (sentinel-filled) followed by the cross-rank accumulators (zero-filled)
    int total_ctas = 0;  // CTAs of all ranks (krotov_comm_connect)
    int max_ctas = 0;    // largest CTA count of a rank
    // replicated forward sweep (every rank holds all trajectories; backward sweep sharded, chi written to all ranks)
    bool rf = false;
    double ms_rank_wait = 0.0;
    int sm_clock_khz = 1965000;
    int bw_lo = 0, bw_hi = 0;
    bool rf_wanted = false;                       // krotov_problem.replicated_forward: d_X holds TWO chi trajectories
    size_t x_slab = 0;                            // elements of one chi trajectory
    DevBuf d_rfcount;                             // arrival counter of the rank barrier
    double2 *peer_Xbase[kr::kMaxRanks] = {};      // chi trajectories of every rank (parity p at + p * x_slab)
    unsigned long long *peer_flag[kr::kMaxRanks] = {};
    int xchg_last = 0;   // cross-rank protocol of the last launch: 0 none, 1 hier, 2 onehop, 3 mailboxes
    int kernel_last = 0, lanes_last = 0;  // enum krotov_kernel and threads per trajectory of the last warp-path launch
    // non-linear control amplitudes (krotov_set_amplitudes, krotov_set_amplitude_saturation)
    bool amp_set = false;           // poly, shape or saturation present
    std::vector<double> amp_poly;   // [L][kAmpMaxDeg+1], ascending powers (empty = a(eps) = eps)
    std::vector<double> amp_shape;  // [L][N_T] (empty = 1)
    std::vector<double> amp_sat;    // [L] s_l: the polynomial is evaluated at tanh(s_l eps) where s_l > 0 (empty = none)
    std::vector<double> amp_rows;   // [L][kAmpRow]: the warp kernels' table, amp_poly rows (a(eps) = eps if empty) then s_l
    std::vector<double> amp_old_host, amp_dfac_host;  // a(eps_old), a'(eps_old): sources of the stream-ordered uploads
    DevBuf d_amp_poly, d_amp_shape, d_amp_sat, d_amp_rows, d_amp_old, d_amp_dfac, d_amp_new;
    // tied control terms (krotov_set_control_terms)
    std::vector<int> tie_ctrl;               // [L] control of every term; empty = every term is its own control
    std::vector<int> tie_first;              // [L] 1 at the first term of its control
    std::vector<double> tie_host;            // the tie table of the coming sweep: [L] tie_ctrl, then [L][N_T] a_t'(eps_old)
    std::vector<double> update_shape_host, lambda_host;  // krotov_problem.update_shape / lambda_a (the setter's checks)
    DevBuf d_tie;
    DevBuf d_emul;       // krotov_group_iterate: per-rank parameter blocks of the emulated multi-rank launch
    long long iter_count = 0;
    // the peers' mailboxes and chi trajectories mapped by krotov_comm_connect (peer_mbox / peer_Xbase point into them)
    std::vector<kr::IpcMapping> peer_maps;
    // dense path
    kr::DenseEngine *dense = nullptr;
    // misc
    int sm_count = 0;
    long long launches_total = 0, launches_last = 0, fallback_steps = 0;
    double ms_last = 0.0, ms_last_bw = 0.0;
    std::string err;

    // peer mappings first, then the dense engine; the buffers (members) and the stream (base) follow
    ~krotov_handle_s() {
        peer_maps.clear();
        kr::dense_destroy(dense);
    }
};

namespace {

#define KR_CUDA(h, call)                                                                             \
    do {                                                                                             \
        cudaError_t e_ = (call);                                                                     \
        if (e_ != cudaSuccess) {                                                                     \
            (h)->err = std::string(#call) + ": " + cudaGetErrorString(e_);                           \
            return KROTOV_ERR_CUDA;                                                                  \
        }                                                                                            \
    } while (0)

int fail(krotov_handle h, int code, const std::string &msg) {
    if (h)
        h->err = msg;
    else
        g_create_error = msg;
    return code;
}

int dev_alloc(krotov_handle h, DevBuf &b, size_t bytes) {
    if (bytes == 0) bytes = 16;
    if (b && b.bytes() >= bytes) return KROTOV_OK;  // reuse: cudaFree/cudaMalloc cost up to 100 ms
    // small tables (Chebyshev coefficients, ...) grow by a few entries when a spectral range widens: give them
    // headroom so that a re-derived polynomial never re-allocates in the middle of an optimisation
    if (bytes < (1u << 20)) {
        size_t cap = 4096;
        while (cap < 2 * bytes) cap <<= 1;
        bytes = cap;
    }
    const cudaError_t e = b.allocate(bytes);
    if (e != cudaSuccess) {
        h->err = std::string("cudaMalloc(") + std::to_string(bytes) + "): " + cudaGetErrorString(e);
        return e == cudaErrorMemoryAllocation ? KROTOV_ERR_NOMEM : KROTOV_ERR_CUDA;
    }
    return KROTOV_OK;
}

// v into b (grown as needed), ordered on the handle's stream (kr::copy_to_device).  wait = false only for a vector the
// handle owns and does not rewrite before its stream is next synchronised; locals wait.
template <typename T>
int upload(krotov_handle h, DevBuf &b, const std::vector<T> &v, bool wait) {
    int rc = dev_alloc(h, b, v.size() * sizeof(T));
    if (rc) return rc;
    if (!v.empty()) KR_CUDA(h, kr::copy_to_device(b.get<void>(), v.data(), v.size() * sizeof(T), h->stream, wait));
    return KROTOV_OK;
}

// ---- kernel table (instances are compiled in warp_inst_*.cu, one translation unit per family) ------------------
using kr::KernelKey;
using kr::WarpKernel;
const std::map<KernelKey, WarpKernel> &kernel_table() {
    static const std::map<KernelKey, WarpKernel> tab = [] {
        std::map<KernelKey, WarpKernel> t;
        kr::add_warp_instances_runtime(t);
        kr::add_warp_instances_preg1(t);
        kr::add_warp_instances_preg2(t);
        kr::add_warp_instances_wide64(t);
        kr::add_warp_instances_wide128(t);
        return t;
    }();
    return tab;
}

// the same kernel serving several emulated ranks in one launch (krotov_group_iterate)
const std::map<KernelKey, WarpKernel> &kernel_emul_table() {
    static const std::map<KernelKey, WarpKernel> tab = [] {
        std::map<KernelKey, WarpKernel> t;
        kr::add_warp_instances_emul(t);
        return t;
    }();
    return tab;
}

// instances with the replicated forward sweep of several ranks compiled in (regular / emulated ranks)
const std::map<KernelKey, WarpKernel> &kernel_rf_table() {
    static const std::map<KernelKey, WarpKernel> tab = [] {
        std::map<KernelKey, WarpKernel> t;
        kr::add_warp_instances_rf(t);
        kr::add_warp_instances_rf2(t);
        return t;
    }();
    return tab;
}
const std::map<KernelKey, WarpKernel> &kernel_rf_emul_table() {
    static const std::map<KernelKey, WarpKernel> tab = [] {
        std::map<KernelKey, WarpKernel> t;
        kr::add_warp_instances_rf_emul(t);
        return t;
    }();
    return tab;
}

// truncated-Taylor instances (prop_method=Expmv): regular and emulated-ranks, in maps of their own
struct TaylorTables {
    std::map<KernelKey, WarpKernel> regular, emul;
};
const TaylorTables &kernel_taylor_tables() {
    static const TaylorTables tab = [] {
        TaylorTables t;
        kr::add_warp_instances_taylor(t.regular, t.emul);
        return t;
    }();
    return tab;
}

// the regular instances serving the handle's propagator
const std::map<KernelKey, WarpKernel> &warp_table(const krotov_handle h) {
    return h->taylor ? kernel_taylor_tables().regular : kernel_table();
}

// pair kernel (two trajectories of one generator per warp): register-resident rows only
const std::map<KernelKey, WarpKernel> &kernel2_table() {
    static const std::map<KernelKey, WarpKernel> tab = [] {
        std::map<KernelKey, WarpKernel> t;
        kr::add_warp2_instances(t);
        return t;
    }();
    return tab;
}

const int kWidths[] = {1, 2, 3, 4, 5, 6, 7, 8, 10, 12, 16, 20, 24, 31};
const int kWidthsWide64[] = {4, 6, 8, 10, 12, 16, 20, 24};
const int kWidthsWide128[] = {4, 6, 8, 12, 16, 24};

int pick_width(int W, int lpt = 32) {
    if (lpt == 64) {
        for (int w : kWidthsWide64)
            if (w >= W) return w;
        return -1;
    }
    if (lpt == 128) {
        for (int w : kWidthsWide128)
            if (w >= W) return w;
        return -1;
    }
    for (int w : kWidths)
        if (w >= W) return w;
    return -1;
}

cplx Hval(const krotov_handle h, int g, int t, int i, int j) {
    return h->Hdense[(((size_t)g * (1 + h->L) + t) * h->d + i) * h->d + j];
}

// ---- pattern + slot assignment -------------------------------------------------------------
int build_pattern(krotov_handle h) {
    const int d = h->d, lpt = h->lpt;
    std::vector<char> pat((size_t)d * d, 0);
    for (int g = 0; g < h->n_gen; ++g)
        for (int t = 0; t <= h->L; ++t)
            for (int i = 0; i < d; ++i)
                for (int j = 0; j < d; ++j)
                    if (Hval(h, g, t, i, j) != cplx(0.0, 0.0)) pat[(size_t)i * d + j] = 1;
    // adjoint pattern must be covered too (backward sweep uses H^dagger): symmetrise
    for (int i = 0; i < d; ++i)
        for (int j = 0; j < d; ++j)
            if (pat[(size_t)i * d + j]) pat[(size_t)j * d + i] = 1;
    int nnz = 0, wmax = 0;
    std::set<int> diags;
    for (int i = 0; i < d; ++i) {
        int w = 0;
        for (int j = 0; j < d; ++j)
            if (pat[(size_t)i * d + j]) {
                ++nnz;
                if (i != j) {
                    ++w;
                    diags.insert(j - i);
                }
            }
        wmax = std::max(wmax, w);
        if (!pat[(size_t)i * d + i]) ++nnz;  // diagonal is always kept
    }
    h->nnz_union = nnz;
    const bool use_dia = (int)diags.size() <= std::max(wmax, 1) + 1 && pick_width((int)diags.size(), lpt) > 0 &&
                         (pick_width(std::max(wmax, 1), lpt) < 0 ||
                          pick_width((int)diags.size(), lpt) <= pick_width(std::max(wmax, 1), lpt));
    h->W = std::max(1, use_dia ? (int)diags.size() : wmax);
    h->Wt = pick_width(h->W, lpt);
    if (h->Wt < 0) return fail(h, KROTOV_ERR_UNSUPPORTED, "row too wide for the warp path");
    h->cols.assign((size_t)h->Wt * h->lpt, 0);
    h->slot_valid.assign((size_t)h->Wt * h->lpt, 0);
    for (int s = 0; s < h->Wt; ++s)
        for (int i = 0; i < lpt; ++i) h->cols[(size_t)s * lpt + i] = i;  // padding: own column, value 0
    if (use_dia) {
        // one slot per matrix diagonal; EVERY lane reads x[(i + off) mod 32] so that a warp's LDS.128
        // gather always touches 32 consecutive 16-byte words (bank-conflict free); entries that are not
        // in the pattern (or wrapped around) carry the value 0
        int s = 0;
        for (int off : diags) {
            for (int i = 0; i < lpt; ++i) {
                const int j = i + off;
                h->cols[(size_t)s * lpt + i] = ((j % lpt) + lpt) % lpt;
                if (i < d && j >= 0 && j < d && pat[(size_t)i * d + j]) h->slot_valid[(size_t)s * lpt + i] = 1;
            }
            ++s;
        }
    } else {
        for (int i = 0; i < d; ++i) {
            int s = 0;
            for (int j = 0; j < d; ++j)
                if (i != j && pat[(size_t)i * d + j]) {
                    h->cols[(size_t)s * lpt + i] = j;
                    h->slot_valid[(size_t)s * lpt + i] = 1;
                    ++s;
                }
        }
    }
    return KROTOV_OK;
}

// rows P_t for one direction: [g][1+L][Wt+1][32].  The factor 2c = -/+ 4i/Delta is purely imaginary, so the product
// is written out (std::complex multiplication goes through __muldc3); generators are spread over a few threads.
void build_rows(krotov_handle h, int dir, std::vector<cplx> &out) {
    const int d = h->d, L = h->L, Wt = h->Wt, lpt = h->lpt;
    const ChebyTables &ct = h->cheb[dir];
    out.assign((size_t)h->n_gen * (1 + L) * (Wt + 1) * lpt, cplx(0, 0));
    const bool fw = (dir == KROTOV_FORWARD);
    auto work = [&](int g0, int g1) {
        for (int g = g0; g < g1; ++g) {
            const double s = 4.0 / ct.Delta[g];
            const double beta = ct.Delta[g] / 2 + ct.E_min[g];
            const double fy = fw ? -s : s;  // f = (0, fy);  f * (a + i b) = -fy b + i fy a
            for (int t = 0; t <= L; ++t) {
                cplx *row = &out[((size_t)g * (1 + L) + t) * (Wt + 1) * lpt];
                const cplx *H = &h->Hdense[(((size_t)g * (1 + L) + t) * d) * d];
                for (int sl = 0; sl < Wt; ++sl)
                    for (int i = 0; i < d; ++i) {
                        if (!h->slot_valid[(size_t)sl * lpt + i]) continue;
                        const int j = h->cols[(size_t)sl * lpt + i];
                        const cplx v = fw ? H[(size_t)i * d + j] : std::conj(H[(size_t)j * d + i]);
                        row[(size_t)sl * lpt + i] = cplx(-fy * v.imag(), fy * v.real());
                    }
                for (int i = 0; i < d; ++i) {
                    const cplx hv = H[(size_t)i * d + i];
                    const double re = hv.real() - (t == 0 ? beta : 0.0), im = fw ? hv.imag() : -hv.imag();
                    row[(size_t)Wt * lpt + i] = cplx(-fy * im, fy * re);
                }
            }
        }
    };
    const int nt = (h->n_gen >= 64) ? 4 : 1;
    if (nt == 1) {
        work(0, h->n_gen);
    } else {
        std::vector<std::thread> pool;
        for (int t = 0; t < nt; ++t) pool.emplace_back(work, (h->n_gen * t) / nt, (h->n_gen * (t + 1)) / nt);
        for (auto &th : pool) th.join();
    }
}

// The same rows WITHOUT the Chebyshev scaling (entry values as build_rows picks them; diagonal in the last slot), uploaded
// once per direction at krotov_create.  krotov_set_cheby then forms P_t = f (H_t - beta delta_t0) on the device from the
// per-generator numbers (fy, beta) -- 2 n_gen doubles instead of building and uploading all rows on the host (C4: 2.75 MB
// and 1.0-1.5 ms per direction and spectral-range event).  Same arithmetic as build_rows: one product per component.
void build_raw_rows(krotov_handle h, int dir, std::vector<cplx> &out) {
    const int d = h->d, L = h->L, Wt = h->Wt, lpt = h->lpt;
    out.assign((size_t)h->n_gen * (1 + L) * (Wt + 1) * lpt, cplx(0, 0));
    const bool fw = (dir == KROTOV_FORWARD);
    for (int g = 0; g < h->n_gen; ++g)
        for (int t = 0; t <= L; ++t) {
            cplx *row = &out[((size_t)g * (1 + L) + t) * (Wt + 1) * lpt];
            const cplx *H = &h->Hdense[(((size_t)g * (1 + L) + t) * d) * d];
            for (int sl = 0; sl < Wt; ++sl)
                for (int i = 0; i < d; ++i) {
                    if (!h->slot_valid[(size_t)sl * lpt + i]) continue;
                    const int j = h->cols[(size_t)sl * lpt + i];
                    row[(size_t)sl * lpt + i] = fw ? H[(size_t)i * d + j] : std::conj(H[(size_t)j * d + i]);
                }
            for (int i = 0; i < d; ++i) {
                const cplx hv = H[(size_t)i * d + i];
                row[(size_t)Wt * lpt + i] = cplx(hv.real(), fw ? hv.imag() : -hv.imag());
            }
        }
}

// P[g][t][slot][lane] = (0, fy_g) * (raw - beta_g on the diagonal of term 0); rows beyond d stay zero
__global__ void scale_rows_kernel(const double2 *__restrict__ raw, const double2 *__restrict__ fy_beta, double2 *__restrict__ out,
                                  const int n_terms, const int Wt, const int lpt, const int d, const size_t total) {
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int lane = (int)(idx % lpt);
    const int sl = (int)((idx / lpt) % (Wt + 1));
    const size_t gt = idx / ((size_t)lpt * (Wt + 1));
    const int t = (int)(gt % n_terms);
    const int g = (int)(gt / n_terms);
    const double2 v = raw[idx];
    const double2 fb = fy_beta[g];
    double2 o = make_double2(0.0, 0.0);
    if (sl == Wt) {
        if (lane < d) {
            const double re = v.x - (t == 0 ? fb.y : 0.0);
            o = make_double2(__dmul_rn(-fb.x, v.y), __dmul_rn(fb.x, re));
        }
    } else if (v.x != 0.0 || v.y != 0.0) {
        o = make_double2(__dmul_rn(-fb.x, v.y), __dmul_rn(fb.x, v.x));
    }
    out[idx] = o;
}

// Spectral envelope on the device (krotov_envelope_extremes_device): one warp per (generator, corner).  The warp forms
// A = H_0 + sum_l amp_l H_l from the unscaled forward rows in shared memory (lane i owns row i) and runs cyclic Jacobi
// rotations on the complex Hermitian matrix until the off-diagonal norm is below 1e-30 ||A||_F^2 (eigenvalues to a few
// ulp of the norm); the extreme diagonal entries are the extreme eigenvalues.  out[(g * n_corner + c)] = (lo, hi).
__global__ void __launch_bounds__(32) jacobi_extremes_kernel(const double2 *__restrict__ raw, const int *__restrict__ cols,
                                                             const double *__restrict__ amps, double2 *__restrict__ out,
                                                             const int L, const int Wt, const int d, const int n_corner) {
    constexpr int LD = 33;
    __shared__ double2 A[32 * LD];
    const int lane = threadIdx.x;
    const int g = blockIdx.x / n_corner, c = blockIdx.x % n_corner;
    for (int j = 0; j < 32; ++j) A[lane * LD + j] = make_double2(0.0, 0.0);
    __syncwarp();
    const size_t rowstride = (size_t)(Wt + 1) * 32;
    for (int sl = 0; sl <= Wt; ++sl) {
        double2 v = raw[((size_t)g * (1 + L)) * rowstride + (size_t)sl * 32 + lane];
        for (int l = 0; l < L; ++l) {
            const double a = amps[c * L + l];
            const double2 w = raw[((size_t)g * (1 + L) + l + 1) * rowstride + (size_t)sl * 32 + lane];
            v.x = fma(a, w.x, v.x);
            v.y = fma(a, w.y, v.y);
        }
        const int j = (sl == Wt) ? lane : cols[sl * 32 + lane];
        if (lane < d && j < d) {  // (each lane owns its row: no two lanes touch the same element)
            A[lane * LD + j].x += v.x;
            A[lane * LD + j].y += v.y;
        }
    }
    __syncwarp();
    // Frobenius norm (for the stopping rule)
    double nrm = 0.0;
    if (lane < d)
        for (int j = 0; j < d; ++j) nrm += A[lane * LD + j].x * A[lane * LD + j].x + A[lane * LD + j].y * A[lane * LD + j].y;
    for (int o = 16; o > 0; o >>= 1) nrm += __shfl_xor_sync(0xffffffffu, nrm, o);
    for (int sweep = 0; sweep < 30; ++sweep) {
        double off = 0.0;
        if (lane < d)
            for (int j = 0; j < d; ++j)
                if (j != lane) off += A[lane * LD + j].x * A[lane * LD + j].x + A[lane * LD + j].y * A[lane * LD + j].y;
        for (int o = 16; o > 0; o >>= 1) off += __shfl_xor_sync(0xffffffffu, off, o);
        if (off <= 1e-30 * nrm) break;
        for (int p = 0; p < d - 1; ++p)
            for (int q = p + 1; q < d; ++q) {
                const double2 cpq = A[p * LD + q];
                const double ac2 = cpq.x * cpq.x + cpq.y * cpq.y;
                // (warp-uniform: every lane reads the same element.)  Elements below 1e-17 ||A||_F are left alone: all 300
                // of them together stay under the stopping rule, and the last sweeps consist of little else
                if (ac2 <= 1e-34 * nrm || ac2 < 1e-300) continue;
                const double ac = sqrt(ac2), iac = 1.0 / ac;
                const double app = A[p * LD + p].x, aqq = A[q * LD + q].x;
                const double tau = 0.5 * (aqq - app) * iac;
                const double t = (tau >= 0.0 ? 1.0 : -1.0) / (fabs(tau) + sqrt(1.0 + tau * tau));
                const double cs = 1.0 / sqrt(1.0 + t * t), sn = t * cs;
                const double wr = cpq.x * iac, wi = cpq.y * iac;  // w = e^{i phi}
                __syncwarp();
                if (lane < d && lane != p && lane != q) {
                    const double2 akp = A[lane * LD + p], akq = A[lane * LD + q];
                    // A'_kp = cs A_kp - sn conj(w) A_kq ;  A'_kq = sn w A_kp + cs A_kq
                    const double2 nkp = make_double2(cs * akp.x - sn * (wr * akq.x + wi * akq.y),
                                                     cs * akp.y - sn * (wr * akq.y - wi * akq.x));
                    const double2 nkq = make_double2(sn * (wr * akp.x - wi * akp.y) + cs * akq.x,
                                                     sn * (wr * akp.y + wi * akp.x) + cs * akq.y);
                    A[lane * LD + p] = nkp;
                    A[lane * LD + q] = nkq;
                    A[p * LD + lane] = make_double2(nkp.x, -nkp.y);
                    A[q * LD + lane] = make_double2(nkq.x, -nkq.y);
                } else if (lane == p) {
                    A[p * LD + p] = make_double2(app - t * ac, 0.0);
                    A[p * LD + q] = make_double2(0.0, 0.0);
                } else if (lane == q) {
                    A[q * LD + q] = make_double2(aqq + t * ac, 0.0);
                    A[q * LD + p] = make_double2(0.0, 0.0);
                }
                __syncwarp();
            }
    }
    double lo = (lane < d) ? A[lane * LD + lane].x : INFINITY, hi = (lane < d) ? A[lane * LD + lane].x : -INFINITY;
    for (int o = 16; o > 0; o >>= 1) {
        lo = fmin(lo, __shfl_xor_sync(0xffffffffu, lo, o));
        hi = fmax(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    }
    if (lane == 0) out[blockIdx.x] = make_double2(lo, hi);
}

// dense prepared terms of one direction for the tiny kernel: [g][1+L][d*d] row-major, same numbers as build_rows
void build_dense_terms(krotov_handle h, int dir, std::vector<cplx> &out) {
    const int d = h->d, L = h->L;
    const ChebyTables &ct = h->cheb[dir];
    out.assign((size_t)h->n_gen * (1 + L) * d * d, cplx(0, 0));
    for (int g = 0; g < h->n_gen; ++g) {
        const double s = 4.0 / ct.Delta[g];
        const double beta = ct.Delta[g] / 2 + ct.E_min[g];
        const cplx f = (dir == KROTOV_FORWARD) ? cplx(0.0, -s) : cplx(0.0, s);
        for (int t = 0; t <= L; ++t)
            for (int i = 0; i < d; ++i)
                for (int j = 0; j < d; ++j) {
                    cplx v = (dir == KROTOV_FORWARD) ? Hval(h, g, t, i, j) : std::conj(Hval(h, g, t, j, i));
                    if (t == 0 && i == j) v -= beta;
                    out[(((size_t)g * (1 + L) + t) * d + i) * d + j] = f * v;
                }
    }
}

using TinyKernel = void (*)(const kr::TinyParams);
TinyKernel tiny_kernel_for(int d, int L, bool gimag = false) {
#define KR_TINY(D, LT)                                                                                              \
    if (d == D && L == LT)                                                                                          \
        return gimag ? (TinyKernel)kr::krotov_tiny_kernel<D, LT, ((1 + LT) * D * D <= 12), true>                     \
                     : (TinyKernel)kr::krotov_tiny_kernel<D, LT, ((1 + LT) * D * D <= 12), false>
    KR_TINY(2, 1); KR_TINY(2, 2); KR_TINY(3, 1); KR_TINY(3, 2); KR_TINY(4, 1); KR_TINY(4, 2);
#undef KR_TINY
    return nullptr;
}

__global__ void chi_coef_kernel(int functional, int N, int N_global, const double2 *tau, const double *w,
                                double2 *coef) {
    // one warp; fixed summation order
    const int lane = threadIdx.x;
    const double Ng = (double)N_global;
    if (functional == KROTOV_CHI_SM) {
        double sr = 0.0, si = 0.0;
        for (int k = lane; k < N; k += 32) {
            sr += w[k] * tau[k].x;
            si += w[k] * tau[k].y;
        }
        sr = kr::warp_sum_xor(sr);
        si = kr::warp_sum_xor(si);
        for (int k = lane; k < N; k += 32) {
            const double f = w[k] / (Ng * Ng);
            coef[k] = make_double2(f * sr, f * si);
        }
    } else if (functional == KROTOV_CHI_SS) {
        for (int k = lane; k < N; k += 32) {
            const double f = w[k] / Ng;
            coef[k] = make_double2(f * tau[k].x, f * tau[k].y);
        }
    } else {
        for (int k = lane; k < N; k += 32) coef[k] = make_double2(w[k] / (2.0 * Ng), 0.0);
    }
}

int choose_launch(krotov_handle h) {
    // One trajectory per warp while they fit on the chip (<= sm_count CTAs, co-resident for the
    // in-kernel grid exchange); register-resident term rows (PREG) when an instance exists and the
    // CTA stays <= 7 trajectory warps; otherwise rows are re-read per use and a warp may own several
    // trajectories.  KROTOV_WPC overrides the warps-per-CTA heuristic (experiments).
    const int N = h->N, sm = h->sm_count;
    const int lpt = h->lpt;
    // groups per CTA (named barriers 3..15); the wide-row instances of one-warp groups are built for 256 threads
    const int cap_preg = (256 - 32) / lpt, cap = (lpt == 32 && h->Wt >= 16) ? 7 : std::min(13, (512 - 32) / lpt);
    const bool preg_possible = warp_table(h).count(KernelKey{h->Wt, h->L, lpt}) > 0;
    // Pair mode: when there are more trajectories than one-per-warp CTAs with register-resident rows can hold
    // (N > 7 per SM) and they come in generator-sharing pairs (ensembles over basis states), one warp runs two
    // of them interleaved and keeps the rows in registers.  Measured on B200: +19 % at N = 2048 against the
    // row-reloading variant; at N = 1024 two independent warps per sub-partition overlap better than one warp
    // with two interleaved recursions (13.7 vs 15.3 ms), so the pair kernel is not used there.
    // KROTOV_NO_PAIR=1 disables it, KROTOV_FORCE_PAIR=1 uses it whenever the pairing exists.
    h->pair = false;
    if (lpt == 32 && !h->taylor && kernel2_table().count(KernelKey{h->Wt, h->L, 32}) > 0 && N % 2 == 0 &&
        (N > cap_preg * sm || getenv("KROTOV_FORCE_PAIR")) && N / 2 <= cap_preg * sm &&
        !getenv("KROTOV_NO_PAIR") && !getenv("KROTOV_NO_PREG") && !getenv("KROTOV_SEQ_PREG")) {
        bool ok = true;
        for (int k = 0; k < N; k += 2) ok = ok && (h->gen_of_traj[k] == h->gen_of_traj[k + 1]);
        if (ok) {
            int wpc2 = std::max(1, (N / 2 + sm - 1) / sm);
            if (const char *env = getenv("KROTOV_WPC")) wpc2 = std::max(1, std::min(cap_preg, atoi(env)));
            h->pair = true; h->preg = true; h->tpw = 1; h->wpc = wpc2;
            h->nCTA = (N / 2 + wpc2 - 1) / wpc2;
            return KROTOV_OK;
        }
    }
    // Larger ensembles whose trajectories come in runs sharing a generator (the basis states of an ensemble sample):
    // one warp runs `tpw` trajectories of ONE generator one after the other and keeps that generator's rows in
    // registers, instead of re-reading rows from L2 for every trajectory and time step (21 row loads of 512 bytes
    // per trajectory and step: ~5 TB/s of L2 traffic at N = 4096, which is what bound the row-reloading variant).
    if (lpt == 32 && !h->taylor && preg_possible && N > cap_preg * sm && !getenv("KROTOV_NO_PREG") &&
        !getenv("KROTOV_NO_SEQ_PREG")) {
        for (int tpw = 2; tpw <= 16; ++tpw) {
            if (N % tpw != 0 || N / tpw > cap_preg * sm) continue;
            bool ok = true;
            for (int k = 0; k < N && ok; k += tpw)
                for (int t = 1; t < tpw; ++t) ok = ok && (h->gen_of_traj[k + t] == h->gen_of_traj[k]);
            if (!ok) continue;
            const int warps = N / tpw;
            int wpc = std::max(1, (warps + sm - 1) / sm);
            if (const char *env = getenv("KROTOV_WPC")) wpc = std::max(1, std::min(cap_preg, atoi(env)));
            h->preg = true; h->tpw = tpw; h->wpc = wpc;
            h->nCTA = (warps + wpc - 1) / wpc;
            return KROTOV_OK;
        }
    }
    int wpc = (N <= 8 && N <= cap_preg) ? N : std::max(std::min(std::min(N, 4), cap_preg), (N + sm - 1) / sm);
    if (const char *env = getenv("KROTOV_WPC")) wpc = std::max(1, atoi(env));
    h->tpw = 1;
    if (preg_possible && wpc <= cap_preg && (N + wpc - 1) / wpc <= sm && !getenv("KROTOV_NO_PREG")) {
        h->preg = true;
    } else {
        h->preg = false;
        wpc = std::min(wpc, cap);
        if ((N + wpc - 1) / wpc > sm) {
            wpc = cap;
            h->tpw = (N + sm * wpc - 1) / (sm * wpc);
        }
    }
    h->wpc = wpc;
    h->nCTA = (N + wpc * h->tpw - 1) / (wpc * h->tpw);
    return KROTOV_OK;
}

size_t warp_smem_bytes(const krotov_handle h) {
    if (h->pair)
        return (size_t)h->wpc * (128 + 64) * 16 + (size_t)h->L * h->wpc * 32 * 8 + kr::kMaxCtrl * 8 +
               (size_t)kr::kMaxCtrl * 160 * 8;
    return (size_t)h->wpc * 2 * h->lpt * 16 + (size_t)h->wpc * h->tpw * h->lpt * 16 + (size_t)h->L * h->wpc * h->lpt * 8 +
           kr::kMaxCtrl * 8 + (size_t)kr::kMaxCtrl * 160 * 8 + (size_t)h->wpc * h->lpt * 16 +
           (h->rf_wanted ? (size_t)h->wpc * kr::kRfRing * (32 * 16 + 8) + (size_t)h->wpc * 2 * 4 + 16 : 0);  // forwarder rings + barriers
}

void fill_warp_params(krotov_handle h, int mode, kr::WarpParams &p) {
    memset(&p, 0, sizeof(p));
    p.d = h->d; p.N = h->N; p.L = h->L; p.N_T = h->N_T; p.n_gen = h->n_gen;
    p.wpc = h->wpc; p.tpw = h->tpw; p.nCTA = h->nCTA; p.mode = mode; p.store_fw = h->store_fw;
    p.mu_hermitian = (h->mu_hermitian && !h->taylor && !getenv("KROTOV_NO_FAST")) ? 1 : 0;
    p.ndtc_f = h->cheb[0].ndtc; p.ndtc_b = h->cheb[1].set ? h->cheb[1].ndtc : 1; p.mmax_f = h->cheb[0].mmax; p.mmax_b = h->cheb[1].set ? h->cheb[1].mmax : 1;
    p.gen_of_traj = h->d_gen.get<const int>();
    p.cols = h->d_cols.get<const int>();
    p.Pf = h->d_Pf.get<const double2>(); p.Pb = h->d_Pb.get<const double2>();
    p.inv_s_f = h->d_inv_s.get<const double>();
    p.coef_f = h->cheb[0].coef.get<const double>(); p.m_f = h->cheb[0].m.get<const int>();
    p.phase_f = h->cheb[0].phase.get<const double2>();
    p.coef_b = h->cheb[1].coef.get<const double>(); p.m_b = h->cheb[1].m.get<const int>();
    p.phase_b = h->cheb[1].phase.get<const double2>();
    p.dtc_f = h->cheb[0].dtc.get<const int>(); p.dtc_b = h->cheb[1].dtc.get<const int>(); p.dt = h->d_dt.get<const double>();
    p.alpha = h->d_alpha.get<const double>();
    p.eps_old = h->d_eps_old.get<const double>(); p.eps_new = h->d_eps_new.get<double>();
    p.amp_old = h->amp_set ? h->d_amp_old.get<const double>() : p.eps_old;
    p.amp_dfac = h->amp_set ? h->d_amp_dfac.get<const double>() : nullptr;
    p.amp_poly = (h->amp_set && !h->amp_rows.empty()) ? h->d_amp_rows.get<const double>() : nullptr;
    p.amp_shape = (h->amp_set && !h->amp_shape.empty()) ? h->d_amp_shape.get<const double>() : nullptr;
    p.tie = h->tie_ctrl.empty() ? nullptr : h->d_tie.get<const double>();
    p.g_a_int = h->d_ga.get<double>();
    p.X = h->d_X.get<double2>(); p.Phi = h->d_Phi.get<double2>();
    p.psi0 = h->d_psi0.get<const double2>();
    p.target = h->has_target ? h->d_target.get<const double2>() : nullptr;
    p.chiT = h->chiT_valid ? h->d_chiT.get<const double2>() : nullptr;
    p.chi_coef = h->d_chicoef.get<const double2>();
    p.psi_final = h->d_psif.get<double2>(); p.tau = h->d_tau.get<double2>();
    p.R = h->d_R.get<double>();
    p.E = h->d_R.get<double>() + (size_t)h->N_T * h->nCTA * h->L;
    p.acc = (h->nCTA > 1 && h->nCTA < 256 && !getenv("KROTOV_NO_ATOMIC_SUM")) ? h->d_acc.get<unsigned long long>() : nullptr;
    p.rank = h->rank; p.world = h->world;
    // Who polls the rank's mailbox: every CTA (no broadcast hop) while pollers x writers stay few, else the reducer
    // alone, which then broadcasts through E.  Measured on C4 (ms per iteration, all-poll / reducer-poll): 2 GPUs x
    // 128 CTAs 14.0 / 14.6, 2 x 147 16.4 / 16.9, 8 x 32 14.9 / 17.2, 8 x 147 23.3 / 18.7.
    p.mbox_all = (h->nCTA * h->world <= 400) ? 1 : 0;
    if (const char *e = getenv("KROTOV_MBOX_ALL")) p.mbox_all = atoi(e);
    const int par = (int)(h->iter_count & 1);
    for (int r = 0; r < h->world && r < kr::kMaxRanks; ++r) p.mbox[r] = h->peer_mbox[par][r];
    // The cross-rank sum of a time step -- the same decision on every rank (it only reads what all ranks know):
    //   hier   (default)  every CTA adds into its own rank's accumulator; the add that completes a word forwards the
    //                     rank sum with ONE add per rank over NVLink (xrank_hier_sum): `world` adds per word and rank
    //   onehop            every CTA of every rank adds into every rank's accumulator (xrank_atomic_sum): total_ctas
    //                     adds per word and rank, up to KROTOV_XACC_MAX (512) CTAs in total
    //   mbox              rank sums pushed into the peers' mailboxes by the reducer CTA (also the fallback of both)
    // KROTOV_XCHG=hier|onehop|mbox selects one (experiments, tests); KROTOV_NO_XACC=1 is the old spelling of mbox.
    p.total_ctas = h->total_ctas;
    p.xacc_stride = 1;
    if (const char *e = getenv("KROTOV_XACC_STRIDE")) p.xacc_stride = std::max(1, std::min(kXaccMaxStride, atoi(e)));
    int xacc_max = 512;
    if (const char *e = getenv("KROTOV_XACC_MAX")) xacc_max = std::min(atoi(e), kr::kXMaxArrivals);
    // default: the one-hop sum while the ranks' CTAs are few (measured on C4, ms per iteration, one-hop / hier / hier
    // with stores / mailboxes: 2 GPUs x 128 CTAs 12.85 / 13.4 / 13.7 / 15.6; 8 GPUs x 32 CTAs 13.9 / 14.2 / 14.5 / -),
    // the hierarchical sum beyond (every rank then receives `world` adds per word instead of `total_ctas`)
    std::string xchg = getenv("KROTOV_XCHG") ? getenv("KROTOV_XCHG") : (h->total_ctas <= xacc_max ? "onehop" : "hier");
    if (getenv("KROTOV_NO_XACC")) xchg = "mbox";
    const bool hier_ok = h->max_ctas < 256 && h->total_ctas <= kr::kXMaxArrivals && !getenv("KROTOV_NO_ATOMIC_SUM");
    if ((xchg == "hier" || xchg == "hierst") && !hier_ok) xchg = "onehop";
    if (xchg == "onehop" && h->total_ctas > xacc_max) xchg = "mbox";
    if (h->world > 1 && h->xacc_bytes && xchg != "mbox") {
        for (int r = 0; r < h->world; ++r) p.xacc[r] = (unsigned long long *)((char *)h->peer_mbox[par][r] + h->mail_bytes);
        p.xchg_hier = (xchg == "hier") ? 1 : (xchg == "hierst") ? 2 : 0;
    }
    h->xchg_last = h->world > 1 ? (p.xacc[0] ? (p.xchg_hier == 1 ? 1 : p.xchg_hier == 2 ? 4 : 2) : 3) : 0;
    if (h->rf) {
        // replicated forward sweep: no per-step exchange between the ranks at all
        p.world = 1;
        p.rank = 0;
        for (int r = 0; r < kr::kMaxRanks; ++r) {
            p.xacc[r] = nullptr;
            p.mbox[r] = nullptr;
        }
        p.xchg_hier = 0;
        p.rf_world = h->world;
        p.rf_rank = h->rank;
        p.bw_lo = h->bw_lo;
        p.bw_hi = h->bw_hi;
        for (int r = 0; r < h->world; ++r) {
            p.Xr[r] = h->peer_Xbase[r] + (size_t)par * h->x_slab;
            p.rf_flag[r] = h->peer_flag[r];
        }
        p.X = p.Xr[h->rank];
        p.rf_count = h->d_rfcount.get<unsigned int>();
        p.rf_iter = (unsigned long long)(h->iter_count + 1);
        p.rf_stride = getenv("KROTOV_RF_STRIDE") ? std::max(1, atoi(getenv("KROTOV_RF_STRIDE"))) : 1;
        p.rf_pack = getenv("KROTOV_RF_PACK") ? (h->bw_hi - h->bw_lo + h->nCTA - 1) / h->nCTA : 0;
        // forwarder warps (the value is their polling interval in ns); KROTOV_RF_DIRECT=1: producers store to all ranks
        p.rf_fwd = (h->lpt == 32 && !getenv("KROTOV_RF_DIRECT")) ? (getenv("KROTOV_RF_SLEEP") ? std::max(1, atoi(getenv("KROTOV_RF_SLEEP"))) : 1000) : 0;
        h->xchg_last = 5;
    }
    p.err_flag = h->d_err.get<int>();
    p.prof = h->d_prof.get<long long>();
    p.timeout_cycles = 20000000000ll;  // ~10 s
    if (const char *e = getenv("KROTOV_TIMEOUT_CYCLES")) p.timeout_cycles = atoll(e);
}

// enum krotov_kernel of the persistent warp kernel choose_launch selected (the tiny kernel aside)
int warp_kernel_kind(const krotov_handle h) {
    if (h->taylor) return KROTOV_KERNEL_TAYLOR;
    if (h->pair) return KROTOV_KERNEL_PAIR;
    if (h->preg) return h->tpw > 1 ? KROTOV_KERNEL_SEQ_PREG : KROTOV_KERNEL_PREG;
    return KROTOV_KERNEL_RELOAD;
}

int launch_warp(krotov_handle h, int mode) {
    kr::WarpParams p;
    fill_warp_params(h, mode, p);
    if (h->tiny && h->world == 1 && !h->amp_set) {
        kr::TinyParams tp;
        tp.w = p;
        tp.Tf = h->d_Tf.get<const double2>();
        tp.Tb = h->d_Tb.get<const double2>();
        const int te = (1 + h->L) * h->d * h->d;
        const size_t term_bytes = te <= 12 ? 0 : (size_t)te * 32 * 16;
        const size_t coef_bytes = ((size_t)p.ndtc_f * p.mmax_f + (size_t)p.ndtc_b * p.mmax_b) * 32 * 8;
        tp.coef_in_smem = (term_bytes + coef_bytes <= 160 * 1024) ? 1 : 0;
        const size_t smem = term_bytes + (tp.coef_in_smem ? coef_bytes : 0) + 16;
        TinyKernel fn = tiny_kernel_for(h->d, h->L, h->tiny_imag[0] && h->tiny_imag[1]);
        KR_CUDA(h, cudaFuncSetAttribute((const void *)fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        void *args[] = {(void *)&tp};
        KR_CUDA(h, cudaLaunchKernel((const void *)fn, dim3(1), dim3(32), args, smem, h->stream));
        h->launches_last += 1;
        h->kernel_last = KROTOV_KERNEL_TINY;
        h->lanes_last = 1;
        return KROTOV_OK;
    }
    KernelKey key{h->Wt, h->preg ? h->L : 0, h->pair ? 32 : h->lpt};
    const auto &table = h->pair ? kernel2_table() : warp_table(h);
    auto it = table.find(key);
    if (it == table.end()) return fail(h, KROTOV_ERR_UNSUPPORTED, "no kernel instance for this (W, L)");
    WarpKernel fn = it->second;
    const size_t smem = warp_smem_bytes(h);
    KR_CUDA(h, cudaFuncSetAttribute((const void *)fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid(h->nCTA), block(h->wpc * h->lpt + 32);
    if (h->rf && mode == 1) {
        // replicated forward sweep, stage 1: the RF instance runs this rank's shard of the backward sweep, writes chi to
        // every rank and ends behind the rank barrier; stage 2 below: the regular instance runs the forward sweep
        auto itr = kernel_rf_table().find(key);
        if (itr == kernel_rf_table().end()) return fail(h, KROTOV_ERR_UNSUPPORTED, "no RF kernel instance for this (W, L)");
        KR_CUDA(h, cudaFuncSetAttribute((const void *)itr->second, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        void *args1[] = {(void *)&p};
        KR_CUDA(h, cudaLaunchCooperativeKernel((const void *)itr->second, grid, block, args1, smem, h->stream));
        h->launches_last += 1;
        p.skip_bw = 1;
    }
    p.rf_world = 0;  // (the regular instances carry no RF code; the field is theirs to ignore)
    void *args[] = {(void *)&p};
    if (h->nCTA > 1 && mode == 1) {
        KR_CUDA(h, cudaLaunchCooperativeKernel((const void *)fn, grid, block, args, smem, h->stream));
    } else {
        KR_CUDA(h, cudaLaunchKernel((const void *)fn, grid, block, args, smem, h->stream));
    }
    h->launches_last += 1;
    h->kernel_last = warp_kernel_kind(h);
    h->lanes_last = h->lpt;
    return KROTOV_OK;
}

int check_err_flag(krotov_handle h) {
    int flags[4] = {0, 0, 0, 0};  // [0] exchange timed out, [1] time steps redone with the gather protocol,
                                  // [2..3] SM cycles CTA 0 waited at the rank barrier (replicated forward sweep)
    KR_CUDA(h, cudaMemcpy(flags, h->d_err.get<void>(), sizeof(flags), cudaMemcpyDeviceToHost));
    const int flag = flags[0];
    h->fallback_steps = flags[1];
    long long wait_cycles;
    memcpy(&wait_cycles, flags + 2, 8);
    h->ms_rank_wait = h->rf ? (double)wait_cycles / (double)h->sm_clock_khz : 0.0;
    if (flags[1]) KR_CUDA(h, cudaMemsetAsync(h->d_err.get<int>() + 1, 0, sizeof(int), h->stream));
    if (flag) {
        KR_CUDA(h, cudaMemsetAsync(h->d_err.get<void>(), 0, sizeof(int), h->stream));
        return fail(h, KROTOV_ERR_TIMEOUT, "in-kernel exchange timed out waiting for a partial sum");
    }
    return KROTOV_OK;
}

}  // namespace

// ============================================================================== C ABI
extern "C" {

int krotov_abi_version(void) { return KROTOV_ABI_VERSION; }

const char *krotov_last_error(krotov_handle h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int krotov_destroy(krotov_handle h) {
    if (!h) return KROTOV_OK;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    delete h;
    return KROTOV_OK;
}

int64_t krotov_live_device_objects(void) { return kr::g_live_device_objects.load(); }

// krotov_create past its argument checks: fills the fresh handle h; on failure h->err holds the message
static int create_handle(krotov_handle h, const krotov_problem *pb) {
    h->d = pb->d; h->N = pb->n_traj; h->L = pb->n_ctrl; h->N_T = pb->n_steps; h->n_gen = pb->n_gen;
    h->functional = pb->functional;
    h->N_global = pb->n_traj_global > 0 ? pb->n_traj_global : pb->n_traj;
    h->store_fw = pb->store_fw; h->device = pb->device;
    h->rf_wanted = pb->replicated_forward != 0;
    if (pb->propagator != KROTOV_PROP_CHEBY && pb->propagator != KROTOV_PROP_EXPMV)
        return fail(h, KROTOV_ERR_ARG, "unknown krotov_problem.propagator");
    h->taylor = pb->propagator == KROTOV_PROP_EXPMV;
    const int d = h->d, N = h->N, L = h->L, N_T = h->N_T;
    if (h->taylor && (d > 32 || (pb->force_path != 0 && pb->force_path != KROTOV_PATH_WARP) || h->rf_wanted))
        return fail(h, KROTOV_ERR_UNSUPPORTED, "KROTOV_PROP_EXPMV runs on the persistent one-warp-per-trajectory kernel "
                                               "only (d <= 32, no replicated_forward)");
    if (cudaSetDevice(h->device) != cudaSuccess) return fail(h, KROTOV_ERR_CUDA, "cudaSetDevice failed");
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, h->device);
    h->sm_count = prop.multiProcessorCount;
    {
        int khz = 0;
        if (cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, h->device) == cudaSuccess && khz > 0) h->sm_clock_khz = khz;
    }
    if (prop.major < 10) return fail(h, KROTOV_ERR_UNSUPPORTED, "libkrotov_cuda is built for sm_100a only");
    if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreate(&h->ev0) != cudaSuccess || cudaEventCreate(&h->ev1) != cudaSuccess)
        return fail(h, KROTOV_ERR_CUDA, "stream/event creation failed");

    h->tlist.assign(pb->tlist, pb->tlist + N_T + 1);
    h->dt.resize(N_T);
    for (int n = 0; n < N_T; ++n) {
        h->dt[n] = h->tlist[n + 1] - h->tlist[n];
        if (!(h->dt[n] > 0)) return fail(h, KROTOV_ERR_ARG, "tlist must be strictly increasing");
    }
    h->gen_of_traj.assign(pb->gen_of_traj, pb->gen_of_traj + N);
    for (int k = 0; k < N; ++k)
        if (h->gen_of_traj[k] < 0 || h->gen_of_traj[k] >= h->n_gen)
            return fail(h, KROTOV_ERR_ARG, "gen_of_traj out of range");
    h->weight.assign(N, 1.0);
    if (pb->weight) h->weight.assign(pb->weight, pb->weight + N);
    h->has_target = pb->target != nullptr;

    // ---- generator ingestion.  `for_each_entry` walks the non-zeros of term (g, t) in either wire format.
    const cplx *vals = reinterpret_cast<const cplx *>(pb->gen_values);
    if (pb->gen_format != KROTOV_GEN_DENSE_COLMAJOR && pb->gen_format != KROTOV_GEN_CSR)
        return fail(h, KROTOV_ERR_ARG, "unknown gen_format");
    if (pb->gen_format == KROTOV_GEN_CSR)
        for (int q = 0; q < pb->csr_rowptr[d]; ++q)
            if (pb->csr_colind[q] < 0 || pb->csr_colind[q] >= d)
                return fail(h, KROTOV_ERR_ARG, "CSR column out of range");
    auto for_each_entry = [&](int g, int t, auto &&fn) {
        if (pb->term_present && !pb->term_present[(size_t)g * (1 + L) + t]) return;
        if (pb->gen_format == KROTOV_GEN_DENSE_COLMAJOR) {
            const cplx *src = vals + ((size_t)g * (1 + L) + t) * d * d;
            for (int j = 0; j < d; ++j)
                for (int i = 0; i < d; ++i)
                    if (src[(size_t)j * d + i] != cplx(0.0, 0.0)) fn(i, j, src[(size_t)j * d + i]);
        } else {
            const cplx *src = vals + ((size_t)g * (1 + L) + t) * pb->nnz;
            for (int i = 0; i < d; ++i)
                for (int q = pb->csr_rowptr[i]; q < pb->csr_rowptr[i + 1]; ++q) fn(i, pb->csr_colind[q], src[q]);
        }
    };

    int path = pb->force_path;
    if (path == KROTOV_PATH_WARP && d > 128)
        return fail(h, KROTOV_ERR_UNSUPPORTED, "warp path needs d <= 128");
    if (path != 0 && path != KROTOV_PATH_WARP && path != KROTOV_PATH_DENSE && path != KROTOV_PATH_SPARSE)
        return fail(h, KROTOV_ERR_ARG, "bad force_path");
    auto fill_dense = [&]() {  // dense host copy of every term (row-major)
        h->Hdense.assign((size_t)h->n_gen * (1 + L) * d * d, cplx(0, 0));
        for (int g = 0; g < h->n_gen; ++g)
            for (int t = 0; t <= L; ++t) {
                cplx *dst = &h->Hdense[((size_t)g * (1 + L) + t) * d * d];
                for_each_entry(g, t, [&](int i, int j, cplx v) { dst[(size_t)i * d + j] += v; });
            }
    };
    // persistent one-launch kernel: one row per thread, 32 / 64 / 128 threads per trajectory; needs narrow rows
    // beyond d = 32 (the generator row lives in registers)
    h->lpt = d <= 32 ? 32 : (d <= 64 ? 64 : 128);
    bool pattern_built = false;
    if ((path == 0 || path == KROTOV_PATH_WARP) && d <= 128) {
        fill_dense();
        const int prc = build_pattern(h);
        if (prc == KROTOV_OK) {
            path = KROTOV_PATH_WARP;
            pattern_built = true;
        } else if (path == KROTOV_PATH_WARP) {
            return prc;
        } else {
            h->err.clear();
        }
    }

    // d > 32: union sparsity pattern (symmetrised: the backward sweep needs the adjoint; diagonal always present)
    HostSparse hs;
    if (path == 0 || path == KROTOV_PATH_SPARSE) {
        std::vector<std::vector<int>> pat(d);
        for (int i = 0; i < d; ++i) pat[i].push_back(i);
        for (int g = 0; g < h->n_gen; ++g)
            for (int t = 0; t <= L; ++t)
                for_each_entry(g, t, [&](int i, int j, cplx) {
                    if (i != j) {
                        pat[i].push_back(j);
                        pat[j].push_back(i);
                    }
                });
        size_t nnz = 0;
        int W = 1;
        for (int i = 0; i < d; ++i) {
            std::sort(pat[i].begin() + 1, pat[i].end());
            pat[i].erase(std::unique(pat[i].begin() + 1, pat[i].end()), pat[i].end());
            nnz += pat[i].size();
            W = std::max(W, (int)pat[i].size());
        }
        // sparse path when the generator is sparse enough for ELL rows to pay off against DMMA tiles
        bool sparse_ok = (double)nnz <= 0.25 * (double)d * d && W <= 512;
        // Dense generators just beyond the cluster sweep's reach (256 < d <= 448) with many trajectories: the one-launch
        // ELL sweep with full-width rows beats the launch-per-term DMMA stream (measured, us per time step and direction,
        // 64 trajectories: d = 288 202 / 336, d = 400 267 / 452; at d = 512 the stream wins again, and with 16
        // trajectories it always does -- profiles/r2_dense_cluster_sweep.txt).  KROTOV_NO_DENSE_ELL=1 disables the rule.
        if (!sparse_ok && d > 256 && d <= 448 && N >= 48 && W <= 512 && !getenv("KROTOV_NO_DENSE_ELL")) sparse_ok = true;
        if (path == 0) path = sparse_ok ? KROTOV_PATH_SPARSE : KROTOV_PATH_DENSE;
        if (path == KROTOV_PATH_SPARSE) {
            hs.W = W;
            hs.nnz_union = (int)std::min<size_t>(nnz, 0x7fffffff);
            hs.cols.assign((size_t)d * W, 0);
            for (int i = 0; i < d; ++i)
                for (int sl = 0; sl < W; ++sl) hs.cols[(size_t)i * W + sl] = sl < (int)pat[i].size() ? pat[i][sl] : i;
            auto slot_of = [&](int i, int j) -> int {
                if (i == j) return 0;
                auto it = std::lower_bound(pat[i].begin() + 1, pat[i].end(), j);
                return (int)(it - pat[i].begin());
            };
            const size_t per_term = (size_t)d * W;
            hs.vals_f.assign((size_t)h->n_gen * (1 + L) * per_term, cplx(0, 0));
            hs.vals_b.assign(hs.vals_f.size(), cplx(0, 0));
            for (int g = 0; g < h->n_gen; ++g)
                for (int t = 0; t <= L; ++t) {
                    const size_t base = ((size_t)g * (1 + L) + t) * per_term;
                    for_each_entry(g, t, [&](int i, int j, cplx v) {
                        hs.vals_f[base + (size_t)i * W + slot_of(i, j)] += v;
                        hs.vals_b[base + (size_t)j * W + slot_of(j, i)] += std::conj(v);
                    });
                }
            hs.hermitian = (hs.vals_f == hs.vals_b);
            if (hs.hermitian) std::vector<cplx>().swap(hs.vals_b);
        }
    }
    h->path = path;
    if (h->taylor && path != KROTOV_PATH_WARP)
        return fail(h, KROTOV_ERR_UNSUPPORTED, "KROTOV_PROP_EXPMV: the generator does not fit the persistent warp kernel");

    if (path != KROTOV_PATH_SPARSE && h->Hdense.empty()) fill_dense();

    int rc;
    // ---- buffers common to both paths
    std::vector<double> alpha((size_t)L * N_T);
    for (int l = 0; l < L; ++l) {
        if (!(pb->lambda_a[l] != 0.0)) return fail(h, KROTOV_ERR_ARG, "lambda_a must be non-zero");
        for (int n = 0; n < N_T; ++n) alpha[(size_t)l * N_T + n] = pb->update_shape[(size_t)l * N_T + n] / pb->lambda_a[l];
    }
    if ((rc = upload(h, h->d_alpha, alpha, true))) return rc;
    h->update_shape_host.assign(pb->update_shape, pb->update_shape + (size_t)L * N_T);
    h->lambda_host.assign(pb->lambda_a, pb->lambda_a + L);
    if ((rc = upload(h, h->d_dt, h->dt, false))) return rc;
    if ((rc = upload(h, h->d_gen, h->gen_of_traj, false))) return rc;
    if ((rc = upload(h, h->d_weight, h->weight, false))) return rc;
    if ((rc = dev_alloc(h, h->d_eps_old, (size_t)L * N_T * 8))) return rc;
    if ((rc = dev_alloc(h, h->d_eps_new, (size_t)L * N_T * 8))) return rc;
    if ((rc = dev_alloc(h, h->d_ga, kr::kMaxCtrl * 8))) return rc;
    if ((rc = dev_alloc(h, h->d_tau, (size_t)N * 16))) return rc;
    if ((rc = dev_alloc(h, h->d_chicoef, (size_t)N * 16))) return rc;
    if ((rc = dev_alloc(h, h->d_err, 16))) return rc;
    KR_CUDA(h, cudaMemsetAsync(h->d_err.get<void>(), 0, 16, h->stream));
    KR_CUDA(h, cudaMemsetAsync(h->d_tau.get<void>(), 0, (size_t)N * 16, h->stream));
    // peer mailboxes for the per-time-step exchange between ranks: [N_T][L][rank], one per iteration parity
    // behind them (warp path): the accumulators of the one-hop cross-rank sum, word stride up to one 128-byte line
    h->mail_bytes = (size_t)N_T * kr::kMaxRanks * L * 8;
    h->xacc_bytes = (path == KROTOV_PATH_WARP && L * kr::kXLimbs <= 32) ? (size_t)N_T * L * kr::kXLimbs * kXaccMaxStride * 8 : 0;
    for (int par = 0; par < 2; ++par) {
        if ((rc = dev_alloc(h, h->d_mbox[par], h->mail_bytes + h->xacc_bytes + 256))) return rc;
        // rank-barrier flags (parity 0 only)
        KR_CUDA(h, cudaMemsetAsync(h->d_mbox[par].get<char>() + h->mail_bytes + h->xacc_bytes, 0, 256, h->stream));
        KR_CUDA(h, cudaMemsetAsync(h->d_mbox[par].get<void>(), 0xFF, h->mail_bytes, h->stream));
        if (h->xacc_bytes) KR_CUDA(h, cudaMemsetAsync(h->d_mbox[par].get<char>() + h->mail_bytes, 0, h->xacc_bytes, h->stream));
        h->peer_mbox[par][0] = h->d_mbox[par].get<double>();
    }

    // are all control terms Hermitian?  (mu_l^dagger = mu_l lets the kernel form mu_l chi ahead of time)
    h->mu_hermitian = (path == KROTOV_PATH_WARP);
    for (int g = 0; path == KROTOV_PATH_WARP && g < h->n_gen && h->mu_hermitian; ++g)
        for (int t = 1; t <= L && h->mu_hermitian; ++t)
            for (int i = 0; i < d && h->mu_hermitian; ++i)
                for (int j = i; j < d; ++j)
                    if (Hval(h, g, t, i, j) != std::conj(Hval(h, g, t, j, i))) {
                        h->mu_hermitian = false;
                        break;
                    }
    if (path == KROTOV_PATH_WARP) {
        if (!pattern_built && (rc = build_pattern(h))) return rc;
        if ((rc = upload(h, h->d_cols, h->cols, false))) return rc;
        {
            std::vector<cplx> raw;
            build_raw_rows(h, KROTOV_FORWARD, raw);
            if ((rc = upload(h, h->d_rawf, raw, true))) return rc;
            build_raw_rows(h, KROTOV_BACKWARD, raw);
            if ((rc = upload(h, h->d_rawb, raw, true))) return rc;
        }
        choose_launch(h);
        if (h->taylor && h->tpw > 1)  // (several trajectories per warp, one after another: not served by the Taylor step)
            return fail(h, KROTOV_ERR_UNSUPPORTED, "KROTOV_PROP_EXPMV: more trajectories than one per warp of a co-resident "
                                                   "grid (" + std::to_string(N) + ")");
        // (the one-thread kernel propagates with the Chebyshev series only: Expmv problems run on the warp kernel)
        h->tiny = !h->taylor && d >= 2 && d <= 4 && N <= 32 && tiny_kernel_for(d, L) != nullptr && !getenv("KROTOV_NO_TINY");
        // padded state arrays [N][32]
        auto pad_states = [&](const double *src, std::vector<cplx> &dst) {
            dst.assign((size_t)N * h->lpt, cplx(0, 0));
            const cplx *s = reinterpret_cast<const cplx *>(src);
            for (int k = 0; k < N; ++k)
                for (int i = 0; i < d; ++i) dst[(size_t)k * h->lpt + i] = s[(size_t)k * d + i];
        };
        std::vector<cplx> tmp;
        pad_states(pb->psi0, tmp);
        if ((rc = upload(h, h->d_psi0, tmp, true))) return rc;
        if (h->has_target) {
            pad_states(pb->target, tmp);
            if ((rc = upload(h, h->d_target, tmp, true))) return rc;
        }
        const size_t slab = (size_t)N * (N_T + 1) * h->lpt * 16;
        h->x_slab = slab / 16;
        // (replicated forward sweep: two chi trajectories, by iteration parity -- a peer that is one iteration ahead
        // writes the other one)
        if ((rc = dev_alloc(h, h->d_X, slab * (h->rf_wanted ? 2 : 1)))) return rc;
        if (h->store_fw && (rc = dev_alloc(h, h->d_Phi, slab))) return rc;
        if ((rc = dev_alloc(h, h->d_chiT, (size_t)N * h->lpt * 16))) return rc;
        if ((rc = dev_alloc(h, h->d_psif, (size_t)N * h->lpt * 16))) return rc;
        // Freshly initialised propagators hold the initial states: that is what `skip_initial_forward_propagation`
        // (src/optimize.jl:171-181) leaves for the first chi(T) (:297) and update_result! (:378-381)
        KR_CUDA(h, cudaMemcpyAsync(h->d_psif.get<void>(), h->d_psi0.get<void>(), (size_t)N * h->lpt * 16, cudaMemcpyDeviceToDevice,
                                   h->stream));
        if (h->has_target) {
            std::vector<cplx> tau0(N);
            const cplx *s0 = reinterpret_cast<const cplx *>(pb->psi0), *tg = reinterpret_cast<const cplx *>(pb->target);
            for (int k = 0; k < N; ++k) {
                cplx a(0, 0);
                for (int i = 0; i < d; ++i) a += std::conj(tg[(size_t)k * d + i]) * s0[(size_t)k * d + i];
                tau0[k] = a;
            }
            if ((rc = upload(h, h->d_tau, tau0, true))) return rc;
        }
        h->swept = true;
        if ((rc = dev_alloc(h, h->d_R, ((size_t)N_T * h->nCTA * L + (size_t)N_T * L) * 8))) return rc;
        if ((rc = dev_alloc(h, h->d_acc, (size_t)N_T * L * kr::kFixLimbs * 8))) return rc;
        if (getenv("KROTOV_PROF")) {
            if ((rc = dev_alloc(h, h->d_prof, (size_t)h->nCTA * 8 * 8))) return rc;
            KR_CUDA(h, cudaMemsetAsync(h->d_prof.get<void>(), 0, h->d_prof.bytes(), h->stream));
        }
    } else {
        kr::SparseDesc sd;
        if (path == KROTOV_PATH_SPARSE) {
            sd.W = hs.W; sd.nnz_union = hs.nnz_union; sd.hermitian = hs.hermitian;
            sd.cols = &hs.cols; sd.vals_f = &hs.vals_f; sd.vals_b = &hs.vals_b;
        }
        h->dense = kr::dense_create(h->d, h->N, h->L, h->N_T, h->n_gen, h->Hdense, h->gen_of_traj, pb->psi0,
                                    pb->target, h->store_fw, h->stream, h->err,
                                    path == KROTOV_PATH_SPARSE ? &sd : nullptr);
        if (!h->dense) return KROTOV_ERR_UNSUPPORTED;
        std::vector<cplx>().swap(h->Hdense);  // the device holds the generators now
        if (!kr::dense_seed(h->dense, h->d_tau.get<double2>(), h->err)) return KROTOV_ERR_CUDA;
        h->swept = true;
    }
    if (cudaDeviceSynchronize() != cudaSuccess) return fail(h, KROTOV_ERR_CUDA, "device sync after create failed");
    return KROTOV_OK;
}

int krotov_create(const krotov_problem *pb, krotov_handle *out) {
    if (!pb || !out) return fail(nullptr, KROTOV_ERR_ARG, "null argument");
    *out = nullptr;
    if (pb->struct_size != (int32_t)sizeof(krotov_problem))
        return fail(nullptr, KROTOV_ERR_ARG, "krotov_problem.struct_size mismatch (ABI version?)");
    if (pb->d < 1 || pb->n_traj < 1 || pb->n_steps < 1 || pb->n_gen < 1)
        return fail(nullptr, KROTOV_ERR_ARG, "d, n_traj, n_steps, n_gen must be >= 1");
    if (pb->n_ctrl < 1) return fail(nullptr, KROTOV_ERR_ARG, "no controls in trajectories: cannot optimize");
    if (pb->n_ctrl > kr::kMaxCtrl) return fail(nullptr, KROTOV_ERR_UNSUPPORTED, "more than 8 controls");
    if (!pb->tlist || !pb->gen_of_traj || !pb->gen_values || !pb->psi0 || !pb->update_shape || !pb->lambda_a)
        return fail(nullptr, KROTOV_ERR_ARG, "null array in krotov_problem");
    if (pb->gen_format == KROTOV_GEN_CSR && (!pb->csr_rowptr || !pb->csr_colind))
        return fail(nullptr, KROTOV_ERR_ARG, "CSR pattern missing");
    if (pb->functional != KROTOV_CHI_HOST && !pb->target)
        return fail(nullptr, KROTOV_ERR_ARG, "built-in functional needs target states");
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev == 0)
        return fail(nullptr, KROTOV_ERR_CUDA, std::string("no CUDA device: ") + cudaGetErrorString(ce));
    if (pb->device < 0 || pb->device >= ndev) return fail(nullptr, KROTOV_ERR_ARG, "bad device ordinal");

    std::unique_ptr<krotov_handle_s> h(new krotov_handle_s());
    const int rc = create_handle(h.get(), pb);
    if (rc != KROTOV_OK) {
        g_create_error = h->err;
        return rc;
    }
    *out = h.release();
    return KROTOV_OK;
}

int krotov_get_info(krotov_handle h, krotov_info *out) {
    if (!h || !out) return KROTOV_ERR_ARG;
    memset(out, 0, sizeof(*out));
    out->struct_size = sizeof(krotov_info);
    out->path = h->path;
    out->ell_width = h->Wt;
    out->nnz_union = h->nnz_union;
    out->grid_blocks = h->nCTA;
    out->block_threads = h->wpc * h->lpt + 32;
    if (h->tiny && h->world == 1 && !h->amp_set) {
        out->grid_blocks = 1;
        out->block_threads = 32;
    }
    out->m_fw = h->cheb[0].m_max_used;
    out->m_bw = h->cheb[1].m_max_used;
    out->sm_count = h->sm_count;
    out->exchange = h->rf ? 5 : h->xchg_last;
    out->launches_total = h->launches_total;
    out->launches_last = h->launches_last;
    out->ms_last = h->ms_last;
    out->ms_last_backward = h->ms_last_bw;
    out->hbm_bytes_state = (int64_t)h->d_X.bytes();
    out->fallback_steps = h->fallback_steps;
    out->ms_rank_wait = h->ms_rank_wait;
    out->kernel = h->kernel_last;
    out->lanes_per_traj = h->lanes_last;
    if (h->dense) kr::dense_info(h->dense, out);
    return KROTOV_OK;
}

int krotov_set_cheby(krotov_handle h, int direction, int n_dt_class, const int32_t *dt_class_of_step,
                     const double *dt_of_class, const double *E_min, const double *Delta, const int32_t *m,
                     const double *coeffs, int m_max) {
    if (!h) return KROTOV_ERR_ARG;
    if (direction != KROTOV_FORWARD && direction != KROTOV_BACKWARD) return fail(h, KROTOV_ERR_ARG, "bad direction");
    if (n_dt_class < 1 || !dt_class_of_step || !dt_of_class || !E_min || !Delta || !m || !coeffs || m_max < 1)
        return fail(h, KROTOV_ERR_ARG, "bad argument to krotov_set_cheby");
    if (h->taylor) return fail(h, KROTOV_ERR_STATE, "the handle propagates with KROTOV_PROP_EXPMV: use krotov_set_taylor");
    Trace tr("set_cheby");
    cudaSetDevice(h->device);
    ChebyTables &ct = h->cheb[direction];
    for (int n = 0; n < h->N_T; ++n)
        if (dt_class_of_step[n] < 0 || dt_class_of_step[n] >= n_dt_class)
            return fail(h, KROTOV_ERR_ARG, "dt_class_of_step out of range");
    for (int c = 0; c < n_dt_class; ++c) {
        if (direction == KROTOV_FORWARD && !(dt_of_class[c] > 0)) return fail(h, KROTOV_ERR_ARG, "forward dt must be > 0");
        if (direction == KROTOV_BACKWARD && !(dt_of_class[c] < 0)) return fail(h, KROTOV_ERR_ARG, "backward dt must be < 0");
    }
    ct.ndtc = n_dt_class;
    ct.mmax = m_max;
    ct.E_min.assign(E_min, E_min + h->n_gen);
    ct.Delta.assign(Delta, Delta + h->n_gen);
    ct.m_host.assign(m, m + (size_t)h->n_gen * n_dt_class);
    ct.coef_host.assign(coeffs, coeffs + (size_t)h->n_gen * n_dt_class * m_max);
    ct.m_max_used = 0;
    for (int g = 0; g < h->n_gen; ++g) {
        if (!(Delta[g] > 0)) return fail(h, KROTOV_ERR_ARG, "Delta must be > 0");
        for (int c = 0; c < n_dt_class; ++c) {
            int mm = ct.m_host[(size_t)g * n_dt_class + c];
            if (mm < 1 || mm > m_max) return fail(h, KROTOV_ERR_ARG, "m out of range");
            ct.m_max_used = std::max(ct.m_max_used, mm);
        }
    }
    ct.phase_host.resize((size_t)h->n_gen * n_dt_class);
    for (int g = 0; g < h->n_gen; ++g) {
        const double beta = Delta[g] / 2 + E_min[g];
        for (int c = 0; c < n_dt_class; ++c)
            ct.phase_host[(size_t)g * n_dt_class + c] = std::exp(cplx(0.0, -beta * dt_of_class[c]));
    }
    ct.dtc_of_step.assign(dt_class_of_step, dt_class_of_step + h->N_T);
    int rc;
    if ((rc = upload(h, ct.dtc, ct.dtc_of_step, false))) return rc;
    if ((rc = upload(h, ct.coef, ct.coef_host, false))) return rc;
    if ((rc = upload(h, ct.m, ct.m_host, false))) return rc;
    if ((rc = upload(h, ct.phase, ct.phase_host, true))) return rc;  // (waits for all four: the next call rewrites ct)
    ct.set = true;
    tr.lap("tables uploaded");
    if (h->path == KROTOV_PATH_WARP) {
        std::vector<cplx> rows;
        DevBuf &dP = direction == KROTOV_FORWARD ? h->d_Pf : h->d_Pb;
        const DevBuf &raw = direction == KROTOV_FORWARD ? h->d_rawf : h->d_rawb;
        if (raw && !getenv("KROTOV_HOST_ROWS")) {
            // rows scaled on the device from the unscaled rows uploaded at krotov_create
            std::vector<double> fb((size_t)2 * h->n_gen);
            for (int g = 0; g < h->n_gen; ++g) {
                const double sc = 4.0 / Delta[g];
                fb[2 * g] = direction == KROTOV_FORWARD ? -sc : sc;
                fb[2 * g + 1] = Delta[g] / 2 + E_min[g];
            }
            if ((rc = upload(h, h->d_rowscale, fb, true))) return rc;
            const size_t total = (size_t)h->n_gen * (1 + h->L) * (h->Wt + 1) * h->lpt;
            if ((rc = dev_alloc(h, dP, total * 16))) return rc;
            scale_rows_kernel<<<(unsigned)((total + 255) / 256), 256, 0, h->stream>>>(
                raw.get<const double2>(), h->d_rowscale.get<const double2>(), dP.get<double2>(), 1 + h->L, h->Wt, h->lpt, h->d, total);
            KR_CUDA(h, cudaStreamSynchronize(h->stream));  // the next call may rewrite d_rowscale
            h->launches_total += 1;
            tr.lap("rows scaled on the device");
        } else {
            build_rows(h, direction, rows);
            tr.lap("rows built");
            if ((rc = upload(h, dP, rows, true))) return rc;
        }
        if (direction == KROTOV_FORWARD) {
            std::vector<double> inv_s(h->n_gen);
            for (int g = 0; g < h->n_gen; ++g) inv_s[g] = Delta[g] / 4.0;
            if ((rc = upload(h, h->d_inv_s, inv_s, true))) return rc;
        }
        if (h->tiny) {
            build_dense_terms(h, direction, rows);
            bool imag = !getenv("KROTOV_NO_TINY_IMAG");
            for (const cplx &v : rows) imag = imag && (v.real() == 0.0);
            h->tiny_imag[direction] = imag;
            if ((rc = upload(h, direction == KROTOV_FORWARD ? h->d_Tf : h->d_Tb, rows, true))) return rc;
        }
        tr.lap("rows uploaded");
    } else {
        std::string e;
        if (!kr::dense_set_cheby(h->dense, direction, n_dt_class, ct.dtc_of_step, ct.E_min, ct.Delta, ct.m_host,
                                 ct.coef_host, m_max, ct.phase_host, e))
            return fail(h, KROTOV_ERR_CUDA, e);
    }
    return KROTOV_OK;
}

int krotov_set_taylor(krotov_handle h, int direction, int n_dt_class, const int32_t *dt_class_of_step,
                      const double *dt_of_class, const double *mu, const double *scale, const int32_t *s,
                      const int32_t *m, const double *coeffs, int m_max) {
    if (!h) return KROTOV_ERR_ARG;
    if (direction != KROTOV_FORWARD && direction != KROTOV_BACKWARD) return fail(h, KROTOV_ERR_ARG, "bad direction");
    if (n_dt_class < 1 || !dt_class_of_step || !dt_of_class || !mu || !scale || !s || !m || !coeffs || m_max < 1)
        return fail(h, KROTOV_ERR_ARG, "bad argument to krotov_set_taylor");
    if (!h->taylor) return fail(h, KROTOV_ERR_STATE, "krotov_set_taylor needs a handle created with KROTOV_PROP_EXPMV");
    cudaSetDevice(h->device);
    for (int n = 0; n < h->N_T; ++n)
        if (dt_class_of_step[n] < 0 || dt_class_of_step[n] >= n_dt_class)
            return fail(h, KROTOV_ERR_ARG, "dt_class_of_step out of range");
    for (int c = 0; c < n_dt_class; ++c) {
        if (direction == KROTOV_FORWARD && !(dt_of_class[c] > 0)) return fail(h, KROTOV_ERR_ARG, "forward dt must be > 0");
        if (direction == KROTOV_BACKWARD && !(dt_of_class[c] < 0)) return fail(h, KROTOV_ERR_ARG, "backward dt must be < 0");
    }
    const int n_gen = h->n_gen;
    for (int g = 0; g < n_gen; ++g) {
        if (!(std::isfinite(scale[g]) && scale[g] > 0)) return fail(h, KROTOV_ERR_ARG, "scale must be finite and > 0");
        if (!std::isfinite(mu[g])) return fail(h, KROTOV_ERR_ARG, "mu must be finite");
        for (int c = 0; c < n_dt_class; ++c) {
            const size_t i = (size_t)g * n_dt_class + c;
            if (m[i] < 1 || m[i] > m_max) return fail(h, KROTOV_ERR_ARG, "m out of range");
            if (s[i] < 1) return fail(h, KROTOV_ERR_ARG, "s must be >= 1");
        }
    }
    // the tables of krotov_set_cheby, with (m, s) pairs in the count table and the phase of one repeat
    ChebyTables &ct = h->cheb[direction];
    ct.ndtc = n_dt_class;
    ct.mmax = m_max;
    ct.m_host.resize((size_t)2 * n_gen * n_dt_class);
    ct.phase_host.resize((size_t)n_gen * n_dt_class);
    ct.m_max_used = 0;
    for (int g = 0; g < n_gen; ++g)
        for (int c = 0; c < n_dt_class; ++c) {
            const size_t i = (size_t)g * n_dt_class + c;
            ct.m_host[2 * i] = m[i];
            ct.m_host[2 * i + 1] = s[i];
            ct.m_max_used = (int)std::min<long long>(INT32_MAX, std::max<long long>(ct.m_max_used, (long long)m[i] * s[i]));
            ct.phase_host[i] = std::exp(cplx(0.0, -mu[g] * dt_of_class[c] / s[i]));
        }
    ct.coef_host.assign(coeffs, coeffs + (size_t)n_gen * n_dt_class * m_max);
    ct.dtc_of_step.assign(dt_class_of_step, dt_class_of_step + h->N_T);
    int rc;
    if ((rc = upload(h, ct.dtc, ct.dtc_of_step, false))) return rc;
    if ((rc = upload(h, ct.coef, ct.coef_host, false))) return rc;
    if ((rc = upload(h, ct.m, ct.m_host, false))) return rc;
    if ((rc = upload(h, ct.phase, ct.phase_host, true))) return rc;  // (waits for all four: the next call rewrites ct)
    ct.set = true;
    // R_t = -i scale_g (H_t - mu_g delta_t0) in both directions (the backward rows hold the adjoint generator and the
    // coefficients carry the negative dt): scale_rows_kernel with (fy, beta) = (-scale_g, mu_g)
    std::vector<double> fb((size_t)2 * n_gen);
    for (int g = 0; g < n_gen; ++g) {
        fb[2 * g] = -scale[g];
        fb[2 * g + 1] = mu[g];
    }
    if ((rc = upload(h, h->d_rowscale, fb, true))) return rc;
    DevBuf &dP = direction == KROTOV_FORWARD ? h->d_Pf : h->d_Pb;
    const DevBuf &raw = direction == KROTOV_FORWARD ? h->d_rawf : h->d_rawb;
    const size_t total = (size_t)n_gen * (1 + h->L) * (h->Wt + 1) * h->lpt;
    if ((rc = dev_alloc(h, dP, total * 16))) return rc;
    scale_rows_kernel<<<(unsigned)((total + 255) / 256), 256, 0, h->stream>>>(
        raw.get<const double2>(), h->d_rowscale.get<const double2>(), dP.get<double2>(), 1 + h->L, h->Wt, h->lpt, h->d, total);
    KR_CUDA(h, cudaStreamSynchronize(h->stream));  // the next call may rewrite d_rowscale
    KR_CUDA(h, cudaGetLastError());
    h->launches_total += 1;
    if (direction == KROTOV_FORWARD) {  // overlaps: Im<chi|H_l|psi> = Re<chi|R_l psi> / scale
        std::vector<double> inv_s(n_gen);
        for (int g = 0; g < n_gen; ++g) inv_s[g] = 1.0 / scale[g];
        if ((rc = upload(h, h->d_inv_s, inv_s, true))) return rc;
    }
    return KROTOV_OK;
}

// a_l(eps_old) and a_l'(eps_old) for the pulses of the coming sweep: O(L N_T) host work, uploaded on the launch stream
static int prepare_amplitudes(krotov_handle h, const double *pulses) {
    if (!h->amp_set) return KROTOV_OK;
    const int L = h->L, N_T = h->N_T, D = kr::kAmpMaxDeg;
    for (int t = 0; t < (int)h->tie_ctrl.size(); ++t) {  // tied terms carry their control's pulse: one row per term
        const int t0 = (int)(std::find(h->tie_ctrl.begin(), h->tie_ctrl.end(), h->tie_ctrl[t]) - h->tie_ctrl.begin());
        if (t0 != t && memcmp(pulses + (size_t)t * N_T, pulses + (size_t)t0 * N_T, (size_t)N_T * 8) != 0)
            return fail(h, KROTOV_ERR_ARG, "pulse rows of tied control terms " + std::to_string(t0) + " and " +
                                               std::to_string(t) + " differ");
    }
    std::vector<double> &a = h->amp_old_host, &da = h->amp_dfac_host;
    a.resize((size_t)L * N_T);
    da.resize((size_t)L * N_T);
    for (int l = 0; l < L; ++l) {
        const double s = h->amp_sat.empty() ? 0.0 : h->amp_sat[l];
        for (int n = 0; n < N_T; ++n) {
            const double e = pulses[(size_t)l * N_T + n];
            double v = e, dv = 1.0;
            if (s > 0.0) {  // saturating: x = tanh(s e), a = shape P(x), a' = shape P'(x) s (1 - x)(1 + x)
                const double x = std::tanh(s * e);
                v = x;
                if (!h->amp_poly.empty()) {
                    const double *q = &h->amp_poly[(size_t)l * (D + 1)];
                    v = q[D];
                    for (int p = D - 1; p >= 0; --p) v = std::fma(v, x, q[p]);  // same Horner form as the kernels
                    dv = 0.0;
                    for (int p = D; p >= 1; --p) dv = dv * x + p * q[p];
                }
                dv = dv * s * ((1.0 - x) * (1.0 + x));
            } else if (!h->amp_poly.empty()) {
                const double *q = &h->amp_poly[(size_t)l * (D + 1)];
                v = q[D];
                for (int p = D - 1; p >= 0; --p) v = std::fma(v, e, q[p]);  // same Horner form as the kernels
                dv = 0.0;
                for (int p = D; p >= 1; --p) dv = dv * e + p * q[p];
            }
            if (!h->amp_shape.empty()) {
                const double sh = h->amp_shape[(size_t)l * N_T + n];
                v = sh * v;
                dv = sh * dv;
            }
            a[(size_t)l * N_T + n] = v;
            da[(size_t)l * N_T + n] = dv;
        }
    }
    int rc;
    if (!h->tie_ctrl.empty()) {
        // tied control terms: a' goes into the tie table, the kernels' per-term factor becomes 1 (WarpParams::tie)
        h->tie_host.assign(h->tie_ctrl.begin(), h->tie_ctrl.end());
        h->tie_host.insert(h->tie_host.end(), da.begin(), da.end());
        std::fill(da.begin(), da.end(), 1.0);
        if ((rc = upload(h, h->d_tie, h->tie_host, false))) return rc;
    }
    if ((rc = upload(h, h->d_amp_old, a, false))) return rc;
    if ((rc = upload(h, h->d_amp_dfac, da, false))) return rc;
    return KROTOV_OK;
}

static int begin_timed(krotov_handle h) {
    h->launches_last = 0;
    KR_CUDA(h, cudaEventRecord(h->ev0, h->stream));
    return KROTOV_OK;
}
static int end_timed(krotov_handle h) {
    KR_CUDA(h, cudaEventRecord(h->ev1, h->stream));
    KR_CUDA(h, cudaStreamSynchronize(h->stream));
    float ms = 0.f;
    KR_CUDA(h, cudaEventElapsedTime(&ms, h->ev0, h->ev1));
    h->ms_last = ms;
    h->launches_total += h->launches_last;
    KR_CUDA(h, cudaGetLastError());
    return KROTOV_OK;
}

int krotov_forward(krotov_handle h, const double *pulses) {
    if (!h || !pulses) return KROTOV_ERR_ARG;
    if (!h->cheb[0].set)
        return fail(h, KROTOV_ERR_STATE, h->taylor ? "krotov_set_taylor(FORWARD) must be called before krotov_forward"
                                                   : "krotov_set_cheby(FORWARD) must be called before krotov_forward");
    cudaSetDevice(h->device);
    KR_CUDA(h, cudaMemcpyAsync(h->d_eps_old.get<void>(), pulses, (size_t)h->L * h->N_T * 8, cudaMemcpyHostToDevice, h->stream));
    int rc;
    if ((rc = prepare_amplitudes(h, pulses))) return rc;
    if ((rc = begin_timed(h))) return rc;
    if (h->path == KROTOV_PATH_WARP) {
        if ((rc = launch_warp(h, 0))) return rc;
    } else {
        std::string e;
        if (!kr::dense_forward(h->dense, h->d_eps_old.get<const double>(), h->d_tau.get<double2>(), h->launches_last, e))
            return fail(h, KROTOV_ERR_CUDA, e);
    }
    if ((rc = end_timed(h))) return rc;
    h->swept = true;
    h->chiT_valid = false;
    h->chicoef_valid = false;
    return KROTOV_OK;
}

int krotov_set_chi(krotov_handle h, const double *chi) {
    if (!h || !chi) return KROTOV_ERR_ARG;
    cudaSetDevice(h->device);
    const int N = h->N, d = h->d;
    if (h->path == KROTOV_PATH_WARP) {
        std::vector<cplx> tmp((size_t)N * h->lpt, cplx(0, 0));
        const cplx *s = reinterpret_cast<const cplx *>(chi);
        for (int k = 0; k < N; ++k)
            for (int i = 0; i < d; ++i) tmp[(size_t)k * h->lpt + i] = s[(size_t)k * d + i];
        int rc;
        if ((rc = upload(h, h->d_chiT, tmp, true))) return rc;
    } else {
        std::string e;
        if (!kr::dense_set_chi(h->dense, chi, e)) return fail(h, KROTOV_ERR_CUDA, e);
    }
    h->chiT_valid = true;
    return KROTOV_OK;
}

int krotov_set_chi_coeffs(krotov_handle h, const double *coef) {
    if (!h || !coef) return KROTOV_ERR_ARG;
    if (!h->has_target) return fail(h, KROTOV_ERR_STATE, "krotov_set_chi_coeffs needs target states");
    cudaSetDevice(h->device);
    const cplx *c = reinterpret_cast<const cplx *>(coef);
    int rc;
    if ((rc = upload(h, h->d_chicoef, std::vector<cplx>(c, c + h->N), true))) return rc;
    h->chicoef_valid = true;
    h->chiT_valid = false;
    return KROTOV_OK;
}

// what krotov_iterate does before its launch(es): argument / state checks, pulses to the device, chi coefficients,
// exchange arrays reset.  Leaves the timed region open (begin_timed).
static int iterate_prepare(krotov_handle h, const double *guess_pulses) {
    if (!h->cheb[0].set || !h->cheb[1].set)
        return fail(h, KROTOV_ERR_STATE, h->taylor ? "krotov_set_taylor must be called for both directions before krotov_iterate"
                                                   : "krotov_set_cheby must be called for both directions before krotov_iterate");
    cudaSetDevice(h->device);
    const bool need_device_coef = !h->chiT_valid && !h->chicoef_valid;
    if (need_device_coef) {
        if (h->functional == KROTOV_CHI_HOST)
            return fail(h, KROTOV_ERR_STATE, "functional is KROTOV_CHI_HOST: call krotov_set_chi before krotov_iterate");
        if (!h->swept) return fail(h, KROTOV_ERR_STATE, "krotov_forward must run before the first krotov_iterate");
        if (h->world > 1 && !h->rf && h->functional == KROTOV_CHI_SM)
            return fail(h, KROTOV_ERR_STATE, "multi-rank J_T_sm needs krotov_set_chi_coeffs (global sum of tau)");
    }
    const size_t pbytes = (size_t)h->L * h->N_T * 8;
    KR_CUDA(h, cudaMemcpyAsync(h->d_eps_old.get<void>(), guess_pulses, pbytes, cudaMemcpyHostToDevice, h->stream));
    int rc;
    if ((rc = prepare_amplitudes(h, guess_pulses))) return rc;
    if ((rc = begin_timed(h))) return rc;
    if (need_device_coef) {
        chi_coef_kernel<<<1, 32, 0, h->stream>>>(h->functional, h->N, h->N_global, h->d_tau.get<const double2>(),
                                                 h->d_weight.get<const double>(), h->d_chicoef.get<double2>());
        h->launches_last += 1;
    }
    if (h->rf) KR_CUDA(h, cudaMemsetAsync(h->d_rfcount.get<void>(), 0, 16, h->stream));
    if (h->world > 1 && !h->rf) {
        // the mailbox of the NEXT iteration's parity is cleared now (peers are at most one iteration ahead)
        const int nxt = (int)((h->iter_count + 1) & 1);
        KR_CUDA(h, cudaMemsetAsync(h->d_mbox[nxt].get<void>(), 0xFF, h->mail_bytes, h->stream));
        if (h->xacc_bytes) KR_CUDA(h, cudaMemsetAsync(h->d_mbox[nxt].get<char>() + h->mail_bytes, 0, h->xacc_bytes, h->stream));
    }
    if (h->path == KROTOV_PATH_WARP) {
        if (h->nCTA > 1 || h->world > 1) KR_CUDA(h, cudaMemsetAsync(h->d_R.get<void>(), 0xFF, h->d_R.bytes(), h->stream));
        if (h->nCTA > 1) KR_CUDA(h, cudaMemsetAsync(h->d_acc.get<void>(), 0, h->d_acc.bytes(), h->stream));
    }
    return KROTOV_OK;
}

static int iterate_finish(krotov_handle h, double *new_pulses, double *g_a_int) {
    int rc;
    if ((rc = end_timed(h))) return rc;
    h->iter_count += 1;
    if ((rc = check_err_flag(h))) return rc;
    KR_CUDA(h, cudaMemcpy(new_pulses, h->d_eps_new.get<void>(), (size_t)h->L * h->N_T * 8, cudaMemcpyDeviceToHost));
    KR_CUDA(h, cudaMemcpy(g_a_int, h->d_ga.get<void>(), (size_t)h->L * 8, cudaMemcpyDeviceToHost));
    for (int t = 0; t < (int)h->tie_first.size(); ++t)  // tied terms: the control's integral sits at its first term
        if (!h->tie_first[t]) g_a_int[t] = 0.0;
    h->chiT_valid = false;
    h->chicoef_valid = false;
    h->swept = true;
    return KROTOV_OK;
}

int krotov_iterate(krotov_handle h, const double *guess_pulses, double *new_pulses, double *g_a_int) {
    if (!h || !guess_pulses || !new_pulses || !g_a_int) return KROTOV_ERR_ARG;
    int rc;
    if ((rc = iterate_prepare(h, guess_pulses))) return rc;
    if (h->path == KROTOV_PATH_WARP) {
        if ((rc = launch_warp(h, 1))) return rc;
    } else {
        std::string e;
        double ms_bw = 0.0;
        kr::DenseComm dc;
        dc.rank = h->rank;
        dc.world = h->world;
        dc.err_flag = h->d_err.get<int>();
        dc.timeout_cycles = 20000000000ll;
        for (int r = 0; r < kr::kMaxRanks; ++r) dc.mbox[r] = h->peer_mbox[(int)(h->iter_count & 1)][r];
        kr::dense_set_comm(h->dense, dc);
        if (!kr::dense_iterate(h->dense, h->d_eps_old.get<const double>(), h->d_eps_new.get<double>(),
                               h->d_alpha.get<const double>(), h->d_dt.get<const double>(), h->d_ga.get<double>(),
                               h->chiT_valid ? nullptr : h->d_chicoef.get<const double2>(), h->d_tau.get<double2>(),
                               h->launches_last, e))
            return fail(h, KROTOV_ERR_CUDA, e);
        h->ms_last_bw = ms_bw;
    }
    return iterate_finish(h, new_pulses, g_a_int);
}

// Replicated forward sweep: possible when this handle holds ALL trajectories of the problem and runs the persistent
// kernel with one trajectory per warp (KROTOV_NO_RF=1 keeps the sharded forward sweep with its per-step exchange).
static bool rf_eligible(krotov_handle h) {
    return h->rf_wanted && h->path == KROTOV_PATH_WARP && h->N == h->N_global && h->tpw == 1 && !h->pair && h->lpt == 32 &&
           kernel_rf_table().count(KernelKey{h->Wt, h->preg ? h->L : 0, 32}) && !getenv("KROTOV_NO_RF");
}

// this rank's share of the backward sweep: a contiguous block cut at generator boundaries where that is possible
static void rf_shard(krotov_handle h, int rank, int world, int *lo, int *hi) {
    const int N = h->N;
    std::vector<int> cuts{0};
    for (int k = 1; k < N; ++k)
        if (h->gen_of_traj[k] != h->gen_of_traj[k - 1]) cuts.push_back(k);
    cuts.push_back(N);
    std::vector<int> b(world + 1);
    for (int r = 0; r <= world; ++r) {
        const long long ideal = (long long)r * N / world;
        int best = cuts[0];
        for (int c : cuts)
            if (std::llabs(c - ideal) < std::llabs(best - ideal)) best = c;
        b[r] = best;
    }
    b[0] = 0;
    b[world] = N;
    bool ok = true;
    for (int r = 0; r < world; ++r) ok = ok && b[r + 1] > b[r];
    if (!ok)
        for (int r = 0; r <= world; ++r) b[r] = (int)((long long)r * N / world);
    *lo = b[rank];
    *hi = b[rank + 1];
}

// arrival counter + backward shard of the replicated forward sweep (when the mode is chosen at connect time)
static int rf_prepare(krotov_handle h, int rank, int world) {
    int rc;
    if ((rc = dev_alloc(h, h->d_rfcount, 16))) return rc;
    rf_shard(h, rank, world, &h->bw_lo, &h->bw_hi);
    h->rf = true;
    return KROTOV_OK;
}

// ---- several ranks emulated on ONE device (diagnostics / tests) ---------------------------------------------------------
// Ranks that wait for one another inside their persistent kernels cannot run as separate launches on one GPU (nothing
// makes them co-resident).  A group of handles created on the same device is instead driven by ONE cooperative launch
// whose grid is the union of the ranks' grids; every CTA picks its rank's parameter block and runs the UNCHANGED
// multi-rank code: the cross-rank accumulators / mailboxes are then plain device pointers instead of NVLink mappings.
int krotov_group_connect(krotov_handle *hs, int world) {
    if (!hs || world < 1 || world > kr::kMaxRanks) return KROTOV_ERR_ARG;
    int total = 0, mx = 0;
    for (int r = 0; r < world; ++r) {
        krotov_handle h = hs[r];
        if (!h) return KROTOV_ERR_ARG;
        if (h->path != KROTOV_PATH_WARP || h->pair || (h->tiny && world == 1))
            return fail(h, KROTOV_ERR_UNSUPPORTED, "krotov_group_connect: warp path (one trajectory per warp) only");
        if (h->device != hs[0]->device || h->L != hs[0]->L || h->N_T != hs[0]->N_T || h->Wt != hs[0]->Wt ||
            h->lpt != hs[0]->lpt || h->preg != hs[0]->preg || h->wpc != hs[0]->wpc || h->tpw != hs[0]->tpw ||
            h->taylor != hs[0]->taylor)
            return fail(h, KROTOV_ERR_ARG, "krotov_group_connect: ranks must share device, grid shape and kernel instance");
        total += h->nCTA;
        mx = std::max(mx, h->nCTA);
    }
    if (total > hs[0]->sm_count) return fail(hs[0], KROTOV_ERR_UNSUPPORTED, "krotov_group_connect: more CTAs than SMs");
    bool rf_all = world > 1;
    for (int r = 0; r < world; ++r) rf_all = rf_all && rf_eligible(hs[r]) && hs[r]->N == hs[0]->N;
    rf_all = rf_all && kernel_rf_emul_table().count(KernelKey{hs[0]->Wt, hs[0]->preg ? hs[0]->L : 0, hs[0]->lpt});
    if (!rf_all && world > 1)
        for (int r = 0; r < world; ++r)
            if (hs[r]->rf_wanted)  // handles that hold ALL trajectories must never run the sharded exchange
                return fail(hs[r], KROTOV_ERR_UNSUPPORTED, "replicated_forward was requested but cannot be used by this group");
    for (int r = 0; r < world; ++r) {
        krotov_handle h = hs[r];
        h->rank = r;
        h->world = world;
        h->total_ctas = total;
        h->max_ctas = mx;
        h->iter_count = 0;
        h->rf = false;
        for (int q = 0; q < world; ++q)
            for (int par = 0; par < 2; ++par) h->peer_mbox[par][q] = hs[q]->d_mbox[par].get<double>();
        if (rf_all) {
            int rc = rf_prepare(h, r, world);
            if (rc) return rc;
            for (int q = 0; q < world; ++q) {
                h->peer_Xbase[q] = hs[q]->d_X.get<double2>();
                h->peer_flag[q] = (unsigned long long *)(hs[q]->d_mbox[0].get<char>() + hs[q]->mail_bytes + hs[q]->xacc_bytes);
            }
        }
    }
    return KROTOV_OK;
}

int krotov_group_iterate(krotov_handle *hs, int world, const double *guess_pulses, double *new_pulses, double *g_a_int) {
    if (!hs || world < 1 || world > kr::kMaxRanks || !guess_pulses || !new_pulses || !g_a_int) return KROTOV_ERR_ARG;
    krotov_handle h0 = hs[0];
    const size_t pn = (size_t)h0->L * h0->N_T;
    int rc;
    for (int r = 0; r < world; ++r) {
        if (hs[r]->world != world || hs[r]->rank != r) return fail(hs[r], KROTOV_ERR_STATE, "krotov_group_connect first");
        if ((rc = iterate_prepare(hs[r], guess_pulses))) return rc;
    }
    std::vector<kr::WarpParams> pv(world);
    int base = 0;
    for (int r = 0; r < world; ++r) {
        fill_warp_params(hs[r], 1, pv[r]);
        pv[r].cta_base = base;
        base += hs[r]->nCTA;
        KR_CUDA(hs[r], cudaStreamSynchronize(hs[r]->stream));  // the ranks' preparation ran on their own streams
    }
    // (replicated forward sweep: two stages -- the RF instance for the backward shards, the regular one for the forward sweeps;
    // the parameter blocks of stage 2 sit behind those of stage 1)
    const bool rf = h0->rf;
    if (rf) {
        pv.resize(2 * world);
        for (int r = 0; r < world; ++r) {
            pv[world + r] = pv[r];
            pv[world + r].skip_bw = 1;
            pv[world + r].rf_world = 0;
        }
    }
    if ((rc = upload(h0, h0->d_emul, pv, true))) return rc;
    kr::WarpParams p0;
    memset(&p0, 0, sizeof(p0));
    p0.emul = h0->d_emul.get<const kr::WarpParams>();
    p0.emul_ranks = world;
    p0.wpc = h0->wpc;
    const KernelKey key{h0->Wt, h0->preg ? h0->L : 0, h0->lpt};
    const auto &emul_table = h0->taylor ? kernel_taylor_tables().emul : kernel_emul_table();
    auto it = emul_table.find(key);
    if (it == emul_table.end())
        return fail(h0, KROTOV_ERR_UNSUPPORTED, "no emulated-ranks instance of this kernel (W, L)");
    size_t smem = 0;
    for (int r = 0; r < world; ++r) smem = std::max(smem, warp_smem_bytes(hs[r]));
    dim3 grid(base), block(h0->wpc * h0->lpt + 32);
    if (rf) {
        auto itr = kernel_rf_emul_table().find(key);
        if (itr == kernel_rf_emul_table().end())
            return fail(h0, KROTOV_ERR_UNSUPPORTED, "no emulated-ranks RF instance of this kernel (W, L)");
        KR_CUDA(h0, cudaFuncSetAttribute((const void *)itr->second, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        void *args1[] = {(void *)&p0};
        KR_CUDA(h0, cudaLaunchCooperativeKernel((const void *)itr->second, grid, block, args1, smem, h0->stream));
        h0->launches_last += 1;
        p0.emul = h0->d_emul.get<const kr::WarpParams>() + world;
    }
    KR_CUDA(h0, cudaFuncSetAttribute((const void *)it->second, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    void *args[] = {(void *)&p0};
    KR_CUDA(h0, cudaLaunchCooperativeKernel((const void *)it->second, grid, block, args, smem, h0->stream));
    KR_CUDA(h0, cudaStreamSynchronize(h0->stream));
    h0->launches_last += 1;
    for (int r = 0; r < world; ++r) {
        hs[r]->kernel_last = warp_kernel_kind(hs[r]);
        hs[r]->lanes_last = hs[r]->lpt;
    }
    for (int r = 0; r < world; ++r)
        if ((rc = iterate_finish(hs[r], new_pulses + (size_t)r * pn, g_a_int + (size_t)r * h0->L))) return rc;
    return KROTOV_OK;
}

static int amp_commit(krotov_handle h);

int krotov_set_amplitudes(krotov_handle h, int degree, const double *poly, const double *shape) {
    if (!h) return KROTOV_ERR_ARG;
    if (poly && (degree < 1 || degree > kr::kAmpMaxDeg))
        return fail(h, KROTOV_ERR_UNSUPPORTED, "amplitude polynomials of degree 1..4 only");
    cudaSetDevice(h->device);
    const int L = h->L, N_T = h->N_T, D = kr::kAmpMaxDeg;
    h->amp_poly.clear();
    h->amp_shape.clear();
    if (poly) {
        h->amp_poly.assign((size_t)L * (D + 1), 0.0);
        for (int l = 0; l < L; ++l)
            for (int p = 0; p <= degree; ++p) {
                const double v = poly[(size_t)l * (degree + 1) + p];
                if (!std::isfinite(v)) return fail(h, KROTOV_ERR_ARG, "amplitude polynomial coefficient is not finite");
                h->amp_poly[(size_t)l * (D + 1) + p] = v;
            }
    }
    if (shape) h->amp_shape.assign(shape, shape + (size_t)L * N_T);
    int rc;
    if (!h->amp_poly.empty() && (rc = upload(h, h->d_amp_poly, h->amp_poly, false))) return rc;
    if (!h->amp_shape.empty() && (rc = upload(h, h->d_amp_shape, h->amp_shape, false))) return rc;
    return amp_commit(h);
}

int krotov_set_amplitude_saturation(krotov_handle h, const double *s) {
    if (!h) return KROTOV_ERR_ARG;
    cudaSetDevice(h->device);
    const int L = h->L;
    if (s)
        for (int l = 0; l < L; ++l)
            if (!std::isfinite(s[l]) || s[l] < 0.0)
                return fail(h, KROTOV_ERR_ARG, "amplitude saturation s[l] must be finite and >= 0");
    h->amp_sat.clear();
    if (s && std::any_of(s, s + L, [](double v) { return v > 0.0; })) h->amp_sat.assign(s, s + L);
    int rc;
    if (!h->amp_sat.empty() && (rc = upload(h, h->d_amp_sat, h->amp_sat, false))) return rc;
    return amp_commit(h);
}

// after either amplitude entry point: the non-linear flag, the per-sweep tables and the block paths' view of them
static int amp_commit(krotov_handle h) {
    const int L = h->L, N_T = h->N_T;
    // tied control terms run on the non-linear code path (with a(eps) = eps where no amplitude is set)
    h->amp_set = !h->amp_poly.empty() || !h->amp_shape.empty() || !h->amp_sat.empty() || !h->tie_ctrl.empty();
    int rc;
    // the warp kernels' table: one row per control, the polynomial (identity where only saturation is set) then s_l
    h->amp_rows.clear();
    if (!h->amp_poly.empty() || !h->amp_sat.empty()) {
        const int D = kr::kAmpMaxDeg, R = kr::kAmpRow;
        h->amp_rows.assign((size_t)L * R, 0.0);
        for (int l = 0; l < L; ++l) {
            for (int p = 0; p <= D; ++p)
                h->amp_rows[(size_t)l * R + p] = h->amp_poly.empty() ? (p == 1 ? 1.0 : 0.0) : h->amp_poly[(size_t)l * (D + 1) + p];
            h->amp_rows[(size_t)l * R + D + 1] = h->amp_sat.empty() ? 0.0 : h->amp_sat[l];
        }
        if ((rc = upload(h, h->d_amp_rows, h->amp_rows, false))) return rc;
    }
    if (h->amp_set) {
        if ((rc = dev_alloc(h, h->d_amp_old, (size_t)L * N_T * 8))) return rc;
        if ((rc = dev_alloc(h, h->d_amp_dfac, (size_t)L * N_T * 8))) return rc;
        if ((rc = dev_alloc(h, h->d_amp_new, (size_t)L * N_T * 8))) return rc;
    }
    if (!h->tie_ctrl.empty() && (rc = dev_alloc(h, h->d_tie, ((size_t)L + (size_t)L * N_T) * 8))) return rc;
    if (h->dense) {
        kr::AmpDev a;
        if (h->amp_set) {
            a.amp_old = h->d_amp_old.get<const double>();
            a.dfac = h->d_amp_dfac.get<const double>();
            a.poly = h->amp_poly.empty() ? nullptr : h->d_amp_poly.get<const double>();
            a.shape = h->amp_shape.empty() ? nullptr : h->d_amp_shape.get<const double>();
            a.sat = h->amp_sat.empty() ? nullptr : h->d_amp_sat.get<const double>();
            a.amp_new = h->d_amp_new.get<double>();
            a.tie = h->tie_ctrl.empty() ? nullptr : h->d_tie.get<const double>();
        }
        kr::dense_set_amp(h->dense, a);
    }
    return KROTOV_OK;
}

int krotov_set_control_terms(krotov_handle h, const int32_t *control_of_term) {
    if (!h) return KROTOV_ERR_ARG;
    cudaSetDevice(h->device);
    const int L = h->L, N_T = h->N_T;
    std::vector<int> ctrl, first(L, 0);
    bool tied = false;
    if (control_of_term) {
        int next = 0;  // ids are numbered in order of first appearance: term t opens control `next` or joins an earlier one
        for (int t = 0; t < L; ++t) {
            const int c = control_of_term[t];
            if (c < 0 || c > next)
                return fail(h, KROTOV_ERR_ARG, "control_of_term[" + std::to_string(t) + "] = " + std::to_string(c) +
                                                   ": ids must be 0..C-1 in order of first appearance");
            if (c == next) {
                first[t] = 1;
                ++next;
                continue;
            }
            tied = true;
            const int t0 = (int)(std::find(control_of_term, control_of_term + t, c) - control_of_term);
            if (h->lambda_host[t] != h->lambda_host[t0] ||
                memcmp(&h->update_shape_host[(size_t)t * N_T], &h->update_shape_host[(size_t)t0 * N_T], (size_t)N_T * 8) != 0)
                return fail(h, KROTOV_ERR_ARG, "tied control terms " + std::to_string(t0) + " and " + std::to_string(t) +
                                                   " have different update_shape rows or lambda_a");
        }
        if (tied) ctrl.assign(control_of_term, control_of_term + L);
    }
    // the identity map (or NULL) is the untied state itself
    h->tie_ctrl = ctrl;
    if (tied) h->tie_first = first; else h->tie_first.clear();
    return amp_commit(h);
}

int krotov_get_states(krotov_handle h, double *states) {
    if (!h || !states) return KROTOV_ERR_ARG;
    cudaSetDevice(h->device);
    const int N = h->N, d = h->d;
    if (h->path == KROTOV_PATH_WARP) {
        std::vector<cplx> tmp((size_t)N * h->lpt);
        KR_CUDA(h, cudaMemcpy(tmp.data(), h->d_psif.get<void>(), tmp.size() * 16, cudaMemcpyDeviceToHost));
        cplx *o = reinterpret_cast<cplx *>(states);
        for (int k = 0; k < N; ++k)
            for (int i = 0; i < d; ++i) o[(size_t)k * d + i] = tmp[(size_t)k * h->lpt + i];
    } else {
        std::string e;
        if (!kr::dense_get_states(h->dense, states, e)) return fail(h, KROTOV_ERR_CUDA, e);
    }
    return KROTOV_OK;
}

int krotov_get_tau(krotov_handle h, double *tau) {
    if (!h || !tau) return KROTOV_ERR_ARG;
    cudaSetDevice(h->device);
    KR_CUDA(h, cudaMemcpy(tau, h->d_tau.get<void>(), (size_t)h->N * 16, cudaMemcpyDeviceToHost));
    return KROTOV_OK;
}

int krotov_get_storage(krotov_handle h, int which, int k, int n0, int n1, double *out) {
    if (!h || !out) return KROTOV_ERR_ARG;
    if (k < 0 || k >= h->N || n0 < 0 || n1 > h->N_T + 1 || n0 >= n1) return fail(h, KROTOV_ERR_ARG, "bad storage range");
    if (which == KROTOV_FORWARD && !h->store_fw) return fail(h, KROTOV_ERR_STATE, "forward storage was not requested (store_fw)");
    cudaSetDevice(h->device);
    const int d = h->d;
    if (h->path == KROTOV_PATH_WARP) {
        const DevBuf &b = which == KROTOV_FORWARD ? h->d_Phi : h->d_X;
        std::vector<cplx> tmp((size_t)(n1 - n0) * h->lpt);
        const char *src = b.get<const char>() + ((size_t)k * (h->N_T + 1) + n0) * h->lpt * 16;
        if (h->rf && which == KROTOV_BACKWARD && h->iter_count > 0)  // the chi trajectory of the LAST iteration's parity
            src += (size_t)((h->iter_count - 1) & 1) * h->x_slab * 16;
        KR_CUDA(h, cudaMemcpy(tmp.data(), src, tmp.size() * 16, cudaMemcpyDeviceToHost));
        cplx *o = reinterpret_cast<cplx *>(out);
        for (int n = 0; n < n1 - n0; ++n)
            for (int i = 0; i < d; ++i) o[(size_t)n * d + i] = tmp[(size_t)n * h->lpt + i];
    } else {
        std::string e;
        if (!kr::dense_get_storage(h->dense, which, k, n0, n1, out, e)) return fail(h, KROTOV_ERR_CUDA, e);
    }
    return KROTOV_OK;
}

int krotov_envelope_extremes_device(krotov_handle h, int n_corner, const double *amps, double *e_min, double *e_max) {
    if (!h) return KROTOV_ERR_ARG;
    if (n_corner < 1 || !amps || !e_min || !e_max) return fail(h, KROTOV_ERR_ARG, "bad argument to krotov_envelope_extremes_device");
    if (h->path != KROTOV_PATH_WARP || h->lpt != 32 || !h->d_rawf)
        return fail(h, KROTOV_ERR_UNSUPPORTED, "krotov_envelope_extremes_device: persistent kernel path with d <= 32 only");
    cudaSetDevice(h->device);
    int rc;
    const size_t n_out = (size_t)h->n_gen * n_corner;
    if ((rc = dev_alloc(h, h->d_envamps, (size_t)n_corner * h->L * 8 + 16))) return rc;
    if ((rc = dev_alloc(h, h->d_envout, n_out * 16))) return rc;
    KR_CUDA(h, cudaMemcpyAsync(h->d_envamps.get<void>(), amps, (size_t)n_corner * h->L * 8, cudaMemcpyHostToDevice, h->stream));
    jacobi_extremes_kernel<<<(unsigned)n_out, 32, 0, h->stream>>>(h->d_rawf.get<const double2>(), h->d_cols.get<const int>(),
                                                                  h->d_envamps.get<const double>(), h->d_envout.get<double2>(),
                                                                  h->L, h->Wt, h->d, n_corner);
    std::vector<double> out(2 * n_out);
    KR_CUDA(h, cudaMemcpyAsync(out.data(), h->d_envout.get<void>(), n_out * 16, cudaMemcpyDeviceToHost, h->stream));
    KR_CUDA(h, cudaStreamSynchronize(h->stream));
    h->launches_total += 1;
    for (int g = 0; g < h->n_gen; ++g) {
        double lo = out[2 * ((size_t)g * n_corner)], hi = out[2 * ((size_t)g * n_corner) + 1];
        for (int c = 1; c < n_corner; ++c) {
            lo = std::min(lo, out[2 * ((size_t)g * n_corner + c)]);
            hi = std::max(hi, out[2 * ((size_t)g * n_corner + c) + 1]);
        }
        e_min[g] = lo;
        e_max[g] = hi;
    }
    return KROTOV_OK;
}

int krotov_get_profile(krotov_handle h, int cta, int64_t *out) {
    if (!h || !out) return KROTOV_ERR_ARG;
    for (int i = 0; i < 8; ++i) out[i] = 0;
    if (!h->d_prof) return fail(h, KROTOV_ERR_STATE, "profiling counters are off (set KROTOV_PROF=1 before krotov_create)");
    cudaSetDevice(h->device);
    std::vector<long long> tmp((size_t)h->nCTA * 8);
    KR_CUDA(h, cudaMemcpy(tmp.data(), h->d_prof.get<void>(), tmp.size() * 8, cudaMemcpyDeviceToHost));
    if (cta >= h->nCTA) return fail(h, KROTOV_ERR_ARG, "cta out of range");
    for (int c = 0; c < h->nCTA; ++c)
        if (cta < 0 || c == cta)
            for (int i = 0; i < 8; ++i) out[i] = std::max<int64_t>(out[i], tmp[(size_t)c * 8 + i]);
    return KROTOV_OK;
}

// ---- multi-GPU mailbox exchange over CUDA IPC -------------------------------------------------
struct CommDesc {
    cudaIpcMemHandle_t mh[2];
    cudaIpcMemHandle_t xh;  // the chi trajectory (replicated forward sweep: peers write it)
};
struct CommDescTail {  // behind the handles, in the descriptor's spare bytes
    int nCTA;
    int n_traj, n_traj_global;
    int rf_ok;  // this rank could run the replicated forward sweep (warp path, one trajectory per warp, all trajectories held)
};
static_assert(sizeof(CommDesc) + sizeof(CommDescTail) <= KROTOV_COMM_DESC_BYTES, "descriptor too large");

int krotov_comm_export(krotov_handle h, void *desc) {
    if (!h || !desc) return KROTOV_ERR_ARG;
    cudaSetDevice(h->device);
    CommDesc cd;
    memset(&cd, 0, sizeof(cd));
    for (int par = 0; par < 2; ++par) KR_CUDA(h, cudaIpcGetMemHandle(&cd.mh[par], h->d_mbox[par].get<void>()));
    if (h->path == KROTOV_PATH_WARP) KR_CUDA(h, cudaIpcGetMemHandle(&cd.xh, h->d_X.get<void>()));
    memset(desc, 0, KROTOV_COMM_DESC_BYTES);
    memcpy(desc, &cd, sizeof(cd));
    CommDescTail tail{h->path == KROTOV_PATH_WARP ? h->nCTA : 0, h->N, h->N_global, rf_eligible(h) ? 1 : 0};
    memcpy((char *)desc + sizeof(cd), &tail, sizeof(tail));
    return KROTOV_OK;
}

int krotov_comm_connect(krotov_handle h, int rank, int world, const void *descs) {
    if (!h || !descs) return KROTOV_ERR_ARG;
    if (world < 1 || world > kr::kMaxRanks || rank < 0 || rank >= world) return fail(h, KROTOV_ERR_ARG, "bad rank/world");
    cudaSetDevice(h->device);
    h->peer_maps.clear();  // the mappings of an earlier connect
    h->rank = rank;
    h->world = world;
    h->total_ctas = 0;
    h->max_ctas = 0;
    bool rf_all = world > 1;
    for (int r = 0; r < world; ++r) {
        CommDescTail tail;
        memcpy(&tail, (const char *)descs + (size_t)r * KROTOV_COMM_DESC_BYTES + sizeof(CommDesc), sizeof(tail));
        h->total_ctas += tail.nCTA;
        h->max_ctas = std::max(h->max_ctas, tail.nCTA);
        rf_all = rf_all && tail.rf_ok && tail.n_traj == h->N && tail.n_traj_global == h->N_global;
    }
    h->rf = false;
    if (rf_all) {  // every rank holds the whole problem: replicated forward sweep (same decision on every rank)
        int rc = rf_prepare(h, rank, world);
        if (rc) return rc;
    } else if (world > 1 && h->rf_wanted) {
        // a handle that holds ALL trajectories must never run the sharded exchange (every trajectory would count
        // `world` times): fail loudly instead
        return fail(h, KROTOV_ERR_UNSUPPORTED, "replicated_forward was requested but cannot be used (needs the persistent "
                                               "kernel with one trajectory per warp and the same full problem on every rank)");
    }
    for (int r = 0; r < world; ++r) {
        if (r == rank) {
            for (int par = 0; par < 2; ++par) h->peer_mbox[par][r] = h->d_mbox[par].get<double>();
            continue;
        }
        CommDesc cd;
        memcpy(&cd, (const char *)descs + (size_t)r * KROTOV_COMM_DESC_BYTES, sizeof(cd));
        for (int par = 0; par < 2; ++par) {
            KR_CUDA(h, h->peer_maps.emplace_back().open(cd.mh[par]));
            h->peer_mbox[par][r] = h->peer_maps.back().get<double>();
        }
    }
    h->iter_count = 0;
    if (h->rf) {  // the peers' chi trajectories (both parities in one allocation) and their rank-barrier flags
        for (int r = 0; r < world; ++r) {
            if (r == rank) {
                h->peer_Xbase[r] = h->d_X.get<double2>();
            } else {
                CommDesc cd;
                memcpy(&cd, (const char *)descs + (size_t)r * KROTOV_COMM_DESC_BYTES, sizeof(cd));
                KR_CUDA(h, h->peer_maps.emplace_back().open(cd.xh));
                h->peer_Xbase[r] = h->peer_maps.back().get<double2>();
            }
            h->peer_flag[r] = (unsigned long long *)((char *)h->peer_mbox[0][r] + h->mail_bytes + h->xacc_bytes);
        }
    }
    return KROTOV_OK;
}

}  // extern "C"
