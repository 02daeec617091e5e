/*
 * libkrotov_cuda -- C ABI of the B200-native Krotov iteration.
 *
 * This is the drop-in boundary for the hot path of JuliaQuantumControl/Krotov.jl:
 *   krotov_initial_fw_prop!   src/optimize.jl:247-265
 *   krotov_iteration          src/optimize.jl:279-371
 * plus the slice of QuantumPropagators.jl those functions call (prop_step!/reinit_prop! of
 * the `Cheby` propagator, the bw/fw storage arrays, dot(chi, mu, psi)).  The reference has NO
 * FFI for this path (it is pure Julia); the entry points below are what the Julia `Krotov`
 * module binds with `ccall` in place of those functions (see INTEGRATION.md for the stubs).
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a HOST pointer owned by the caller; the
 *     library copies during the call and never retains a host pointer.
 *   - complex numbers are interleaved (re, im) Float64 pairs == Julia ComplexF64 == C99
 *     `double complex`; "cplx[n]" below means 2*n doubles.
 *   - pulses, update shapes: Float64, [L][N_T] row-major (control-major), values on the N_T
 *     intervals of tlist (the layout of KrotovWrk.pulses0/pulses1, src/workspace.jl:37-40).
 *   - states: cplx[N][d] row-major (trajectory-major; one contiguous state per trajectory).
 *   - every function returns KROTOV_OK (0) or an error code; krotov_last_error() has the text.
 *     The Julia side turns non-zero into an ErrorException inside the try block of
 *     src/optimize.jl:206-226.
 *   - a handle may be used from any OS thread, one call at a time (Julia tasks migrate).
 *   - all device work of a call has completed when the call returns.
 */
#ifndef KROTOV_CUDA_H
#define KROTOV_CUDA_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KROTOV_ABI_VERSION 1

typedef struct krotov_handle_s *krotov_handle;

enum krotov_status {
    KROTOV_OK = 0,
    KROTOV_ERR_ARG = 1,         /* bad argument / inconsistent sizes            */
    KROTOV_ERR_CUDA = 2,        /* CUDA runtime error (text in last_error)      */
    KROTOV_ERR_STATE = 3,       /* call order violated (e.g. iterate before set_cheby) */
    KROTOV_ERR_UNSUPPORTED = 4, /* problem shape outside what the kernels cover */
    KROTOV_ERR_TIMEOUT = 5,     /* in-kernel exchange timed out (peer never arrived) */
    KROTOV_ERR_NOMEM = 6
};

enum krotov_gen_format {
    KROTOV_GEN_DENSE_COLMAJOR = 0, /* values: cplx[n_gen][1+L][d*d], column-major (Julia Matrix) */
    KROTOV_GEN_CSR = 1             /* one shared CSR pattern; values: cplx[n_gen][1+L][nnz]      */
};

enum krotov_direction { KROTOV_FORWARD = 0, KROTOV_BACKWARD = 1 };

enum krotov_propagator { /* krotov_problem.propagator */
    KROTOV_PROP_CHEBY = 0, /* Chebyshev series (krotov_set_cheby); the default of a zeroed problem              */
    KROTOV_PROP_EXPMV = 1  /* truncated Taylor series with scaling (krotov_set_taylor): exact for non-Hermitian
                              generators; persistent one-warp-per-trajectory kernel only (d <= 32, sharded ranks,
                              at most one trajectory per warp of a co-resident grid: 13 x SMs with rows of <= 12
                              entries, 7 x SMs with wider ones) */
};

enum krotov_functional { /* built-in chi = -dJ_T/d<psi| (QuantumControl.Functionals.make_chi analytic forms) */
    KROTOV_CHI_HOST = 0, /* caller supplies chi_k(T) every iteration via krotov_set_chi            */
    KROTOV_CHI_SM = 1,   /* J_T_sm : chi_k = w_k/N^2 (sum_j w_j tau_j) |tgt_k>                     */
    KROTOV_CHI_SS = 2,   /* J_T_ss : chi_k = w_k/N tau_k |tgt_k>                                   */
    KROTOV_CHI_RE = 3    /* J_T_re : chi_k = w_k/(2N) |tgt_k>                                      */
};

enum krotov_path { /* which kernel family serves the handle (krotov_info.path) */
    KROTOV_PATH_WARP = 1, /* d <= 32 (or d <= 128 with narrow rows): 1/2/4 warps per trajectory, whole iteration in one persistent launch */
    KROTOV_PATH_DENSE = 2, /* larger d, dense generators: FP64 DMMA complex GEMM per Chebyshev term             */
    KROTOV_PATH_SPARSE = 3 /* larger d, sparse generators: ELL SpMM over the state block per Chebyshev term      */
};

enum krotov_kernel { /* which kernel served the last forward/iterate call (krotov_info.kernel); 0 before the first */
    KROTOV_KERNEL_TINY = 1,          /* WARP: d <= 4, one thread per trajectory, everything in registers        */
    KROTOV_KERNEL_PREG = 2,          /* WARP: one trajectory per thread group, term rows held in registers      */
    KROTOV_KERNEL_SEQ_PREG = 3,      /* WARP: several trajectories of one generator per warp, one after another */
    KROTOV_KERNEL_PAIR = 4,          /* WARP: two trajectories of one generator per warp, interleaved           */
    KROTOV_KERNEL_RELOAD = 5,        /* WARP: term rows re-read from memory for every use                       */
    KROTOV_KERNEL_DMMA_STREAM = 6,   /* DENSE: one DMMA GEMM launch per Chebyshev term                          */
    KROTOV_KERNEL_DENSE_SWEEP = 7,   /* DENSE: persistent cluster sweep                                         */
    KROTOV_KERNEL_SPARSE_SWEEP = 8,  /* SPARSE: persistent sweep                                                */
    KROTOV_KERNEL_SPARSE_STREAM = 9, /* SPARSE: one ELL SpMM launch per Chebyshev term                          */
    KROTOV_KERNEL_TAYLOR = 10        /* WARP: one trajectory per warp, truncated-Taylor step (KROTOV_PROP_EXPMV)  */
};

/*
 * The control problem, reduced to arrays.  Replaces what KrotovWrk's constructor collects
 * (src/workspace.jl:65-131): trajectories (initial/target state, generator), tlist, update
 * shapes S_l, lambda_a, control derivatives.  Term l of generator k is a static operator H_kl (term 0 the drift); a term
 * flagged absent is the reference's `nothing` (src/optimize.jl:344).  By default term l is control l and enters linearly,
 * mu_kl = dH_k/d eps_l = H_kl (src/optimize.jl:275-276); krotov_set_amplitudes / krotov_set_amplitude_saturation give a
 * term a non-linear amplitude and krotov_set_control_terms ties several terms to one control.
 */
typedef struct {
    int32_t struct_size; /* = sizeof(krotov_problem), for ABI evolution */
    int32_t d;           /* Hilbert-space dimension                     */
    int32_t n_traj;      /* N: trajectories held by THIS handle (this rank's shard) */
    int32_t n_ctrl;      /* L: control terms (= controls unless krotov_set_control_terms ties terms) */
    int32_t n_steps;     /* N_T = length(tlist) - 1                      */
    int32_t n_gen;       /* distinct generators (ensemble members sharing a Hamiltonian share one) */
    int32_t gen_format;  /* enum krotov_gen_format                       */
    int32_t nnz;         /* CSR only                                     */
    const double *tlist;        /* [N_T+1]                                */
    const int32_t *gen_of_traj; /* [N] generator index of each trajectory */
    const int32_t *csr_rowptr;  /* [d+1]  (CSR only)                      */
    const int32_t *csr_colind;  /* [nnz]  (CSR only)                      */
    const double *gen_values;   /* cplx, see krotov_gen_format; term 0 = drift, 1..L = controls */
    const uint8_t *term_present; /* [n_gen][1+L] or NULL (= all present)   */
    const double *psi0;         /* cplx[N][d] initial states              */
    const double *target;       /* cplx[N][d] target states or NULL       */
    const double *weight;       /* [N] trajectory weights or NULL (= 1)   */
    const double *update_shape; /* [L][N_T]  S_l on the intervals         */
    const double *lambda_a;     /* [L]                                    */
    int32_t functional;         /* enum krotov_functional                 */
    int32_t n_traj_global;      /* N over all ranks (the N of J_T / chi); 0 = n_traj */
    int32_t store_fw;           /* keep the forward storage Phi (src/optimize.jl:367); 0 = skip */
    int32_t device;             /* CUDA device ordinal                    */
    int32_t force_path;         /* 0 = auto, else enum krotov_path        */
    int32_t replicated_forward; /* several ranks, every rank creates the handle with ALL trajectories: the backward sweep
                                   is sharded and chi written to every rank over NVLink, the time-serial forward sweep
                                   runs on every rank (no per-step exchange).  Chosen at krotov_comm_connect when every
                                   rank asked for it and runs the persistent kernel with one trajectory per warp. */
    int32_t propagator;         /* enum krotov_propagator; 0 = Chebyshev.  KROTOV_PROP_EXPMV on a problem the persistent
                                   one-warp-per-trajectory kernel does not serve (d > 32, block paths, replicated_forward)
                                   -> KROTOV_ERR_UNSUPPORTED */
    int32_t reserved[5];
} krotov_problem;

typedef struct {
    int32_t struct_size;
    int32_t path;            /* enum krotov_path                                     */
    int32_t ell_width;       /* WARP path: padded nonzeros per row                   */
    int32_t nnz_union;       /* nonzeros of the union pattern                        */
    int32_t grid_blocks;     /* CTAs of the persistent kernel                        */
    int32_t block_threads;
    int32_t m_fw;            /* Chebyshev coefficient counts currently loaded (max over generators): forward, */
                             /* (KROTOV_PROP_EXPMV: the largest m * s, Taylor terms per step; (m - 1) s products) */
    int32_t m_bw;            /* backward */
    int32_t sm_count;
    int32_t exchange;        /* cross-rank protocol of the last launch: 0 none (one rank), 1 hierarchical sum (local
                                accumulator, then one add per rank over NVLink), 2 one-hop sum (every CTA adds into every
                                rank's accumulator), 3 rank sums through the peers' mailboxes, 4 hierarchical sum forwarded with plain
                                stores into per-rank slots, 5 replicated forward sweep (no per-step exchange: sharded backward sweep
                                writes chi to every rank, one rank barrier per iteration) */
    int64_t launches_total;  /* kernels launched by this handle since creation       */
    int64_t launches_last;   /* kernels launched by the last forward/iterate call    */
    double ms_last;          /* device time of the last forward/iterate call (CUDA events on the launch stream) */
    double ms_last_backward; /* DENSE path: share of ms_last spent in the backward sweep, else 0 */
    int64_t hbm_bytes_state; /* bytes of the chi trajectory in HBM                   */
    int64_t fallback_steps;  /* WARP path: time steps of the last krotov_iterate whose grid sum left the fixed-point
                                range of the one-hop all-reduce and was redone with the gather protocol */
    int64_t graph_replays;   /* block paths: iterations served by replaying the captured CUDA graph since creation */
    double ms_rank_wait;     /* replicated forward sweep: time CTA 0 of this rank spent at the rank barrier behind the backward
                                sweep in the last krotov_iterate (launch skew between the ranks + the slowest backward shard) */
    int32_t kernel;          /* enum krotov_kernel of the last forward/iterate call, 0 before the first */
    int32_t lanes_per_traj;  /* WARP path: threads per trajectory of that kernel (32, 64 or 128; 1 for the tiny kernel);
                                0 on the block paths */
    int64_t reserved[2];
} krotov_info;

/* ---- lifetime ------------------------------------------------------------------------ */
int krotov_abi_version(void);
/* Build the device-side problem.  Replaces KrotovWrk(problem) for the device-owned fields
 * (src/workspace.jl:123-131: pulses, storages) and init_prop_trajectory (:136-161). */
int krotov_create(const krotov_problem *problem, krotov_handle *out);
int krotov_destroy(krotov_handle h);
/* Text of the last error on this handle (h == NULL: last error of a failed krotov_create on
 * the calling thread).  Never NULL. */
const char *krotov_last_error(krotov_handle h);
int krotov_get_info(krotov_handle h, krotov_info *out);
/* Device allocations and peer mappings the library currently owns, over all handles of the process.  Every
 * krotov_destroy (and every failed krotov_create) gives back what its handle took, so a test can check for leaks
 * by comparing this count before and after, which device-wide free memory cannot show on a shared GPU. */
int64_t krotov_live_device_objects(void);

/* ---- propagator settings --------------------------------------------------------------
 * Chebyshev polynomial of one direction.  Replaces what init_prop/reinit_prop! leave in
 * ChebyWrk (called at src/optimize.jl:251,306,324): per generator the spectral radius Delta,
 * E_min and the coefficients a_0..a_{m-1} for the time step dt.  The host side keeps the
 * reference's control-range logic (transform_control_ranges, src/optimize.jl:238-244) and
 * calls this again whenever the range had to be widened.
 *   n_dt_class          : distinct |dt| values of the time grid (1 for a uniform grid)
 *   dt_class_of_step[N_T]: class of every interval
 *   dt_of_class[n_dt_class] : signed step of each class as the propagator uses it (dt > 0
 *                         forward, dt < 0 backward)
 *   E_min, Delta        : [n_gen]
 *   m                   : [n_gen][n_dt_class]
 *   coeffs              : [n_gen][n_dt_class][m_max]
 */
int krotov_set_cheby(krotov_handle h, int direction, int n_dt_class, const int32_t *dt_class_of_step,
                     const double *dt_of_class, const double *E_min, const double *Delta, const int32_t *m,
                     const double *coeffs, int m_max);

/* Truncated Taylor series with scaling (Al-Mohy & Higham, SIAM J. Sci. Comput. 33 (2011); the algorithm of
 * scipy.sparse.linalg.expm_multiply) for handles created with propagator = KROTOV_PROP_EXPMV; the counterpart of
 * krotov_set_cheby, with the same dt classes.  One interval of generator g and class c applies
 *     psi <- [ e^{-i mu_g dt/s} sum_{j<m} coeffs[g][c][j] R_g^j ]^s psi,   R_g = -i scale_g (H_g(eps) - mu_g),
 * with coeffs[j] = (dt / (scale_g s))^j / j! (dt signed as in krotov_set_cheby, H_g the adjoint generator backward):
 * s times the first m terms of exp(B), B = -i dt/s (H_g - mu_g).  Exact to double-precision backward error for any
 * generator, Hermitian or not, when (m - 1, s) are chosen for ||B||_1 (the caller's part; theta table of the paper).
 * A fixed number of products per step, (m - 1) s, without early termination.
 *   mu, scale : [n_gen]    shift (real; tr(H0)/d is a good choice) and row scale (> 0, e.g. 1/||H - mu||_1)
 *   s, m      : [n_gen][n_dt_class]   repeats (>= 1) and terms (1 <= m <= m_max)
 *   coeffs    : [n_gen][n_dt_class][m_max]
 * KROTOV_ERR_STATE on a Chebyshev handle (and krotov_set_cheby on an Expmv handle); KROTOV_ERR_ARG for m or s out of
 * range, a scale that is not finite and > 0 or a mu that is not finite. */
int krotov_set_taylor(krotov_handle h, int direction, int n_dt_class, const int32_t *dt_class_of_step,
                      const double *dt_of_class, const double *mu, const double *scale, const int32_t *s,
                      const int32_t *m, const double *coeffs, int m_max);

/* Non-linear control amplitudes.  Replaces what `evaluate(generator, tlist, n; vals_dict)` and `_eval_mu`
 * (src/optimize.jl:268-276, 337-346) do for generators whose control terms carry amplitude objects: control term l
 * enters the generator of interval n as  a_l(eps, n) H_l  with
 *     a_l(eps, n) = shape[l][n] * sum_{p=0..degree} poly[l][p] eps^p          (one operator per control)
 * and the derivative  mu_l = dH/d eps_l = a_l'(eps^(i)_l[n], n) H_l  is evaluated at the GUESS pulse of the interval, as
 * the reference does (:337).  poly: [L][degree+1], ascending powers, degree 1..4, or NULL (a = eps); shape: [L][N_T]
 * or NULL (1) -- QuantumPropagators' ShapedAmplitude is (poly NULL, shape given).  Both NULL restores linear controls.
 * Takes effect with the next krotov_forward / krotov_iterate.  The caller derives the spectral envelope passed to
 * krotov_set_cheby from the amplitudes' range. */
int krotov_set_amplitudes(krotov_handle h, int degree, const double *poly, const double *shape);

/* Saturating (bounded) control amplitudes: pulse parametrizations such as QuantumControl's TanhParametrization.
 * s: [L] or NULL.  s[l] > 0: control l enters as shape[l][n] * poly_l(tanh(s[l] * eps)); s[l] == 0: as today.
 * NULL restores s = 0 for all controls.  Non-finite or negative s -> KROTOV_ERR_ARG.  A control with s[l] > 0 makes
 * the problem non-linear even when krotov_set_amplitudes left poly and shape NULL (poly_l(x) = x then).  Independent of
 * krotov_set_amplitudes (either may be called first); takes effect with the next krotov_forward / krotov_iterate. */
int krotov_set_amplitude_saturation(krotov_handle h, const double *s);

/* Control terms: one control that enters the generators through several (operator, amplitude) pairs, e.g. a drive in a
 * rotating frame, cos(Dt) eps X + sin(Dt) eps Y, or a drive together with its quadratic ac-Stark shift.  The handle's
 * n_ctrl counts TERMS: gen_values, term_present, update_shape, lambda_a, the amplitude polynomial, shape and saturation
 * are per term.  control_of_term[n_ctrl] says which control each term belongs to (ids 0..C-1, numbered in order of first
 * appearance); NULL = every term is its own control (the default; the identity map is the same state).  The overlap
 * sums stay per term, S_t(n) = sum_k Im<chi_k| H_t |psi_k>; the update ties them (src/optimize.jl:351-358 with
 * mu = sum_t a_t' H_t, as QuantumPropagators' get_control_deriv returns it):
 *     du_c(n) = sum over the terms t of control c, ascending t, of a_t'(eps_c^(i)[n], n) S_t(n)
 *     eps_c^(i+1)[n] = eps_c^(i)[n] + alpha_c[n] du_c(n),    H_t enters the forward step as a_t(eps_c^(i+1)[n], n) H_t.
 * Pulses stay [n_ctrl][N_T], one row per term: the guess rows of tied terms must be bitwise equal (else krotov_forward /
 * krotov_iterate return KROTOV_ERR_ARG), and the rows of one control in new_pulses are.  g_a_int[t] holds the control's
 * integral at the control's first term and 0 at its other terms, so that sum_t g_a_int[t] = sum_c g_a_c.
 * KROTOV_ERR_ARG: an id out of range or out of first-appearance order, or tied terms with different update_shape rows or
 * lambda_a.  Takes effect with the next krotov_forward / krotov_iterate. */
int krotov_set_control_terms(krotov_handle h, const int32_t *control_of_term);

/* ---- the hot path ----------------------------------------------------------------------
 * krotov_forward: forward propagation of every trajectory under `pulses` without update.
 * Replaces the loop over krotov_initial_fw_prop! (src/optimize.jl:182-184, 247-265).  Leaves
 * Psi_k(T) and tau_k on the device; fills the forward storage when store_fw != 0. */
int krotov_forward(krotov_handle h, const double *pulses /* [L][N_T] */);

/* chi_k(T) for the next iteration, when functional == KROTOV_CHI_HOST or to override.
 * Replaces the result of `chi(Psi, trajectories; tau)` (src/optimize.jl:297-302). */
int krotov_set_chi(krotov_handle h, const double *chi /* cplx[N][d] */);
/* chi_k(T) = coef_k * |tgt_k>: the analytic forms with the (possibly multi-rank) sums done by
 * the caller.  coef: cplx[N]. */
int krotov_set_chi_coeffs(krotov_handle h, const double *coef);

/* One Krotov iteration: backward sweep under `guess_pulses` storing chi_k(t_n) for all n,
 * then the time-serial update + forward sweep.  Replaces krotov_iteration
 * (src/optimize.jl:279-371).  On return new_pulses holds eps^(i+1) ([L][N_T]) and g_a_int
 * the running-cost integrals (src/optimize.jl:357).  With a built-in functional and no
 * krotov_set_chi* call since the last sweep, chi_k(T) is formed on the device from tau. */
int krotov_iterate(krotov_handle h, const double *guess_pulses, double *new_pulses, double *g_a_int);

/* ---- results ---------------------------------------------------------------------------
 * Psi_k(T) of the last sweep (`propagator.state`, src/optimize.jl:379) and tau_k
 * (taus!, src/optimize.jl:381; zero when no target was given). */
int krotov_get_states(krotov_handle h, double *states /* cplx[N][d] */);
int krotov_get_tau(krotov_handle h, double *tau /* cplx[N] */);
/* Columns n0..n1-1 (0-based time-grid index) of the storage of trajectory k:
 * which = KROTOV_BACKWARD -> bw_storage (chi_k(t_n)); KROTOV_FORWARD -> fw_storage (needs
 * store_fw).  out: cplx[n1-n0][d].  Backs wrk.fw_storage / wrk.bw_storage for callbacks. */
int krotov_get_storage(krotov_handle h, int which, int k, int n0, int n1, double *out);

/* Diagnostic cycle counters of the last krotov_iterate on the WARP path (of CTA `cta`, or the max over
 * all CTAs for cta = -1), available
 * when the environment variable KROTOV_PROF=1 was set at krotov_create:
 *   out[0] backward sweep, out[1] forward sweep, out[2] trajectory warp 0 waiting for the updated pulse,
 *   out[3] comm warp waiting for its CTA's partials, out[4] CTA-local reduction, out[5] grid/peer gather,
 *   out[6] overlap computation of trajectory warp 0, out[7] its whole forward steps (sum over steps).
 * SM clock cycles; out has 8 entries. */
int krotov_get_profile(krotov_handle h, int cta, int64_t *out);

/* ---- multi-GPU (one process per GPU; trajectories sharded across ranks) ----------------
 * The only per-step cross-GPU dependency is the L-vector of overlap sums
 * (src/optimize.jl:340-349).  Each rank exports an IPC descriptor of its mailbox; after the
 * descriptors of all ranks have been gathered (any transport), krotov_comm_connect maps the
 * peers' mailboxes and the forward sweep exchanges partial sums in-kernel over NVLink. */
#define KROTOV_COMM_DESC_BYTES 256
int krotov_comm_export(krotov_handle h, void *desc /* KROTOV_COMM_DESC_BYTES */);
int krotov_comm_connect(krotov_handle h, int rank, int world, const void *descs /* [world][DESC_BYTES] */);

/* Several ranks emulated on ONE device, for tests and diagnostics (a single-GPU box must be able to exercise the
 * multi-rank exchange protocols; ranks that wait for one another cannot be separate launches on one GPU).  The handles
 * -- created on the same device, one shard each, same grid shape -- are connected in-process and one cooperative launch
 * runs all ranks' CTAs; every rank's kernel code, accumulators and mailboxes are those of the multi-GPU path.
 * new_pulses: [world][L][N_T] (every rank's copy, to be compared), g_a_int: [world][L].  WARP path only. */
int krotov_group_connect(krotov_handle *handles, int world);
int krotov_group_iterate(krotov_handle *handles, int world, const double *guess_pulses, double *new_pulses,
                         double *g_a_int);

/* ---- host utility -----------------------------------------------------------------------
 * Smallest and largest eigenvalue of n_mat complex Hermitian d x d matrices (cplx[n_mat][d][d]; the Hermitian
 * part is taken, so row- and column-major callers agree), spread over n_threads host threads (0 = all cores).
 * Pure host code.  It is the arithmetic behind the spectral envelope that `reinit_prop!` re-derives
 * (QuantumPropagators `specrange(...; method=:diag)`, reached from src/optimize.jl:251,306,324 through the range
 * hook :238-244) for every ensemble member at once; a Julia caller may keep using `eigvals`. */
int krotov_hermitian_extremes(int n_mat, int d, const double *mats, double *e_min, double *e_max, int n_threads);
/* The spectral envelope of every generator of an ensemble in one call: for generator g the smallest and largest
 * eigenvalue over the `n_corner` amplitude corners of  H0[g] + sum_l amps[corner][l] * Hc[l][g]  (Hermitian part).
 * H0: cplx[n_gen][d][d], Hc: cplx[n_ctrl][n_gen][d][d], amps: [n_corner][n_ctrl], e_min/e_max: [n_gen]. */
int krotov_envelope_extremes(int n_gen, int d, int n_ctrl, const double *H0, const double *Hc, int n_corner,
                             const double *amps, double *e_min, double *e_max, int n_threads);

/* The same envelope on the DEVICE, from the generator terms the handle already holds (persistent kernel path, d <= 32,
 * Hermitian generators -- the caller's duty, as for krotov_envelope_extremes): one warp per (generator, corner) forms
 * H0[g] + sum_l amps[corner][l] Hc[l][g] in shared memory and diagonalises it with cyclic Jacobi rotations.  Agrees
 * with LAPACK to a few ulp of the matrix norm.  Returns KROTOV_ERR_UNSUPPORTED on the other paths (use the host solver).
 * amps: [n_corner][L], e_min/e_max: [n_gen]. */
int krotov_envelope_extremes_device(krotov_handle h, int n_corner, const double *amps, double *e_min, double *e_max);

#ifdef __cplusplus
}
#endif
#endif /* KROTOV_CUDA_H */
